"""One rank of the sharded range-search and id-filter suite (launched by tests/test_sharded_range.py under
torch.distributed.run, one process per GPU), over peer memory or, with VIX_NO_P2P=1, over NCCL.

The harness is tests/mp_sharded_edges.py's: `Problem.full` is one GPU holding every row in the slot the shards hold it in,
and vix_sharded_range_search / vix_sharded_search_filtered must return its vix_index_range_search /
vix_index_search_filtered answer bit for bit on every rank (lims, ids, distance bits with the sign of zero), and every
rank rank 0's answer.  The "[vix range]" line (VIX_SCAN_DEBUG=1) proves the local scan's route on every rank, the
"[vix sharded range]" line the exchange (peer memory or NCCL), the region growth and the long rows.  Every check is
collective.

    python -m torch.distributed.run ... tests/mp_sharded_range.py [case ...]      (no case: all of them)
"""
import ctypes as C
import os
import re
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from mp_sharded_edges import (METRICS, CaseFailure, Env, Problem, Ranks, bits, block_sizes, clustered,  # noqa: E402
                              hand_out, np_of, random_problem, with_stderr)

LOCAL = re.compile(r"\[vix range\] kind ivfpq, kernel (fast G \d|generic), filter (\d), passes (\d), total (\d+)")
SHARDED = re.compile(r"\[vix sharded range\] world (\d+), peer (\d), local (\d+), total (\d+), max_row (\d+), grown (\d)")
ERR_INVALID_K, ERR_INVALID_PARAM = -2, -5


def first_diff(a, b):
    n = min(len(a), len(b))
    bad = np.nonzero(a[:n] != b[:n])[0]
    return int(bad[0]) if bad.size else n


def compare_range(P, what, q, radius, nprobe, filt=None, device=False, route=None):
    """sharded range search == one GPU (bits) on every rank == rank 0's; returns (lims, dist, ids, sharded-line fields)"""
    import torch
    R = P.R
    with Env(VIX_SCAN_DEBUG="1"):
        wl, wd, wi = P.full.range_search(q, radius, nprobe=nprobe, filter=filt)
        qq = torch.from_numpy(np.ascontiguousarray(q)).to(R.dev) if device else q

        def run():
            got, text = with_stderr(lambda: P.sh.range_search(qq, radius, nprobe=nprobe, filter=filt))
            if device:
                assert all(t.is_cuda for t in got), "device queries: the result must stay on the device"
            return [np_of(t) for t in got], text
        got, text = R.step(f"{what}: sharded range search", run)
    lims, dist, ids = got
    info = {}

    def local():
        assert np.array_equal(lims, wl), f"lims differ at row {first_diff(lims, wl)}: totals {lims[-1]} vs one GPU {wl[-1]}"
        j = first_diff(ids, wi)
        assert np.array_equal(ids, wi), f"ids differ at entry {j}: {ids[j:j + 4]} vs one GPU {wi[j:j + 4]}"
        j = first_diff(bits(dist), bits(wd))
        assert np.array_equal(bits(dist), bits(wd)), f"distance bits differ at entry {j}: {dist[j]!r} vs one GPU {wd[j]!r}"
        runs = LOCAL.findall(text)
        if route is not None:
            assert [r[0] for r in runs] == [route], f"local range scans {runs}, expected one [{route}]"
        assert all(int(r[1]) == (filt is not None) for r in runs), f"filter flag {runs}"
        lines = SHARDED.findall(text)
        if R.world == 1 or len(q) == 0:
            assert not lines, "one rank, or nq 0: no exchange"
            return
        assert len(lines) == 1, f"{len(lines)} [vix sharded range] lines"
        w, peer, mine, total, max_row, grown = (int(v) for v in lines[0])
        assert w == R.world and peer == R.want_peer, f"world {w} peer {peer}, expected {R.world} / {R.want_peer}"
        assert total == len(wi) and mine == int(runs[0][3]), f"totals {lines[0]} vs one GPU {len(wi)}, local {runs}"
        rows = np.diff(wl)
        assert max_row == (int(rows.max()) if rows.size else 0), f"max_row {max_row}"
        info.update(local=mine, max_row=max_row, grown=grown)
    R.step(f"{what}: against one GPU", local)
    R.same_everywhere(f"{what}: every rank's answer", [lims, bits(dist), ids])
    return lims, dist, ids, info


def radii(P, q, nprobe):
    """radius quantiles of the probed distances: 0.2 %, 2 %, 20 %; below every distance; +inf"""
    _, d, _ = P.full.range_search(q, float("inf"), nprobe=nprobe)
    qs = [float(np.quantile(d, f)) for f in (0.002, 0.02, 0.2)]
    return qs + [float(d.min()) - 1.0, float("inf")]


# ------------------------------------------------------------------------------------------------ cases
def case_radii(R):
    """L2 and IP, the fast kernel at m = 48: radii at quantiles, below all (total 0), +inf; a zero IP query (-0)"""
    for metric in (0, 1):
        P = random_problem(R, 211 + metric, metric, 96, 48, 64, 6000)
        q = clustered(P.rng, P.coarse, 4 * R.world + 1)
        for i, rad in enumerate(radii(P, q, 9)):
            lims, _, _, _ = compare_range(P, f"radius {rad:.4g} {METRICS[metric]}", q, rad, 9, route="fast G 3")
            if i == 3:
                R.step("radius below all: total 0", lambda: Problem._expect(lims[-1] == 0, f"total {lims[-1]}"))
        if metric == 1:
            z = np.zeros((3, 96), np.float32)
            _, dz, _, _ = compare_range(P, "zero IP query", z, 0.0, 9, route="fast G 3")
            R.step("zero IP query: -0", lambda: Problem._expect(dz.size > 0 and (bits(dz) == 0x80000000).all(),
                                                               "zero IP distances must come back as -0"))
    R.log("ok radii: quantiles 0.2 / 2 / 20 %, below all, +inf, zero IP query; L2 and IP")


def case_blocks(R):
    """nq 0, 1, world - 1, 4 world +- 1, 333 (ranks with empty query blocks), host and device queries"""
    for metric in (0, 1):
        P = random_problem(R, 221 + metric, metric, 96, 48, 64, 6000, skip=(R.world - 1,) if metric == 0 else (0,))
        rad = radii(P, clustered(P.rng, P.coarse, 16), 9)[1]
        for nq in [0] + block_sizes(R.world):
            q = clustered(P.rng, P.coarse, nq)
            compare_range(P, f"blocks {METRICS[metric]} nq {nq}", q, rad, 9, route=None if nq == 0 else "fast G 3")
        q = clustered(P.rng, P.coarse, 333)
        compare_range(P, f"blocks {METRICS[metric]} device queries", q, rad, 9, device=True, route="fast G 3")
    R.log(f"ok blocks: nq 0 and {block_sizes(R.world)}, host and device queries, L2 and IP")


def case_partitions(R):
    """a rank owning no list, a rank whose lists are all empty"""
    w, kc = R.world, 48
    eq = np.array([kc * r // w for r in range(w + 1)])
    none = eq.copy()
    none[1] = 0
    P = random_problem(R, 231, 0, 32, 16, kc, 4000, bounds=none)
    q = clustered(P.rng, P.coarse, 4 * w + 1)
    compare_range(P, "rank 0 owns no list", q, radii(P, q, 8)[2], 8, route="fast G 1")
    home = np.random.default_rng(232).integers(0, int(eq[w - 1]) if w > 1 else kc, 4000)
    P = random_problem(R, 233, 1, 32, 16, kc, 4000, bounds=eq, home=home, noise=0.1)
    q = clustered(P.rng, P.coarse, 4 * w + 1)
    compare_range(P, "last rank's lists empty", q, radii(P, q, kc)[2], kc, route="fast G 1")
    R.log("ok partitions: a rank owning no list, a rank with only empty lists")


def case_routes(R):
    """the local scan's routes: fast G 3 (m 48), generic (m 12, d 36), ks 16 (generic)"""
    for metric in (0, 1):
        for name, d, m, ks, route in (("fast48", 96, 48, 256, "fast G 3"), ("generic", 36, 12, 256, "generic"),
                                      ("ks16", 32, 16, 16, "generic")):
            P = random_problem(R, 241 + 7 * metric + m, metric, d, m, 24, 3000, ks=ks)
            q = clustered(P.rng, P.coarse, 4 * R.world + 1)
            compare_range(P, f"{name} {METRICS[metric]}", q, radii(P, q, 6)[2], 6, route=route)
    R.log("ok routes: fast G 3 (m 48), generic (m 12), ks 16; L2 and IP")


def case_filter(R):
    """allow and deny filters, for range search and for the filtered k-NN call (== IVFPQIndex.batch_search(filter=))"""
    from vectorindex_b200.index import IDFilter
    for metric in (0, 1):
        P = random_problem(R, 251 + metric, metric, 96, 48, 64, 6000)
        q = clustered(P.rng, P.coarse, 4 * R.world + 1)
        rad = radii(P, q, 9)[2]
        rng = np.random.default_rng(252)
        _, _, stored, _ = P.lists()
        for mode in ("allow", "deny"):
            f = IDFilter(int(stored.max()) + 10, mode)
            f.set(rng.choice(stored, stored.size // 3, replace=False))
            compare_range(P, f"filter {mode} {METRICS[metric]}", q, rad, 9, filt=f, route="fast G 3")
            for k in (10, 512):
                fd, fi = P.full.batch_search(q, k, nprobe=9, filter=f)
                sd, si = R.step(f"filtered k-NN {mode} k {k}", lambda: P.sh.batch_search(q, k, nprobe=9, filter=f))

                def same():
                    assert np.array_equal(si, fi), f"ids differ from one GPU ({mode}, k {k})"
                    assert np.array_equal(bits(sd), bits(fd)), f"distance bits differ from one GPU ({mode}, k {k})"
                R.step(f"filtered k-NN {mode} {METRICS[metric]} k {k}: against one GPU", same)
                R.same_everywhere("filtered k-NN on every rank", [bits(sd), si])
    R.log("ok filter: allow and deny, range search and filtered k-NN (k 10 / 512), L2 and IP")


def case_long_rows(R):
    """rows longer than 2048 keys, drawn from every rank's lists"""
    P = random_problem(R, 261, 0, 32, 16, 8 * R.world, 12000)
    q = clustered(P.rng, P.coarse, 2 * R.world + 1)
    _, _, _, info = compare_range(P, "long rows", q, float("inf"), P.kc, route="fast G 1")
    if R.world > 1:
        R.step("long rows: max_row", lambda: Problem._expect(info["max_row"] > 2048 and info["local"] > 0,
                                                             f"max_row {info['max_row']}, local {info['local']}"))
    R.log("ok long_rows: rows of every stored row (> 2048 keys) from every rank")


def case_capacity(R):
    """small -> large -> small answers on a fresh communicator: the region grows once (grown 1), the repeat does not, and
    repeated calls give the same bits"""
    from vectorindex_b200.index import Comm
    comm = Comm.from_torch()
    try:
        P = random_problem(R, 271, 0, 32, 16, 16, 20000, comm=comm)
        q = clustered(P.rng, P.coarse, 64)
        rs = radii(P, q, 16)
        seen = []
        for name, rad in (("small", rs[0]), ("large", float("inf")), ("small again", rs[0]), ("large again", float("inf"))):
            out = compare_range(P, f"capacity {name}", q, rad, 16, route="fast G 1")
            seen.append(out)
        if R.world > 1 and R.want_peer == 1:
            g = [o[3]["grown"] for o in seen]
            R.step("capacity: growth", lambda: Problem._expect(g[1] == 1 and g[2] == 0 and g[3] == 0, f"grown flags {g}"))
        R.step("capacity: repeats", lambda: Problem._expect(
            all(np.array_equal(bits(seen[i][1]), bits(seen[i + 2][1])) and np.array_equal(seen[i][2], seen[i + 2][2])
                for i in (0, 1)), "repeated calls differ"))
    finally:
        comm.close()
    R.log("ok capacity: small, large (the region grows), small, large again (no growth); same bits")


def case_mutate(R):
    """adds and removals between range calls"""
    w = R.world
    P = random_problem(R, 281, 1, 32, 16, 32, 4000)
    q = clustered(P.rng, P.coarse, 4 * w + 1)
    rad = radii(P, q, 8)[2]
    compare_range(P, "before the second add", q, rad, 8, route="fast G 1")
    rng = np.random.default_rng(282)
    xb = clustered(rng, P.coarse, 1500, noise=0.1)
    ids = rng.permutation(1500).astype(np.int64) * 3 + 8
    ids[:40] = 7 + 3 * np.arange(40)                                     # some ids stored twice
    P.add("second add", xb, ids, hand_out(rng, 1500, w), device=True)
    compare_range(P, "after the second add", q, rad, 8, route="fast G 1")
    P.remove("removal", np.concatenate([ids[::7], 7 + 3 * np.arange(0, 4000, 5)]).astype(np.int64))
    compare_range(P, "after the removal", q, rad, 8, route="fast G 1")
    R.log("ok mutate: add (ids stored twice) and removal between range calls")


def case_knn_prefix(R):
    """the sharded k-NN entries within the radius are the first entries of each sharded range row"""
    from test_range_search import knn_prefix
    for metric in (0, 1):
        P = random_problem(R, 291 + metric, metric, 96, 48, 64, 6000)
        q = clustered(P.rng, P.coarse, 4 * R.world + 1)
        for rad in radii(P, q, 9)[:3]:
            lims, dist, ids, _ = compare_range(P, f"knn prefix {METRICS[metric]}", q, rad, 9)
            kd, ki = R.step("sharded k-NN", lambda: P.sh.batch_search(q, 10, nprobe=9))
            R.step(f"knn prefix {METRICS[metric]} radius {rad:.4g}", lambda: knn_prefix((lims, dist, ids), np_of(kd),
                                                                                       np_of(ki), rad))
    R.log("ok knn_prefix: sharded k-NN within the radius heads every sharded range row, L2 and IP")


def case_refusals(R):
    """NaN radius, nprobe 513, a bad filter mode: every rank the same code, and the next call succeeds; replicas refuse"""
    from vectorindex_b200 import _lib
    from vectorindex_b200.index import ReplicatedIVFPQIndex
    P = random_problem(R, 301, 0, 32, 16, 16, 3000)
    q = clustered(P.rng, P.coarse, 4 * R.world + 1)
    L = _lib.lib()
    words = np.zeros(4, np.uint64)
    for name, rad, nprobe, fw, mode, want in (("NaN radius", float("nan"), 8, None, 0, ERR_INVALID_PARAM),
                                              ("nprobe 513", 1.0, 513, None, 0, ERR_INVALID_K),
                                              ("filter mode 2", 1.0, 8, words, 2, ERR_INVALID_PARAM),
                                              ("negative capacity", 1.0, 8, words, 0, ERR_INVALID_PARAM)):
        def call():
            res = C.c_void_p(0)
            rc = L.vix_sharded_range_search(P.local._h, P.sh.comm._c, _lib.ptr(q), C.c_int64(len(q)), C.c_float(rad),
                                            C.c_int(nprobe), _lib.ptr(fw), C.c_int64(-1 if name == "negative capacity" else 256),
                                            C.c_int(mode), C.byref(res))
            L.vix_range_result_destroy(res)
            assert rc == want, f"{name}: status {rc}, expected {want}"
            assert not res.value, f"{name}: a result object was returned"
        R.step(f"refusal: {name}", call)
        compare_range(P, f"after the refusal ({name})", q, 1.0, 8, route="fast G 1")

    def filtered_bad():
        d = np.empty((len(q), 10), np.float32)
        i = np.empty((len(q), 10), np.int64)
        rc = L.vix_sharded_search_filtered(P.local._h, P.sh.comm._c, _lib.ptr(q), C.c_int64(len(q)), 10, 8, _lib.ptr(words),
                                           C.c_int64(256), 3, _lib.ptr(d), _lib.ptr(i))
        assert rc == ERR_INVALID_PARAM, f"filtered k-NN, filter mode 3: status {rc}"
    R.step("refusal: filtered k-NN, bad mode", filtered_bad)
    rp = ReplicatedIVFPQIndex(32, "euclidean", nlist=16, nprobe=8, m=16)

    def replicated():
        for fn in (lambda: rp.range_search(q, 1.0), lambda: rp.batch_search(q, 10, filter=object())):
            try:
                fn()
            except NotImplementedError:
                continue
            raise AssertionError("ReplicatedIVFPQIndex accepted a range search / filter")
    R.step("replicated refuses", replicated)
    R.log("ok refusals: NaN radius, nprobe 513, bad filter mode, negative capacity (same code everywhere, next call fine); "
          "replicas refuse range search and filters")


CASES = {"radii": case_radii, "blocks": case_blocks, "partitions": case_partitions, "routes": case_routes,
         "filter": case_filter, "long_rows": case_long_rows, "capacity": case_capacity, "mutate": case_mutate,
         "knn_prefix": case_knn_prefix, "refusals": case_refusals}


def main():
    import torch.distributed as dist
    names = sys.argv[1:] or list(CASES)
    R = Ranks()
    failed = []
    try:
        R.agree("start", None)
        for name in names:
            try:
                CASES[name](R)
            except CaseFailure as e:                                   # raised on every rank at the same point
                failed.append(f"{name}: {e}")
                R.log(f"FAILED {name}: {e}")
        R.log(f"range: world {R.world}, peer memory {R.comm.uses_peer_memory}, {len(names) - len(failed)} of {len(names)} "
              "cases ok")
    finally:
        R.comm.close()
        dist.barrier()
        dist.destroy_process_group()
    if failed:
        sys.exit(1)


if __name__ == "__main__":
    main()
