"""One rank of the sharded large-k suite (launched by tests/test_sharded_large_k.py under torch.distributed.run, one process
per GPU), over peer memory or, with VIX_NO_P2P=1, over NCCL.

The harness is tests/mp_sharded_edges.py's: `Problem.full` is one GPU holding every row in the slot the shards hold it in,
and vix_sharded_search / vix_sharded_search_filtered with VIX_MAX_K < k <= VIX_MAX_K_LARGE must return its
vix_index_search / vix_index_search_filtered answer bit for bit on every rank (ids, distance bits with the sign of zero,
-1 / NaN padding), and every rank rank 0's answer.  The "[vix sharded knn]" line (VIX_SCAN_DEBUG=1) proves the exchange
taken on every rank: world, peer memory, k, at most nq x k entries sent per rank, and the merged total equal to the sum of
what the ranks sent.  Every check is collective.

    python -m torch.distributed.run ... tests/mp_sharded_large_k.py [case ...]      (no case: all of them)
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

SHARDED = re.compile(r"\[vix sharded knn\] world (\d+), peer (\d), k (\d+), seed (\d+), local (\d+), sent (\d+), total (\d+), "
                     r"max_row (\d+), grown (\d)")
ONE_GPU = re.compile(r"\[vix knn\] kind ivfpq, kernel (fast G \d|generic), filter (\d)")
ERR_INVALID_K = -2


def first_bad(a, b):
    if a.size == 0:
        return -1
    bad = np.nonzero((a != b).reshape(len(a), -1).any(1))[0]
    return int(bad[0]) if bad.size else -1


def compare_knn(P, what, q, k, nprobe, filt=None, device=False, route=None):
    """sharded k-NN == one GPU (bits) on every rank == rank 0's; returns (dist, ids, sharded-line fields)"""
    import torch
    import torch.distributed as dist
    R = P.R
    with Env(VIX_SCAN_DEBUG="1"):
        fd, fi = P.full.batch_search(q, k, nprobe=nprobe, filter=filt)
        qq = torch.from_numpy(np.ascontiguousarray(q)).to(R.dev) if device else q

        def run():
            (sd, si), text = with_stderr(lambda: P.sh.batch_search(qq, k, nprobe=nprobe, filter=filt))
            if device:
                assert sd.is_cuda and si.is_cuda, "device queries: the result must stay on the device"
                torch.cuda.synchronize()
            return np_of(sd), np_of(si), text
        sd, si, text = R.step(f"{what}: sharded search", run)
    lines = SHARDED.findall(text)
    info = {}

    def local():
        assert sd.shape == (len(q), k) and si.shape == (len(q), k), f"shape {sd.shape}"
        r = first_bad(si, fi)
        assert r < 0, f"ids differ from one GPU, row {r}: {si[r][:6]} vs {fi[r][:6]}"
        r = first_bad(bits(sd), bits(fd))
        assert r < 0, f"distance bits differ from one GPU, row {r}"
        runs = ONE_GPU.findall(text)
        if route is not None and k > 512:
            assert runs == [] or all(x[0] == route for x in runs), f"local kernels {runs}, expected {route}"
        if R.world == 1 or len(q) == 0 or k <= 512:
            assert not lines, f"no [vix sharded knn] line expected: {lines}"
            return
        assert len(lines) == 1, f"{len(lines)} [vix sharded knn] lines"
        w, peer, kk, seed, loc, sent, total, max_row, grown = (int(v) for v in lines[0])
        assert w == R.world and peer == R.want_peer and kk == k, f"line {lines[0]}: expected world {R.world}, peer {R.want_peer}"
        assert sent <= min(loc, len(q) * k), f"sent {sent} > min(local {loc}, nq k {len(q) * k})"
        assert total <= R.world * len(q) * k and max_row <= R.world * k, f"total {total}, max_row {max_row}"
        info.update(sent=sent, total=total, grown=grown, seed=seed, local=loc)
    R.step(f"{what}: against one GPU", local)
    if R.world > 1 and len(q) and k > 512:
        import torch
        t = torch.tensor([info.get("sent", 0)], dtype=torch.int64, device=R.dev)
        dist.all_reduce(t)
        R.step(f"{what}: merged total", lambda: Problem._expect(int(t.item()) == info.get("total", -1),
                                                                f"sum of sent {int(t.item())} != total {info.get('total')}"))
    R.same_everywhere(f"{what}: every rank's answer", [bits(sd), si])
    return sd, si, info


# ------------------------------------------------------------------------------------------------ cases
def case_ks(R):
    """k 513 .. 16384, L2 and IP, the fast G 3, generic and ks 16 local routes; search(k)[:, :512] == the k = 512 step"""
    for metric in (0, 1):
        for name, d, m, ks, route, n in (("fast48", 96, 48, 256, "fast G 3", 20000), ("generic", 36, 12, 256, "generic", 6000),
                                         ("ks16", 32, 16, 16, "generic", 6000)):
            P = random_problem(R, 411 + 7 * metric + m, metric, d, m, 32, n, ks=ks)
            q = clustered(P.rng, P.coarse, 4 * R.world + 1)
            for k in ((513, 1000, 2048, 4097, 16384) if name == "fast48" else (513, 4097)):
                sd, si, _ = compare_knn(P, f"{name} {METRICS[metric]} k {k}", q, k, 12, route=route)
                if k == 513:
                    d5, i5, _ = compare_knn(P, f"{name} {METRICS[metric]} k 512", q, 512, 12)
                    R.step("prefix of the k = 512 step", lambda: Problem._expect(
                        np.array_equal(si[:, :512], i5) and np.array_equal(bits(sd[:, :512]), bits(d5)),
                        "search(513)[:, :512] differs from search(512)"))
    R.log("ok ks: k 513 / 1000 / 2048 / 4097 / 16384, fast G 3, generic, ks 16; prefix of k 512; L2 and IP")


def case_blocks(R):
    """nq 0, 1, world - 1, 4 world +- 1, 333 (ranks with empty query blocks), host and device queries"""
    for metric in (0, 1):
        P = random_problem(R, 421 + metric, metric, 96, 48, 64, 12000, skip=(R.world - 1,) if metric == 0 else (0,))
        for nq in [0] + block_sizes(R.world):
            compare_knn(P, f"blocks {METRICS[metric]} nq {nq}", clustered(P.rng, P.coarse, nq), 1000, 9)
        compare_knn(P, f"blocks {METRICS[metric]} device", clustered(P.rng, P.coarse, 333), 1000, 9, device=True)
    R.log(f"ok blocks: nq 0 and {block_sizes(R.world)}, host and device queries, L2 and IP")


def case_partitions(R):
    """a rank owning no list, a rank whose lists are all empty (its bound all ones), every candidate on one rank, k above
    every probed vector"""
    w, kc = R.world, 48
    eq = np.array([kc * r // w for r in range(w + 1)])
    none = eq.copy()
    none[1] = 0
    P = random_problem(R, 431, 0, 32, 16, kc, 8000, bounds=none)
    compare_knn(P, "rank 0 owns no list", clustered(P.rng, P.coarse, 4 * w + 1), 1000, 8)
    home = np.random.default_rng(432).integers(0, int(eq[w - 1]) if w > 1 else kc, 8000)
    P = random_problem(R, 433, 1, 32, 16, kc, 8000, bounds=eq, home=home, noise=0.1)
    q = clustered(P.rng, P.coarse, 4 * w + 1)
    compare_knn(P, "last rank's lists empty", q, 1000, kc)
    one = np.random.default_rng(434).integers(0, int(eq[1]), 8000)
    P = random_problem(R, 435, 0, 32, 16, kc, 8000, bounds=eq, home=one, noise=0.1)
    q = clustered(P.rng, P.coarse, 4 * w + 1, home=np.random.default_rng(436).integers(0, int(eq[1]), 4 * w + 1))
    compare_knn(P, "every candidate on rank 0", q, 1000, max(int(eq[1]), 1))
    _, fi, _ = compare_knn(P, "k above every probed vector", q, 9000, kc)
    R.step("padding", lambda: Problem._expect((fi[:, -1] == -1).all(), "rows must be padded"))
    R.log("ok partitions: no list, only empty lists, every candidate on one rank, k above every probed vector")


def case_ties(R):
    """ties: every row stored twice under its id (equal distances in one list), and other rows under the same ids in other
    lists (one id in lists of several ranks)"""
    w = R.world
    P = random_problem(R, 441, 0, 32, 16, 16, 4000)
    rng = np.random.default_rng(442)
    xb = clustered(rng, P.coarse, 3000, noise=0.05)
    other = clustered(rng, P.coarse, 3000, noise=0.05)
    ids = rng.permutation(3000).astype(np.int64) * 3 + 9
    P.add("duplicates", np.concatenate([xb, xb, other]), np.concatenate([ids, ids, ids]), hand_out(rng, 9000, w))
    q = clustered(rng, P.coarse, 4 * w + 1, noise=0.05)
    for k in (513, 2048, 4097):
        sd, _, _ = compare_knn(P, f"ties k {k}", q, k, 16)
        R.step(f"ties k {k}: equal distances", lambda: Problem._expect((np.diff(sd, axis=1) == 0).any(), "no tie in any row"))
    R.log("ok ties: rows stored twice, one id in lists of several ranks")


def case_filter(R):
    """allow and deny filters with k > 512, one passing fewer than k: == IVFPQIndex.batch_search(filter=)"""
    from vectorindex_b200.index import IDFilter
    for metric in (0, 1):
        P = random_problem(R, 451 + metric, metric, 96, 48, 64, 12000)
        q = clustered(P.rng, P.coarse, 4 * R.world + 1)
        rng = np.random.default_rng(452)
        _, _, stored, _ = P.lists()
        for mode, frac in (("allow", 3), ("deny", 3), ("allow", 40)):
            f = IDFilter(int(stored.max()) + 10, mode)
            f.set(rng.choice(stored, stored.size // frac, replace=False))
            for k in (1000, 4097):
                compare_knn(P, f"filter {mode} 1/{frac} {METRICS[metric]} k {k}", q, k, 9, filt=f)
    R.log("ok filter: allow and deny with k 1000 / 4097, a filter passing fewer than k; L2 and IP")


def case_nonfinite(R):
    """a NaN query (the k smallest probed ids, NaN distances) and a zero IP query (-0)"""
    for metric in (0, 1):
        P = random_problem(R, 461 + metric, metric, 32, 16, 16, 6000)
        q = clustered(P.rng, P.coarse, 4 * R.world + 1)
        q[1] = np.nan
        if metric == 1:
            q[2] = 0.0
        sd, si, _ = compare_knn(P, f"nonfinite {METRICS[metric]}", q, 1000, 8)
        if metric == 1:
            R.step("zero IP query: -0", lambda: Problem._expect((bits(sd[2][si[2] >= 0]) == 0x80000000).all(),
                                                               "zero IP distances must come back as -0"))
    R.log("ok nonfinite: NaN query, zero IP query (-0)")


def case_capacity(R):
    """small -> large -> small k on a fresh communicator: the range region grows once, a repeat gives the same bits"""
    from vectorindex_b200.index import Comm
    comm = Comm.from_torch()
    try:
        P = random_problem(R, 471, 0, 32, 16, 16, 30000, comm=comm)
        q = clustered(P.rng, P.coarse, 64)
        seen = [compare_knn(P, f"capacity k {k}", q, k, 16) for k in (513, 16384, 513, 16384)]
        if R.world > 1 and R.want_peer == 1:
            g = [s[2]["grown"] for s in seen]
            R.step("capacity: growth", lambda: Problem._expect(g[2] == 0 and g[3] == 0 and sum(g) >= 1, f"grown flags {g}"))
        R.step("capacity: repeats", lambda: Problem._expect(
            all(np.array_equal(bits(seen[i][0]), bits(seen[i + 2][0])) and np.array_equal(seen[i][1], seen[i + 2][1])
                for i in (0, 1)), "repeated calls differ"))
    finally:
        comm.close()
    R.log("ok capacity: small, large (the region grows), small, large again (no growth); same bits")


def case_mutate(R):
    """adds and removals between calls"""
    w = R.world
    P = random_problem(R, 481, 1, 32, 16, 32, 6000)
    q = clustered(P.rng, P.coarse, 4 * w + 1)
    compare_knn(P, "before the second add", q, 1000, 8)
    rng = np.random.default_rng(482)
    xb = clustered(rng, P.coarse, 2500, noise=0.1)
    ids = rng.permutation(2500).astype(np.int64) * 3 + 8
    P.add("second add", xb, ids, hand_out(rng, 2500, w), device=True)
    compare_knn(P, "after the second add", q, 1000, 8)
    P.remove("removal", np.concatenate([ids[::7], 7 + 3 * np.arange(0, 6000, 5)]).astype(np.int64))
    compare_knn(P, "after the removal", q, 1000, 8)
    R.log("ok mutate: add and removal between calls")


def case_refusals(R):
    """k 16385 and nprobe 513: the same code on every rank, and the next call succeeds; k 512 prints no large-k line"""
    from vectorindex_b200 import _lib
    P = random_problem(R, 491, 0, 32, 16, 16, 4000)
    q = clustered(P.rng, P.coarse, 4 * R.world + 1)
    L = _lib.lib()
    for name, k, nprobe in (("k 16385", 16385, 8), ("nprobe 513", 1000, 513)):
        def call():
            d = np.empty((len(q), k), np.float32)
            i = np.empty((len(q), k), np.int64)
            rc = L.vix_sharded_search(P.local._h, P.sh.comm._c, _lib.ptr(q), C.c_int64(len(q)), C.c_int(k), C.c_int(nprobe),
                                      _lib.ptr(d), _lib.ptr(i))
            assert rc == ERR_INVALID_K, f"{name}: status {rc}, expected {ERR_INVALID_K}"
        R.step(f"refusal: {name}", call)
        compare_knn(P, f"after the refusal ({name})", q, 1000, 8)
    compare_knn(P, "k 512: the fused step", q, 512, 8)
    R.log("ok refusals: k 16385, nprobe 513 (same code everywhere, next call fine); k 512 takes the fused step")


CASES = {"ks": case_ks, "blocks": case_blocks, "partitions": case_partitions, "ties": case_ties, "filter": case_filter,
         "nonfinite": case_nonfinite, "capacity": case_capacity, "mutate": case_mutate, "refusals": case_refusals}


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
        R.log(f"large k: world {R.world}, peer memory {R.comm.uses_peer_memory}, {len(names) - len(failed)} of {len(names)} "
              "cases ok")
    finally:
        R.comm.close()
        dist.barrier()
        dist.destroy_process_group()
    if failed:
        sys.exit(1)


if __name__ == "__main__":
    main()
