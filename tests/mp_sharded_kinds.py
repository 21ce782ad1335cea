"""One rank of the sharded flat / IVF-Flat suite (launched by tests/test_sharded_kinds.py under torch.distributed.run, one
process per GPU), over peer memory or, with VIX_NO_P2P=1, over NCCL.

Every rank builds the same data (same seeds) and the one-GPU reference from all rows: flat in rank order (rank r contributes
the r-th contiguous block, so that is the original order), IVF-Flat in the original order (its answer does not depend on the
slots).  ShardedFlatIndex / ShardedIVFFlatIndex must return the reference's answer bit for bit on every rank, and every
rank rank 0's answer: k-NN at k = 1 .. 2048 (the large-k route above 512), filtered, host and device queries, range search,
back-to-back searches with device outputs (nothing but the library orders one call's stores into a peer after that peer's
reads of the previous call), and the collective refusals.

    python -m torch.distributed.run ... tests/mp_sharded_kinds.py [case ...]      (no case: all of them)
"""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from mp_sharded_edges import CaseFailure, Ranks, bits, np_of  # noqa: E402

METRICS = {0: "euclidean", 1: "dotProduct", 2: "cosine"}
ERR_INVALID_PARAM, ERR_NOT_TRAINED = -5, -6


def data(seed, n, d, nq):
    rng = np.random.default_rng(seed)
    x = rng.integers(-2, 3, (n, d)).astype(np.float32)             # many ties at one raw score
    dup = rng.choice(n // 2, 20, replace=False)
    x[n - 20:] = x[dup]                                              # rows stored twice, on different ranks
    ids = (np.arange(n, dtype=np.int64)[::-1] * 3 + 11).copy()      # ids opposite to the rank order
    q = rng.integers(-2, 3, (nq, d)).astype(np.float32)
    q[0] = 0.0
    return x, ids, q


def id_filter(ids, seed):
    from vectorindex_b200.index import IDFilter
    f = IDFilter(int(ids.max()) + 1, "allow")
    f.set(np.random.default_rng(seed).choice(np.unique(ids), len(ids) // 2, replace=False))
    return f


def compare(R, what, got, want):
    """got == want bit for bit on every rank, and every rank's answer == rank 0's"""
    got = [np_of(a) for a in got]

    def check():
        for g, w in zip(got, want):
            if g.dtype == np.float32:
                assert np.array_equal(bits(g), bits(w)), f"distance bits differ at {np.flatnonzero(bits(g).ravel() != bits(w).ravel())[:4]}"
            else:
                assert np.array_equal(g, w), f"ids / lims differ at {np.flatnonzero(g.ravel() != w.ravel())[:4]}"
    R.step(what, check)
    R.same_everywhere(what + " (rank 0)", got)


def exercise(R, name, sh, one, q, ids, nprobe):
    """k-NN, filtered, device queries, range, back-to-back device searches"""
    import torch
    filt = id_filter(ids, 5)
    for k in (1, 10, 512, 513, 2048):
        compare(R, f"{name} k {k}", R.step(f"{name} k {k}: search", lambda: sh.batch_search(q, k, nprobe)),
                one.batch_search(q, k, nprobe))
        compare(R, f"{name} k {k} filtered", R.step(f"{name} k {k}: filtered", lambda: sh.batch_search(q, k, nprobe, filter=filt)),
                one.batch_search(q, k, nprobe, filter=filt))
    qd = torch.from_numpy(q).to(R.dev)
    for k in (10, 700):
        compare(R, f"{name} k {k} device", R.step(f"{name} k {k}: device", lambda: sh.batch_search(qd, k, nprobe)),
                one.batch_search(q, k, nprobe))
    ref = one.batch_search(q, 64, nprobe)[0]
    v = np.sort(ref[np.isfinite(ref)].ravel())
    for radius in (float(v[len(v) // 50]), float(v[len(v) // 4])):
        compare(R, f"{name} range {radius}", R.step(f"{name} range: search", lambda: sh.range_search(q, radius, nprobe)),
                one.range_search(q, radius, nprobe))
        compare(R, f"{name} range {radius} filtered",
                R.step(f"{name} range: filtered", lambda: sh.range_search(q, radius, nprobe, filter=filt)),
                one.range_search(q, radius, nprobe, filter=filt))
    # back to back: device queries and outputs, no host synchronisation between the calls
    ks = [10, 3, 10, 512, 7, 10] * 4

    def burst():
        outs = [sh.batch_search(qd, k, nprobe) for k in ks]
        torch.cuda.synchronize()
        return outs
    outs = R.step(f"{name} back-to-back", burst)
    refs = {k: one.batch_search(q, k, nprobe) for k in set(ks)}
    for j, (k, o) in enumerate(zip(ks, outs)):
        compare(R, f"{name} back-to-back call {j} (k {k})", o, refs[k])


def case_flat(R):
    from vectorindex_b200.index import FlatIndex, ShardedFlatIndex
    n, d, nq = 4000, 24, 29
    for metric in (0, 1, 2):
        x, ids, q = data(100 + metric, n, d, nq)
        one = FlatIndex(d, METRICS[metric])
        one.batch_insert(x, ids)
        cuts = np.linspace(0, n, R.world + 1).astype(int)
        if R.world > 2:
            cuts[1] = 0                                              # rank 0 holds nothing
        sh = ShardedFlatIndex(d, METRICS[metric])
        lo, hi = cuts[R.rank], cuts[R.rank + 1]
        R.step(f"flat {metric}: add", lambda: sh.add(x[lo:hi].copy(), ids[lo:hi].copy()))
        exercise(R, f"flat {METRICS[metric]}", sh, one, q, ids, 0)
    R.log("ok flat: three metrics, k 1 .. 2048, filtered, device queries, range, back to back")


def case_ivfflat(R):
    from vectorindex_b200.index import IVFIndex, ShardedIVFFlatIndex
    n, d, nq, kc, nprobe = 4000, 24, 29, 24, 6
    for metric in (0, 1, 2):
        x, ids, q = data(200 + metric, n, d, nq)
        rng = np.random.default_rng(300 + metric)
        coarse = x[rng.choice(n, kc, replace=False)] + 0.25 * rng.standard_normal((kc, d)).astype(np.float32)
        one = IVFIndex(d, METRICS[metric], nlist=kc, nprobe=nprobe)
        one.set_coarse(coarse)
        one.batch_insert(x, ids)
        sh = ShardedIVFFlatIndex(d, METRICS[metric], nlist=kc, nprobe=nprobe)
        sh.set_coarse(coarse)
        if R.world > 2:                                              # rank 1 owns no list
            b = np.linspace(0, kc, R.world + 1).astype(np.int64)
            b[2] = b[1]
            sh.set_list_bounds(b)
        src = rng.integers(0, R.world, n)                            # any rank may contribute any row
        mine = np.flatnonzero(src == R.rank)
        R.step(f"ivfflat {metric}: add", lambda: sh.add(x[mine].copy(), ids[mine].copy()))
        total = R.step("ivfflat count", lambda: _sum(R, sh.count))
        R.step("ivfflat rows", lambda: _expect(total == n, f"{total} rows over the ranks, {n} added"))
        exercise(R, f"ivfflat {METRICS[metric]}", sh, one, q, ids, nprobe)
    R.log("ok ivfflat: three metrics, rows routed to their lists' owners, k 1 .. 2048, filtered, device queries, range")


def _sum(R, v):
    import torch
    import torch.distributed as dist
    t = torch.tensor([v], dtype=torch.int64, device=R.dev)
    dist.all_reduce(t)
    return int(t.item())


def _expect(cond, msg):
    assert cond, msg


def case_refusals(R):
    """collective: a bad id on rank 0 only refuses the call on every rank with nothing stored; list bounds for a flat index
    and an IVF-Flat index without centroids are refused on every rank before any exchange"""
    from vectorindex_b200 import _lib
    from vectorindex_b200._lib import VectorIndexError
    from vectorindex_b200.index import FlatIndex, IVFIndex, ShardedFlatIndex, ShardedIVFFlatIndex
    d = 8
    rng = np.random.default_rng(7)
    x = rng.standard_normal((5, d)).astype(np.float32)
    ids = 100 * R.rank + np.arange(5, dtype=np.int64)
    if R.rank == 0:
        ids[2] = 2 ** 32 - 1

    def status(fn):
        try:
            fn()
        except VectorIndexError as e:
            return e.status, str(e)
        return 0, ""
    for kind in ("flat", "ivfflat"):
        if kind == "flat":
            sh = ShardedFlatIndex(d, "euclidean")
        else:
            sh = ShardedIVFFlatIndex(d, "euclidean", nlist=4, nprobe=2)
            sh.set_coarse(np.eye(4, d, dtype=np.float32))

        def refused():
            st, msg = status(lambda: sh.add(x, ids))
            assert st == ERR_INVALID_PARAM, f"status {st}: {msg}"
            if R.world > 1:
                assert "rank 0" in msg, f"the error does not name rank 0: {msg}"
            assert sh.count == 0, f"{sh.count} rows stored"
        R.step(f"{kind}: an id 2^32 - 1 on rank 0", refused)
    flat = FlatIndex(d, "euclidean")
    comm = None
    if R.world > 1:
        comm = ShardedFlatIndex(d, "euclidean")._native()

    def bounds_refused():
        if comm is None:
            return
        b = np.array([0] * R.world + [1], np.int64)
        st = int(_lib.lib().vix_sharded_add(flat._h, comm._c, _lib.ptr(b), _lib.ptr(x), _lib.ptr(ids), C.c_int64(5)))
        assert st == ERR_INVALID_PARAM, f"status {st}"
        assert flat.count == 0
    R.step("flat: list bounds refused", bounds_refused)
    ivf = IVFIndex(d, "euclidean", nlist=4, nprobe=2)

    def untrained():
        if comm is None:
            return
        dd, di = np.empty((2, 3), np.float32), np.empty((2, 3), np.int64)
        st = int(_lib.lib().vix_sharded_search(ivf._h, comm._c, _lib.ptr(x[:2].copy()), C.c_int64(2), C.c_int(3), C.c_int(0),
                                               _lib.ptr(dd), _lib.ptr(di)))
        assert st == ERR_NOT_TRAINED, f"status {st}"
    R.step("ivfflat without centroids refused", untrained)
    R.log("ok refusals: a bad id on one rank refused everywhere, list bounds on flat, IVF-Flat without centroids")


CASES = {"flat": case_flat, "ivfflat": case_ivfflat, "refusals": case_refusals}


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
        R.log(f"kinds: world {R.world}, {len(names) - len(failed)} of {len(names)} cases ok")
    finally:
        R.comm.close()
        dist.barrier()
        dist.destroy_process_group()
    if failed:
        sys.exit(1)


if __name__ == "__main__":
    main()
