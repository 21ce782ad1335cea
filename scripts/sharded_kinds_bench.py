"""Sharded flat and IVF-Flat search on ONE GPU: what the ranks' local passes and the merge cost, emulated.

  - world 1: vix_sharded_search on a one-rank communicator (the real entry point, which is then the one-GPU search)
    returns vix_index_search's answer (checked bit for bit) and costs the same call;
  - emulated world W in {2, 4, 8}: vix_debug_sharded_emulate runs every rank's local pass at n / W rows one after the other
    on this GPU plus the merge, so (emulated time) / W approximates one rank's local pass with the merge; the exchange
    between GPUs is not in these numbers, and nothing here is a multi-GPU measurement.

Shapes: flat 1M x 128 with 1k queries, IVF-Flat 1M x 128 with nlist 4096 (centroids: a sample of the rows), nprobe 32 and
10k queries, k in {10, 512, 2048}.  Times: median wall time of `reps` calls, host queries and outputs (the copies are in).
Usage: python scripts/sharded_kinds_bench.py [--n 1000000] [--reps 3]
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from vectorindex_b200 import _lib  # noqa: E402
from vectorindex_b200.index import FlatIndex, IVFIndex  # noqa: E402


def timed(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)) * 1e3


def emulate(shards, q, k, nprobe):
    arr = (C.c_void_p * len(shards))(*[s._h.value for s in shards])
    nq = q.shape[0]
    d = np.empty((nq, k), np.float32)
    i = np.empty((nq, k), np.int64)
    _lib.check(_lib.lib().vix_debug_sharded_emulate(arr, C.c_int(len(shards)), _lib.ptr(q), C.c_int64(nq), C.c_int(k),
                                                    C.c_int(nprobe), C.c_float(0), None, C.c_int64(0), C.c_int(0),
                                                    _lib.ptr(d), _lib.ptr(i), None))
    return d, i


def sharded_search(h, comm, q, k, nprobe):
    nq = q.shape[0]
    d = np.empty((nq, k), np.float32)
    i = np.empty((nq, k), np.int64)
    _lib.check(_lib.lib().vix_sharded_search(h._h, comm._c, _lib.ptr(q), C.c_int64(nq), C.c_int(k), C.c_int(nprobe),
                                             _lib.ptr(d), _lib.ptr(i)))
    return d, i


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    import torch  # noqa: F401 -- loads the libnccl the one-rank communicator binds
    from vectorindex_b200.index import Comm
    comm = Comm(0, 1, Comm.unique_id())
    rng = np.random.default_rng(0)
    n, d = a.n, 128
    x = rng.standard_normal((n, d)).astype(np.float32)
    ids = np.arange(n, dtype=np.int64)
    rows = []
    for kind, nq, nprobe in (("flat", 1000, 0), ("ivfflat", 10000, 32)):
        q = rng.standard_normal((nq, d)).astype(np.float32)
        coarse = x[rng.choice(n, 4096, replace=False)].copy()

        def make(lo, hi):
            if kind == "flat":
                ix = FlatIndex(d, "euclidean")
            else:
                ix = IVFIndex(d, "euclidean", nlist=4096, nprobe=nprobe)
                ix.set_coarse(coarse)
            if hi > lo:
                ix.batch_insert(x[lo:hi], ids[lo:hi])
            return ix

        one = make(0, n)
        for k in (10, 512, 2048):
            ref = one.batch_search(q, k, nprobe)
            got = sharded_search(one, comm, q, k, nprobe)
            assert np.array_equal(ref[1], got[1]) and np.array_equal(ref[0].view(np.uint32), got[0].view(np.uint32))
            rows.append({"kind": kind, "n": n, "nq": nq, "k": k, "world": 1,
                         "ms_index_search": timed(lambda: one.batch_search(q, k, nprobe), a.reps),
                         "ms_sharded_search_world1": timed(lambda: sharded_search(one, comm, q, k, nprobe), a.reps),
                         "ms_emulated_one_shard": timed(lambda: emulate([one], q, k, nprobe), a.reps)})
            print(json.dumps(rows[-1]), flush=True)
        del one
        for w in (2, 4, 8):
            cuts = np.linspace(0, n, w + 1).astype(int)
            shards = [make(cuts[r], cuts[r + 1]) for r in range(w)]
            for k in (10, 512, 2048):
                ms = timed(lambda: emulate(shards, q, k, nprobe), a.reps)
                rows.append({"kind": kind, "n": n, "nq": nq, "k": k, "world_emulated": w, "ms_all_ranks_and_merge": ms,
                             "ms_per_rank_emulated": ms / w})
                print(json.dumps(rows[-1]), flush=True)
            del shards
    comm.close()


if __name__ == "__main__":
    main()
