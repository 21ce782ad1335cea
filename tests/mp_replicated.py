"""One rank of the replicated suite (launched by tests/test_replicated.py under torch.distributed.run, one process per GPU),
over peer memory or, with VIX_NO_P2P=1, over NCCL.

Every rank builds the same data and a one-GPU reference holding all rows in rank order (rank r contributes the r-th slice;
the slices are ragged and one is empty).  ReplicatedFlatIndex / ReplicatedIVFFlatIndex / ReplicatedNativeIVFPQIndex must
hold identical lists on every rank and return the reference's answer bit for bit on every rank: k-NN at k = 1 .. 2048 (the
route beyond 512 included), filtered, host and device queries and outputs, range search, back-to-back bursts with device
outputs in asynchronous mode, remove on every replica, and a bad id on one rank refused by all.  Comparisons are local, so
every rank runs the same collective calls whatever fails; the failures are summed at the end.  Prints "replicated ok".
"""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

METRICS = {0: "euclidean", 1: "dotProduct", 2: "cosine"}
KINDS = [("flat", 0), ("flat", 1), ("flat", 2), ("ivfflat", 0), ("ivfflat", 1), ("ivfflat", 2), ("ivfpq", 0), ("ivfpq", 1)]
FAILURES = []


def np_of(a):
    import torch
    return a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)


def check(what, got, want):
    try:
        for g, w in zip(got, want):
            g, w = np_of(g), np_of(w)
            assert g.shape == w.shape, f"shape {g.shape} vs {w.shape}"
            if g.dtype == np.float32:
                bad = np.flatnonzero(g.view(np.uint32).ravel() != w.view(np.uint32).ravel())
            else:
                bad = np.flatnonzero(g.ravel() != w.ravel())
            assert bad.size == 0, f"{bad.size} entries differ, first at {bad[:4]}"
    except AssertionError as e:
        FAILURES.append(f"{what}: {e}")


def slices(n, world):
    """ragged contiguous slices in rank order; rank 1 contributes nothing when there are three ranks or more"""
    cuts = [0]
    for r in range(world):
        share = 0 if (world >= 3 and r == 1) else (n // world + (7 if r == 0 else 0))
        cuts.append(min(n, cuts[-1] + share) if r < world - 1 else n)
    return [(cuts[r], cuts[r + 1]) for r in range(world)]


def main():
    import torch
    import torch.distributed as dist
    from vectorindex_b200 import _lib
    from vectorindex_b200.index import (FlatIndex, IDFilter, IVFIndex, IVFPQIndex, ReplicatedFlatIndex, ReplicatedIVFFlatIndex,
                                        ReplicatedNativeIVFPQIndex, VectorIndexError)
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    _lib.check(_lib.lib().vix_set_device(local))
    dist.init_process_group("nccl")
    rank, world = dist.get_rank(), dist.get_world_size()
    dev = torch.device("cuda", local)
    n, d, nq, kc = 4000, 32, 45, 32
    rng = np.random.default_rng(11)
    cent = rng.standard_normal((24, d)).astype(np.float32)
    x = (cent[rng.integers(0, 24, n)] + 0.3 * rng.standard_normal((n, d))).astype(np.float32)
    ids = (np.arange(n, dtype=np.int64)[::-1] * 3 + 11).copy()
    x[n - 30:] = x[:30]
    ids[n - 30:] = ids[:30]                                         # rows stored twice, contributed by different ranks
    q = (cent[rng.integers(0, 24, nq)] + 0.3 * rng.standard_normal((nq, d))).astype(np.float32)
    filt = IDFilter(int(ids.max()) + 1, "allow")
    filt.set(rng.choice(np.unique(ids), n // 2, replace=False))
    lo, hi = slices(n, world)[rank]

    for kind, metric in KINDS:
        tag = f"{kind}/{METRICS[metric]}"
        if kind == "flat":
            ref, rep = FlatIndex(d, METRICS[metric]), ReplicatedFlatIndex(d, METRICS[metric])
        elif kind == "ivfflat":
            ref, rep = IVFIndex(d, METRICS[metric], nlist=kc, nprobe=6), ReplicatedIVFFlatIndex(d, METRICS[metric], nlist=kc, nprobe=6)
            coarse = torch.from_numpy(x[rng.choice(n, kc, replace=False)]).to(dev)
            dist.broadcast(coarse, 0)
            ref.set_coarse(coarse.cpu().numpy())
            rep.set_coarse(coarse.cpu().numpy())
        else:
            ref = IVFPQIndex(d, METRICS[metric], nlist=kc, nprobe=6, m=16)
            rep = ReplicatedNativeIVFPQIndex(d, METRICS[metric], nlist=kc, nprobe=6, m=16)
            ref.optimize(x[:2500])                                   # rank 0's parameters everywhere
            cb, norms = ref.get_codebooks()
            parts = [torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in (ref.get_coarse(), cb, norms)]
            for t in parts:
                dist.broadcast(t, 0)
            coarse, cb, norms = (t.cpu().numpy() for t in parts)
            ref = IVFPQIndex(d, METRICS[metric], nlist=kc, nprobe=6, m=16)
            ref.set_coarse(coarse)
            ref.set_codebooks(cb, norms)
            rep.set_parameters(coarse, cb, norms)
        ref.batch_insert(x, ids)
        rep.add(x[lo:hi], ids[lo:hi])
        # identical replicas
        if kind == "flat":
            mine = np.array([rep.count], np.int64)
        else:
            mine = np.concatenate([[rep.count], rep.local.list_sizes()]).astype(np.int64)
        if kind == "ivfpq":
            off, codes, lids, _ = rep.local.export_lists()
            mine = np.concatenate([mine, off, lids, codes.astype(np.int64).ravel()])
        t = torch.from_numpy(mine).to(dev)
        allv = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(allv, t)
        check(f"{tag} identical replicas", [allv[r] for r in range(world)], [t] * world)
        check(f"{tag} count", [np.array([rep.count])], [np.array([ref.count])])
        for k in (1, 10, 512, 513, 2048):
            check(f"{tag} k={k}", rep.batch_search(q, k), ref.batch_search(q, k))
        for k in (10, 700):
            check(f"{tag} filtered k={k}", rep.batch_search(q, k, filter=filt), ref.batch_search(q, k, filter=filt))
        radius = float(np.nanmedian(ref.batch_search(q, 10)[0][:, -1]))
        check(f"{tag} range", rep.range_search(q, radius), ref.range_search(q, radius))
        check(f"{tag} range filtered", rep.range_search(q, radius, filter=filt), ref.range_search(q, radius, filter=filt))
        f0, c0 = rep.query_block(nq)
        check(f"{tag} gather=False", rep.batch_search(q, 10, gather=False), ref.batch_search(q[f0:f0 + c0], 10))
        # device queries and outputs; back-to-back bursts with device outputs in asynchronous mode
        dq = torch.from_numpy(q).to(dev)
        check(f"{tag} device", rep.batch_search(dq, 10), ref.batch_search(q, 10))
        L = _lib.lib()
        L.vix_set_async(1)
        try:
            outs = [rep.batch_search(dq[j:], 10 + j) for j in range(6)]
            dl, dd_, di_ = rep.range_search(dq, radius)
            torch.cuda.synchronize()
            _lib.check(L.vix_synchronize())
        finally:
            L.vix_set_async(0)
        for j, o in enumerate(outs):
            check(f"{tag} burst {j}", o, ref.batch_search(q[j:], 10 + j))
        check(f"{tag} range device", (dl, dd_, di_), ref.range_search(q, radius))
        # remove on every replica
        check(f"{tag} removed", [np.array([rep.remove(ids[:60])])], [np.array([ref.batch_remove(ids[:60])])])
        check(f"{tag} after remove", rep.batch_search(q, 10), ref.batch_search(q, 10))
        # a bad id on the last rank: every rank refuses, nothing is stored
        bad = ids[lo:hi][:5].copy()
        if rank == world - 1:
            bad = np.append(bad, (1 << 32) - 1).astype(np.int64)
        before = rep.count
        try:
            rep.add(x[lo:lo + bad.size] if bad.size <= hi - lo else x[:bad.size], bad)
            FAILURES.append(f"{tag}: a bad id on rank {world - 1} was not refused")
        except VectorIndexError as e:
            if e.status != -5 or f"rank {world - 1}" not in str(e):
                FAILURES.append(f"{tag}: refusal {e.status} {e}")
        check(f"{tag} nothing stored", [np.array([rep.count])], [np.array([before])])
        dist.barrier()

    fails = torch.tensor([len(FAILURES)], device=dev)
    dist.all_reduce(fails)
    for f in FAILURES:
        print(f"rank {rank} FAIL {f}", flush=True)
    dist.destroy_process_group()
    if int(fails.item()) == 0:
        print(f"rank {rank}: replicated ok (world {world}, peer memory {'no' if os.environ.get('VIX_NO_P2P') else 'yes'})", flush=True)
        return 0
    return 1


if __name__ == "__main__":
    sys.exit(main())
