"""One rank of the multi-GPU parity check (launched by tests/test_sharded_gpu.py under torch.distributed.run, one process
per GPU): the native sharded step (vix_sharded_add / vix_sharded_search behind ShardedIVFPQIndex) against a single-GPU
index holding all rows and against the oracle, over peer memory or, with VIX_NO_P2P=1, over NCCL all-gathers."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def same_as_single(si, sd, fi, fd, what):
    np.testing.assert_allclose(sd, fd, rtol=2e-6, atol=0, err_msg=what)
    diff = np.nonzero((si != fi).any(axis=1))[0]
    for r in diff:                                                          # ids may swap only at a tie inside the tolerance
        assert set(si[r]) == set(fi[r]) or abs(sd[r][-1] - fd[r][-1]) <= 2e-6 * abs(fd[r][-1]), f"{what}: row {r}"
    assert diff.size <= max(1, si.shape[0] // 50), f"{what}: {diff.size} rows differ in ids"


def padded_shard_case(rank, world):
    """The last rank owns one list of 4 vectors, so every query's local top-10 there is mostly padding keys: the merged
    result must still equal a single-GPU index holding the same rows."""
    import torch
    from vectorindex_b200.index import IVFPQIndex, ShardedIVFPQIndex

    n, d, m, kc, nq, k, nprobe, few = 6000, 96, 48, 64, 200, 10, 9, 4
    rng = np.random.default_rng(8)
    centres = rng.standard_normal((kc, d)).astype(np.float32)
    home = np.concatenate([rng.integers(0, kc - 1, n - few), np.full(few, kc - 1)])     # list kc - 1 gets `few` rows
    xb = (centres[home] + 0.3 * rng.standard_normal((n, d))).astype(np.float32)
    qhome = np.concatenate([np.full(20, kc - 1), rng.integers(0, kc, nq - 20)])         # 20 queries probe the small list
    q = (centres[qhome] + 0.3 * rng.standard_normal((nq, d))).astype(np.float32)
    cb = (0.3 * rng.standard_normal((m, 256, d // m))).astype(np.float32)
    ids = np.arange(n, dtype=np.int64) * 5 + 2
    full = IVFPQIndex(d, "euclidean", nlist=kc, nprobe=nprobe, m=m)
    full.set_coarse(centres)
    full.set_codebooks(cb)
    full.batch_insert(xb, ids)
    assert np.bincount(full.export_lists()[3], minlength=kc)[kc - 1] == few
    fd, fi = full.batch_search(q, k)
    local = IVFPQIndex(d, "euclidean", nlist=kc, nprobe=nprobe, m=m)
    local.set_coarse(centres)
    local.set_codebooks(cb)
    sh = ShardedIVFPQIndex.wrap(local, kc, nprobe)
    sh.set_list_bounds(np.concatenate([np.linspace(0, kc - 1, world).round(), [kc]]).astype(np.int64))
    mine = np.arange(rank, n, world)
    sh.add(torch.from_numpy(xb[mine]).cuda(), torch.from_numpy(ids[mine]).cuda())
    if rank == world - 1:
        assert local.count == few, local.count
    sd, si = sh.batch_search(q, k)
    assert (si >= 0).all() and np.array_equal(si, fi), "padded shard: ids"
    same_as_single(si, sd, fi, fd, "padded shard")
    if rank == 0:
        print(f"ok padded shard: world {world}, the last rank holds {few} rows", flush=True)
    sh.comm.close()


def main():
    import torch
    import torch.distributed as dist
    from oracle import oracle
    from vectorindex_b200 import _lib
    from vectorindex_b200.index import IVFPQIndex, ShardedIVFPQIndex, balanced_list_bounds

    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
    _lib.check(_lib.lib().vix_set_device(int(os.environ["LOCAL_RANK"])))
    dist.init_process_group("nccl", device_id=torch.device("cuda", int(os.environ["LOCAL_RANK"])))
    for metric in ("euclidean", "dotProduct"):
        n, d, m, kc, nq, k, nprobe = 20000, 96, 48, 64, 333, 10, 9
        rng = np.random.default_rng(7)
        centres = rng.standard_normal((kc, d)).astype(np.float32)
        xb = (centres[rng.integers(0, kc, n)] + 0.3 * rng.standard_normal((n, d))).astype(np.float32)
        q = (centres[rng.integers(0, kc, nq)] + 0.3 * rng.standard_normal((nq, d))).astype(np.float32)
        cb = (0.3 * rng.standard_normal((m, 256, d // m))).astype(np.float32)
        ids = (np.arange(n, dtype=np.int64) * 3 + 11)
        full = IVFPQIndex(d, metric, nlist=kc, nprobe=nprobe, m=m)
        full.set_coarse(centres)
        full.set_codebooks(cb)
        full.batch_insert(xb, ids)
        fd, fi = full.batch_search(q, k)
        local = IVFPQIndex(d, metric, nlist=kc, nprobe=nprobe, m=m)
        local.set_coarse(centres)
        local.set_codebooks(cb)
        sh = ShardedIVFPQIndex.wrap(local, kc, nprobe)
        counts = np.bincount(full.export_lists()[3], minlength=kc)
        sh.set_list_bounds(balanced_list_bounds(counts, world))
        mine = np.arange(rank, n, world)                                   # ragged, interleaved contributions
        sh.add(torch.from_numpy(xb[mine]).cuda(), torch.from_numpy(ids[mine]).cuda())
        sizes = torch.tensor([local.count], device="cuda")
        dist.all_reduce(sizes)
        assert int(sizes.item()) == n, (int(sizes.item()), n)
        # host queries in, host results out
        sd, si = sh.batch_search(q, k)
        # same ids; distances agree to fp32 rounding (a vector's 48 table entries are summed in the order of its rotated code
        # layout, which depends on its slot inside its list -- and the shards receive their rows in another order)
        same_as_single(si, sd, fi, fd, f"{metric}: host path")
        if metric == "euclidean":
            # the list-major tensor-core scan on every rank (dsub = 2; forced, the batch is below its threshold): the per-query
            # bounds of the filter are reduced over the ranks (peer memory: stores + barrier; else an NCCL all-reduce), and the
            # result is the query-major scan's on the same shards, bit for bit
            os.environ["VIX_TC_SCAN"] = "1"
            before = _lib.lib().vix_scan_tc_launches()
            td, ti = sh.batch_search(q, k)
            td2, ti2 = sh.batch_search(q, k)                                # the bound slots were reset for the next call
            assert _lib.lib().vix_scan_tc_launches() == before + 2
            del os.environ["VIX_TC_SCAN"]
            assert np.array_equal(ti, si) and np.array_equal(td.view(np.uint32), sd.view(np.uint32)), "list-major != query-major"
            assert np.array_equal(ti2, si) and np.array_equal(td2.view(np.uint32), sd.view(np.uint32)), "list-major, second call"
        # device queries, asynchronous mode
        _lib.lib().vix_set_async(1)
        qd = torch.from_numpy(q).cuda()
        dd, di = sh.batch_search(qd, k)
        dd2, di2 = sh.batch_search(qd[:50].contiguous(), 3, nprobe=4)     # another shape through the same regions
        torch.cuda.synchronize()
        _lib.lib().vix_set_async(0)
        same_as_single(di.cpu().numpy(), dd.cpu().numpy(), fi, fd, f"{metric}: device path")
        f2d, f2i = full.batch_search(q[:50], 3, nprobe=4)
        same_as_single(di2.cpu().numpy(), dd2.cpu().numpy(), f2i, f2d, f"{metric}: second shape")
        # the oracle on the same lists (stage-wise parity of the merged result)
        off, codes, lids, _ = full.export_lists()
        _, norms = full.get_codebooks()
        od, oi, _ = oracle.ivfpq_search(q, centres, cb, norms, off, codes, lids, m, 256, nprobe, k, 1 if metric == "dotProduct" else 0)
        np.testing.assert_allclose(sd, od, rtol=1e-5, atol=1e-6)
        same = np.mean([len(set(si[r]) & set(oi[r])) / k for r in range(nq)])
        assert same > 0.999, same
        peer = sh.comm.uses_peer_memory
        want_peer = 0 if os.environ.get("VIX_NO_P2P") else 1
        assert peer == want_peer, f"peer memory state {peer}, expected {want_peer}"
        # empty batch on every rank
        ed, ei = sh.batch_search(np.zeros((0, d), np.float32), k)
        assert ed.shape == (0, k)
        if rank == 0:
            print(f"ok {metric}: world {world}, peer memory {peer}, {n} rows, top-k overlap with the oracle {same:.4f}", flush=True)
        sh.comm.close()
    padded_shard_case(rank, world)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
