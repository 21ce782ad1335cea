"""One rank of the multi-GPU removal check (launched by tests/test_remove.py under torch.distributed.run, one process per
GPU): rows added through the native sharded step, the same ids removed on every rank by ShardedIVFPQIndex.remove; the
summed count and vix_sharded_search equal a single-GPU index holding all rows after the same removal."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    import torch
    import torch.distributed as dist
    from mp_sharded_check import same_as_single
    from vectorindex_b200 import _lib
    from vectorindex_b200.index import IVFPQIndex, ShardedIVFPQIndex

    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
    _lib.check(_lib.lib().vix_set_device(int(os.environ["LOCAL_RANK"])))
    dist.init_process_group("nccl", device_id=torch.device("cuda", int(os.environ["LOCAL_RANK"])))
    n, d, m, kc, nq, k, nprobe = 20000, 96, 48, 64, 333, 10, 9
    rng = np.random.default_rng(17)
    centres = rng.standard_normal((kc, d)).astype(np.float32)
    xb = (centres[rng.integers(0, kc, n)] + 0.3 * rng.standard_normal((n, d))).astype(np.float32)
    q = (centres[rng.integers(0, kc, nq)] + 0.3 * rng.standard_normal((nq, d))).astype(np.float32)
    cb = (0.3 * rng.standard_normal((m, 256, d // m))).astype(np.float32)
    ids = np.arange(n, dtype=np.int64) * 3 + 11
    ids[::97] = ids[1::97][: ids[::97].size]                               # some ids stored twice
    S = np.concatenate([rng.choice(ids, n // 5, replace=False), [0, 1, 2 ** 32 - 2], ids[1::97][:5]])
    full = IVFPQIndex(d, "euclidean", nlist=kc, nprobe=nprobe, m=m)
    full.set_coarse(centres)
    full.set_codebooks(cb)
    full.batch_insert(xb, ids)
    want = full.batch_remove(S)
    fd, fi = full.batch_search(q, k)
    local = IVFPQIndex(d, "euclidean", nlist=kc, nprobe=nprobe, m=m)
    local.set_coarse(centres)
    local.set_codebooks(cb)
    sh = ShardedIVFPQIndex.wrap(local, kc, nprobe)
    mine = np.arange(rank, n, world)
    sh.add(torch.from_numpy(xb[mine]).cuda(), torch.from_numpy(ids[mine]).cuda())
    sd, si = sh.batch_search(q, k)                                          # lists built before the removal
    got = sh.remove(torch.from_numpy(S).cuda())
    assert got == want, (got, want)
    sizes = torch.tensor([local.count], device="cuda")
    dist.all_reduce(sizes)
    assert int(sizes.item()) == full.count, (int(sizes.item()), full.count)
    sd, si = sh.batch_search(q, k)
    same_as_single(si, sd, fi, fd, "after the removal")
    assert not np.isin(si, S).any()
    if rank == 0:
        print(f"ok remove: world {world}, {want} of {n} rows removed", flush=True)
    sh.comm.close()
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
