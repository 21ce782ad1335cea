"""Sharded range search against sharded k-NN search on bench.py's IVF-PQ workloads, one process per GPU.

Builds the list-sharded index of a bench.py preset (its own PRESETS / Synth / build_index, the partition bench.py uses),
picks radii at which the mean number of results per query is about 10, 100 and 1000 (bisection on a sample of the queries,
every rank alike), and times with CUDA events, after a warm-up, over the whole query batch (queries and results on the
device):
  - ShardedIVFPQIndex.range_search at each radius (vix_sharded_range_search);
  - ShardedIVFPQIndex.batch_search, k = 10 (vix_sharded_search).
With more than one rank it also reads the three phases of one call of each (vix_comm_trace: probes exchanged | local scan
and sort | exchange, merge and decode) and counts the bytes that reach each rank in the exchanges.  Rank 0 prints one JSON
line per preset with the card name and power limit read in the same run.

    python -m torch.distributed.run --nproc-per-node=N scripts/sharded_range_bench.py [--workloads c5s] [--reps 5]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
from datetime import timedelta

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
        return name, power
    except Exception as e:                                     # report, do not guess
        return f"unknown ({e})", "unknown"


def timed(fn, reps):
    import torch
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def pick_radius(sh, q, target, hi):
    """radius whose mean results per query over q is about `target` (bisection; collective, every rank takes the same
    steps because every rank receives the same answer)"""
    while True:
        if float(sh.range_search(q, hi)[0][-1]) / q.shape[0] >= target:
            break
        hi = hi * 2.0 if hi > 0 else hi / 2.0 + 1.0
    lo = 0.0 if hi > 0 else hi * 2
    for _ in range(30):
        mid = 0.5 * (lo + hi)
        mean = float(sh.range_search(q, mid)[0][-1]) / q.shape[0]
        if abs(mean - target) <= 0.02 * target:
            return mid
        lo, hi = (mid, hi) if mean < target else (lo, mid)
    return 0.5 * (lo + hi)


def phases(sh, fn):
    """the three vix_comm_trace phases (ms) of one call of fn"""
    from vectorindex_b200 import _lib
    comm = sh.__dict__.get("comm")
    if comm is None:
        return None
    L = _lib.lib()
    _lib.check(L.vix_comm_trace(comm._c, 1))
    fn()
    ph = (C.c_float * 3)()
    _lib.check(L.vix_comm_trace_get(comm._c, ph))
    _lib.check(L.vix_comm_trace(comm._c, 0))
    return [round(float(v), 4) for v in ph]


def run(name, reps, rank, world, bcast):
    import torch
    import bench
    cfg = dict(bench.PRESETS[name])
    dev = torch.device("cuda", torch.cuda.current_device())
    synth = bench.Synth(cfg, dev)
    idx, sh, _, times = bench.build_index(cfg, synth, rank, world, bcast)
    if sh is None:
        from vectorindex_b200.index import ShardedIVFPQIndex
        sh = ShardedIVFPQIndex.wrap(idx, cfg["nlist"], cfg["nprobe"])
    q = synth.queries(cfg["nq"]).contiguous()
    nq, nprobe = q.shape[0], cfg["nprobe"]
    sample = q[:500].contiguous()
    knn = sh.batch_search if world > 1 else idx.batch_search      # (one rank: vix_sharded_search is the local search)
    kd, _ = knn(sample, 10)
    out = dict(workload=name, label=cfg.get("label", name), world=world, nq=nq, nprobe=nprobe, build=times)
    out["knn_ms"] = round(timed(lambda: knn(q, 10), reps), 4)
    out["knn_phases_ms"] = phases(sh, lambda: knn(q, 10))
    rows = []
    for target in (10, 100, 1000):
        r = pick_radius(sh, sample, target, float(kd[:, -1].median().item()))
        ms = timed(lambda: sh.range_search(q, r), reps)
        lims = sh.range_search(q, r)[0]
        total = int(lims[-1])
        local = 0
        if world > 1:                                          # entries this rank found itself (its own lists)
            loc = idx.range_search(q, r, nprobe=nprobe)[0]     # (probes equal: every rank holds every centroid)
            local = int(loc[-1])
            t = torch.tensor([local], dtype=torch.int64, device=dev)
            allt = torch.empty(world, dtype=torch.int64, device=dev)
            import torch.distributed as dist
            dist.all_gather_into_tensor(allt, t)
            locs = allt.cpu().tolist()
        else:
            locs = [total]
        # bytes that reach rank 0 from its peers: probes of the other blocks, the peers' row starts, the peers' keys
        per = -(-nq // world)
        recv = ((world - 1) * per * nprobe * 4 + (world - 1) * (nq + 2) * 8 + 8 * (total - locs[0])) if world > 1 else 0
        rows.append(dict(target=target, radius=r, mean_results=round(total / nq, 1), ms=round(ms, 4),
                         queries_per_s=round(nq / ms * 1e3), results_per_s=round(total / ms * 1e3),
                         local_results=locs, bytes_received_rank0=recv, vs_knn=round(ms / out["knn_ms"], 3),
                         phases_ms=phases(sh, lambda: sh.range_search(q, r))))
    out["range"] = rows
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", nargs="+", default=["c5s"])
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    import torch
    import torch.distributed as dist
    from vectorindex_b200 import _lib
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    _lib.check(_lib.lib().vix_set_device(local))
    bcast = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local), timeout=timedelta(seconds=1800))
        bcast = lambda t: dist.broadcast(t, 0)
    name, power = card()
    try:
        for w in args.workloads:
            res = run(w, args.reps, rank, world, bcast)
            res["gpu"], res["power_limit"] = name, power
            if rank == 0:
                print(json.dumps(res), flush=True)
    finally:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
