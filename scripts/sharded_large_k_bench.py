"""Sharded k-NN search beyond 512 neighbours on bench.py's IVF-PQ workloads, one process per GPU.

Builds the list-sharded index of a bench.py preset (its own PRESETS / Synth / build_index, the partition bench.py uses) and
times ShardedIVFPQIndex.batch_search over the whole query batch with CUDA events after a warm-up call (queries and results
on the device), for k in 10 and 512 (the fused step) and 513, 1000, 4096 (the two-pass route with one bound per query shared
by all ranks).  Run it at N ranks and at one to compare: with one rank the call is the one-GPU search.  For k > 512 it
reads the VIX_SCAN_DEBUG line of one more call and reports, per query over k: the seed entries, the collected entries, the
entries sent after the cut at k (summed over the ranks) and the merged entries (with more than one rank; with one rank the
"[vix knn]" line's seed and collected entries), and the three vix_comm_trace phases.  Rank 0 prints one JSON line per
preset with the card name and power limit read in the same run.

    python -m torch.distributed.run --nproc-per-node=N scripts/sharded_large_k_bench.py [--workloads c3 c5s] [--reps 3]
"""
import argparse
import ctypes as C
import json
import os
import re
import subprocess
import sys
import tempfile
from datetime import timedelta

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

KS = [10, 512, 513, 1000, 4096]


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


def debug_line(fn):
    """one call with VIX_SCAN_DEBUG=1 -> the text it printed on stderr"""
    os.environ["VIX_SCAN_DEBUG"] = "1"
    with tempfile.TemporaryFile(mode="w+") as f:
        saved = os.dup(2)
        os.dup2(f.fileno(), 2)
        try:
            fn()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            del os.environ["VIX_SCAN_DEBUG"]
        f.seek(0)
        return f.read()


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
    import torch.distributed as dist
    import bench
    cfg = dict(bench.PRESETS[name])
    dev = torch.device("cuda", torch.cuda.current_device())
    synth = bench.Synth(cfg, dev)
    idx, sh, _, times = bench.build_index(cfg, synth, rank, world, bcast)
    if sh is None:
        from vectorindex_b200.index import ShardedIVFPQIndex
        sh = ShardedIVFPQIndex.wrap(idx, cfg["nlist"], cfg["nprobe"])
    q = synth.queries(cfg["nq"]).contiguous()
    nq = q.shape[0]
    knn = sh.batch_search if world > 1 else idx.batch_search      # (one rank: vix_sharded_search is the local search)
    out = dict(workload=name, label=cfg.get("label", name), world=world, nq=nq, nprobe=cfg["nprobe"], build=times)
    rows = []
    for k in KS:
        ms = timed(lambda: knn(q, k), reps)
        row = dict(k=k, ms=round(ms, 4), queries_per_s=round(nq / ms * 1e3))
        if k > 512:
            text = debug_line(lambda: knn(q, k))
            m = re.findall(r"\[vix sharded knn\] .*seed (\d+), local (\d+), sent (\d+), total (\d+), max_row (\d+)", text)
            if m:
                seed, local, sent, total, _ = (int(x) for x in m[-1])
                t = torch.tensor([seed, local, sent], dtype=torch.int64, device=dev)
                dist.all_reduce(t)
                seed, local, sent = t.cpu().tolist()
                row.update(seed_over_k=round(seed / (nq * k), 3), collected_over_k=round(local / (nq * k), 3),
                           sent_over_k=round(sent / (nq * k), 3), merged_over_k=round(total / (nq * k), 3))
            else:
                m = re.findall(r"\[vix knn\] .*seed (\d+), total (\d+)", text)
                if m:
                    seed, total = (int(x) for x in m[-1])
                    row.update(seed_over_k=round(seed / (nq * k), 3), collected_over_k=round(total / (nq * k), 3))
        if world > 1:
            row["phases_ms"] = phases(sh, lambda: knn(q, k))
        rows.append(row)
    out["rows"] = rows
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", nargs="+", default=["c3", "c5s"])
    ap.add_argument("--reps", type=int, default=3)
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
