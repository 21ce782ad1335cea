"""List shards against replicas, side by side, through the library's exchange (vix_sharded_* / vix_replicated_*).

Run under torch.distributed.run with one process per GPU (world = every GPU of the box), or as a plain script for one
rank.  For each workload every rank generates the same data on its GPU (a clustered mixture; inner product on unit rows for
the C4 shape), rank 0 trains the quantisers and broadcasts them, and both layouts are filled through their collective adds
(every rank contributes its slice of the rows).  Then, with device-resident queries and outputs:
  - ms per batch (median of `reps` calls, host clock around calls that end in a device synchronise, after warm-up) and
    queries/s, for ShardedIVFPQIndex / ShardedFlatIndex and ReplicatedNativeIVFPQIndex / ReplicatedFlatIndex;
  - the vix_comm_trace phases of one call of each layout (sharded: probes + exchange | scan | merge; replicated: queries in |
    local search | assembly);
  - the card's name and power limit, read in the same run.
Workloads (--scale scales the database of each): C4-shaped IVF-PQ inner product, 768-d, nlist 16384, nprobe 32, M 64;
C5s-shaped IVF-PQ L2 96-d, nlist 8192, nprobe 8, M 48; flat L2 1M x 128.  10k queries, k = 10.  Prints one JSON line per
workload on rank 0 and writes them to --out.
Usage: torchrun --nproc-per-node=G scripts/replicated_bench.py [--scale 0.1] [--reps 10] [--out replicated.json]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

WORKLOADS = {
    "c4": dict(n=10_000_000, d=768, nlist=16384, nprobe=32, m=64, metric="dotProduct", kind="ivfpq"),
    "c5s": dict(n=12_500_000, d=96, nlist=8192, nprobe=8, m=48, metric="euclidean", kind="ivfpq"),
    "flat": dict(n=1_000_000, d=128, metric="euclidean", kind="flat"),
}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def make_data(torch, dev, n, d, nq, unit, seed):
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    nc = 4096
    cent = torch.randn((nc, d), generator=g, device=dev)
    cent = cent / cent.norm(dim=1, keepdim=True)
    sigma = 0.3 / d ** 0.5 * 4
    x = torch.empty((n, d), device=dev)
    for a in range(0, n, 1 << 20):
        b = min(n, a + (1 << 20))
        lab = torch.randint(0, nc, (b - a,), generator=g, device=dev)
        x[a:b] = cent[lab] + sigma * torch.randn((b - a, d), generator=g, device=dev)
    lab = torch.randint(0, nc, (nq,), generator=g, device=dev)
    q = cent[lab] + sigma * torch.randn((nq, d), generator=g, device=dev)
    if unit:
        x = x / x.norm(dim=1, keepdim=True)
        q = q / q.norm(dim=1, keepdim=True)
    return x.contiguous(), q.contiguous()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of each workload's database size")
    ap.add_argument("--nq", type=int, default=10_000)
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--workloads", default="c4,c5s,flat")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch
    import torch.distributed as dist
    from vectorindex_b200 import _lib
    from vectorindex_b200.index import (IVFPQIndex, ReplicatedFlatIndex, ReplicatedNativeIVFPQIndex, ShardedFlatIndex,
                                        ShardedIVFPQIndex)
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    _lib.check(_lib.lib().vix_set_device(local))
    if "WORLD_SIZE" not in os.environ:                                  # a plain run: a one-rank group
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT="29611", RANK="0", WORLD_SIZE="1")
    dist.init_process_group("nccl")
    rank, world = dist.get_rank(), dist.get_world_size()
    dev = torch.device("cuda", local)
    name = card()
    lines = []
    for wl in args.workloads.split(","):
        cfg = dict(WORKLOADS[wl])
        n = max(int(cfg["n"] * args.scale), 65536)
        d = cfg["d"]
        x, q = make_data(torch, dev, n, d, args.nq, cfg["metric"] == "dotProduct", 7)
        ids = torch.arange(n, dtype=torch.int64, device=dev)
        per = (n + world - 1) // world
        lo, hi = min(n, rank * per), min(n, (rank + 1) * per)
        if cfg["kind"] == "ivfpq":
            ref = IVFPQIndex(d, cfg["metric"], nlist=cfg["nlist"], nprobe=cfg["nprobe"], m=cfg["m"])
            if rank == 0:
                ref.optimize(x[:min(n, max(32 * cfg["nlist"], 65536))])
                cb, norms = ref.get_codebooks()
                parts = [torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in (ref.get_coarse(), cb, norms)]
            else:
                parts = [torch.empty((cfg["nlist"], d), device=dev), torch.empty((cfg["m"], 256, d // cfg["m"]), device=dev),
                         torch.empty((cfg["m"], 256), device=dev)]
            if world > 1:
                for t in parts:
                    dist.broadcast(t, 0)
            coarse, cb, norms = (t.cpu().numpy() for t in parts)
            sh = ShardedIVFPQIndex(d, cfg["metric"], nlist=cfg["nlist"], nprobe=cfg["nprobe"], m=cfg["m"])
            sh.set_parameters(coarse, cb, norms)
            rep = ReplicatedNativeIVFPQIndex(d, cfg["metric"], nlist=cfg["nlist"], nprobe=cfg["nprobe"], m=cfg["m"])
            rep.set_parameters(coarse, cb, norms)
        else:
            sh, rep = ShardedFlatIndex(d, cfg["metric"]), ReplicatedFlatIndex(d, cfg["metric"])
        sh.add(x[lo:hi], ids[lo:hi])
        rep.add(x[lo:hi], ids[lo:hi])
        del x
        torch.cuda.synchronize()
        row = {"workload": wl, "n": n, "d": d, "nq": args.nq, "k": args.k, "world": world, "card": name,
               "nprobe": cfg.get("nprobe"), "m": cfg.get("m"), "nlist": cfg.get("nlist"), "metric": cfg["metric"]}
        for label, ix in (("sharded", sh), ("replicated", rep)):
            def call():
                return ix.batch_search(q, args.k)
            for _ in range(3):
                call()
            torch.cuda.synchronize()
            ts = []
            for _ in range(args.reps):
                if world > 1:
                    dist.barrier()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                call()
                torch.cuda.synchronize()
                ts.append(time.perf_counter() - t0)
            ms = float(np.median(ts)) * 1e3
            row[f"{label}_ms"] = round(ms, 3)
            row[f"{label}_qps"] = round(args.nq / (ms / 1e3))
            comm = ix.__dict__.get("comm")
            if comm is not None:
                L = _lib.lib()
                _lib.check(L.vix_comm_trace(comm._c, 1))
                call()
                ph = (C.c_float * 3)()
                _lib.check(L.vix_comm_trace_get(comm._c, ph))
                _lib.check(L.vix_comm_trace(comm._c, 0))
                row[f"{label}_phases_ms"] = [round(v, 3) for v in ph]
            else:
                row[f"{label}_phases_ms"] = "not measured (one rank: the local index, no exchange)"
        del sh, rep
        torch.cuda.empty_cache()
        if rank == 0:
            print(json.dumps(row), flush=True)
        lines.append(row)
    if rank == 0 and args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for row in lines:
                f.write(json.dumps(row) + "\n")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
