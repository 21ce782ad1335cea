#!/usr/bin/env python
"""Removal on the headline index: bench.py's C5 (IVF-PQ 100M x 96, nlist 65536, M = 48) built on one GPU, then

  - batch_remove of 1 % of the ids (1M, random) and of 10 ids, each followed by the first search (which rebuilds the lists)
    and a steady-state search, timed with CUDA events;
  - one more 1 % removal under torch.profiler: the compaction kernels' time and achieved bytes/s against 7.7 TB/s;
  - no removed id in any result, and recall@10 of the first 256 queries against the exact top-10 of the remaining rows.

Prints one JSON line with the GPU's name and power limit read in the same run.

    python scripts/remove_bench.py [--workload c5|c5s|tiny] [--searches 5]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (bench.main runs only as a script)

B200_HBM = 7.7e12


def power_limit_w():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i",
                              os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0]],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return float(out[0])
    except Exception:  # noqa: BLE001
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="c5", choices=["c5", "c5s", "tiny"])
    ap.add_argument("--searches", type=int, default=5)
    args = ap.parse_args()
    import torch
    from vectorindex_b200 import kernels as vk

    cfg = dict(bench.PRESETS[args.workload])
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    synth = bench.Synth(cfg, dev)
    t0 = time.time()
    idx, _, _, build_t = bench.build_index(cfg, synth, 0, 1)
    n, k, nq = cfg["n"], cfg["k"], cfg["nq"]
    q = synth.queries(nq)
    ev = lambda: torch.cuda.Event(enable_timing=True)                      # noqa: E731

    def timed(fn):
        torch.cuda.synchronize()
        a, b = ev(), ev()
        a.record()
        out = fn()
        b.record()
        torch.cuda.synchronize()
        return out, a.elapsed_time(b)

    def steady():
        ms = [timed(lambda: idx.batch_search(q, k))[1] for _ in range(args.searches)]
        return float(np.median(ms))

    for _ in range(3):
        idx.batch_search(q, k)
    before = {"search_ms": steady(), "qps": None}
    before["qps"] = nq / before["search_ms"] * 1e3
    gen = torch.Generator(device=dev)
    gen.manual_seed(2024)
    removed_all = []
    report = {}
    for name, count in (("remove_1pct", n // 100), ("remove_10", 10)):
        ids = torch.randperm(n, generator=gen, device=dev)[:count].to(torch.int64)
        if removed_all:                                                      # ids not removed before
            ids = ids[~torch.isin(ids, torch.cat(removed_all))]
        removed_all.append(ids)
        got, ms_remove = timed(lambda: idx.batch_remove(ids))
        (_, ri), ms_first = timed(lambda: idx.batch_search(q, k))
        ms_steady = steady()
        report[name] = {"ids": int(ids.numel()), "removed": got, "ms_remove": round(ms_remove, 3),
                        "ms_first_search": round(ms_first, 3), "ms_steady_search": round(ms_steady, 3),
                        "ms_list_rebuild_est": round(ms_first - ms_steady, 3),
                        "removed_id_in_results": bool(torch.isin(ri, torch.cat(removed_all)).any())}
    # the compaction kernels of one more 1 % removal
    ids = torch.randperm(n, generator=gen, device=dev)[: n // 100].to(torch.int64)
    ids = ids[~torch.isin(ids, torch.cat(removed_all))]
    removed_all.append(ids)
    rows_before = idx.count
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        got = idx.batch_remove(ids)
        torch.cuda.synchronize()
    kt = {}
    for e in prof.key_averages():
        if e.device_type.name == "CUDA":
            kt[e.key] = kt.get(e.key, 0.0) + e.device_time_total / 1e3            # ms
    compact_ms = sum(v for kname, v in kt.items() if "compact_rows_kernel" in kname)
    kept = rows_before - got
    row_bytes = 8 + 4 + cfg["m"]                                              # ids, assign, codes
    moved = rows_before * row_bytes + kept * row_bytes + 3 * rows_before * 8   # read all, write kept, keep + pos per array
    report["remove_1pct_profiled"] = {
        "removed": got, "kernel_ms": {kname: round(v, 3) for kname, v in sorted(kt.items(), key=lambda x: -x[1])[:8]},
        "compaction_ms": round(compact_ms, 3), "compaction_bytes": moved,
        "compaction_tb_s": round(moved / (compact_ms * 1e-3) / 1e12, 3) if compact_ms else None,
        "compaction_share_of_7.7tb_s": round(moved / (compact_ms * 1e-3) / B200_HBM, 3) if compact_ms else None}
    # recall@10 of the remaining rows: exact top-10 over the rows not removed, first bench.GT_QUERIES queries
    gone = torch.cat(removed_all)
    qgt = q[: bench.GT_QUERIES].contiguous()
    deep = 64
    gd = torch.full((qgt.shape[0], deep), float("inf"), device=dev)
    gi = torch.full((qgt.shape[0], deep), -1, dtype=torch.int64, device=dev)
    for b, c in bench.chunks_of(n):
        dd, ii = vk.flat_search_f32(qgt, synth.rows(b, c), deep, 0)
        alld, alli = torch.cat([gd, dd], 1), torch.cat([gi, ii + b], 1)
        o = torch.argsort(alld, dim=1, stable=True)[:, :deep]
        gd, gi = torch.gather(alld, 1, o), torch.gather(alli, 1, o)
    truth = np.stack([r[~np.isin(r, gone.cpu().numpy())][:k] for r in gi.cpu().numpy()])
    _, ri = idx.batch_search(q, k)
    after = {"search_ms": steady()}
    after["qps"] = nq / after["search_ms"] * 1e3
    line = {"workload": cfg["label"], "gpu": torch.cuda.get_device_name(dev), "power_limit_w": power_limit_w(),
            "rows_before": n, "rows_after": idx.count, "build": build_t, "steady_before": before, "steady_after": after,
            **report,
            "removed_id_in_final_results": bool(torch.isin(ri, gone).any()),
            "recall_at_10_remaining_rows": bench.recall_at_k(ri[: bench.GT_QUERIES], torch.from_numpy(truth), k),
            "wall_s": round(time.time() - t0, 1)}
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
