"""Range search against k-NN search on bench.py's IVF-PQ workloads (one GPU).

Builds the index of a bench.py preset (its own PRESETS / Synth / build_index), picks radii at which the mean number of
results per query is about 10, 100 and 1000 (bisection on a sample of the queries), and times with CUDA events, after a
warm-up, over the whole query batch:
  - range_search at each radius (queries and results on the device);
  - k-NN batch_search (k = 10) on the query-major scan (VIX_TC_SCAN=0), the scan range search shares;
  - k-NN batch_search on the default path.
Prints one JSON line per preset: card name and power limit (read in the same run), queries/s and results/s per radius, the
passes and rows sorted in global memory of each range call (its "[vix range]" line), and the k-NN times.

    python scripts/range_bench.py [--workloads c3 c5] [--reps 5]
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile

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


def route_of(idx, q, radius):
    """one range call with VIX_SCAN_DEBUG=1; its [vix range] fields (stderr captured through a temporary file)"""
    os.environ["VIX_SCAN_DEBUG"] = "1"
    with tempfile.TemporaryFile(mode="w+") as f:
        saved = os.dup(2)
        os.dup2(f.fileno(), 2)
        try:
            idx.range_search(q, radius)
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            del os.environ["VIX_SCAN_DEBUG"]
        f.seek(0)
        m = re.findall(r"\[vix range\] .*passes (\d), total (\d+), max_row (\d+), sorted_long (\d+)", f.read())
    p, t, mx, sl = (int(x) for x in m[-1])
    return dict(passes=p, total=t, max_row=mx, sorted_long=sl)


def pick_radius(idx, q, target, hi):
    """radius whose mean results per query over q is about `target` (bisection)"""
    while True:
        lims = idx.range_search(q, hi)[0]
        if float(lims[-1]) / q.shape[0] >= target:
            break
        hi *= 2.0
    lo = 0.0 if hi > 0 else hi * 2
    for _ in range(30):
        mid = 0.5 * (lo + hi)
        mean = float(idx.range_search(q, mid)[0][-1]) / q.shape[0]
        if abs(mean - target) <= 0.02 * target:
            return mid
        lo, hi = (mid, hi) if mean < target else (lo, mid)
    return 0.5 * (lo + hi)


def run(name, reps):
    import torch
    import bench
    cfg = dict(bench.PRESETS[name])
    dev = torch.device("cuda:0")
    synth = bench.Synth(cfg, dev)
    idx, _, _, times = bench.build_index(cfg, synth, 0, 1)
    q = synth.queries(cfg["nq"]).contiguous()
    nq = q.shape[0]
    sample = q[:500].contiguous()
    kd, _ = idx.batch_search(sample, 10)
    out = dict(workload=name, label=cfg.get("label", name), nq=nq, nprobe=cfg["nprobe"], build=times)
    os.environ["VIX_TC_SCAN"] = "0"
    out["knn_query_major_ms"] = round(timed(lambda: idx.batch_search(q, 10), reps), 4)
    del os.environ["VIX_TC_SCAN"]
    out["knn_default_ms"] = round(timed(lambda: idx.batch_search(q, 10), reps), 4)
    rows = []
    for target in (10, 100, 1000):
        r = pick_radius(idx, sample, target, float(kd[:, -1].median().item()))
        ms = timed(lambda: idx.range_search(q, r), reps)
        info = route_of(idx, q, r)
        rows.append(dict(target=target, radius=r, mean_results=round(info["total"] / nq, 1), ms=round(ms, 4),
                         queries_per_s=round(nq / ms * 1e3), results_per_s=round(info["total"] / ms * 1e3),
                         passes=info["passes"], sorted_long=info["sorted_long"], max_row=info["max_row"],
                         vs_query_major_knn=round(ms / out["knn_query_major_ms"], 3)))
    out["range"] = rows
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", nargs="+", default=["c3"])
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    name, power = card()
    for w in args.workloads:
        res = run(w, args.reps)
        res["gpu"], res["power_limit"] = name, power
        print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
