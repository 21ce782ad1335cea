"""k-NN search beyond 512 neighbours (the two-pass route over the range-search scans) against the fused route (one GPU).

Shapes: bench.py's IVF-PQ presets (c3: 1M x 128, nprobe 32, 10k queries; c5s), built with bench.py's own PRESETS / Synth /
build_index, and flat indexes of 100k x 128 (the c1 shape, 1k queries) and 1M x 128 (1k queries) of standard-normal rows.
For k in 10, 512 (the fused route) and 513, 1000, 2048, 4096 (the two-pass route) it times batch_search over the whole
query batch with CUDA events after a warm-up call (queries and results on the device), and reads the "[vix knn]" line of
one more call: seed entries and collected entries per query over k (how loose the seed is) and the passes of the collect.
Prints one JSON line per shape with the card's name and power limit, read in the same run.

    python scripts/large_k_bench.py [--workloads c3 c5s flat100k flat1m] [--reps 5]
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

KS = [10, 512, 513, 1000, 2048, 4096]


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


def route_of(fn):
    """one call with VIX_SCAN_DEBUG=1; the fields of its [vix knn] line (stderr captured through a temporary file)"""
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
        m = re.findall(r"\[vix knn\] .*seed (\d+), total (\d+), passes (\d), max_row (\d+)", f.read())
    if not m:
        return None
    s, t, p, mx = (int(x) for x in m[-1])
    return dict(seed=s, total=t, passes=p, max_row=mx)


def sweep(search, nq, reps):
    rows = []
    for k in KS:
        ms = timed(lambda: search(k), reps)
        row = dict(k=k, ms=round(ms, 4), queries_per_s=round(nq / ms * 1e3))
        info = route_of(lambda: search(k)) if k > 512 else None
        if info:
            row.update(seed_over_k=round(info["seed"] / (nq * k), 3), total_over_k=round(info["total"] / (nq * k), 3),
                       passes=info["passes"], max_row=info["max_row"])
        rows.append(row)
    return rows


def run_ivfpq(name, reps):
    import torch
    import bench
    cfg = dict(bench.PRESETS[name])
    synth = bench.Synth(cfg, torch.device("cuda:0"))
    idx, _, _, times = bench.build_index(cfg, synth, 0, 1)
    q = synth.queries(cfg["nq"]).contiguous()
    out = dict(workload=name, label=cfg.get("label", name), nq=q.shape[0], nprobe=cfg["nprobe"], build=times)
    out["rows"] = sweep(lambda k: idx.batch_search(q, k), q.shape[0], reps)
    return out


def run_flat(name, n, reps):
    import torch
    from vectorindex_b200.index import FlatIndex
    g = torch.Generator(device="cuda:0")
    g.manual_seed(123)
    d, nq = 128, 1000
    xb = torch.randn(n, d, device="cuda:0", generator=g)
    q = torch.randn(nq, d, device="cuda:0", generator=g)
    idx = FlatIndex(d, "euclidean")
    idx.batch_insert(xb)
    out = dict(workload=name, label=f"flat L2 {n} x {d} standard-normal rows, {nq} queries", nq=nq)
    out["rows"] = sweep(lambda k: idx.batch_search(q, k), nq, reps)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", nargs="+", default=["c3", "c5s", "flat100k", "flat1m"])
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    name, power = card()
    for w in args.workloads:
        if w == "flat100k":
            res = run_flat(w, 100_000, args.reps)
        elif w == "flat1m":
            res = run_flat(w, 1_000_000, args.reps)
        else:
            res = run_ivfpq(w, args.reps)
        res["gpu"], res["power_limit"] = name, power
        print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
