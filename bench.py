#!/usr/bin/env python
"""bench.py -- IVF-PQ batched search throughput (BASELINE.json's metric) on 1..8 B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c5|c5s|c3|tiny] [--impl reference]
                    [--dump-outputs DIR]

One "step" = one pass of the search hot path (probe selection -> query-only LUT -> fused ADC list scan +
top-k [-> all-gather + mergeTopK at N > 1]) over ONE batch of nq synthetic queries against a device-resident
IVF-PQ index.  The default workload is BASELINE.json's headline configuration (configs[4], "c5"):
IVF-PQ 100M x 96 Deep-shaped, nlist=65536, nprobe=64, M=48, 10k queries, k=10.  The database is FIXED as N
grows (strong scaling): it is partitioned over the ranks, queries are replicated, each rank scans its
partition and the per-rank top-k lists are merged after one all-gather.  (`--partition replicate`: every rank keeps a
full replica and the batch is split by query instead -- for indexes that fit one GPU; not the default.)

Printed JSON line (rank 0): `value` = queries/s with queries and results resident in HBM; `e2e` = the same
through the public API with pinned HOST query/result buffers (H2D + D2H inside the timed region);
`roofline` = the fused ADC-scan kernel against the measured HBM peak (algorithmic bytes = sum over
(query, probed list) of list length x M code bytes, SURVEY.md 8d); `cpu_baseline` = the oracle (C
restatement of the reference arithmetic, OpenMP over queries) on a bounded sample of the same queries.
`--impl reference` times only that CPU path (all host threads) on the same index.

`--dump-outputs DIR` writes what the last timed step returned to its caller as DIR/<name>.npy (float32; ids as float64,
which holds every id exactly): the inputs depend only on the workload and fixed seeds, so two builds of the
project can be compared output for output.  An output above DUMP_LIMIT bytes is cut to a fixed, seeded sample of rows,
whose row numbers are written beside it.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

PRESETS = {
    # BASELINE.json configs[4]; data: unit-norm Gaussian-cluster mixture (recipe of the reference bench,
    # Sources/VectorIndexBenchmarks/main.swift:129-144), generated on the device chunk by chunk
    "c5": dict(n=100_000_000, d=96, nlist=65536, nprobe=64, m=48, nq=10_000, k=10, shape="deep", clusters=100_000,
               label="IVF-PQ 100M x 96 Deep-shaped, nlist=65536, nprobe=64, M=48, batch 10k queries, k=10 (BASELINE configs[4])"),
    # one eighth of c5 (what one GPU holds at N = 8), for kernel work on one GPU
    "c5s": dict(n=12_500_000, d=96, nlist=8192, nprobe=8, m=48, nq=10_000, k=10, shape="deep", clusters=12_500,
                label="one-eighth shard of configs[4]: IVF-PQ 12.5M x 96, nlist=8192, nprobe=8, M=48, batch 10k, k=10"),
    # BASELINE.json configs[3]: inner-product, embedding-shaped; nprobe / batch are not specified there (32 / 10k assumed)
    # data: "embed" = the deep recipe plus near-duplicate structure (groups of 8 rows share a seed vector, queries are
    # perturbed base rows): with isotropic 768-d noise alone every cluster-mate is equidistant from a query and recall@10 of
    # ANY 64-byte code is ~0.05 (round 1), which measures nothing
    "c4": dict(n=10_000_000, d=768, nlist=16384, nprobe=32, m=64, nq=10_000, k=10, shape="embed", clusters=16384, metric="dotProduct",
               label="IVF-PQ inner-product 10M x 768 embedding-shaped, nlist=16384, nprobe=32 (assumed), M=64, batch 10k queries, k=10 (BASELINE configs[3])"),
    "c3": dict(n=1_000_000, d=128, nlist=4096, nprobe=32, m=16, nq=10_000, k=10, shape="sift", clusters=4096,
               label="IVF-PQ 1M x 128 SIFT-shaped, nlist=4096, nprobe=32, M=16, batch 10k queries, k=10 (BASELINE configs[2])"),
    "tiny": dict(n=200_000, d=96, nlist=512, nprobe=8, m=48, nq=1000, k=10, shape="deep", clusters=1000,
                 label="tiny self-test"),
    # BASELINE.json configs[0] / configs[1]: the parity-test configurations, measurable through the same contract
    # (one GPU; `python bench.py --workload c1|c2`); data = the reference benchmark's LCG vectors (main.swift:535-548)
    "c1": dict(kind="flat", n=100_000, d=128, nq=1000, k=10,
               label="Flat exact L2 search, 100k x 128 fp32 synthetic base, 1k queries, k=10 (BASELINE configs[0])"),
    "c2": dict(kind="pq_encode", n=1_000_000, d=128, m=16, ks=256,
               label="PQ train+encode 1M x 128 fp32, M=16 subquantizers x 256 centroids (BASELINE configs[1])"),
}
CHUNK = 1_000_000
GT_QUERIES = 256
SEED = 123
DUMP_LIMIT = 60_000_000                                               # bytes written by --dump-outputs, in all (< 64 MB)


def dump_outputs(out_dir, arrays):
    """Writes name -> host array as out_dir/<name>.npy: integers wider than 16 bits as float64 (exact up to 2^53), the rest
    as float32.  When the whole set would exceed DUMP_LIMIT, every array keeps the same fixed, seeded sample of rows,
    listed in rows.npy."""
    arrays = {name: a.astype(np.float64 if np.issubdtype(a.dtype, np.integer) and a.dtype.itemsize > 2 else np.float32)
              for name, a in arrays.items()}
    n = next(iter(arrays.values())).shape[0]
    row_bytes = sum(a.nbytes for a in arrays.values()) // max(n, 1)
    if row_bytes * n > DUMP_LIMIT:
        rows = np.sort(np.random.default_rng(SEED).choice(n, DUMP_LIMIT // (row_bytes + 8), replace=False))
        arrays = {name: a[rows] for name, a in arrays.items()}
        arrays["rows"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    log(f"[bench] wrote {sorted(arrays)} ({sum(a.nbytes for a in arrays.values())} bytes) to {out_dir}")


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """SM clock + throttle reasons DURING the timed region.  The K timed steps are enqueued asynchronously;
    while the GPU works through them the host polls NVML from the main thread (samples 2 ms apart).
    NVML queries take the driver lock that CUDA API calls need, so polling from a second thread (or an
    `nvidia-smi -lms` child) while the host is still launching stalls the launches -- measured: a 6 ms step
    became 60 ms.  Polling only after everything is enqueued perturbs nothing."""
    NAMES = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, device_index: int):
        self.clocks, self.power, self.reasons, self.max_mhz, self.nv = [], [], set(), None, None
        if os.environ.get("VIX_BENCH_NO_CLOCKS"):
            return
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = device_index
            if vis:
                parts = vis.split(",")
                if device_index < len(parts) and parts[device_index].strip().isdigit():
                    phys = int(parts[device_index])
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nv = pynvml
        except Exception as e:  # noqa: BLE001
            log(f"[bench] NVML unavailable: {e}")

    def sample(self):
        nv = self.nv
        if nv is None:
            return
        try:
            self.clocks.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
            self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
            try:
                r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
            except Exception:  # noqa: BLE001
                r = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
            for bit, name in self.NAMES.items():
                if r & bit:
                    self.reasons.add(name)
        except Exception as e:  # noqa: BLE001
            log(f"[bench] NVML sample failed: {e}")

    def poll_until(self, done, period_s=0.002, max_samples=64):
        """Sample while `done()` is false (at least once)."""
        self.sample()
        while not done() and len(self.clocks) < max_samples:
            time.sleep(period_s)
            self.sample()

    def stop(self):
        pass

    def summary(self):
        return {"sm_mhz": float(np.median(self.clocks)) if self.clocks else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.clocks),
                "power_w_max": max(self.power) if self.power else None}


# ------------------------------------------------------------------------------------------------ data
class Synth:
    """Deterministic synthetic base/query generator on the device (torch is plumbing here: RNG + memory)."""

    def __init__(self, cfg, dev):
        import torch
        self.t, self.cfg, self.dev = torch, cfg, dev
        g = torch.Generator(device=dev)
        g.manual_seed(SEED)
        c = torch.randn((cfg["clusters"], cfg["d"]), generator=g, device=dev)
        if cfg["shape"] in ("deep", "embed"):
            self.centres = c / c.norm(dim=1, keepdim=True)
        else:  # SIFT-shaped: non-negative integer-valued components in [0, 218] with heavy ties
            self.centres = (c.abs() * 40).floor().clamp_(0, 218)

    def rows(self, start: int, count: int, seed: int = SEED):
        torch, cfg = self.t, self.cfg
        g = torch.Generator(device=self.dev)
        g.manual_seed(seed * 1_000_003 + start)
        which = torch.randint(0, cfg["clusters"], (count,), generator=g, device=self.dev)
        noise = torch.randn((count, cfg["d"]), generator=g, device=self.dev)
        if cfg["shape"] == "deep":
            v = self.centres[which] + (0.3 / cfg["d"] ** 0.5) * noise
            v /= v.norm(dim=1, keepdim=True)
            return v.contiguous()
        if cfg["shape"] == "embed":
            # groups of 8 consecutive rows: one cluster, one seed vector (centre + 0.3-norm noise), 0.06-norm noise per row
            grp = torch.arange(count, device=self.dev) // 8
            first = grp * 8                                               # the row whose draws define the group
            v = self.centres[which[first]] + (0.3 / cfg["d"] ** 0.5) * noise[first]
            v += (0.06 / cfg["d"] ** 0.5) * torch.randn((count, cfg["d"]), generator=g, device=self.dev)
            v /= v.norm(dim=1, keepdim=True)
            return v.contiguous()
        return (self.centres[which] + 12.0 * noise).abs_().floor_().clamp_(0, 218).contiguous()

    def queries(self, nq: int):
        if self.cfg["shape"] == "embed":                                   # perturbed base rows (every 7th row of the first chunk)
            torch = self.t
            n0 = min(self.cfg["n"], CHUNK)
            base = self.rows(0, n0)
            pick = (torch.arange(nq, device=self.dev) * 7) % n0
            g = torch.Generator(device=self.dev)
            g.manual_seed(321)
            v = base[pick] + (0.06 / self.cfg["d"] ** 0.5) * torch.randn((nq, self.cfg["d"]), generator=g, device=self.dev)
            v /= v.norm(dim=1, keepdim=True)
            return v.contiguous()
        return self.rows(0, nq, seed=321)


def chunks_of(n):
    return [(b, min(CHUNK, n - b)) for b in range(0, n, CHUNK)]


# ------------------------------------------------------------------------------------------------ build
def build_index(cfg, synth, rank, world, bcast=None, partition="lists"):
    """Train on the first chunks (rank 0, parameters broadcast), then build: every rank generates, assigns and
    encodes ITS chunks of the database; rows travel to the rank owning their inverted list (all-to-all).
    Returns (per-rank index, sharded view or None, exact ground truth of the first GT_QUERIES queries over the
    rows this rank generated, timings)."""
    import torch
    from vectorindex_b200 import kernels as vk
    from vectorindex_b200._lib import KMeansCfg, PQTrainCfg
    from vectorindex_b200.index import IVFPQIndex, ReplicatedIVFPQIndex, ShardedIVFPQIndex

    n, d, nlist, m = cfg["n"], cfg["d"], cfg["nlist"], cfg["m"]
    idx = IVFPQIndex(d, cfg.get("metric", "euclidean"), nlist=nlist, nprobe=cfg["nprobe"], m=m)
    t0 = time.time()
    ntrain = min(n, max(32 * nlist, 65536))
    if rank == 0:
        parts = [synth.rows(b, c) for b, c in chunks_of(ntrain)]
        xt = torch.cat(parts) if len(parts) > 1 else parts[0]
        del parts
        idx.optimize(xt, KMeansCfg(1024, 6, 1e-4, 42, 0, False, 1), PQTrainCfg(0, 8, 1e-4, 1024, 65536, 42, 0, 0, 1))
        del xt
        coarse = torch.from_numpy(idx.get_coarse()).to(synth.dev)
        cb, cn = idx.get_codebooks()
        cb, cn = torch.from_numpy(cb).to(synth.dev), torch.from_numpy(cn).to(synth.dev)
    else:
        coarse = torch.empty((nlist, d), dtype=torch.float32, device=synth.dev)
        cb = torch.empty((m, 256, d // m), dtype=torch.float32, device=synth.dev)
        cn = torch.empty((m, 256), dtype=torch.float32, device=synth.dev)
    sh = None
    if world > 1:
        for t in (coarse, cb, cn):
            bcast(t)
        if rank != 0:
            idx.set_coarse(coarse)
            idx.set_codebooks(cb, cn)
        sh = (ReplicatedIVFPQIndex if partition == "replicate" else ShardedIVFPQIndex).wrap(idx, nlist, cfg["nprobe"])
    if world > 1 and partition != "replicate":
        # list-block boundaries that equalise the ranks' expected scan work (sum of squared list lengths), from the list
        # sizes of a sample: rank 0 assigns its training chunk, every rank gets the boundaries
        from vectorindex_b200.index import balanced_list_bounds
        bounds = torch.zeros(world + 1, dtype=torch.int64, device=synth.dev)
        if rank == 0:
            sample = synth.rows(0, min(n, 2_000_000))
            asg = vk.ivf_assign_f32(sample, coarse) if cfg.get("metric") != "dotProduct" else \
                vk.ivf_assign_metric_f32(sample, coarse, 1, None)
            counts = torch.bincount(asg.to(torch.int64), minlength=nlist).cpu().numpy()
            bounds.copy_(torch.from_numpy(balanced_list_bounds(counts, world)))
            del sample, asg
        bcast(bounds)
        sh.set_list_bounds(bounds.cpu().numpy())
    torch.cuda.synchronize()
    t_train = time.time() - t0

    t0 = time.time()
    qgt = synth.queries(cfg["nq"])[:GT_QUERIES].contiguous()
    k = cfg["k"]
    gt_d = torch.full((GT_QUERIES, k), float("inf"), device=synth.dev)
    gt_i = torch.full((GT_QUERIES, k), -1, dtype=torch.int64, device=synth.dev)
    chunks = chunks_of(n)
    for c0 in range(0, len(chunks), world):                          # one collective round per `world` chunks
        ci = c0 + rank
        if ci < len(chunks):
            b, c = chunks[ci]
            x = synth.rows(b, c)
            ids = torch.arange(b, b + c, dtype=torch.int64, device=synth.dev)
            dd, ii = vk.flat_search_f32(qgt, x, k, 1 if cfg.get("metric") == "dotProduct" else 0)   # exact ground truth
            alld = torch.cat([gt_d, dd], 1)
            alli = torch.cat([gt_i, ii + b], 1)
            o = torch.argsort(alld, dim=1, stable=True)[:, :k]
            gt_d, gt_i = torch.gather(alld, 1, o), torch.gather(alli, 1, o)
        else:
            x = torch.empty((0, d), dtype=torch.float32, device=synth.dev)
            ids = torch.empty((0,), dtype=torch.int64, device=synth.dev)
        if sh is not None:
            sh.add(x, ids)
        else:
            idx.batch_insert(x, ids)
        del x, ids
    idx.list_sizes()                                                 # forces the list build (untimed)
    torch.cuda.synchronize()
    t_add = time.time() - t0
    return idx, sh, (gt_d, gt_i), dict(train_s=round(t_train, 2), add_s=round(t_add, 2))


def recall_at_k(found, truth, k):
    f, t = found.cpu().numpy(), truth.cpu().numpy()
    return float(np.mean([len(set(f[r, :k]) & set(t[r, :k])) / k for r in range(t.shape[0])]))


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_search_arm(cfg, idx, q_host, budget_s=12.0, gpu_ids=None):
    """The oracle's IVF-PQ search (reference arithmetic, OpenMP over queries) on a bounded sample."""
    from oracle import oracle
    coarse = idx.get_coarse()
    cb, norms = idx.get_codebooks()
    off, codes, lids, _ = idx.export_lists()
    # every host core this process may run on, whatever OMP_NUM_THREADS the launcher exported (torchrun sets it to 1)
    want = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    cores = oracle.set_threads(want)                                 # = omp_get_max_threads() after the call
    args = (coarse, cb, norms, off, codes, lids, cfg["m"], 256, cfg["nprobe"], cfg["k"], 1 if cfg.get("metric") == "dotProduct" else 0)
    probe = min(q_host.shape[0], 2 * cores)
    t0 = time.perf_counter()
    oracle.ivfpq_search(q_host[:probe], *args)
    per_q = (time.perf_counter() - t0) / probe
    s = int(max(probe, min(q_host.shape[0], budget_s / max(per_q, 1e-9))))
    t0 = time.perf_counter()
    od, oi, _ = oracle.ivfpq_search(q_host[:s], *args)
    dt = time.perf_counter() - t0
    out = {"value": s / dt, "unit": "queries/s", "cores": cores, "kind": "port",
           "sample": f"first {s} of the {q_host.shape[0]} queries, full index, oracle/ C restatement with OpenMP over queries "
                     f"({dt:.1f} s, {cores} OpenMP threads)"}
    if gpu_ids is not None:
        g = gpu_ids[:s]
        out["topk_overlap_with_gpu"] = float(np.mean([len(set(g[r]) & set(oi[r])) / cfg["k"] for r in range(s)]))
    return out, dt, s


# ------------------------------------------------------------------------------------------------ configs[0..1]
def run_side_workload(args, cfg, K, W):
    """BASELINE configs[0] (flat exact search) and configs[1] (PQ train + encode) on ONE GPU through the same contract:
    value = device-resident throughput (CUDA events), e2e = host buffers in and out, roofline, cpu_baseline (the oracle /
    the reference's own compiled encoder on a bounded sample).  Parity of both is covered by tests/test_gpu_fullsize.py."""
    import torch
    from oracle import oracle
    from vectorindex_b200 import _lib, datagen, kernels as vk
    L = _lib.lib()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    _lib.check(L.vix_set_device(0))
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    _lib.check(L.vix_set_stream(C.c_void_p(stream.cuda_stream)))
    clk = ClockSampler(0)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:  # noqa: BLE001
        pass
    cores = oracle.set_threads(len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1))
    n, d = cfg["n"], cfg["d"]
    detail = {}
    if cfg["kind"] == "flat":
        nq, k = cfg["nq"], cfg["k"]
        xb_h = datagen.bench_vectors(n, d, 123)
        q_pin = torch.empty((nq, d), dtype=torch.float32, pin_memory=True)
        q_pin.copy_(torch.from_numpy(datagen.bench_vectors(nq, d, 321)))
        xb, q = torch.from_numpy(xb_h).to(dev), q_pin.to(dev)
        o_pin = (torch.empty((nq, k), dtype=torch.float32, pin_memory=True).numpy(),
                 torch.empty((nq, k), dtype=torch.int64, pin_memory=True).numpy())
        od, oi = torch.empty((nq, k), dtype=torch.float32, device=dev), torch.empty((nq, k), dtype=torch.int64, device=dev)

        def step():
            _lib.check(L.vix_flat_search_f32(_lib.ptr(q), C.c_int64(nq), _lib.ptr(xb), C.c_int64(n), C.c_int(d), C.c_int(0),
                                             C.c_int(k), _lib.ptr(od), _lib.ptr(oi)))

        def api():      # host queries in, host results out (the base stays resident: it is the index)
            _lib.check(L.vix_flat_search_f32(_lib.ptr(q_pin.numpy()), C.c_int64(nq), _lib.ptr(xb), C.c_int64(n), C.c_int(d),
                                             C.c_int(0), C.c_int(k), _lib.ptr(o_pin[0]), _lib.ptr(o_pin[1])))
        units, unit, metric = nq, "queries/s", "queries/sec (flat exact L2, k=10)"
        h2d, d2h = nq * d * 4, nq * k * 12
        work = 2.0 * nq * n * d                                       # SURVEY 8d: 2 Q N d flop
        t0 = time.perf_counter()
        cd, ci, _ = oracle.flat_search(q_pin.numpy(), xb_h, k, 0)
        cpu_dt = time.perf_counter() - t0
        cpu = {"value": nq / cpu_dt, "unit": unit, "cores": cores, "kind": "port",
               "sample": f"all {nq} queries against the full base, oracle/ C restatement of L2Sqr + selectTopK ({cpu_dt:.1f} s)"}
        check = lambda: bool(np.array_equal(o_pin[1], ci) and np.array_equal(o_pin[0].view(np.uint32), cd.view(np.uint32)))   # noqa: E731
        outputs = lambda: {"distances": od.cpu().numpy(), "ids": oi.cpu().numpy()}   # noqa: E731
        detail["parity_with_cpu_baseline"] = "ids and distance bits equal"
        # two TF32 tensor-core passes dominate the step; TF32 runs at half the bf16 rate
        peak = float(peaks.get("bf16_tflops_sustained", 1385.9)) / 2.0
        roof = {"kernel": "tc_score_kernel (two passes: group minima, emission) + exact rescoring", "bound": "tensor",
                "unit": "TFLOP/s", "peak": peak, "traffic": None,
                "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained / 2 (kind::tf32)" if peaks else "fallback"}
    else:
        m, ks = cfg["m"], cfg["ks"]
        x_h = datagen.bench_vectors(n, d, 123, normalize=False)
        x = torch.from_numpy(x_h).to(dev)
        x_pin = torch.empty((n, d), dtype=torch.float32, pin_memory=True)
        x_pin.copy_(torch.from_numpy(x_h))
        t0 = time.perf_counter()
        tcfg = vk.pq_train_cfg(algorithm=0, max_iters=25, sample_n=65536, mode=1)   # GPU Lloyd, 25 iterations (DESIGN.md 7)
        cb, norms = vk.pq_train_f32(x, m, ks, cfg=tcfg)
        torch.cuda.synchronize()
        detail["train_s"] = round(time.perf_counter() - t0, 3)
        cbf, nf = cb.reshape(-1).contiguous(), norms.reshape(-1).contiguous()
        codes = torch.empty((n, m), dtype=torch.uint8, device=dev)
        c_pin = torch.empty((n, m), dtype=torch.uint8, pin_memory=True).numpy()

        def step():
            L.cpq_encode_u8_f32_with_csq(_lib.ptr(x), C.c_int64(n), C.c_int(d), C.c_int(m), C.c_int(ks), _lib.ptr(cbf), _lib.ptr(nf),
                                         _lib.ptr(codes), None)

        def api():      # the reference's own entry point with HOST pointers, as the Swift wrapper calls it
            L.cpq_encode_u8_f32_with_csq(_lib.ptr(x_pin.numpy()), C.c_int64(n), C.c_int(d), C.c_int(m), C.c_int(ks), _lib.ptr(cbf),
                                         _lib.ptr(nf), _lib.ptr(c_pin), None)
        units, unit, metric = n, "vectors/s", "vectors/sec (PQ encode, M=16 x 256, bit-exact codes)"
        h2d, d2h = n * d * 4, n * m
        work = 4.0 * n * d + n * m                                    # SURVEY 8d: bytes in + out
        ns = n                                                        # the CPU arm: the reference's C encoder on the whole input (~1.3 s)
        cbh, nh = cbf.cpu().numpy(), nf.cpu().numpy()
        t0 = time.perf_counter()
        try:
            ref = oracle.ref_encode("cpq_encode_u8_f32_with_csq", x_h[:ns], cbh, m, ks, centroid_sq=nh, omp=True)
            kind = "reference"
            what = "the reference's pq_encode.c compiled unmodified with OpenMP (oracle/_ref)"
        except Exception:  # noqa: BLE001  (oracle/_ref not built on this box)
            ref = oracle.pq_encode_u8(x_h[:ns], cbh, m, ks, centroid_sq=nh)
            kind, what = "port", "oracle/ C restatement of pq_encode.c"
        cpu_dt = time.perf_counter() - t0
        cpu = {"value": ns / cpu_dt, "unit": unit, "cores": cores, "kind": kind,
               "sample": f"all {ns} vectors, {what} ({cpu_dt:.1f} s)"}
        check = lambda: bool(np.array_equal(c_pin[:ns], ref))        # noqa: E731
        outputs = lambda: {"codes": codes.cpu().numpy()}             # noqa: E731
        detail["parity_with_cpu_baseline"] = "codes bit-identical on all vectors"
        peak = float(peaks.get("hbm_gbs", 6650.0))
        roof = {"kernel": "pq_tc_encode_kernel (tcgen05 shortlist + exact finalists)", "bound": "hbm", "unit": "GB/s", "peak": peak,
                "traffic": None, "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s",
                "note": "compute-bound by the per-codeword epilogue, far from the HBM floor: see DESIGN.md 4.4"}
    _lib.check(L.vix_set_async(1))
    for _ in range(W):
        step()
    torch.cuda.synchronize()
    L.vix_kernel_launches(1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        step()
    e1.record()
    clk.poll_until(e1.query)
    torch.cuda.synchronize()
    launches = int(L.vix_kernel_launches(0))
    ms = e0.elapsed_time(e1) / K
    last = outputs() if args.dump_outputs else None
    _lib.check(L.vix_set_async(0))
    for _ in range(W):
        api()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(K):
        api()
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / K
    _lib.check(L.vix_synchronize())
    assert check(), "GPU result differs from the CPU baseline on the same inputs"
    achieved = work / (ms * 1e-3) / (1e12 if roof["bound"] == "tensor" else 1e9)
    roof.update({"achieved": achieved, "frac": achieved / roof["peak"], "algorithmic_per_launch": work, "ms_per_launch": ms,
                 "timing": "algorithmic work / the whole step (the named kernels dominate it)"})
    shape = {k2: v for k2, v in cfg.items() if k2 not in ("kind", "label")}
    line = {"metric": metric, "value": units / (ms * 1e-3), "unit": unit, "n_gpus": 1, "steps": K, "warmup": W, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32 (tf32 shortlist, exact fp32 finalists)", "data": "synthetic",
            "config": dict({"workload": cfg["label"]}, **shape,
                           l2_policy="flat: the 51 MB base is L2-resident by design (it is read once per batch); "
                                     "pq_encode: 512 MB input > L2, no flush between steps"),
            "detail": detail, "clocks": clk.summary(),
            "e2e": {"value": units / (e2e_ms * 1e-3), "unit": unit, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_ms},
            "gpu_launches": launches, "roofline": roof, "cpu_baseline": cpu}
    if args.impl == "reference":
        line = {"impl": "reference", "metric": metric, "value": cpu["value"], "unit": unit, "n_gpus": args.gpus, "steps": K, "warmup": W,
                "ms_per_step": None, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic", "config": line["config"], "cpu_baseline": cpu,
                "e2e": {"value": cpu["value"], "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if last is not None:
        dump_outputs(args.dump_outputs, last)
    emit(line)
    return 0


# ------------------------------------------------------------------------------------------------ main
def emit(line: dict):
    """The ONE JSON line of the contract, on the process's real stdout (see main: fd 1 is pointed at stderr while
    the bench runs, so that banners of libraries -- NCCL's version line -- cannot land on stdout)."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default=os.environ.get("VIX_BENCH_WORKLOAD", "c5"), choices=sorted(PRESETS))
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--partition", default=os.environ.get("VIX_BENCH_PARTITION", "lists"), choices=["lists", "replicate"],
                    help="N > 1: inverted lists sharded over the ranks (default, what north_star names) or every rank a full "
                         "replica with the batch split by query (indexes that fit one GPU)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--profile", action="store_true",
                    help="bracket the timed steps with cudaProfilerStart/Stop (for ncu --profile-from-start off) "
                         "and skip the e2e / CPU legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned as DIR/<name>.npy (float32 / float64, at most 64 MB)")
    args = ap.parse_args()
    cfg = dict(PRESETS[args.workload])
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path; --impl reference has none")
    K, W = args.steps, max(3, args.warmup)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference" and rank != 0:
        return 0                                                     # rank 0 alone runs the CPU arm

    import torch
    from vectorindex_b200 import _lib
    from vectorindex_b200.index import merge_shard_results

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback for the product path")
    if cfg.get("kind") in ("flat", "pq_encode"):
        if rank != 0:
            return 0                                                 # single-GPU workloads: the other ranks have nothing to do
        return run_side_workload(args, cfg, K, W)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    L = _lib.lib()
    _lib.check(L.vix_set_device(local_rank))
    dist = None
    if world > 1 and args.impl == "ours":
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")      # keep NCCL's banner / logs off stdout (ONE JSON line there)
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    _lib.check(L.vix_set_stream(C.c_void_p(stream.cuda_stream)))

    clk = ClockSampler(local_rank)                                   # started early: see ClockSampler.summary
    synth = Synth(cfg, dev)
    eff_world = world if args.impl == "ours" else 1
    bcast = (lambda t: dist.broadcast(t, 0)) if dist else None
    idx, sh, (gt_d, gt_i), build_t = build_index(cfg, synth, rank if args.impl == "ours" else 0, eff_world, bcast,
                                                 args.partition)
    log(f"[bench] rank {rank}: built {idx.count} vectors ({build_t})")
    nq, k, d = cfg["nq"], cfg["k"], cfg["d"]
    q_dev = synth.queries(nq)
    q_pin = torch.empty((nq, d), dtype=torch.float32, pin_memory=True)
    q_pin.copy_(q_dev)
    torch.cuda.synchronize()
    q_host = q_pin.numpy()

    base_cfg = {"workload": cfg["label"], "n": cfg["n"], "d": d, "nlist": cfg["nlist"], "nprobe": cfg["nprobe"],
                "M": cfg["m"], "ks": 256, "batch_queries": nq, "k": k, "metric": cfg.get("metric", "euclidean"),
                "l2_policy": "inputs larger than L2 (code arrays >> 126 MB); no flush between steps"}
    # run-dependent facts live OUTSIDE `config`, so that both arms print the same `config` object
    detail = {"partition": (f"inverted lists in contiguous blocks over {eff_world} rank(s); queries replicated; probe selection "
                            "split by query block + exchange of list ids; per-rank top-k exchanged + mergeTopK")
              if args.partition == "lists" or eff_world == 1 else
              f"full replica on each of {eff_world} rank(s); batch split by query block; all-gather of the "
              "finished [nq/world x k] blocks",
              "build": build_t}

    # ---------------------------------------------------------------- reference arm (CPU only)
    if args.impl == "reference":
        steps = []
        info = None
        for s in range(W + K):
            info, dt, ns = cpu_search_arm(cfg, idx, q_host, budget_s=max(2.0, 60.0 / (W + K)))
            if s >= W:
                steps.append((ns, dt))
        tot_q, tot_t = sum(a for a, _ in steps), sum(b for _, b in steps)
        val = tot_q / tot_t
        info["value"] = val
        line = {"impl": "reference", "metric": "queries/sec at matched recall@10 (IVF-PQ)", "value": val,
                "unit": "queries/s", "n_gpus": args.gpus, "steps": K, "warmup": W, "ms_per_step": 1e3 * tot_t / K,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": base_cfg, "detail": detail, "cpu_baseline": info,
                "e2e": {"value": val, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        emit(line)
        clk.stop()
        return 0

    # ---------------------------------------------------------------- our arm
    out_d = torch.empty((nq, k), dtype=torch.float32, device=dev)
    out_i = torch.empty((nq, k), dtype=torch.int64, device=dev)
    st = _lib.SearchStats()
    _lib.check(L.vix_set_async(1))
    qp, dp, ip = _lib.ptr(q_dev), _lib.ptr(out_d), _lib.ptr(out_i)

    def step_device():
        # asynchronous: nothing here waits for the GPU (stage events are traced inside the library)
        if world == 1:
            _lib.check(L.vix_index_search(idx._h, qp, C.c_int64(nq), C.c_int(k), C.c_int(0), dp, ip))
            return out_d, out_i
        return sh.batch_search(q_dev, k)

    def barrier():
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(W):
        res_d, res_i = step_device()
    barrier()
    _lib.check(L.vix_index_trace(idx._h, K))
    L.vix_kernel_launches(1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if args.profile:
        torch.cuda.profiler.start()
    e0.record()
    for _ in range(K):
        res_d, res_i = step_device()
    e1.record()
    clk.poll_until(e1.query)                                         # GPU still busy with the queued steps
    barrier()
    if args.profile:
        torch.cuda.profiler.stop()
    last = {"distances": res_d.cpu().numpy(), "ids": res_i.cpu().numpy()} if args.dump_outputs and rank == 0 else None
    launches = int(L.vix_kernel_launches(0))
    ms_total = e0.elapsed_time(e1)
    scan_ms = coarse_ms = kern_ms = 0.0
    scan_bytes = 0
    scan_path = 0
    for i in range(K):
        _lib.check(L.vix_index_trace_get(idx._h, i, C.byref(st)))
        scan_ms += st.ms_scan
        coarse_ms += st.ms_coarse
        kern_ms += st.ms_scan_kernel                                 # the dominant kernel alone (events around its launch)
        scan_bytes += st.code_bytes_scanned
        scan_path = st.scan_path
    _lib.check(L.vix_index_trace(idx._h, 0))

    # ---- end to end through the public API with pinned host buffers
    _lib.check(L.vix_set_async(0))
    if world > 1 and args.partition == "lists":
        # pinned host result buffers, as a host that cares about the copy back would pass them
        o_pin = (torch.empty((nq, k), dtype=torch.float32, pin_memory=True).numpy(),
                 torch.empty((nq, k), dtype=torch.int64, pin_memory=True).numpy())
        api = lambda: sh.batch_search(q_host, k, out=o_pin)           # noqa: E731
    elif world > 1:
        api = lambda: sh.batch_search(q_host, k)                      # noqa: E731
    else:
        o_pin = (torch.empty((nq, k), dtype=torch.float32, pin_memory=True).numpy(),
                 torch.empty((nq, k), dtype=torch.int64, pin_memory=True).numpy())
        api = lambda: idx.batch_search(q_host, k, out=o_pin)          # noqa: E731
    for _ in range(1 if args.profile else W):
        api()
    barrier()
    t0 = time.perf_counter()
    for _ in range(1 if args.profile else K):
        h_d, h_i = api()
    barrier()
    e2e_s = (time.perf_counter() - t0) * (K if args.profile else 1)

    times = torch.tensor([ms_total, e2e_s * 1e3, scan_ms, coarse_ms, float(scan_bytes)], dtype=torch.float64, device=dev)
    if dist:
        tmax = times.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = times.clone()
        dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        ms_total, e2e_ms = float(tmax[0]), float(tmax[1])
        scan_bytes_all = float(tsum[4])
    else:
        e2e_ms = e2e_s * 1e3
        scan_bytes_all = float(scan_bytes)

    # diagnostic (untimed): where a sharded step spends its time on this rank, and the per-rank scan times
    phase_ms = None
    if dist:
        comm = getattr(sh, "comm", None)
        if comm is not None and args.partition == "lists":         # the library's own phase events (vix_comm_trace)
            _lib.check(L.vix_comm_trace(comm._c, 1))
            acc = np.zeros(3)
            ph = (C.c_float * 3)()
            for _ in range(3):
                sh.batch_search(q_dev, k)
                _lib.check(L.vix_comm_trace_get(comm._c, ph))
                acc += np.array(list(ph))
            _lib.check(L.vix_comm_trace(comm._c, 0))
            phase_ms = dict(zip(("probe_select+exchange", "scan", "exchange+merge"), (round(float(v) / 3, 3) for v in acc)))
            phase_ms["peer_memory"] = comm.uses_peer_memory
        else:
            sh.phase_times = {}
            for _ in range(3):
                sh.batch_search(q_dev, k)
            phase_ms = {kk: round(v / 3, 3) for kk, v in sh.phase_times.items()}
            sh.phase_times = None
        per_rank = torch.zeros(world, dtype=torch.float64, device=dev)
        per_rank[rank] = scan_ms / K
        dist.all_reduce(per_rank)
        phase_ms["scan_ms_per_rank"] = [round(float(v), 3) for v in per_rank]

    # recall of the (merged) result against the exact ground truth
    if dist:
        _lib.check(L.vix_set_async(0))
        gt_d, gt_i = merge_shard_results(sh._all_gather(gt_d.contiguous()), sh._all_gather(gt_i.contiguous()), k)
    torch.cuda.synchronize()
    recall = recall_at_k(res_i[:GT_QUERIES], gt_i, k)
    assert np.array_equal(np.asarray(h_i), res_i.cpu().numpy()), "host-path ids differ from the device-path ids"

    if rank != 0:
        clk.stop()
        if dist:
            dist.barrier()
            dist.destroy_process_group()
        return 0

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:  # noqa: BLE001
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    # dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the scan kernel from the committed `ncu --set full`
    # captures (profiles/): known only for the configurations that were captured
    # (a CONSTANT from that capture, not a per-run measurement: the traffic of a launch depends only on the index and the batch)
    list_major = scan_path == 1
    if list_major:
        captures = {("c5", 1, "lists"): (3.807961e9 + 12.889856e6, "profiles/r02_final_scan_c5_n1_ncu_summary.txt (ncu --set full, one "
                                                                     "launch of tc_scan_kernel; a constant from that capture, not measured in this run)")}
    else:
        captures = {("c5", 1, "lists"): (87.148642e9 + 7.127e6, "profiles/r02_scan_c5_n1_ncu_summary.txt (ncu --set full, one launch; a "
                                                                  "constant from that capture, not measured in this run)"),
                    ("c5s", 1, "lists"): (5.486273e9 + 5.3e6, "profiles/r01_scan_c5s_ncu_summary.txt (ncu --set full, one launch)"),
                    # one rank's share of an 8-way list-sharded C5, captured on ONE GPU holding the first equal-count eighth of the
                    # lists (the bench's work-balanced boundaries move the block edges by a few lists: approximate for this run)
                    ("c5", 8, "lists"): (6.422206e9 + 6.883328e6, "profiles/r01_scan_shard8_ncu_summary.txt (ncu --set full, one launch "
                                                                   "of an equal-count one-eighth share, scripts/shard_emul.py 8 0; approximate)")}
    traffic, traffic_src = captures.get((args.workload, world, args.partition if world > 1 else "lists"), (None, None))
    per_launch_bytes = scan_bytes / K                                  # rank 0's scan kernel, one launch per step
    per_launch_ms = kern_ms / K if kern_ms > 0 else scan_ms / K
    achieved = per_launch_bytes / (per_launch_ms * 1e-3) / 1e9 if per_launch_ms > 0 else 0.0
    kernel_name = "tc_scan_kernel (list-major: decode once per list, tcgen05 shortlist)" if list_major else "ivfpq_scan_kernel"
    note = None
    if list_major:
        # SURVEY 8d: "any list-major schedule reuses code tiles across queries, so measured DRAM bytes will be below the
        # algorithmic figure -- report both".  The algorithmic bytes stay sum_q sum_l len(l) * M (what a query-major scan must
        # read); this kernel reads every probed list ONCE per batch, so `achieved` may exceed the HBM peak: the bound that
        # applies to it is the shared-memory pipe of the decode, quantified in DESIGN 4.1b.
        note = ("list-major: the algorithmic bytes (SURVEY 8d: sum over (query, probed list) of len x M) are what a query-major "
                "scan reads; this kernel decodes every probed list once per batch and scores all its queries on the tensor "
                "cores, so achieved > peak is reuse, not a measurement error; `traffic` is the DRAM bytes it really moves")
    line = {
        "metric": "queries/sec at matched recall@10 (IVF-PQ)", "value": nq * K / (ms_total * 1e-3), "unit": "queries/s",
        "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_total / K, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": base_cfg,
        "detail": dict(detail, recall_at_10=recall, recall_queries=GT_QUERIES,
                       stage_ms_per_step={"probe_select": coarse_ms / K, "lut_adc_scan_topk": scan_ms / K},
                       sharded_phase_ms=phase_ms),
        "clocks": clk.summary(),
        "e2e": {"value": nq * K / (e2e_ms * 1e-3), "unit": "queries/s", "h2d_bytes_per_step": nq * d * 4,
                "d2h_bytes_per_step": nq * k * 12, "ms_per_step": e2e_ms / K},
        "gpu_launches": launches,
        "roofline": {"kernel": kernel_name, "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": traffic,
                     "traffic_source": traffic_src, "note": note, "stage_ms_per_launch": scan_ms / K,
                     "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s",
                     "algorithmic_bytes_per_launch": per_launch_bytes, "ms_per_launch": per_launch_ms,
                     "job_code_bytes_per_step": scan_bytes_all / K},
    }
    if traffic and per_launch_ms > 0:
        # the DRAM side of the same launch: the captured bytes over this run's kernel time
        dram = traffic / (per_launch_ms * 1e-3) / 1e9
        line["roofline"].update(dram_achieved=dram, dram_frac=dram / peak)
    if list_major:
        line["roofline"]["limiter"] = ("ALU pipe of the decode (ncu sm__inst_executed_pipe_alu 73 % at C5 on one GPU; the exchange network's "
                                       "SELs are 22 % of the executed instructions), DESIGN 4.1b")
    if world == 1 and not args.no_cpu_baseline and not args.profile:
        info, _, _ = cpu_search_arm(cfg, idx, q_host, gpu_ids=np.asarray(h_i))
        line["cpu_baseline"] = info
    if last is not None:
        dump_outputs(args.dump_outputs, last)
    emit(line)
    if dist:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
