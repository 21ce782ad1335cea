"""Sharded range search and id filters (vix_sharded_range_search, vix_sharded_search_filtered behind
ShardedIVFPQIndex.range_search / batch_search(filter=)), bit for bit against one GPU holding the rows in the slots the shards
hold them in.

On one GPU: the merge the exchange runs (shard_range_merge_kernel through vix_debug_shard_range_merge) over three shards
emulated on one GPU equals the one-GPU range search bit for bit, and over synthetic adversarial runs equals a numpy stable
merge.  On several GPUs: tests/mp_sharded_range.py under torch.distributed.run, at two ranks and at every GPU of the box (up
to 8), over peer memory and over NCCL (VIX_NO_P2P=1); a box with one GPU runs it at world 1.
"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu

CASES = ["radii", "blocks", "partitions", "routes", "filter", "long_rows", "capacity", "mutate", "knn_prefix", "refusals"]
METRICS = {0: "euclidean", 1: "dotProduct"}


def _ngpus():
    import torch
    return torch.cuda.device_count()


def _launch(world, no_p2p, cases, port):
    env = dict(os.environ)
    env.pop("VIX_NO_P2P", None)
    env.pop("VIX_TC_SCAN", None)
    if no_p2p:
        env["VIX_NO_P2P"] = "1"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr",
           "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "mp_sharded_range.py")] + cases
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=1200, env=env)
    assert out.returncode == 0, out.stdout[-6000:] + out.stderr[-4000:]
    for case in cases:
        assert f"ok {case}:" in out.stdout, f"case {case} did not report: " + out.stdout[-3000:]
    peer = -1 if world == 1 else 0 if no_p2p else 1
    assert f"range: world {world}, peer memory {peer}, {len(cases)} of {len(cases)} cases ok" in out.stdout, out.stdout[-3000:]


@pytest.mark.parametrize("no_p2p", [False, True], ids=["peer", "nccl"])
@pytest.mark.parametrize("size", ["two", "all"])
def test_sharded_range(size, no_p2p):
    n = _ngpus()
    if n < 2:
        pytest.skip("needs two GPUs")
    if size == "all" and n <= 2:
        pytest.skip("the box has two GPUs: the two-rank launch covers it")
    _launch(2 if size == "two" else min(n, 8), no_p2p, CASES, 29571 + 2 * (size == "all") + no_p2p)


def test_sharded_range_single_rank():
    """One rank: the sharded entry points are the one-GPU calls; every case that needs no second rank."""
    if _ngpus() >= 2:
        pytest.skip("the multi-rank launches cover it")
    _launch(1, False, [c for c in CASES if c != "partitions"], 29575)


# ------------------------------------------------------------------------------------------------ the merge on one GPU
def _merge(lims_all, dist_all, ids_all, metric):
    from vectorindex_b200 import _lib
    L = _lib.lib()
    world, nq = lims_all.shape[0], lims_all.shape[1] - 1
    res = C.c_void_p(0)
    try:
        _lib.check(L.vix_debug_shard_range_merge(_lib.ptr(np.ascontiguousarray(lims_all, np.int64)),
                                                 _lib.ptr(np.ascontiguousarray(dist_all, np.float32)),
                                                 _lib.ptr(np.ascontiguousarray(ids_all, np.int64)), world, C.c_int64(nq),
                                                 metric, C.byref(res)))
        total = int(L.vix_range_result_total(res))
        lims = np.empty(nq + 1, np.int64)
        dist = np.empty(total, np.float32)
        ids = np.empty(total, np.int64)
        _lib.check(L.vix_range_result_get(res, _lib.ptr(lims), _lib.ptr(dist) if total else None,
                                          _lib.ptr(ids) if total else None))
        return lims, dist, ids
    finally:
        L.vix_range_result_destroy(res)


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


@pytest.mark.parametrize("metric", [0, 1], ids=["l2", "ip"])
def test_shard_range_merge_on_one_gpu(metric):
    """Three shards emulated on one GPU (all centroids, one list block's rows in the one-GPU slots, as
    test_shard_merge_on_one_gpu builds them) each run the plain range search -- the same probes, the centroids being the
    same -- and their CSRs through vix_debug_shard_range_merge equal the one-GPU range search bit for bit: several radii,
    one below every distance (total 0), +inf, a negative IP radius, a zero IP query (-0)."""
    from vectorindex_b200.index import IVFPQIndex
    rng = np.random.default_rng(17 + metric)
    world, d, m, kc, n = 3, 32, 16, 24, 3000
    coarse = rng.standard_normal((kc, d)).astype(np.float32)
    cb = (0.3 * rng.standard_normal((m, 256, d // m))).astype(np.float32)
    xb = (coarse[rng.integers(0, kc, n)] + 0.3 * rng.standard_normal((n, d))).astype(np.float32)
    ids = rng.permutation(n).astype(np.int64) * 3 + 7

    def index():
        ix = IVFPQIndex(d, METRICS[metric], nlist=kc, nprobe=6, m=m)
        ix.set_coarse(coarse)
        ix.set_codebooks(cb)
        return ix
    full = index()
    full.batch_insert(xb, ids)
    off, codes, lids, _ = full.export_lists()
    asg = np.repeat(np.arange(kc, dtype=np.int32), np.diff(off))
    bounds = [kc * r // world for r in range(world + 1)]
    shards = []
    for r in range(world):
        sel = (asg >= bounds[r]) & (asg < bounds[r + 1])
        sh = index()
        sh.add_encoded(asg[sel], codes[sel], lids[sel])
        shards.append(sh)
    q = np.concatenate([(coarse[rng.integers(0, kc, 20)] + 0.3 * rng.standard_normal((20, d))), np.zeros((3, d))])
    q = q.astype(np.float32)
    _, alld, _ = full.range_search(q, float("inf"), nprobe=6)
    radii = [float(np.quantile(alld, f)) for f in (0.01, 0.1, 0.5)] + [float(alld.min()) - 1.0, float("inf")]
    if metric == 1:
        radii.append(-0.5)
    for nprobe in (6, 24):
        for radius in radii:
            want = full.range_search(q, radius, nprobe=nprobe)
            parts = [s.range_search(q, radius, nprobe=nprobe) for s in shards]
            got = _merge(np.stack([p[0] for p in parts]), np.concatenate([p[1] for p in parts]),
                         np.concatenate([p[2] for p in parts]), metric)
            assert np.array_equal(got[0], want[0]), f"radius {radius}: lims differ"
            assert np.array_equal(got[2], want[2]), f"radius {radius}: ids differ"
            assert np.array_equal(_bits(got[1]), _bits(want[1])), f"radius {radius}: distance bits differ"
            if radius < float(alld.min()):
                assert got[0][-1] == 0
            if metric == 1 and radius >= 0:
                z = got[1][got[0][-4]:]                                      # the three zero queries
                assert z.size and (_bits(z) == 0x80000000).all(), "zero IP distances must be -0"


def _numpy_merge(lims_all, dist_all, ids_all, metric):
    """stable merge of the runs rank by rank, row by row: (distance, id) order, equal keys in rank order"""
    world, nq = lims_all.shape[0], lims_all.shape[1] - 1
    base = np.concatenate([[0], np.cumsum(lims_all[:, -1])])
    lims, dist, ids = [0], [], []
    for qi in range(nq):
        dd = np.concatenate([dist_all[base[r] + lims_all[r, qi]:base[r] + lims_all[r, qi + 1]] for r in range(world)])
        ii = np.concatenate([ids_all[base[r] + lims_all[r, qi]:base[r] + lims_all[r, qi + 1]] for r in range(world)])
        dd = dd + np.float32(0.0)                                           # the keys hold zeros as +0
        o = np.lexsort((ii, dd))
        dist.append(dd[o])
        ids.append(ii[o])
        lims.append(lims[-1] + o.size)
    d = np.concatenate(dist).astype(np.float32) if dist else np.zeros(0, np.float32)
    if metric == 1:
        d[d == 0] = np.float32(-0.0)
    return np.asarray(lims, np.int64), d, np.concatenate(ids) if ids else np.zeros(0, np.int64)


def _runs(rng, world, nq, sizes, values, id_range):
    """world ranks' sorted rows: sizes[r][q] entries with distances from `values` and ids from [0, id_range)"""
    lims, dist, ids = [], [], []
    for r in range(world):
        lr = np.concatenate([[0], np.cumsum(sizes[r])]).astype(np.int64)
        lims.append(lr)
        for q in range(nq):
            n = int(sizes[r][q])
            dd = rng.choice(values, n).astype(np.float32)
            ii = rng.integers(0, id_range, n).astype(np.int64)
            o = np.lexsort((ii, dd))
            dist.append(dd[o])
            ids.append(ii[o])
    cat = lambda xs, t: np.concatenate(xs).astype(t) if xs else np.zeros(0, t)
    return np.stack(lims), cat(dist, np.float32), cat(ids, np.int64)


@pytest.mark.parametrize("world", [1, 2, 8])
def test_shard_range_merge_adversarial(world):
    """Synthetic runs against a numpy stable merge: every key equal across ranks, empty runs, one rank holding everything,
    rows longer than 2048 keys, and (world 2) one row of more than 10^6 keys."""
    rng = np.random.default_rng(40 + world)
    nq = 7
    cases = {
        "all equal": ([np.full(nq, 50) for _ in range(world)], np.array([1.5]), 1),
        "ties": ([rng.integers(0, 300, nq) for _ in range(world)], np.array([0.0, 0.25, 0.5, -1.0]), 20),
        "empty runs": ([rng.integers(0, 3, nq) * rng.integers(0, 2, nq) for _ in range(world)],
                       np.linspace(-2, 2, 9), 1000),
        "one rank": ([np.full(nq, 900) if r == world // 2 else np.zeros(nq, np.int64) for r in range(world)],
                     np.linspace(0, 4, 17), 2 ** 32 - 2),
        "long rows": ([rng.integers(2049, 5000, nq) for _ in range(world)], np.linspace(0, 1, 64), 10 ** 6),
        "nothing": ([np.zeros(nq, np.int64) for _ in range(world)], np.array([1.0]), 1),
    }
    if world == 2:
        cases["row of 10^6"] = ([np.array([600_000, 0, 3]), np.array([500_000, 7, 0])], np.linspace(0, 1, 4096), 2 ** 31)
    for name, (sizes, values, id_range) in cases.items():
        nrow = len(sizes[0])
        lims_all, dist_all, ids_all = _runs(rng, world, nrow, sizes, values, id_range)
        for metric in (0, 1):
            got = _merge(lims_all, dist_all, ids_all, metric)
            want = _numpy_merge(lims_all, dist_all, ids_all, metric)
            assert np.array_equal(got[0], want[0]), f"{name}: lims"
            assert np.array_equal(got[2], want[2]), f"{name} (metric {metric}): ids"
            assert np.array_equal(_bits(got[1]), _bits(want[1])), f"{name} (metric {metric}): distance bits"
