"""Sharded k-NN search beyond 512 neighbours (vix_sharded_search / vix_sharded_search_filtered with VIX_MAX_K < k <=
VIX_MAX_K_LARGE behind ShardedIVFPQIndex.batch_search), bit for bit against one GPU holding the rows in the slots the shards
hold them in.

On one GPU: the merge-and-cut kernel of the exchange (shard_knn_merge_kernel through vix_debug_shard_knn_merge) against a
numpy stable merge plus cut over adversarial runs; over three shards emulated on one GPU, the shards' own large-k rows
merged and cut equal the one-GPU answer; and the bound argument of the route (each shard's candidates within the smallest
of the shards' k-th distances, cut at k, merged) equals it too.  On several GPUs: tests/mp_sharded_large_k.py under
torch.distributed.run, at two ranks and at every GPU of the box (up to 8), over peer memory and over NCCL (VIX_NO_P2P=1); a
box with one GPU runs it at world 1.
"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu

CASES = ["ks", "blocks", "partitions", "ties", "filter", "nonfinite", "capacity", "mutate", "refusals"]
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
           "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "mp_sharded_large_k.py")] + cases
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=1800, env=env)
    assert out.returncode == 0, out.stdout[-6000:] + out.stderr[-4000:]
    for case in cases:
        assert f"ok {case}:" in out.stdout, f"case {case} did not report: " + out.stdout[-3000:]
    peer = -1 if world == 1 else 0 if no_p2p else 1
    assert f"large k: world {world}, peer memory {peer}, {len(cases)} of {len(cases)} cases ok" in out.stdout, \
        out.stdout[-3000:]


@pytest.mark.parametrize("no_p2p", [False, True], ids=["peer", "nccl"])
@pytest.mark.parametrize("size", ["two", "all"])
def test_sharded_large_k(size, no_p2p):
    n = _ngpus()
    if n < 2:
        pytest.skip("needs two GPUs")
    if size == "all" and n <= 2:
        pytest.skip("the box has two GPUs: the two-rank launch covers it")
    _launch(2 if size == "two" else min(n, 8), no_p2p, CASES, 29591 + 2 * (size == "all") + no_p2p)


def test_sharded_large_k_single_rank():
    """One rank: the sharded entry points are the one-GPU calls; every case that needs no second rank."""
    if _ngpus() >= 2:
        pytest.skip("the multi-rank launches cover it")
    _launch(1, False, [c for c in CASES if c != "partitions"], 29595)


# ------------------------------------------------------------------------------------------------ the merge on one GPU
def _merge_cut(lims_all, dist_all, ids_all, k, metric):
    from vectorindex_b200 import _lib
    L = _lib.lib()
    world, nq = lims_all.shape[0], lims_all.shape[1] - 1
    dist = np.empty((nq, k), np.float32)
    ids = np.empty((nq, k), np.int64)
    _lib.check(L.vix_debug_shard_knn_merge(_lib.ptr(np.ascontiguousarray(lims_all, np.int64)),
                                           _lib.ptr(np.ascontiguousarray(dist_all, np.float32)),
                                           _lib.ptr(np.ascontiguousarray(ids_all, np.int64)), world, C.c_int64(nq), k,
                                           metric,
                                           _lib.ptr(dist), _lib.ptr(ids)))
    return dist, ids


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _numpy_merge_cut(lims_all, dist_all, ids_all, k, metric):
    """stable merge of the runs rank by rank ((distance, id) order, equal keys in rank order), cut at k, padded"""
    world, nq = lims_all.shape[0], lims_all.shape[1] - 1
    base = np.concatenate([[0], np.cumsum(lims_all[:, -1])])
    dist = np.full((nq, k), np.nan, np.float32)
    ids = np.full((nq, k), -1, np.int64)
    for qi in range(nq):
        dd = np.concatenate([dist_all[base[r] + lims_all[r, qi]:base[r] + lims_all[r, qi + 1]] for r in range(world)])
        ii = np.concatenate([ids_all[base[r] + lims_all[r, qi]:base[r] + lims_all[r, qi + 1]] for r in range(world)])
        dd = dd.astype(np.float32) + np.float32(0.0)                         # the keys hold zeros as +0
        o = np.lexsort((ii, dd))[:k]
        dist[qi, :o.size] = dd[o]
        ids[qi, :o.size] = ii[o]
    if metric == 1:
        dist[dist == 0] = np.float32(-0.0)
    return dist, ids


def _runs(rng, world, nq, sizes, values, id_range):
    """world ranks' sorted rows: sizes[r][q] entries with distances from `values` and ids from [0, id_range)"""
    lims, dist, ids = [], [], []
    for r in range(world):
        lims.append(np.concatenate([[0], np.cumsum(sizes[r])]).astype(np.int64))
        for q in range(nq):
            n = int(sizes[r][q])
            dd = rng.choice(values, n).astype(np.float32)
            ii = rng.integers(0, id_range, n).astype(np.int64)
            o = np.lexsort((ii, dd))
            dist.append(dd[o])
            ids.append(ii[o])
    cat = lambda xs, t: np.concatenate(xs).astype(t) if xs else np.zeros(0, t)
    return np.stack(lims), cat(dist, np.float32), cat(ids, np.int64)


@pytest.mark.parametrize("k", [513, 1000, 4097, 16384])
@pytest.mark.parametrize("world", [1, 2, 8])
def test_shard_knn_merge_adversarial(world, k):
    """Synthetic runs against a numpy stable merge plus cut: every key equal across ranks, ties at the k-th place split
    across ranks, empty runs, one rank holding everything, rows shorter than k (padding), rows of exactly k on every rank;
    L2 and IP (zero distances -0 for IP)."""
    rng = np.random.default_rng(k + world)
    nq = 5
    split = -(-k // world)                                                 # ceil(k / world)
    cases = {
        "all equal": ([np.full(nq, min(k, 600)) for _ in range(world)], np.array([1.5]), 1),
        "ties at k": ([np.full(nq, split + 3) for _ in range(world)], np.array([0.0, 0.5]), 3),
        "empty runs": ([rng.integers(0, 3, nq) * rng.integers(0, 2, nq) for _ in range(world)], np.linspace(-2, 2, 9), 1000),
        "one rank": ([np.full(nq, k + 50) if r == world // 2 else np.zeros(nq, np.int64) for r in range(world)],
                     np.linspace(0, 4, 17), 2 ** 32 - 2),
        "short rows": ([rng.integers(0, max(k // (2 * world), 1), nq) for _ in range(world)], np.linspace(0, 1, 64),
                       10 ** 6),
        "exactly k": ([np.full(nq, k) for _ in range(world)], np.linspace(-1, 1, 257), 10 ** 9),
        "nothing": ([np.zeros(nq, np.int64) for _ in range(world)], np.array([1.0]), 1),
    }
    for name, (sizes, values, id_range) in cases.items():
        lims_all, dist_all, ids_all = _runs(rng, world, nq, sizes, values, id_range)
        for metric in (0, 1):
            gd, gi = _merge_cut(lims_all, dist_all, ids_all, k, metric)
            wd, wi = _numpy_merge_cut(lims_all, dist_all, ids_all, k, metric)
            assert np.array_equal(gi, wi), f"{name} (metric {metric}): ids"
            assert np.array_equal(_bits(gd), _bits(wd)), f"{name} (metric {metric}): distance bits"
            if name == "ties at k" and world > 1:
                # the k-th place lies inside a run of equal keys that several ranks contribute to
                assert (wd[:, k - 1] == wd[:, k - 2]).all()


# ------------------------------------------------------------------------------------------------ emulated shards
def _emulated(metric, seed, n=6000):
    """three shards on one GPU (all centroids, one list block's rows each, in the one-GPU slots) and the full index"""
    from vectorindex_b200.index import IVFPQIndex
    rng = np.random.default_rng(seed)
    world, d, m, kc = 3, 32, 16, 24
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
    return rng, coarse, full, shards, bounds


def _csr(rows):
    """[(dist row, id row)] per rank -> lims_all, dist_all, ids_all (padding dropped)"""
    lims, dist, ids = [], [], []
    for d, i in rows:
        keep = i >= 0
        lims.append(np.concatenate([[0], np.cumsum(keep.sum(1))]).astype(np.int64))
        dist.append(d[keep])
        ids.append(i[keep])
    return np.stack(lims), np.concatenate(dist).astype(np.float32), np.concatenate(ids).astype(np.int64)


@pytest.mark.parametrize("metric", [0, 1], ids=["l2", "ip"])
def test_shard_knn_merge_on_one_gpu(metric):
    """Each emulated shard's own large-k rows (batch_search(q, k), padding dropped) through the hook equal the full index's
    batch_search(q, k) bit for bit: k 513, 1000, 4097 and above every probed vector, nprobe 1 and nprobe = kc."""
    rng, coarse, full, shards, _ = _emulated(metric, 61 + metric)
    kc = coarse.shape[0]
    q = np.concatenate([coarse[rng.integers(0, kc, 20)] + 0.3 * rng.standard_normal((20, coarse.shape[1])),
                        np.zeros((2, coarse.shape[1]))]).astype(np.float32)
    for nprobe in (1, kc):
        for k in (513, 1000, 4097, 6500):                                 # 6500: above every stored vector
            wd, wi = full.batch_search(q, k, nprobe=nprobe)
            lims_all, dist_all, ids_all = _csr([s.batch_search(q, k, nprobe=nprobe) for s in shards])
            gd, gi = _merge_cut(lims_all, dist_all, ids_all, k, metric)
            assert np.array_equal(gi, wi), f"nprobe {nprobe}, k {k}: ids differ"
            assert np.array_equal(_bits(gd), _bits(wd)), f"nprobe {nprobe}, k {k}: distance bits differ"
            if k == 6500:
                assert (wi[:, -1] == -1).all(), "k above every probed vector: padded rows"


@pytest.mark.parametrize("metric", [0, 1], ids=["l2", "ip"])
def test_shard_knn_bound_argument(metric):
    """The route's argument on one GPU, one query at a time: each shard's range search at the radius min over shards of
    that shard's k-th distance (+inf when no shard holds k), each row cut at k, merged through the hook, equals the full
    index's batch_search(q, k) bit for bit.  Some queries leave a shard with no candidate (nprobe 1)."""
    rng, coarse, full, shards, bounds = _emulated(metric, 71 + metric, n=9000)
    kc, d = coarse.shape
    k = 700
    qs = [(coarse[rng.integers(0, kc)] + 0.3 * rng.standard_normal(d)).astype(np.float32) for _ in range(9)]
    qs += [coarse[bounds[1] - 1].astype(np.float32), coarse[0].astype(np.float32), coarse[kc - 1].astype(np.float32)]
    empty_shard = False
    for j, q1 in enumerate(qs):
        q = q1[None, :]
        nprobe = 1 if j >= 9 else 4
        kth = []
        for s in shards:
            sd, si = s.batch_search(q, k, nprobe=nprobe)
            kth.append(float(sd[0, k - 1]) if si[0, k - 1] >= 0 else float("inf"))
        radius = min(kth)
        rows = []
        for s in shards:
            lims, dd, ii = s.range_search(q, radius, nprobe=nprobe)
            empty_shard |= int(lims[-1]) == 0
            rows.append((dd[:k][None, :], ii[:k][None, :]))
        lims_all = np.stack([np.array([0, r[1].shape[1]], np.int64) for r in rows])
        gd, gi = _merge_cut(lims_all, np.concatenate([r[0].ravel() for r in rows]),
                            np.concatenate([r[1].ravel() for r in rows]), k, metric)
        wd, wi = full.batch_search(q, k, nprobe=nprobe)
        assert np.array_equal(gi, wi), f"query {j}: ids differ"
        assert np.array_equal(_bits(gd), _bits(wd)), f"query {j}: distance bits differ"
    assert empty_shard, "no query left a shard without candidates"
