"""Edge cases of the sharded IVF-PQ step (vix_sharded_add / vix_sharded_search behind ShardedIVFPQIndex, and
ReplicatedIVFPQIndex), bit for bit against one GPU holding the rows in the order the shards receive them.

The cases live in tests/mp_sharded_edges.py, one process per GPU under torch.distributed.run, all of them in one process
group per launch: query blocks at small and ragged batch sizes, k and nprobe at their limits, partitions with ranks that own
no list or only empty ones, every scan route, ties across ranks and the sign of zero inner-product distances, growth of the
exchange region, adds and removals between searches, replicas, and the collective refusal of an out-of-range id.  Each
world size runs over peer memory and over the NCCL fallback (VIX_NO_P2P=1): two ranks, and every GPU of the box (up to 8)
when it has more than two.  A box with one GPU runs the cases that need no second rank at world 1, and the shard merge
itself through its one-GPU entry point.
"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu

CASES = ["blocks", "k_nprobe", "partitions", "routes", "ties", "region", "mutate", "replicated", "bad_id"]
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
           "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "mp_sharded_edges.py")] + cases
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=1200, env=env)
    assert out.returncode == 0, out.stdout[-6000:] + out.stderr[-4000:]
    for case in cases:
        assert f"ok {case}:" in out.stdout, f"case {case} did not report: " + out.stdout[-3000:]
    peer = -1 if world == 1 else 0 if no_p2p else 1
    assert f"edges: world {world}, peer memory {peer}, {len(cases)} of {len(cases)} cases ok" in out.stdout, out.stdout[-3000:]


@pytest.mark.parametrize("no_p2p", [False, True], ids=["peer", "nccl"])
@pytest.mark.parametrize("size", ["two", "all"])
def test_sharded_edges(size, no_p2p):
    n = _ngpus()
    if n < 2:
        pytest.skip("needs two GPUs")
    if size == "all" and n <= 2:
        pytest.skip("the box has two GPUs: the two-rank launch covers it")
    _launch(2 if size == "two" else min(n, 8), no_p2p, CASES, 29561 + 2 * (size == "all") + no_p2p)


def test_sharded_edges_single_rank():
    """One rank: vix_sharded_add's collective validation over a one-rank communicator and the harness's one-GPU references,
    for every case that needs no second rank.  Boxes with two GPUs or more run the multi-rank launches instead."""
    if _ngpus() >= 2:
        pytest.skip("the multi-rank launches cover it")
    _launch(1, False, [c for c in CASES if c != "partitions"], 29565)


@pytest.mark.parametrize("metric", [0, 1], ids=["l2", "ip"])
def test_shard_merge_on_one_gpu(metric):
    """The result merge of vix_sharded_search (pack_result_keys_kernel + merge_shard_keys_kernel, through
    vix_debug_shard_merge) over three shards emulated on one GPU -- one IVFPQIndex per list block holding its lists' rows
    in the one-GPU index's slots, each scanning the one-GPU probes -- equals the one-GPU answer bit for bit: the sign of
    zero distances (a zero query: -0 under IP), NaN / -1 padding (k above the probed vectors), ties to the smaller id."""
    from vectorindex_b200 import _lib
    from vectorindex_b200.index import IVFPQIndex
    rng = np.random.default_rng(7 + metric)
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
    asg = np.repeat(np.arange(kc, dtype=np.int32), np.diff(off))      # the list of every exported row
    bounds = [kc * r // world for r in range(world + 1)]
    shards = []
    for r in range(world):
        sel = (asg >= bounds[r]) & (asg < bounds[r + 1])
        sh = index()
        sh.add_encoded(asg[sel], codes[sel], lids[sel])
        soff, _, sids, _ = sh.export_lists()
        assert np.array_equal(sids, lids[sel]) and np.array_equal(np.diff(soff)[bounds[r]:bounds[r + 1]],
                                                                   np.diff(off)[bounds[r]:bounds[r + 1]])
        shards.append(sh)
    q = np.concatenate([(coarse[rng.integers(0, kc, 20)] + 0.3 * rng.standard_normal((20, d))), np.zeros((3, d))])
    q = q.astype(np.float32)
    L = _lib.lib()
    for k, nprobe in ((10, 6), (64, 24), (512, 2)):
        fd, fi, fp = full.batch_search(q, k, nprobe=nprobe, return_probes=True)
        parts = [s.search_with_probes(q, k, fp) for s in shards]
        dall = np.ascontiguousarray(np.stack([p[0] for p in parts]))
        iall = np.ascontiguousarray(np.stack([p[1] for p in parts]))
        md, mi = np.empty((len(q), k), np.float32), np.empty((len(q), k), np.int64)
        _lib.check(L.vix_debug_shard_merge(_lib.ptr(dall), _lib.ptr(iall), world, C.c_int64(len(q)), k, metric,
                                           _lib.ptr(md), _lib.ptr(mi)))
        assert np.array_equal(mi, fi), f"k {k}: ids differ from one GPU"
        bad = np.argwhere(md.view(np.uint32) != fd.view(np.uint32))
        assert bad.size == 0, f"k {k}: {len(bad)} distances differ in their bits, first {md[tuple(bad[0])]!r} vs {fd[tuple(bad[0])]!r}"
        if metric == 1:
            z = mi[-3:] >= 0                                                 # (past the probed vectors: padding)
            assert z.any() and (md[-3:][z].view(np.uint32) == 0x80000000).all(), "zero IP distances must be -0"
        if k == 512:
            assert (mi[:, -1] == -1).all() and np.isnan(md[:, -1]).all(), "padding"
