"""Replicated indexes (vix_replicated_*), bit for bit against one GPU.

1. The premise of the layout: a query's answer does not depend on the other queries of its batch.  For every kind and
   metric, with and without an id filter, for k in {10, 512, 513, 2048} and for range search, the whole batch's one-GPU
   answer equals the answers of its blocks (vix_sharded_query_block at W = 2, 3 and 8: ragged, single-row and empty
   blocks) concatenated.  Two shapes take a different route for the whole batch than for its blocks, and the counters
   prove it: IVF-PQ through the list-major tensor-core scan (vix_scan_tc_launches), flat through the tensor-core shortlist
   (vix_tc_shortlist_calls).
2. The assembly kernels (vix_debug_replica_assemble) against a numpy concatenation: empty blocks and rows, NaN rows, the
   zero sign of each kind, world up to 256.
3. The calls at one rank (a one-rank communicator) through the C ABI and the Python classes equal vix_index_search /
   _filtered / vix_index_range_search, and every refusal comes before anything runs.
On several GPUs tests/mp_replicated.py runs under torch.distributed.run (two ranks and every GPU, peer memory and NCCL);
tests/c/replicated_smoke.c is a plain-C host of the four calls.
"""
import ctypes as C
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu

METRICS = {0: "euclidean", 1: "dotProduct", 2: "cosine"}
ERR_INVALID_K, ERR_INVALID_PARAM, ERR_NOT_TRAINED, ERR_UNSUPPORTED = -2, -5, -6, -9
KINDS = [("flat", 0), ("flat", 1), ("flat", 2), ("ivfflat", 0), ("ivfflat", 1), ("ivfflat", 2), ("ivfpq", 0), ("ivfpq", 1)]


def _L():
    from vectorindex_b200 import _lib
    return _lib.lib()


def same(a, b):
    """bit for bit: ids, distance bits (sign of zero and NaN included), lims"""
    assert len(a) == len(b)
    for x, y in zip(a, b):
        x, y = np.asarray(x), np.asarray(y)
        assert x.shape == y.shape, (x.shape, y.shape)
        if x.dtype == np.float32:
            bad = np.flatnonzero(x.view(np.uint32).ravel() != y.view(np.uint32).ravel())
            assert bad.size == 0, f"{bad.size} distance bits differ, first at {bad[0]}: {x.ravel()[bad[0]]} vs {y.ravel()[bad[0]]}"
        else:
            assert np.array_equal(x, y), f"{np.count_nonzero(x != y)} ids / lims differ"


def blocks(nq, world):
    out = []
    for r in range(world):
        f, c = C.c_int64(0), C.c_int64(0)
        assert _L().vix_sharded_query_block(C.c_int64(nq), C.c_int(r), C.c_int(world), C.byref(f), C.byref(c)) == 0
        out.append((f.value, c.value))
    return out


def build(kind, metric, seed=0, n=3000, d=32, kc=32, m=16, nprobe=6, dup=True):
    """an index of each kind over clustered rows, some stored twice (ids repeat)"""
    from vectorindex_b200.index import FlatIndex, IVFIndex, IVFPQIndex
    rng = np.random.default_rng(seed)
    cent = rng.standard_normal((24, d)).astype(np.float32)
    x = (cent[rng.integers(0, 24, n)] + 0.3 * rng.standard_normal((n, d))).astype(np.float32)
    ids = np.arange(n, dtype=np.int64) * 3 + 1
    if dup:
        x[n - 40:] = x[:40]
        ids[n - 40:] = ids[:40]
    if kind == "flat":
        ix = FlatIndex(d, METRICS[metric])
    elif kind == "ivfflat":
        ix = IVFIndex(d, METRICS[metric], nlist=kc, nprobe=nprobe)
        ix.set_coarse(x[rng.choice(n, kc, replace=False)])
    else:
        ix = IVFPQIndex(d, METRICS[metric], nlist=kc, nprobe=nprobe, m=m)
        ix.optimize(x[:2000])
    ix.batch_insert(x, ids)
    q = (cent[rng.integers(0, 24, 64)] + 0.3 * rng.standard_normal((64, d))).astype(np.float32)
    return ix, x, ids, q


def a_filter(ids, seed=1):
    from vectorindex_b200.index import IDFilter
    rng = np.random.default_rng(seed)
    f = IDFilter(int(ids.max()) + 1, "allow")
    f.set(rng.choice(ids, ids.size // 2, replace=False))
    return f


def knn_blocks(ix, q, k, nprobe, filt, world):
    parts = [ix.batch_search(q[f:f + c], k, nprobe, filter=filt) for f, c in blocks(q.shape[0], world)]
    return np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts])


def range_blocks(ix, q, radius, nprobe, filt, world):
    lims, ds, ids, at = [np.zeros(1, np.int64)], [], [], 0
    for f, c in blocks(q.shape[0], world):
        l, d, i = ix.range_search(q[f:f + c], radius, nprobe, filter=filt)
        lims.append(l[1:] + at)
        at += d.size
        ds.append(d)
        ids.append(i)
    return np.concatenate(lims), np.concatenate(ds), np.concatenate(ids)


# ---------------------------------------------------------------------------------------------------- 1. the premise
@pytest.mark.parametrize("kind,metric", KINDS)
@pytest.mark.parametrize("filtered", [False, True])
def test_block_independence(kind, metric, filtered):
    ix, x, ids, q = build(kind, metric)
    filt = a_filter(ids) if filtered else None
    for nq in (9, 37):                                   # W = 8 at nq = 9: blocks of 4, 4, 1 and five empty ones
        qq = q[:nq]
        for k in (10, 512, 513, 2048):
            whole = ix.batch_search(qq, k, 0, filter=filt)
            for world in (2, 3, 8):
                same(whole, knn_blocks(ix, qq, k, 0, filt, world))
            if k == 2048:
                same((whole[0][:, :513], whole[1][:, :513]), ix.batch_search(qq, 513, 0, filter=filt))
        d10 = ix.batch_search(qq, 10)[0]
        radius = float(np.nanmedian(d10[:, -1]))
        whole = ix.range_search(qq, radius, 0, filter=filt)
        assert whole[0][-1] > 0
        for world in (2, 3, 8):
            same(whole, range_blocks(ix, qq, radius, 0, filt, world))


def test_block_independence_list_major_scan():
    """the whole batch takes the list-major tensor-core scan (nq x nprobe >= 32768), its blocks the query-major one"""
    from vectorindex_b200.index import IVFPQIndex
    L = _L()
    rng = np.random.default_rng(5)
    n, d, m, kc, nprobe, nq = 20000, 32, 16, 128, 64, 600
    cent = rng.standard_normal((64, d)).astype(np.float32)
    x = (cent[rng.integers(0, 64, n + nq)] + 0.3 * rng.standard_normal((n + nq, d))).astype(np.float32)
    ix = IVFPQIndex(d, "euclidean", nlist=kc, nprobe=nprobe, m=m)
    ix.optimize(x[:8000])
    ix.batch_insert(x[:n])
    q = x[n:]
    for k in (10, 64):
        before = int(L.vix_scan_tc_launches())
        whole = ix.batch_search(q, k)
        assert int(L.vix_scan_tc_launches()) - before == 1, "the whole batch did not take the list-major scan"
        for world in (2, 3, 8):
            before = int(L.vix_scan_tc_launches())
            parts = knn_blocks(ix, q, k, 0, None, world)
            assert int(L.vix_scan_tc_launches()) == before, "a block took the list-major scan"
            same(whole, parts)


def test_block_independence_flat_shortlist():
    """the whole batch takes the flat tensor-core shortlist (nq >= 16), blocks of 8 rows the exact kernel"""
    from vectorindex_b200.index import FlatIndex
    L = _L()
    rng = np.random.default_rng(6)
    n, d, nq = 4096, 64, 40
    x = rng.standard_normal((n, d)).astype(np.float32)
    q = rng.standard_normal((nq, d)).astype(np.float32)
    for metric in (0, 1):
        ix = FlatIndex(d, METRICS[metric])
        ix.batch_insert(x)
        before = int(L.vix_tc_shortlist_calls(1))
        whole = ix.batch_search(q, 10)
        assert int(L.vix_tc_shortlist_calls(1)) > before, "the whole batch did not take the shortlist"
        for world in (2, 3, 8):
            before = int(L.vix_tc_shortlist_calls(1))
            parts = knn_blocks(ix, q, 10, 0, None, world)
            if world == 8:
                assert int(L.vix_tc_shortlist_calls(1)) == before, "a block of 8 rows took the shortlist"
            same(whole, parts)


# ---------------------------------------------------------------------------------------------------- 2. assembly
def assemble_knn(dist, ids, world, k):
    from vectorindex_b200 import _lib
    nq = dist.shape[0]
    od, oi = np.empty((nq, k), np.float32), np.empty((nq, k), np.int64)
    _lib.check(_L().vix_debug_replica_assemble(None, _lib.ptr(dist), _lib.ptr(ids), C.c_int(world), C.c_int64(nq), C.c_int(k),
                                               C.c_int(0), C.c_int(2), _lib.ptr(od), _lib.ptr(oi), None))
    return od, oi


def assemble_range(lims_all, dist, ids, world, nq, metric, kind):
    from vectorindex_b200 import _lib
    res = C.c_void_p(0)
    _lib.check(_L().vix_debug_replica_assemble(_lib.ptr(lims_all), _lib.ptr(dist) if dist.size else None,
                                               _lib.ptr(ids) if ids.size else None, C.c_int(world), C.c_int64(nq), C.c_int(0),
                                               C.c_int(metric), C.c_int(kind), None, None, C.byref(res)))
    try:
        total = int(_L().vix_range_result_total(res))
        lims, d, i = np.empty(nq + 1, np.int64), np.empty(total, np.float32), np.empty(total, np.int64)
        _lib.check(_L().vix_range_result_get(res, _lib.ptr(lims), _lib.ptr(d) if total else None, _lib.ptr(i) if total else None))
        return lims, d, i
    finally:
        _L().vix_range_result_destroy(res)


@pytest.mark.parametrize("world,nq,k", [(1, 5, 3), (2, 9, 10), (3, 37, 7), (8, 9, 513), (256, 300, 4), (256, 5, 2)])
def test_assemble_knn(world, nq, k):
    rng = np.random.default_rng(world + nq)
    d = rng.standard_normal((nq, k)).astype(np.float32)
    i = rng.integers(0, 1 << 31, (nq, k)).astype(np.int64)
    d[0, k // 2:] = np.nan                                         # a padded row
    i[0, k // 2:] = -1
    if nq > 3:
        d[3] = np.float32(np.nan)                                  # a NaN row with real ids
        d[1, 0] = -0.0
    same((d, i), assemble_knn(d, i, world, k))


@pytest.mark.parametrize("world,nq", [(1, 4), (2, 9), (3, 37), (8, 9), (256, 300), (256, 3)])
@pytest.mark.parametrize("metric,kind", [(0, 2), (1, 2), (1, 0), (1, 1), (2, 1)])
def test_assemble_range(world, nq, metric, kind):
    rng = np.random.default_rng(world * 7 + nq + metric)
    lens = rng.integers(0, 5, nq)
    lens[::3] = 0                                                  # empty rows
    rows_d = [np.sort(rng.standard_normal(l).astype(np.float32)) for l in lens]
    for r in rows_d:
        if r.size:
            r[0] = 0.0                                             # a zero distance: its sign is the kind's
    rows_i = [rng.integers(0, 1 << 31, l).astype(np.int64) for l in lens]
    lims_all = []
    for f, c in blocks(nq, world):
        lims_all.append(np.concatenate([[0], np.cumsum(lens[f:f + c])]).astype(np.int64))
    lims_all = np.concatenate(lims_all)
    d = np.concatenate(rows_d) if nq else np.zeros(0, np.float32)
    i = np.concatenate(rows_i) if nq else np.zeros(0, np.int64)
    neg = kind != 1 and metric == 1
    want_d = np.where(d == 0, np.float32(-0.0) if neg else np.float32(0.0), d).astype(np.float32)
    want = (np.concatenate([[0], np.cumsum(lens)]).astype(np.int64), want_d, i)
    same(want, assemble_range(lims_all, d.astype(np.float32), i, world, nq, metric, kind))


# ---------------------------------------------------------------------------------------------------- 3. one rank
def _comm():
    from vectorindex_b200.index import Comm
    return Comm(0, 1, Comm.unique_id())


@pytest.mark.parametrize("kind,metric", KINDS)
def test_one_rank_equals_one_gpu(kind, metric):
    from vectorindex_b200 import _lib
    from vectorindex_b200.index import FlatIndex, IVFIndex, IVFPQIndex
    L = _L()
    ref, x, ids, q = build(kind, metric, seed=3)
    cls = {"flat": FlatIndex, "ivfflat": IVFIndex, "ivfpq": IVFPQIndex}[kind]
    rep = cls(x.shape[1], METRICS[metric], nlist=32, nprobe=6, m=16) if kind != "flat" else FlatIndex(x.shape[1], METRICS[metric])
    if kind == "ivfflat":
        rep.set_coarse(ref.get_coarse())
    elif kind == "ivfpq":
        rep.set_coarse(ref.get_coarse())
        rep.set_codebooks(*ref.get_codebooks())
    comm = _comm()
    n = x.shape[0]
    _lib.check(L.vix_replicated_add(rep._h, comm._c, _lib.ptr(x), _lib.ptr(ids), C.c_int64(n)))
    filt = a_filter(ids)
    for k in (10, 600):
        want = ref.batch_search(q, k)
        got = (np.empty((q.shape[0], k), np.float32), np.empty((q.shape[0], k), np.int64))
        _lib.check(L.vix_replicated_search(rep._h, comm._c, _lib.ptr(q), C.c_int64(q.shape[0]), C.c_int(k), C.c_int(0),
                                           _lib.ptr(got[0]), _lib.ptr(got[1])))
        same(want, got)
        want = ref.batch_search(q, k, filter=filt)
        _lib.check(L.vix_replicated_search_filtered(rep._h, comm._c, _lib.ptr(q), C.c_int64(q.shape[0]), C.c_int(k), C.c_int(0),
                                                    _lib.ptr(filt.words, np.uint64), C.c_int64(filt.capacity), C.c_int(filt.mode),
                                                    _lib.ptr(got[0]), _lib.ptr(got[1])))
        same(want, got)
    radius = float(np.nanmedian(ref.batch_search(q, 10)[0][:, -1]))
    res = C.c_void_p(0)
    _lib.check(L.vix_replicated_range_search(rep._h, comm._c, _lib.ptr(q), C.c_int64(q.shape[0]), C.c_float(radius), C.c_int(0),
                                             None, C.c_int64(0), C.c_int(0), C.byref(res)))
    total = int(L.vix_range_result_total(res))
    got = (np.empty(q.shape[0] + 1, np.int64), np.empty(total, np.float32), np.empty(total, np.int64))
    _lib.check(L.vix_range_result_get(res, _lib.ptr(got[0]), _lib.ptr(got[1]), _lib.ptr(got[2])))
    L.vix_range_result_destroy(res)
    same(ref.range_search(q, radius), got)
    comm.close()


@pytest.mark.parametrize("kind,metric", [("flat", 1), ("ivfflat", 0), ("ivfpq", 1)])
def test_python_classes_one_rank(kind, metric):
    import torch
    from vectorindex_b200.index import ReplicatedFlatIndex, ReplicatedIVFFlatIndex, ReplicatedNativeIVFPQIndex
    ref, x, ids, q = build(kind, metric, seed=4)
    if kind == "flat":
        rep = ReplicatedFlatIndex(x.shape[1], METRICS[metric])
    elif kind == "ivfflat":
        rep = ReplicatedIVFFlatIndex(x.shape[1], METRICS[metric], nlist=32, nprobe=6)
        rep.set_coarse(ref.get_coarse())
    else:
        rep = ReplicatedNativeIVFPQIndex(x.shape[1], METRICS[metric], nlist=32, nprobe=6, m=16)
        rep.set_parameters(ref.get_coarse(), *ref.get_codebooks())
    rep.add(x, ids)
    assert rep.count == ref.count
    filt = a_filter(ids)
    same(ref.batch_search(q, 10), rep.batch_search(q, 10))
    same(ref.batch_search(q, 700, filter=filt), rep.batch_search(q, 700, filter=filt))
    same(ref.batch_search(q, 10), rep.batch_search(q, 10, gather=False))            # one rank: the block is the batch
    dq = torch.from_numpy(q).cuda()
    got = rep.batch_search(dq, 10)
    same(ref.batch_search(q, 10), (got[0].cpu().numpy(), got[1].cpu().numpy()))
    radius = float(np.nanmedian(ref.batch_search(q, 10)[0][:, -1]))
    same(ref.range_search(q, radius, filter=filt), rep.range_search(q, radius, filter=filt))
    assert rep.remove(ids[:100]) == ref.batch_remove(ids[:100])
    same(ref.batch_search(q, 10), rep.batch_search(q, 10))


def test_refusals_before_anything_runs():
    from vectorindex_b200 import _lib
    from vectorindex_b200.index import FlatIndex, IVFIndex, IVFPQIndex
    L = _L()
    comm = _comm()
    ix, x, ids, q = build("ivfflat", 0, seed=7)
    nq = q.shape[0]
    d, i = np.full((nq, 10), 7, np.float32), np.full((nq, 10), 7, np.int64)

    def search(h, k=10, nprobe=0, words=None, cap=0, mode=0):
        return L.vix_replicated_search_filtered(h, comm._c, _lib.ptr(q), C.c_int64(nq), C.c_int(k), C.c_int(nprobe),
                                                _lib.ptr(words, np.uint64), C.c_int64(cap), C.c_int(mode), _lib.ptr(d), _lib.ptr(i))

    def rng_search(h, radius=1.0, nprobe=0, mode=0, cap=0):
        res = C.c_void_p(0)
        rc = L.vix_replicated_range_search(h, comm._c, _lib.ptr(q), C.c_int64(nq), C.c_float(radius), C.c_int(nprobe), None,
                                           C.c_int64(cap), C.c_int(mode), C.byref(res))
        assert not res.value
        return rc

    launches = int(L.vix_kernel_launches(0))
    assert rng_search(ix._h, radius=float("nan")) == ERR_INVALID_PARAM
    assert rng_search(ix._h, mode=2) == ERR_INVALID_PARAM
    assert rng_search(ix._h, cap=-1) == ERR_INVALID_PARAM
    assert rng_search(ix._h, nprobe=513) == ERR_INVALID_K
    assert search(ix._h, mode=2, words=np.zeros(1, np.uint64)) == ERR_INVALID_PARAM
    assert search(ix._h, cap=-1, words=np.zeros(1, np.uint64)) == ERR_INVALID_PARAM
    assert search(ix._h, nprobe=513) == ERR_INVALID_K
    assert search(ix._h, k=16385) == ERR_INVALID_K
    pq = IVFPQIndex(x.shape[1], "euclidean", nlist=16, nprobe=4, m=16)                 # untrained
    assert search(pq._h) == ERR_NOT_TRAINED and rng_search(pq._h) == ERR_NOT_TRAINED
    assert L.vix_replicated_add(pq._h, comm._c, _lib.ptr(x), _lib.ptr(ids), C.c_int64(10)) == ERR_NOT_TRAINED
    raw = IVFIndex(x.shape[1], "euclidean", nlist=16, nprobe=4)                        # IVF-Flat without centroids
    assert L.vix_replicated_add(raw._h, comm._c, _lib.ptr(x), _lib.ptr(ids), C.c_int64(10)) == ERR_NOT_TRAINED
    assert raw.count == 0
    from vectorindex_b200._lib import IndexParams
    p = IndexParams()
    L.vix_index_params_default(C.byref(p))
    p.kind, p.d, p.metric, p.shard_rank, p.shard_world = 0, x.shape[1], 0, 0, 2
    sh = C.c_void_p(0)
    _lib.check(L.vix_index_create(C.byref(p), C.byref(sh)))
    assert search(sh) == ERR_INVALID_PARAM and rng_search(sh) == ERR_INVALID_PARAM
    assert L.vix_replicated_add(sh, comm._c, _lib.ptr(x), _lib.ptr(ids), C.c_int64(10)) == ERR_INVALID_PARAM
    L.vix_index_destroy(sh)
    assert int(L.vix_kernel_launches(0)) == launches, "a refused call launched a kernel"
    assert (d == 7).all() and (i == 7).all(), "a refused call wrote its outputs"
    # collective validation: one id outside [0, 2^32 - 1) refuses the whole add
    fl = FlatIndex(x.shape[1], "euclidean")
    bad = ids[:10].copy()
    bad[3] = (1 << 32) - 1
    assert L.vix_replicated_add(fl._h, comm._c, _lib.ptr(x), _lib.ptr(bad), C.c_int64(10)) == ERR_INVALID_PARAM
    assert fl.count == 0
    assert L.vix_replicated_add(ix._h, comm._c, _lib.ptr(x), _lib.ptr(bad), C.c_int64(10)) == ERR_INVALID_PARAM
    assert ix.count == x.shape[0]
    comm.close()


def test_plain_c_host_one_rank(tmp_path):
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else shutil.which("gcc")
    lib_dir = os.path.join(ROOT, "vectorindex_b200")
    exe = str(tmp_path / "replicated_smoke")
    subprocess.check_call([cc, "-std=c11", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "c", "replicated_smoke.c"), "-o", exe, "-L", lib_dir, "-lvindex_b200",
                           "-Wl,-rpath," + lib_dir, "-lm"])
    out = subprocess.run([exe, "1"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "replicated == single-GPU: yes" in out.stdout


# ---------------------------------------------------------------------------------------------------- several GPUs
def _ngpus():
    import torch
    return torch.cuda.device_count()


@pytest.mark.parametrize("no_p2p", [False, True])
def test_plain_c_host_two_ranks(tmp_path, no_p2p):
    if _ngpus() < 2:
        pytest.skip("needs two GPUs")
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else shutil.which("gcc")
    lib_dir = os.path.join(ROOT, "vectorindex_b200")
    exe = str(tmp_path / "replicated_smoke")
    subprocess.check_call([cc, "-std=c11", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "c", "replicated_smoke.c"), "-o", exe, "-L", lib_dir, "-lvindex_b200",
                           "-Wl,-rpath," + lib_dir, "-lm"])
    env = dict(os.environ)
    if no_p2p:
        env["VIX_NO_P2P"] = "1"
    out = subprocess.run([exe, "2"], capture_output=True, text=True, timeout=600, env=env)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "replicated == single-GPU: yes" in out.stdout


@pytest.mark.parametrize("every_gpu", [False, True])
@pytest.mark.parametrize("no_p2p", [False, True])
def test_ranks_under_torchrun(every_gpu, no_p2p):
    n = _ngpus()
    if n < 2:
        pytest.skip("needs two GPUs")
    world = min(n, 8) if every_gpu else 2
    if every_gpu and world == 2:
        pytest.skip("the box has two GPUs: the two-rank case covers it")
    env = dict(os.environ)
    env.pop("VIX_NO_P2P", None)
    if no_p2p:
        env["VIX_NO_P2P"] = "1"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(29561 + world + (10 if no_p2p else 0)), os.path.join(ROOT, "tests", "mp_replicated.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=1200, env=env)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "replicated ok" in out.stdout
