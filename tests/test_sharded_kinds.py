"""The sharded flat and IVF-Flat indexes, bit for bit against one GPU.

Every rank is emulated on one GPU (vix_debug_sharded_emulate: each rank's local pass of vix_sharded_search /
_filtered / vix_sharded_range_search over its own handle, merged by the kernels the exchange runs; only the transport is
left out).  Flat shards hold contiguous row blocks, and the one-GPU index holds the blocks rank by rank; IVF-Flat shards
hold the rows of their list blocks (one rank owns none), and the answer must equal one GPU holding the rows in the shards'
order and in the original order.  The flat merge is also checked against a numpy stable merge, and each trap of the flat
merge has its own case: ties at one raw score broken by rank (row) rather than id, two raw scores that map to one API
distance, NaN rows beside a short rank, the sign of a zero distance per kind, one row stored on two ranks (the parity
data).  One rank runs through the real entry points (a one-rank communicator) and the Python classes.  On several GPUs:
tests/mp_sharded_kinds.py under torch.distributed.run, at two ranks and at every GPU of the box (up to 8), over peer
memory and over NCCL (VIX_NO_P2P=1); a box with one GPU runs it at world 1.  tests/c/sharded_kinds_smoke.c is the plain-C
host of the same calls.
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
ERR_INVALID_PARAM, ERR_NOT_TRAINED = -5, -6


def _L():
    from vectorindex_b200 import _lib
    return _lib.lib()


def emulate(shards, q, k=0, nprobe=0, filt=None, radius=None):
    """k-NN (radius None) or range search over the shards, every rank on this GPU"""
    from vectorindex_b200 import _lib
    arr = (C.c_void_p * len(shards))(*[s._h.value for s in shards])
    q = np.ascontiguousarray(q, dtype=np.float32)
    nq = q.shape[0]
    words = filt.words if filt is not None else None
    fargs = (_lib.ptr(words, np.uint64), C.c_int64(filt.capacity if filt is not None else 0),
             C.c_int(filt.mode if filt is not None else 0))
    if radius is None:
        d = np.empty((nq, k), np.float32)
        i = np.empty((nq, k), np.int64)
        _lib.check(_L().vix_debug_sharded_emulate(arr, C.c_int(len(shards)), _lib.ptr(q), C.c_int64(nq), C.c_int(k),
                                                  C.c_int(nprobe), C.c_float(0.0), *fargs, _lib.ptr(d), _lib.ptr(i), None))
        return d, i
    res = C.c_void_p(0)
    _lib.check(_L().vix_debug_sharded_emulate(arr, C.c_int(len(shards)), _lib.ptr(q), C.c_int64(nq), C.c_int(0),
                                              C.c_int(nprobe), C.c_float(radius), *fargs, None, None, C.byref(res)))
    try:
        total = int(_L().vix_range_result_total(res))
        lims = np.empty(nq + 1, np.int64)
        d = np.empty(total, np.float32)
        i = np.empty(total, np.int64)
        _lib.check(_L().vix_range_result_get(res, _lib.ptr(lims), _lib.ptr(d) if total else None, _lib.ptr(i) if total else None))
        return lims, d, i
    finally:
        _L().vix_range_result_destroy(res)


def same(a, b):
    """bit for bit: ids, distance bits (sign of zero and NaN included), lims"""
    assert len(a) == len(b)
    for x, y in zip(a, b):
        assert x.shape == y.shape, (x.shape, y.shape)
        if x.dtype == np.float32:
            bad = np.flatnonzero(x.view(np.uint32).ravel() != y.view(np.uint32).ravel())
            assert bad.size == 0, f"{bad.size} distance bits differ, first at {bad[0]}: {x.ravel()[bad[0]]} vs {y.ravel()[bad[0]]}"
        else:
            assert np.array_equal(x, y), f"{np.count_nonzero(x != y)} ids / lims differ"


def _flat(d, metric, x=None, ids=None):
    from vectorindex_b200.index import FlatIndex
    ix = FlatIndex(d, METRICS[metric])
    if x is not None and len(x):
        ix.batch_insert(np.ascontiguousarray(x, np.float32), np.ascontiguousarray(ids, np.int64))
    return ix


def _ivfflat(d, metric, coarse, nprobe, x=None, ids=None):
    from vectorindex_b200.index import IVFIndex
    ix = IVFIndex(d, METRICS[metric], nlist=coarse.shape[0], nprobe=nprobe)
    ix.set_coarse(coarse)
    if x is not None and len(x):
        ix.batch_insert(np.ascontiguousarray(x, np.float32), np.ascontiguousarray(ids, np.int64))
    return ix


def _data(seed, n, d, nq):
    """small integer components: many rows tie at one raw score; a few rows stored twice (same vector; half of them under
    the same id too) so that copies land on different ranks; ids descend with the row, opposite to the ranks' order"""
    rng = np.random.default_rng(seed)
    x = rng.integers(-2, 3, (n, d)).astype(np.float32)
    dup = rng.choice(n // 2, 40, replace=False)
    x[n - 40:] = x[dup]
    ids = (np.arange(n, dtype=np.int64)[::-1] * 3 + 11).copy()
    ids[n - 20:] = ids[dup[20:]]
    q = rng.integers(-2, 3, (nq, d)).astype(np.float32)
    q[0] = 0.0
    return x, ids, q


def _filter(ids, seed):
    from vectorindex_b200.index import IDFilter
    rng = np.random.default_rng(seed)
    f = IDFilter(int(ids.max()) + 1, "allow")
    f.set(rng.choice(np.unique(ids), len(ids) // 2, replace=False))
    return f


def _radii(ref_d):
    v = np.sort(ref_d[np.isfinite(ref_d)].ravel())
    return [float(v[len(v) // 50]), float(v[len(v) // 4])]


# ---------------------------------------------------------------------------------------------------------------- flat
@pytest.mark.parametrize("world", [2, 3, 8])
@pytest.mark.parametrize("metric", [0, 1, 2], ids=["l2", "ip", "cos"])
def test_flat_parity(metric, world):
    n, d, nq = 6000, 24, 37
    x, ids, q = _data(100 + metric, n, d, nq)
    one = _flat(d, metric, x, ids)
    cuts = np.linspace(0, n, world + 1).astype(int)
    cuts[1] = cuts[0]                                                  # rank 0 holds nothing
    shards = [_flat(d, metric, x[cuts[r]:cuts[r + 1]], ids[cuts[r]:cuts[r + 1]]) for r in range(world)]
    filt = _filter(ids, 5)
    for k in (1, 10, 512, 513, 2048):
        ref = one.batch_search(q, k)
        same(emulate(shards, q, k), ref)
        same(emulate(shards, q, k, filt=filt), one.batch_search(q, k, filter=filt))
        if k == 2048:                                                  # search(k)[:, :k2] == search(k2)
            for k2 in (10, 512, 513):
                same([a[:, :k2].copy() for a in ref], one.batch_search(q, k2))
    ref = one.batch_search(q, 64)[0]
    for radius in _radii(ref):
        same(emulate(shards, q, radius=radius), one.range_search(q, radius))
        same(emulate(shards, q, radius=radius, filt=filt), one.range_search(q, radius, filter=filt))


# ------------------------------------------------------------------------------------------------------------ IVF-Flat
@pytest.mark.parametrize("world", [2, 3, 8])
@pytest.mark.parametrize("metric", [0, 1, 2], ids=["l2", "ip", "cos"])
def test_ivfflat_parity(metric, world):
    from vectorindex_b200.index import IVFIndex
    n, d, nq, kc, nprobe = 6000, 24, 37, 32, 6
    x, ids, q = _data(200 + metric, n, d, nq)
    trainer = IVFIndex(d, METRICS[metric], nlist=kc, nprobe=nprobe)
    trainer.optimize(x)
    coarse = trainer.get_coarse()
    kc = coarse.shape[0]
    # the list each row goes to (its first probe: the partition only decides which rank holds a row, the answer does not
    # depend on it), and the ranks' list blocks (rank 1 owns none)
    asg = _first_probe(_ivfflat(d, metric, coarse, 1), x)
    bounds = np.linspace(0, kc, world + 1).astype(int)
    bounds[2] = bounds[1]
    owner = np.searchsorted(bounds[1:-1], asg, side="right")
    rows = [np.flatnonzero(owner == r) for r in range(world)]
    shards = [_ivfflat(d, metric, coarse, nprobe, x[rw], ids[rw]) for rw in rows]
    order = np.concatenate(rows)
    slots = _ivfflat(d, metric, coarse, nprobe, x[order], ids[order])  # the shards' slots
    orig = _ivfflat(d, metric, coarse, nprobe, x, ids)                 # the original order
    filt = _filter(ids, 6)
    for k in (1, 10, 512, 513, 2048):
        ref = slots.batch_search(q, k)
        same(ref, orig.batch_search(q, k))
        same(emulate(shards, q, k), ref)
        same(emulate(shards, q, k, filt=filt), slots.batch_search(q, k, filter=filt))
    ref = slots.batch_search(q, 64)[0]
    for radius in _radii(ref):
        same(emulate(shards, q, radius=radius), slots.range_search(q, radius))
        same(emulate(shards, q, radius=radius, filt=filt), orig.range_search(q, radius, filter=filt))


def _first_probe(ix, x):
    from vectorindex_b200 import _lib
    nq = x.shape[0]
    d = np.empty((nq, 1), np.float32)
    i = np.empty((nq, 1), np.int64)
    pr = np.empty((nq, 1), np.int32)
    _lib.check(_L().vix_index_search_ex(ix._h, _lib.ptr(x), C.c_int64(nq), C.c_int(1), C.c_int(1), _lib.ptr(d), _lib.ptr(i),
                                        _lib.ptr(pr), None))
    return pr[:, 0].astype(np.int64)


# ------------------------------------------------------------------------------------------------ the flat merge vs numpy
def _word(s, order_max):
    s = (s + np.float32(0)).astype(np.float32)                        # -0 -> +0, as make_key
    u = s.view(np.uint32).astype(np.uint64)
    w = np.where(u & 0x80000000, ~u & 0xFFFFFFFF, u | 0x80000000)
    if order_max:
        w = ~w & 0xFFFFFFFF
    return np.where(np.isnan(s), 0xFFFFFFFF, w).astype(np.uint64)


def _api(s, metric):
    s = (s + np.float32(0)).astype(np.float32)
    with np.errstate(invalid="ignore"):
        if metric == 0:
            return np.sqrt(s)
        if metric == 1:
            return -s
        return np.float32(1) - s


@pytest.mark.parametrize("metric", [0, 1, 2], ids=["l2", "ip", "cos"])
@pytest.mark.parametrize("k", [0, 7, 600])
def test_flat_merge_against_numpy(metric, k):
    """vix_debug_shard_flat_merge over adversarial runs (scores from a handful of values, NaN scores, empty and long runs,
    ids in the opposite order to the ranks) against a stable numpy merge by (score word, rank, place in the run)"""
    from vectorindex_b200 import _lib
    rng = np.random.default_rng(11 + metric + k)
    world, nq = 5, 9
    vals = np.array([0.0, -0.0, 0.25, 0.5, 0.5000001, 2.0, np.nan, -1.0], np.float32)
    order_max = metric != 0
    lims, sc, idv = [], [], []
    for r in range(world):
        lr = [0]
        for qq in range(nq):
            m = int(rng.integers(0, 3 if r == 1 else 900))
            s = rng.choice(vals, m).astype(np.float32)
            if metric == 0:
                s = np.abs(s)
            w = _word(s, order_max)
            o = np.argsort(w, kind="stable")                           # a run: word order, then row
            sc.append(s[o])
            idv.append((10000 - 1000 * r - np.arange(m)).astype(np.int64))
            lr.append(lr[-1] + m)
        lims.append(lr)
    lims = np.asarray(lims, np.int64)
    sc, idv = np.concatenate(sc), np.concatenate(idv)
    total = int(lims[:, -1].sum())
    n_out = nq * k if k else total
    od = np.empty(max(n_out, 1), np.float32)
    oi = np.empty(max(n_out, 1), np.int64)
    ol = np.empty(nq + 1, np.int64)
    _lib.check(_L().vix_debug_shard_flat_merge(_lib.ptr(lims), _lib.ptr(sc), _lib.ptr(idv), C.c_int(world), C.c_int64(nq),
                                               C.c_int(k), C.c_int(metric), _lib.ptr(ol), _lib.ptr(od), _lib.ptr(oi)))
    base = np.concatenate([[0], np.cumsum(lims[:, -1])])
    exp_d, exp_i, exp_l = [], [], [0]
    for qq in range(nq):
        ws, rs, ps, ss, ii = [], [], [], [], []
        for r in range(world):
            lo, hi = base[r] + lims[r, qq], base[r] + lims[r, qq + 1]
            ws.append(_word(sc[lo:hi], order_max)); rs.append(np.full(hi - lo, r)); ps.append(np.arange(hi - lo))
            ss.append(sc[lo:hi]); ii.append(idv[lo:hi])
        w, rr, pp, s, i = map(np.concatenate, (ws, rs, ps, ss, ii))
        o = np.lexsort((pp, rr, w))
        dd, di = _api(s[o], metric), i[o]
        if k:
            dd = np.concatenate([dd[:k], np.full(max(0, k - len(dd)), np.nan, np.float32)])
            di = np.concatenate([di[:k], np.full(max(0, k - len(di)), -1, np.int64)])
        exp_d.append(dd); exp_i.append(di); exp_l.append(exp_l[-1] + len(dd))
    exp_d, exp_i = np.concatenate(exp_d), np.concatenate(exp_i)
    od, oi = od[:n_out], oi[:n_out]
    assert np.array_equal(oi, exp_i)
    fin = ~np.isnan(exp_d)
    assert np.array_equal(np.isnan(od), ~fin)
    assert np.array_equal(od[fin].view(np.uint32), exp_d[fin].view(np.uint32))
    if not k:
        assert np.array_equal(ol, np.asarray(exp_l))


# ------------------------------------------------------------------------------------------------------------ the traps
def test_trap_equal_scores_fall_to_the_rank():
    """Equal raw scores on two ranks, ids in the opposite order: one GPU returns the lower RANK's row first (its row index
    is smaller), which a merge on (distance, id) would put second"""
    d = 8
    v = np.zeros((1, d), np.float32); v[0, 0] = 1.0
    q = np.zeros((1, d), np.float32)
    for metric in (0, 1):
        a = _flat(d, metric, v, [900])
        b = _flat(d, metric, v, [5])
        one = _flat(d, metric, np.concatenate([v, v]), [900, 5])
        for k in (2, 600):
            got = emulate([a, b], q, k)
            same(got, one.batch_search(q, k))
            assert list(got[1][0, :2]) == [900, 5]


def test_trap_two_scores_one_distance():
    """Two raw scores that sqrt (L2) or 1 - s (cosine) map to one API distance, the smaller-id row on the lower rank holding
    the worse score: one GPU orders by the raw score, so the higher rank's row comes first"""
    d = 8
    # L2: rows (1, 0, ...) and (1, b, 0, ...) against the zero query score 1 and fl(1 + fl(b * b)) = 1 + 2^-23, whose
    # square roots both round to 1
    b = np.float32(2 ** -11.5)
    s2 = np.float32(1) + b * b
    assert s2 != np.float32(1) and np.sqrt(s2) == np.float32(1)
    x1 = np.zeros((1, d), np.float32); x1[0, 0] = 1.0
    x2 = np.zeros((1, d), np.float32); x2[0, 0] = 1.0; x2[0, 1] = b
    q = np.zeros((1, d), np.float32)
    hi, lo = _flat(d, 0, x2, [3]), _flat(d, 0, x1, [8])                # rank 0: the larger score, the smaller id
    one = _flat(d, 0, np.concatenate([x2, x1]), [3, 8])
    for k in (2, 600):
        got = emulate([hi, lo], q, k)
        same(got, one.batch_search(q, k))
        assert got[0][0, 0] == got[0][0, 1] and list(got[1][0, :2]) == [8, 3]
    # cosine: similarities ~1e-9 and ~2e-9 both give 1 - s = 1
    y1 = np.zeros((1, d), np.float32); y1[0, 0] = 1e-9; y1[0, 1] = 1.0
    y2 = np.zeros((1, d), np.float32); y2[0, 0] = 2e-9; y2[0, 1] = 1.0
    qc = np.zeros((1, d), np.float32); qc[0, 0] = 1.0
    r0, r1 = _flat(d, 2, y1, [3]), _flat(d, 2, y2, [8])
    one = _flat(d, 2, np.concatenate([y1, y2]), [3, 8])
    for k in (2, 600):
        got = emulate([r0, r1], qc, k)
        same(got, one.batch_search(qc, k))
        assert got[0][0, 0] == got[0][0, 1] and list(got[1][0, :2]) == [8, 3]


@pytest.mark.parametrize("metric", [0, 1, 2], ids=["l2", "ip", "cos"])
@pytest.mark.parametrize("nan_rank", [0, 1], ids=["nan_low", "nan_high"])
def test_trap_nan_rows_beside_a_short_rank(metric, nan_rank):
    """NaN rows (scored NaN, kept by one GPU after every number) on one rank, another rank with fewer than k rows: the NaN
    rows are real entries, not padding, and the padding follows them.  nan_high puts the short rank below the NaN rows, so
    that its padding meets them under the lower ranks' <= rule"""
    rng = np.random.default_rng(3)
    d = 8
    x0 = rng.standard_normal((4, d)).astype(np.float32)
    x0[1, 2] = np.nan
    x0[3, 0] = np.nan
    x1 = rng.standard_normal((3, d)).astype(np.float32)
    q = rng.standard_normal((2, d)).astype(np.float32)
    parts = [(x0, [1, 2, 3, 4]), (x1, [5, 6, 7])]
    if nan_rank == 1:
        parts = parts[::-1]
    shards = [_flat(d, metric, xs, ids) for xs, ids in parts]
    one = _flat(d, metric, np.concatenate([p[0] for p in parts]), sum((p[1] for p in parts), []))
    for k in (10, 600):
        got = emulate(shards, q, k)
        same(got, one.batch_search(q, k))
        # (cosine clamps the NaN similarity, so those rows come back with a number, still after every finite row)
        assert (np.sort(got[1][:, 5:7], axis=1) == [2, 4]).all() and (got[1][:, 7:] == -1).all()
        assert metric == 2 or np.isnan(got[0][:, 5:7]).all()


def test_trap_zero_distance_sign():
    """A zero inner-product distance comes back as -0 from the flat kind and +0 from IVF-Flat, in k-NN, beyond 512 and in
    range search, as on one GPU"""
    d = 8
    x = np.zeros((3, d), np.float32); x[0, 1] = 1.0; x[1, 2] = 2.0; x[2, 0] = 1.0
    q = np.zeros((1, d), np.float32); q[0, 0] = 1.0                    # orthogonal to rows 0 and 1: a zero dot
    coarse = np.eye(2, d, dtype=np.float32)
    for kind in ("flat", "ivfflat"):
        mk = (lambda xs, ids: _flat(d, 1, xs, ids)) if kind == "flat" else (lambda xs, ids: _ivfflat(d, 1, coarse, 2, xs, ids))
        a, b = mk(x[:1], [1]), mk(x[1:], [2, 3])
        one = mk(x, [1, 2, 3])
        for k in (3, 600):
            got = emulate([a, b], q, k, nprobe=2)
            same(got, one.batch_search(q, k, nprobe=2))
            zeros = got[0][0][got[0][0] == 0]
            assert zeros.size == 2 and np.all(np.signbit(zeros) == (kind == "flat"))
        got = emulate([a, b], q, nprobe=2, radius=0.0)
        same(got, one.range_search(q, 0.0, nprobe=2))
        assert got[1].size == 3 and np.all(np.signbit(got[1][got[1] == 0]) == (kind == "flat"))


# ----------------------------------------------------------------------------------------------------- refusals, world 1
def _comm1():
    import torch
    torch.cuda.init()
    from vectorindex_b200.index import Comm
    return Comm(0, 1, Comm.unique_id())


def _status(fn, *args):
    return int(getattr(_L(), fn)(*args))


def test_refusals():
    """on every rank alike, before any exchange: an IVF-Flat handle without centroids, list bounds for a flat index, an
    IVF-PQ handle as before (untrained: the same code and message)"""
    from vectorindex_b200 import _lib
    from vectorindex_b200.index import IVFIndex, IVFPQIndex
    comm = _comm1()
    d, n, nq, k = 8, 50, 3, 4
    rng = np.random.default_rng(0)
    x = rng.standard_normal((n, d)).astype(np.float32)
    ids = np.arange(n, dtype=np.int64)
    q = x[:nq].copy()
    dd, di = np.empty((nq, k), np.float32), np.empty((nq, k), np.int64)
    res = C.c_void_p(0)
    bounds = np.array([0, 4], np.int64)
    ivf = IVFIndex(d, "euclidean", nlist=4, nprobe=2)
    for fn, args in (("vix_sharded_add", (ivf._h, comm._c, None, _lib.ptr(x), _lib.ptr(ids), C.c_int64(n))),
                     ("vix_sharded_search", (ivf._h, comm._c, _lib.ptr(q), C.c_int64(nq), C.c_int(k), C.c_int(0), _lib.ptr(dd),
                                             _lib.ptr(di))),
                     ("vix_sharded_range_search", (ivf._h, comm._c, _lib.ptr(q), C.c_int64(nq), C.c_float(1.0), C.c_int(0),
                                                   None, C.c_int64(0), C.c_int(0), C.byref(res)))):
        assert _status(fn, *args) == ERR_NOT_TRAINED
        assert "IVF-Flat" in _lib.last_error()
    flat = _flat(d, 0)
    assert _status("vix_sharded_add", flat._h, comm._c, _lib.ptr(bounds), _lib.ptr(x), _lib.ptr(ids), C.c_int64(n)) == ERR_INVALID_PARAM
    assert flat.count == 0
    bad = ids.copy(); bad[7] = -1
    assert _status("vix_sharded_add", flat._h, comm._c, None, _lib.ptr(x), _lib.ptr(bad), C.c_int64(n)) == ERR_INVALID_PARAM
    assert flat.count == 0
    pq = IVFPQIndex(d, "euclidean", nlist=4, nprobe=2, m=4)
    assert _status("vix_sharded_search", pq._h, comm._c, _lib.ptr(q), C.c_int64(nq), C.c_int(k), C.c_int(0), _lib.ptr(dd),
                   _lib.ptr(di)) == ERR_NOT_TRAINED
    assert "needs a trained IVF-PQ index" in _lib.last_error()
    comm.close()


@pytest.mark.parametrize("metric", [0, 1, 2], ids=["l2", "ip", "cos"])
def test_kinds_single_rank(metric):
    """One rank through the real entry points (a one-rank communicator: vix_sharded_add files the rows through the collective
    path, index_add_assigned_locked for IVF-Flat) and through the Python classes, equal to the one-GPU index"""
    from vectorindex_b200 import _lib
    from vectorindex_b200.index import ShardedFlatIndex, ShardedIVFFlatIndex, IVFIndex
    comm = _comm1()
    n, d, nq = 3000, 16, 21
    x, ids, q = _data(300 + metric, n, d, nq)
    trainer = IVFIndex(d, METRICS[metric], nlist=16, nprobe=4)
    trainer.optimize(x)
    coarse = trainer.get_coarse()
    filt = _filter(ids, 9)
    for kind in ("flat", "ivfflat"):
        one = _flat(d, metric, x, ids) if kind == "flat" else _ivfflat(d, metric, coarse, 4, x, ids)
        sh = _flat(d, metric) if kind == "flat" else _ivfflat(d, metric, coarse, 4)
        _lib.check(_L().vix_sharded_add(sh._h, comm._c, None, _lib.ptr(x), _lib.ptr(ids), C.c_int64(n)))
        py = ShardedFlatIndex(d, METRICS[metric]) if kind == "flat" else ShardedIVFFlatIndex(d, METRICS[metric], 16, 4)
        if kind == "ivfflat":
            py.set_coarse(coarse)
        py.add(x, ids)
        for k in (10, 700):
            ref = one.batch_search(q, k)
            dd, di = np.empty((nq, k), np.float32), np.empty((nq, k), np.int64)
            _lib.check(_L().vix_sharded_search(sh._h, comm._c, _lib.ptr(q), C.c_int64(nq), C.c_int(k), C.c_int(0), _lib.ptr(dd),
                                               _lib.ptr(di)))
            same((dd, di), ref)
            same(py.batch_search(q, k), ref)
            same(py.batch_search(q, k, filter=filt), one.batch_search(q, k, filter=filt))
        radius = _radii(one.batch_search(q, 32)[0])[1]
        same(py.range_search(q, radius), one.range_search(q, radius))
        assert py.remove(ids[:5]) == one.batch_remove(ids[:5])
        same(py.batch_search(q, 10), one.batch_search(q, 10))
    comm.close()


# ---------------------------------------------------------------------------------------------------- several processes
def _ngpus():
    import torch
    return torch.cuda.device_count()


def _launch(world, no_p2p, port):
    env = dict(os.environ)
    env.pop("VIX_NO_P2P", None)
    env.pop("VIX_TC_SCAN", None)
    if no_p2p:
        env["VIX_NO_P2P"] = "1"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr",
           "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "mp_sharded_kinds.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=1200, env=env)
    assert out.returncode == 0, out.stdout[-6000:] + out.stderr[-4000:]
    for case in ("flat", "ivfflat", "refusals"):
        assert f"ok {case}:" in out.stdout, f"case {case} did not report: " + out.stdout[-3000:]
    assert f"kinds: world {world}, 3 of 3 cases ok" in out.stdout, out.stdout[-3000:]


@pytest.mark.parametrize("no_p2p", [False, True], ids=["peer", "nccl"])
@pytest.mark.parametrize("size", ["two", "all"])
def test_sharded_kinds_ranks(size, no_p2p):
    n = _ngpus()
    if n < 2:
        pytest.skip("needs two GPUs")
    if size == "all" and n <= 2:
        pytest.skip("the box has two GPUs: the two-rank launch covers it")
    _launch(2 if size == "two" else min(n, 8), no_p2p, 29581 + 2 * (size == "all") + no_p2p)


def test_sharded_kinds_ranks_single_rank():
    """One rank: the Python classes and the harness on a one-rank process group."""
    if _ngpus() >= 2:
        pytest.skip("the multi-rank launches cover it")
    _launch(1, False, 29585)


def test_c_host_sharded_kinds(tmp_path):
    """flat and IVF-Flat add, search and range search through the C ABI from a plain C11 host, one rank"""
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else shutil.which("gcc")
    if cc is None:
        pytest.skip("no C compiler")
    lib_dir = os.path.join(ROOT, "vectorindex_b200")
    exe = str(tmp_path / "sharded_kinds_smoke")
    subprocess.check_call([cc, "-std=c11", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "c", "sharded_kinds_smoke.c"), "-o", exe, "-L", lib_dir,
                           "-lvindex_b200", "-Wl,-rpath," + lib_dir, "-lm"])
    import torch  # noqa: F401 -- the process that runs the host finds libnccl where torch keeps it
    nccl = _nccl_path()
    env = dict(os.environ)
    if nccl:
        env["VIX_NCCL_PATH"] = nccl
    out = subprocess.run([exe], capture_output=True, text=True, timeout=300, env=env)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "sharded kinds ok" in out.stdout, out.stdout


def _nccl_path():
    """the libnccl.so.2 torch loaded (a plain C host names it through VIX_NCCL_PATH)"""
    try:
        with open("/proc/self/maps") as f:
            for line in f:
                if "libnccl.so" in line:
                    return line.split()[-1]
    except OSError:
        pass
    return None
