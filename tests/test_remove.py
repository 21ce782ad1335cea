"""Removing vectors by id (vix_index_remove / batch_remove) on every index kind.

The property every case checks: after remove(S) an index is indistinguishable from one built by adding only the rows whose
id is not in S, in the same order and with the same ids -- count, exported lists (offsets, codes, ids, assignments), list
sizes, the list-major decode layout, and search results (ids and distance bits; both IVF-PQ scans where the list-major one
can serve the index; filtered and re-ranked searches too).  Further: the IVF-PQ search after a removal against the oracle,
lists that cross a chunk boundary as they shrink, removals interleaved with adds and searches, removing everything, a
removal that matches nothing (no list rebuild follows), invalid input, automatic ids, an index of 2^21 rows, and the
sharded index.
"""
import ctypes as C
import os
import subprocess
import sys
import types

import numpy as np
import pytest

from conftest import ROOT
from test_gpu_parity import _make_ivfpq_problem, bits
from test_tc_scan_edges import Lists, both_paths, queries_near
from test_tc_scan_layout import expected_tc_codes, tc_codes
from vectorindex_b200 import _lib

pytestmark = pytest.mark.gpu

LIST_MAJOR_M = (16, 32, 48, 64)
K = 10


# ------------------------------------------------------------------------------------------------ building blocks
def export(idx):
    """(offsets, codes or None, ids, assignments in add order) of an IVF index, through vix_index_export_lists"""
    L = _lib.lib()
    kc = C.c_int(0)
    _lib.check(L.vix_index_get_coarse(idx._h, None, C.byref(kc)))
    n = idx.count
    off = np.empty(kc.value + 1, np.int64)
    ids = np.empty(n, np.int64)
    asg = np.empty(n, np.int32)
    codes = np.empty((n, idx.code_bytes), np.uint8) if hasattr(idx, "code_bytes") else None
    _lib.check(L.vix_index_export_lists(idx._h, _lib.ptr(off), _lib.ptr(codes), _lib.ptr(ids), _lib.ptr(asg)))
    return off, codes, ids, asg


def ids_with_duplicates(rng, n):
    """n ids = 3 p + 5 in random order, a twentieth of them stored a second (or third) time"""
    ids = rng.permutation(n).astype(np.int64) * 3 + 5
    dup = rng.choice(n, n // 20, replace=False)
    ids[dup] = ids[rng.integers(0, n, dup.size)]
    return ids


def removal_set(rng, ids, share=5):
    """a fifth of the stored ids, three ids stored more than once, ids that are not stored, and repeats -- shuffled"""
    u, c = np.unique(ids, return_counts=True)
    pick = rng.choice(u, u.size // share, replace=False)
    absent = np.array([0, 1, 3, 4, 2 ** 32 - 2], np.int64)            # never 3 p + 5 for the p used here
    s = np.concatenate([pick, u[c > 1][:3], absent, pick[:10], u[c > 1][:1]])
    assert (c > 1).sum() >= 3 and not np.isin(absent, ids).any()
    return rng.permutation(s)


class Problem:
    """rows of one index kind: vectors (FLAT / IVF_FLAT) or lists, codes (IVF-PQ); build(keep) adds the kept ones in order"""

    def __init__(self, oracle, case, rng, n=3000):
        self.oracle, self.case, self.rng = oracle, case, rng
        self.kind = case.split("_")[0]
        self.ids = ids_with_duplicates(rng, n)
        if self.kind in ("flat", "ivfflat"):
            self.d, self.kc = 32, 16
            centres = 3.0 * rng.standard_normal((8, self.d))
            self.x = (centres[rng.integers(0, 8, n)] + rng.standard_normal((n, self.d))).astype(np.float32)
            self.coarse = np.ascontiguousarray(self.x[rng.choice(n, self.kc, replace=False)])
            self.metric = "dotProduct" if case == "flat_ip" else "euclidean"
            self.q = (centres[rng.integers(0, 8, 64)] + rng.standard_normal((64, self.d))).astype(np.float32)
            return
        self.m = {"pq_m16": 16, "pq_m48": 48, "pq_m12": 12, "pq_ip": 48, "pq_u4": 16}[case]
        self.ks = 16 if case == "pq_u4" else 256
        self.metric = "dotProduct" if case == "pq_ip" else "euclidean"
        self.kc, self.d = 12, 2 * self.m
        self.coarse = (rng.standard_normal((self.kc, self.d)) * 2.0).astype(np.float32)
        self.cb = (rng.standard_normal((self.m, self.ks, 2)) * 0.5).astype(np.float32)
        self.assign = rng.integers(0, self.kc, n).astype(np.int32)
        self.codes = rng.integers(0, 256, (n, self.m // 2 if self.ks == 16 else self.m), dtype=np.uint8)
        home = rng.integers(0, self.kc, 200)
        if self.ks == 256:                                                  # (what queries_near reads of a Lists)
            self.q = queries_near(rng, types.SimpleNamespace(coarse=self.coarse, cb=self.cb, m=self.m), home)
        else:
            self.q = (self.coarse[home] + 0.5 * rng.standard_normal((home.size, self.d))).astype(np.float32)
        self.xb = rng.standard_normal((int(self.ids.max()) + 1, self.d)).astype(np.float32)   # re-rank reader: row = id

    @property
    def list_major(self):
        return self.kind == "pq" and self.metric == "euclidean" and self.ks == 256 and self.m in LIST_MAJOR_M

    def build(self, keep=None, coarse_first=True):
        from vectorindex_b200.index import FlatIndex, IVFIndex, IVFPQIndex
        sel = slice(None) if keep is None else keep
        if self.kind == "flat":
            idx = FlatIndex(self.d, self.metric)
            idx.batch_insert(self.x[sel], self.ids[sel])
        elif self.kind == "ivfflat":
            idx = IVFIndex(self.d, self.metric, nlist=self.kc, nprobe=4)
            if coarse_first:
                idx.set_coarse(self.coarse)
            idx.batch_insert(self.x[sel], self.ids[sel])
        elif self.ks == 256:
            idx = Lists(self.oracle, self.coarse, self.cb, self.assign[sel], self.codes[sel], self.ids[sel],
                        metric=self.metric, nprobe=4).idx
        else:
            idx = IVFPQIndex(self.d, self.metric, nlist=self.kc, nprobe=4, m=self.m, ks=16)
            idx.set_coarse(self.coarse)
            idx.set_codebooks(self.cb)
            idx.add_encoded(self.assign[sel], self.codes[sel], self.ids[sel])
        return idx


def search(mp, capfd, idx, q, k, list_major):
    """batch_search; through both IVF-PQ scans (equal bits, the list-major one proven taken) where it can serve the index"""
    if list_major:
        d, i, _ = both_paths(mp, capfd, lambda: idx.batch_search(q, k))
        return d, i
    return idx.batch_search(q, k)


def assert_same_index(a, b, mp, capfd, q, k=K, lists=True, list_major=False, m=None, removed=None, xb=None):
    """a (after removals) indistinguishable from b (rebuilt): count, exported lists, list sizes, decode layout, searches"""
    from vectorindex_b200.index import IDFilter
    assert a.count == b.count
    if lists:
        for x, y in zip(export(a), export(b)):
            assert (x is None and y is None) or np.array_equal(x, y)
        assert np.array_equal(a.list_sizes(), b.list_sizes())
    if hasattr(a, "code_bytes"):
        ta, tb = tc_codes(a), tc_codes(b)
        assert np.array_equal(ta, tb)
        if list_major:
            off, codes, _, _ = export(a)
            assert ta.size > 0 and np.array_equal(ta, expected_tc_codes(off, codes, m))
        else:
            assert ta.size == 0
    da, ia = search(mp, capfd, a, q, k, list_major)
    db, ib = search(mp, capfd, b, q, k, list_major)
    assert np.array_equal(ia, ib), "ids differ from the rebuilt index"
    assert np.array_equal(bits(da), bits(db)), "distance bits differ from the rebuilt index"
    outs = [ia]
    cap = int(max(ia.max(), 1)) + 100
    f = IDFilter(cap, "deny").set(np.random.default_rng(1).choice(cap, cap // 3, replace=False))
    fa, fb = a.batch_search(q, k, filter=f), b.batch_search(q, k, filter=f)
    assert np.array_equal(fa[1], fb[1]) and np.array_equal(bits(fa[0]), bits(fb[0]))
    outs.append(fa[1])
    if xb is not None:
        ra, rb = a.batch_search_rerank(q, k, xb, 40), b.batch_search_rerank(q, k, xb, 40)
        assert np.array_equal(ra[1], rb[1]) and np.array_equal(bits(ra[0]), bits(rb[0]))
        outs.append(ra[1])
    if removed is not None:
        for o in outs:
            assert not np.isin(o, removed).any(), "a removed id was returned"
    return da, ia


# ------------------------------------------------------------------------------------------------ 1. remove == rebuild
CASES = ["flat_l2", "flat_ip", "ivfflat_linear", "ivfflat_lists", "pq_m16", "pq_m48", "pq_m12", "pq_ip", "pq_u4"]


@pytest.mark.parametrize("case", CASES)
def test_remove_equals_rebuild(oracle, monkeypatch, capfd, case):
    """A = all rows, then remove(S); B = the rows whose id is not in S, added in the same order.  S mixes stored ids, ids
    stored twice, ids that are not stored and repeats; IVF-PQ indexes get it as a CUDA tensor."""
    import torch
    rng = np.random.default_rng(CASES.index(case) + 40)
    P = Problem(oracle, case, rng)
    S = removal_set(rng, P.ids)
    keep = ~np.isin(P.ids, S)
    linear = case == "ivfflat_linear"                                   # rows stored before the index has centroids
    a = P.build(coarse_first=not linear)
    got = a.batch_remove(torch.from_numpy(S).cuda() if P.kind == "pq" else S)
    assert got == int((~keep).sum()) and a.count == int(keep.sum())
    b = P.build(keep, coarse_first=not linear)
    pq = P.kind == "pq"
    kw = dict(list_major=P.list_major, m=getattr(P, "m", None), removed=S, xb=P.xb if pq else None)
    assert_same_index(a, b, monkeypatch, capfd, P.q, lists=P.kind != "flat" and not linear, **kw)
    if linear:                                                          # then filed into lists (optimize() with centroids)
        a.set_coarse(P.coarse)
        b.set_coarse(P.coarse)
        assert_same_index(a, b, monkeypatch, capfd, P.q, **kw)


# ------------------------------------------------------------------------------------------------ 2. against the oracle
@pytest.mark.parametrize("m", [16, 12])
def test_ivfpq_search_after_removal_matches_oracle(oracle, m):
    """encoded vectors (batch_insert), a third of them removed: the search is the oracle's over the exported lists"""
    from vectorindex_b200.index import IVFPQIndex
    n, d, kc, nq, k, nprobe = 6000, 48, 32, 40, 10, 6
    xb, q, coarse, cb, norms = _make_ivfpq_problem(oracle, n, d, m, kc, nq, seed=5)
    ids = np.arange(n, dtype=np.int64) * 2 + 1
    idx = IVFPQIndex(d, "euclidean", nlist=kc, nprobe=nprobe, m=m)
    idx.set_coarse(coarse)
    idx.set_codebooks(cb, norms)
    idx.batch_insert(xb, ids)
    idx.batch_search(q, k)                                              # lists built before the removal
    S = np.random.default_rng(3).choice(ids, n // 3, replace=False)
    assert idx.batch_remove(S) == n // 3
    gd, gi = idx.batch_search(q, k)
    off, codes, lids, _ = idx.export_lists()
    assert lids.size == n - n // 3 and not np.isin(lids, S).any()
    od, oi, _ = oracle.ivfpq_search(q, coarse, cb, norms, off, codes, lids, m, 256, nprobe, k, 0)
    np.testing.assert_allclose(gd, od, rtol=1e-5, equal_nan=True)
    same = np.mean([len(set(gi[r]) & set(oi[r])) / k for r in range(nq)])
    assert same > 0.995
    assert not np.isin(gi, S).any()


# ------------------------------------------------------------------------------------------------ 3. chunk boundaries
@pytest.mark.parametrize("m", LIST_MAJOR_M)
def test_lists_shrink_across_chunk_boundaries(oracle, monkeypatch, capfd, m):
    """lists of 33, 32, 1, 4097 and 40 vectors lose one each of the first four: 32, 31, 0, 4096 -- a chunk of 32 slots
    less for three of them.  The decode layout is the stated mapping of the exported lists and the rebuilt index's; both
    scans return the rebuilt index's bits."""
    rng = np.random.default_rng(200 + m)
    sizes = np.array([33, 32, 1, 4097, 40])
    kc = sizes.size
    coarse = (rng.standard_normal((kc, 2 * m)) * 2.0).astype(np.float32)
    cb = (rng.standard_normal((m, 256, 2)) * 0.5).astype(np.float32)
    assign = np.repeat(np.arange(kc, dtype=np.int32), sizes)
    codes = rng.integers(0, 256, (assign.size, m), dtype=np.uint8)
    ids = rng.permutation(assign.size).astype(np.int64) * 7 + 1
    A = Lists(oracle, coarse, cb, assign, codes, ids, nprobe=2)
    starts = np.concatenate([[0], np.cumsum(sizes)])
    pick = np.array([starts[0] + 32, starts[1] + 5, starts[2], starts[3] + 4096])   # last, middle, only, last
    assert A.idx.batch_remove(ids[pick]) == 4
    assert np.array_equal(A.idx.list_sizes(), [32, 31, 0, 4096, 40])
    keep = np.ones(assign.size, bool)
    keep[pick] = False
    B = Lists(oracle, coarse, cb, assign[keep], codes[keep], ids[keep], nprobe=2)
    q = queries_near(rng, A, rng.integers(0, kc, 200))
    assert_same_index(A.idx, B.idx, monkeypatch, capfd, q, list_major=True, m=m, removed=ids[pick])
    assert tc_codes(A.idx).size == (32 + 32 + 0 + 4096 + 64) * m


# ------------------------------------------------------------------------------------------------ 4. order of operations
@pytest.mark.parametrize("order", ["before_first_search", "after_search", "then_add", "twice"])
def test_order_of_operations(oracle, monkeypatch, capfd, order):
    """remove while the lists are still unbuilt, after a search, followed by an add, and twice in a row: each equals the
    index rebuilt from what remains"""
    from vectorindex_b200.index import IVFPQIndex
    rng = np.random.default_rng(300 + len(order))
    P = Problem(oracle, "pq_m48", rng)
    a = IVFPQIndex(P.d, "euclidean", nlist=P.kc, nprobe=4, m=P.m)
    a.set_coarse(P.coarse)
    a.set_codebooks(P.cb, oracle.pq_centroid_sq(P.cb, P.m, 256, 2))
    a.add_encoded(P.assign, P.codes, P.ids)                             # lists dirty from here on
    S = removal_set(rng, P.ids)
    if order == "after_search":
        a.batch_search(P.q, K)
    a.batch_remove(S)
    keep = ~np.isin(P.ids, S)
    rows = [P.assign[keep], P.codes[keep], P.ids[keep]]
    if order == "twice":
        left = P.ids[keep]
        S2 = rng.choice(left, left.size // 4, replace=False)
        assert a.batch_remove(S2) == int(np.isin(left, S2).sum())
        k2 = ~np.isin(rows[2], S2)
        rows = [r[k2] for r in rows]
        S = np.concatenate([S, S2])
    if order == "then_add":
        na = 500
        more = [rng.integers(0, P.kc, na).astype(np.int32), rng.integers(0, 256, (na, P.m), dtype=np.uint8),
                10 ** 7 + np.arange(na, dtype=np.int64)]
        a.add_encoded(*more)
        rows = [np.concatenate([r, s]) for r, s in zip(rows, more)]
    b = Lists(oracle, P.coarse, P.cb, *rows, nprobe=4).idx
    assert_same_index(a, b, monkeypatch, capfd, P.q, list_major=True, m=P.m, removed=S, xb=None)


# ------------------------------------------------------------------------------------------------ 5. remove everything
@pytest.mark.parametrize("case", ["flat_l2", "ivfflat_linear", "ivfflat_lists", "pq_m48", "pq_ip", "pq_u4"])
def test_remove_everything(oracle, case):
    """count 0, every search returns id -1 / NaN (plain and filtered), and the index takes new rows afterwards"""
    from vectorindex_b200.index import IDFilter
    rng = np.random.default_rng(7)
    P = Problem(oracle, case, rng, n=1000)
    linear = case == "ivfflat_linear"
    a = P.build(coarse_first=not linear)
    assert a.batch_remove(P.ids) == 1000 and a.count == 0
    for dd, ii in (a.batch_search(P.q, K), a.batch_search(P.q, K, filter=IDFilter(100, "deny"))):
        assert (ii == -1).all() and np.isnan(dd).all()
    if P.kind != "flat" and not linear:
        off, _, lids, _ = export(a)
        assert (off == 0).all() and lids.size == 0 and (a.list_sizes() == 0).all()
    if P.kind == "pq":
        assert tc_codes(a).size == 0
        a.add_encoded(P.assign[:50], P.codes[:50], P.ids[:50])
    else:
        a.batch_insert(P.x[:50], P.ids[:50])
    assert a.count == 50
    dd, ii = a.batch_search(P.q, K, nprobe=P.kc)
    assert (ii >= 0).all() and np.isin(ii, P.ids[:50]).all()


# ------------------------------------------------------------------------------------------------ 6. nothing matches
def test_removal_that_matches_nothing_changes_nothing(oracle):
    """ids that are not stored: 0 removed, and the next search launches exactly the kernels of the search before it (no
    list rebuild) and returns the same bits"""
    rng = np.random.default_rng(8)
    P = Problem(oracle, "pq_m48", rng)
    a = P.build()
    L = _lib.lib()
    d0, i0 = a.batch_search(P.q, K)
    L.vix_kernel_launches(1)
    d0, i0 = a.batch_search(P.q, K)
    before = int(L.vix_kernel_launches(1))
    assert a.batch_remove(np.array([0, 1, 3, 2 ** 32 - 2], np.int64)) == 0
    assert a.batch_remove(np.zeros(0, np.int64)) == 0
    L.vix_kernel_launches(1)
    d1, i1 = a.batch_search(P.q, K)
    assert int(L.vix_kernel_launches(0)) == before
    assert np.array_equal(i0, i1) and np.array_equal(bits(d0), bits(d1))


# ------------------------------------------------------------------------------------------------ 7. invalid input
@pytest.mark.parametrize("case", ["flat_l2", "pq_m48"])
def test_invalid_input_removes_nothing(oracle, case):
    import torch
    from vectorindex_b200 import VectorIndexError
    rng = np.random.default_rng(9)
    P = Problem(oracle, case, rng, n=500)
    a = P.build()
    d0, i0 = a.batch_search(P.q, K)
    stored = int(P.ids[0])
    for bad in (-1, 2 ** 32 - 1):
        for arr in (np.array([stored, bad], np.int64), torch.tensor([stored, bad], dtype=torch.int64, device="cuda")):
            with pytest.raises(VectorIndexError) as e:
                a.batch_remove(arr)
            assert e.value.kind == "invalidParameter"
            assert a.count == 500
    L = _lib.lib()
    removed = C.c_int64(-7)
    assert L.vix_index_remove(a._h, None, C.c_int64(3), C.byref(removed)) == -3 and removed.value == 0
    assert L.vix_index_remove(a._h, None, C.c_int64(0), C.byref(removed)) == 0 and removed.value == 0
    assert L.vix_index_remove(a._h, None, C.c_int64(0), None) == 0
    d1, i1 = a.batch_search(P.q, K)
    assert np.array_equal(i0, i1) and np.array_equal(bits(d0), bits(d1))


# ------------------------------------------------------------------------------------------------ 8. automatic ids
def test_automatic_ids_after_removal(oracle):
    """10 rows without ids get 0..9; after remove(3) two more get 10 and 11, not 9 and 10.  Without a removal automatic
    ids continue from the count; clear starts them at 0 and an import at the imported count."""
    from vectorindex_b200.index import FlatIndex, IVFIndex, IVFPQIndex
    rng = np.random.default_rng(10)
    d = 16
    x = rng.standard_normal((12, d)).astype(np.float32)
    for make in (lambda: FlatIndex(d), lambda: IVFIndex(d, nlist=3, nprobe=3)):
        idx = make()
        if isinstance(idx, IVFIndex):
            idx.set_coarse(x[:3].copy())
        idx.batch_insert(x[:10])
        assert idx.remove(3) == 1 and idx.remove(3) == 0
        idx.batch_insert(x[10:])
        _, i = idx.batch_search(x, 1, nprobe=3)                        # every stored row is its own nearest neighbour
        assert np.delete(i[:, 0], 3).tolist() == [0, 1, 2, 4, 5, 6, 7, 8, 9, 10, 11]
        assert i[3, 0] != 3 and idx.count == 11
        if isinstance(idx, IVFIndex):
            assert sorted(export(idx)[2].tolist()) == [0, 1, 2, 4, 5, 6, 7, 8, 9, 10, 11]
    plain = FlatIndex(d)
    plain.batch_insert(x[:5])
    plain.batch_insert(x[5:8])
    assert plain.batch_search(x[:8], 1)[1][:, 0].tolist() == list(range(8))
    plain.clear()
    plain.batch_insert(x[8:10])
    assert plain.batch_search(x[8:10], 1)[1][:, 0].tolist() == [0, 1]
    # IVF-PQ: import of 7 rows, then two rows without ids get 7 and 8
    m = 8
    pq = IVFPQIndex(d, nlist=2, nprobe=2, m=m)
    pq.set_coarse(x[:2].copy())
    pq.set_codebooks((0.3 * rng.standard_normal((m, 256, d // m))).astype(np.float32))
    pq.import_lists(np.array([0, 4, 7], np.int64), rng.integers(0, 256, (7, m), dtype=np.uint8), np.arange(100, 107, dtype=np.int64))
    pq.batch_insert(x[:2])
    assert sorted(pq.export_lists()[2].tolist()) == [7, 8] + list(range(100, 107))


# ------------------------------------------------------------------------------------------------ 9. size
def test_large_index_removal_equals_numpy_compaction(oracle, monkeypatch, capfd):
    """2^21 rows at m = 48 (grids of many blocks, a scan of more than one tile): a random tenth removed; the export equals
    a numpy compaction of the export before, the decode layout its stated mapping, and searches the rebuilt index's"""
    rng = np.random.default_rng(11)
    n, m, kc = 1 << 21, 48, 256
    coarse = (rng.standard_normal((kc, 2 * m)) * 2.0).astype(np.float32)
    cb = (rng.standard_normal((m, 256, 2)) * 0.5).astype(np.float32)
    assign = rng.integers(0, kc, n).astype(np.int32)
    codes = rng.integers(0, 256, (n, m), dtype=np.uint8)
    ids = rng.permutation(n).astype(np.int64)
    A = Lists(oracle, coarse, cb, assign, codes, ids, nprobe=4)
    off0, codes0, lids0, asg0 = A.off, A.codes, A.lids, A.idx.export_lists()[3]
    S = rng.choice(n, n // 10, replace=False).astype(np.int64)
    assert A.idx.batch_remove(S) == n // 10
    off, codes1, lids, asg = A.idx.export_lists()
    kl = ~np.isin(lids0, S)
    lens = np.bincount(np.repeat(np.arange(kc), np.diff(off0))[kl], minlength=kc)
    assert np.array_equal(off, np.concatenate([[0], np.cumsum(lens)]))
    assert np.array_equal(codes1, codes0[kl]) and np.array_equal(lids, lids0[kl])
    assert np.array_equal(asg, asg0[~np.isin(ids, S)])
    assert np.array_equal(tc_codes(A.idx), expected_tc_codes(off, codes1, m))
    keep = ~np.isin(ids, S)
    B = Lists(oracle, coarse, cb, assign[keep], codes[keep], ids[keep], nprobe=4)
    q = queries_near(rng, A, rng.integers(0, kc, 2000))
    da, ia, _ = both_paths(monkeypatch, capfd, lambda: A.idx.batch_search(q, K))
    db, ib = B.idx.batch_search(q, K)
    assert np.array_equal(ia, ib) and np.array_equal(bits(da), bits(db))
    assert not np.isin(ia, S).any()


# ------------------------------------------------------------------------------------------------ 10. sharded
def test_sharded_single_rank_remove_equals_plain_index(oracle):
    """ShardedIVFPQIndex.remove over one rank whose rows came through vix_sharded_add on a single-rank Comm: the count and
    vix_sharded_search equal a plain index after the same removal"""
    from vectorindex_b200.index import Comm, IVFPQIndex, ShardedIVFPQIndex
    rng = np.random.default_rng(12)
    n, d, m, kc, nq, k = 5000, 64, 16, 16, 77, 10
    xb = rng.standard_normal((n, d)).astype(np.float32)
    q = rng.standard_normal((nq, d)).astype(np.float32)
    coarse = rng.standard_normal((kc, d)).astype(np.float32)
    cb = (0.4 * rng.standard_normal((m, 256, d // m))).astype(np.float32)
    a, b = (IVFPQIndex(d, "euclidean", nlist=kc, nprobe=4, m=m) for _ in range(2))
    for idx in (a, b):
        idx.set_coarse(coarse)
        idx.set_codebooks(cb)
    ids = ids_with_duplicates(rng, n)
    a.batch_insert(xb, ids)
    comm = Comm(0, 1, Comm.unique_id())
    L = _lib.lib()
    _lib.check(L.vix_sharded_add(b._h, comm._c, None, _lib.ptr(xb), _lib.ptr(ids), C.c_int64(n)))
    S = removal_set(rng, ids)
    sh = ShardedIVFPQIndex.wrap(b, kc, 4)
    want = a.batch_remove(S)
    assert sh.remove(S) == want > 0 and a.count == b.count
    dist, out = np.empty((nq, k), np.float32), np.empty((nq, k), np.int64)
    _lib.check(L.vix_sharded_search(b._h, comm._c, _lib.ptr(q), C.c_int64(nq), C.c_int(k), C.c_int(0), _lib.ptr(dist), _lib.ptr(out)))
    ad, ai = a.batch_search(q, k)
    assert np.array_equal(ai, out) and np.array_equal(bits(ad), bits(dist))
    assert not np.isin(out, S).any()
    comm.close()


def test_two_ranks_remove_under_torchrun():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29541", os.path.join(ROOT, "tests", "mp_remove_check.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=dict(os.environ))
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "ok remove" in out.stdout
