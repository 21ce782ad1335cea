"""k-NN search beyond VIX_MAX_K (512 < k <= VIX_MAX_K_LARGE): the exact two-pass route over the range-search scans.

The route seeds a per-query bound on the distance word, collects every candidate within it through the kind's range
kernel, sorts each row by (distance, id) and cuts it at k.  A case checks
  - flat and IVF-Flat (L2, IP): the oracle's own k-NN search at the same k, ids equal, distance bits equal (IVF-Flat
    cosine: the oracle to 1e-5);
  - the prefix property on every kind, metric and filter mode: search(k)[:, :k2] is search(k2), bit for bit, for k2 = 512
    (the untouched fused route) and 512 < k2 < k;
  - IVF-PQ: a range search whose radius is the row's k-th distance begins with the row, and the oracle agrees outside the
    RTOL band;
  - fewer candidates than k, ties across the k-th position, a NaN query component, adversarial (loose) seeds with a
    first capacity that is too small, filters, the re-rank, and the interface's edges.
The "[vix knn]" line of VIX_SCAN_DEBUG=1 shows the route taken: seed entries, collected entries, passes.
"""
import re
import zlib

import numpy as np
import pytest

from pq_ref64 import RTOL
from test_gpu_parity import bits
from test_range_search import cut, filters, ranged
from test_scan_edges import PQ, TIE_STEP, decode, queries_near, random_pq
from vectorindex_b200 import _lib

gpu = pytest.mark.gpu
KNN = re.compile(r"\[vix knn\] kind (\w+), kernel (fast G \d|generic|ivfflat|flat), filter (\d), k (\d+), seed (\d+), "
                 r"total (\d+), passes (\d), max_row (\d+)")
METRICS = {0: "euclidean", 1: "dotProduct", 2: "cosine"}
ERR_INVALID_K = -2
KS = [513, 1000, 2048, 4097]


# ------------------------------------------------------------------------------------------------ building blocks
def knn(mp, capfd, fn, lines=1):
    """fn() under VIX_SCAN_DEBUG=1 -> (its result, the fields of its [vix knn] lines; `lines` of them expected)"""
    capfd.readouterr()
    mp.setenv("VIX_SCAN_DEBUG", "1")
    try:
        out = fn()
    finally:
        mp.delenv("VIX_SCAN_DEBUG")
    err = capfd.readouterr().err
    found = KNN.findall(err)
    assert len(found) == lines, f"{len(found)} [vix knn] lines"
    assert "[vix range]" not in err
    return out, [dict(kind=g[0], kernel=g[1], filter=int(g[2]), k=int(g[3]), seed=int(g[4]), total=int(g[5]),
                      passes=int(g[6]), max_row=int(g[7])) for g in found]


def same(got, want, cols=None):
    """ids and distance bits equal (over the first `cols` columns of both)"""
    gd, gi = (np.asarray(a) for a in got)
    wd, wi = (np.asarray(a) for a in want)
    if cols is not None:
        gd, gi, wd, wi = gd[:, :cols], gi[:, :cols], wd[:, :cols], wi[:, :cols]
    assert gi.shape == wi.shape
    assert np.array_equal(gi, wi), f"ids differ in {int((gi != wi).sum())} places"
    assert np.array_equal(bits(gd), bits(wd)), "distance bits differ"


def padded(gd, gi, n):
    """columns from n on are padding: id -1, NaN"""
    assert (gi[:, n:] == -1).all() and np.isnan(gd[:, n:]).all()


def prefix_property(search, k):
    """search(k)[:, :k2] == search(k2) for k2 = 512 (the fused route) and one k2 between 512 and k"""
    full = search(k)
    same(full, search(512), cols=512)
    if k > 514:
        k2 = (512 + k) // 2
        same(full, search(k2), cols=k2)
    return full


def oracle_ids(oi, ids):
    return np.where(oi >= 0, ids[np.maximum(oi, 0)], -1)


def filtered_top(od, oi, k, keep):
    """the oracle's full ranking with the filter cut, the first k, padded"""
    nq = od.shape[0]
    wd = np.full((nq, k), np.nan, np.float32)
    wi = np.full((nq, k), -1, np.int64)
    for r in range(nq):
        sel = (oi[r] >= 0) & keep(oi[r])
        d, i = od[r][sel][:k], oi[r][sel][:k]
        wd[r, :d.size], wi[r, :i.size] = d, i
    return wd, wi


# ------------------------------------------------------------------------------------------------ 1. oracle parity, flat
@gpu
@pytest.mark.parametrize("metric,d", [(0, 40), (0, 300), (1, 40), (2, 36)], ids=["l2", "l2_dot", "ip", "cosine"])
def test_flat_oracle(oracle, monkeypatch, capfd, metric, d):
    """A flat index (ids a permutation: ties fall to the smaller row, as in the fused search) and vix_flat_search_f32:
    the oracle's k-NN at the same k, ids and bits; k = 4097 on 8000 rows takes the route without a seed."""
    from vectorindex_b200 import kernels
    from vectorindex_b200.index import FlatIndex
    rng = np.random.default_rng(100 + d + metric)
    n, nq = 8000, 6
    xb = rng.standard_normal((n, d)).astype(np.float32)
    q = rng.standard_normal((nq, d)).astype(np.float32)
    ids = rng.permutation(n).astype(np.int64) * 2 + 7
    idx = FlatIndex(d, METRICS[metric])
    idx.batch_insert(xb, ids)
    for k in KS:
        od, oi, _ = oracle.flat_search(q, xb, k, metric)
        got, lines = knn(monkeypatch, capfd, lambda: idx.batch_search(q, k))
        assert lines[0]["kind"] == "flat" and lines[0]["kernel"] == "flat" and lines[0]["k"] == k
        assert (lines[0]["seed"] > 0) == (n > 2 * k)
        same(got, (od, oracle_ids(oi, ids)))
        raw, _ = knn(monkeypatch, capfd, lambda: kernels.flat_search_f32(q, xb, k, metric))
        same(raw, (od, oi))


# ------------------------------------------------------------------------------------------------ 1. oracle parity, IVF-Flat
@gpu
@pytest.mark.parametrize("metric", [0, 1, 2], ids=["l2", "ip", "cosine"])
def test_ivfflat_oracle(oracle, monkeypatch, capfd, metric):
    """Trained IVF-Flat: the oracle's k-NN at the same k (cosine: to 1e-5 and the prefix property); before optimize() the
    linear scan through the flat engine, the oracle's flat k-NN."""
    from vectorindex_b200.index import IVFIndex
    rng = np.random.default_rng(200 + metric)
    n, d, kc, nq, nprobe = 9000, 32, 24, 8, 8
    xb = rng.standard_normal((n, d)).astype(np.float32)
    q = rng.standard_normal((nq, d)).astype(np.float32)
    coarse = np.ascontiguousarray(xb[rng.choice(n, kc, replace=False)])
    ids = np.arange(n, dtype=np.int64) * 3 + 1
    lin = IVFIndex(d, METRICS[metric], nlist=kc, nprobe=nprobe)
    lin.batch_insert(xb, ids)
    ivf = IVFIndex(d, METRICS[metric], nlist=kc, nprobe=nprobe)
    ivf.set_coarse(coarse)
    ivf.batch_insert(xb, ids)
    asg = oracle.assign(xb, coarse)[0] if metric == 0 else oracle.assign_metric(xb, coarse, metric)
    off, order = oracle.build_lists(asg, kc)
    for k in KS:
        od, oi, _ = oracle.flat_search(q, xb, k, metric)
        got, lines = knn(monkeypatch, capfd, lambda: lin.batch_search(q, k))
        assert lines[0]["kind"] == "ivfflat" and lines[0]["kernel"] == "flat"
        same(got, (od, oracle_ids(oi, ids)))
        od, oi = oracle.ivfflat_search(q, coarse, off, xb[order], ids[order], nprobe, k, metric)
        got, lines = knn(monkeypatch, capfd, lambda: ivf.batch_search(q, k))
        assert lines[0]["kind"] == "ivfflat" and lines[0]["kernel"] == "ivfflat" and lines[0]["seed"] > 0
        if metric != 2:
            same(got, (od, oi))
        else:
            gd, gi = got
            assert np.array_equal(gi >= 0, oi >= 0)
            np.testing.assert_allclose(gd[gi >= 0], od[oi >= 0], rtol=1e-5, atol=1e-5)
            prefix_property(lambda kk: ivf.batch_search(q, kk), k)


# ------------------------------------------------------------------------------------------------ 2. prefix property
@gpu
@pytest.mark.parametrize("fname", ["none", "allow", "deny"])
@pytest.mark.parametrize("kind", ["flat", "ivfflat", "ivfpq"])
@pytest.mark.parametrize("metric", [0, 1, 2], ids=["l2", "ip", "cosine"])
def test_prefix_property(oracle, kind, metric, fname):
    """search(k)[:, :512] == search(512) (the fused route) and search(k1)[:, :k2] == search(k2), every kind, metric, filter"""
    from vectorindex_b200.index import FlatIndex, IVFIndex
    if kind == "ivfpq" and metric == 2:
        pytest.skip("IVF-PQ indexes are L2 / inner product")
    rng = np.random.default_rng(zlib.crc32(f"{kind}/{metric}/{fname}".encode()))
    nq = 10
    if kind == "ivfpq":
        P = random_pq(oracle, rng, 16, 2, rng.integers(300, 600, 16), metric=metric)
        idx, q, cap = P.idx, queries_near(rng, P, rng.integers(0, 16, nq)), int(P.lids.max()) + 1
        search = lambda k, f: idx.batch_search(q, k, nprobe=8, filter=f)
    else:
        n, d = 6000, 24
        xb = rng.standard_normal((n, d)).astype(np.float32)
        q = rng.standard_normal((nq, d)).astype(np.float32)
        ids = rng.permutation(n).astype(np.int64) + 3
        idx = FlatIndex(d, METRICS[metric]) if kind == "flat" else IVFIndex(d, METRICS[metric], nlist=16, nprobe=6)
        if kind == "ivfflat":
            idx.set_coarse(np.ascontiguousarray(xb[rng.choice(n, 16, replace=False)]))
        idx.batch_insert(xb, ids)
        cap = n + 3
        search = lambda k, f: idx.batch_search(q, k, filter=f)
    filt = filters(cap, rng)[fname]
    for k in (1000, 2500):
        prefix_property(lambda kk: search(kk, filt), k)


@gpu
def test_prefix_property_list_major(oracle, monkeypatch):
    """IVF-PQ on an L2 d = 2 m batch large enough for the list-major tensor-core scan: the route (which never takes that
    scan) against k = 512 under the default route selection and with VIX_TC_SCAN=1"""
    rng = np.random.default_rng(31)
    kc, nq = 32, 1200
    P = random_pq(oracle, rng, 48, 2, rng.integers(500, 900, kc))
    q = queries_near(rng, P, rng.integers(0, kc, nq))
    for tc in (None, "1"):
        if tc is None:
            monkeypatch.delenv("VIX_TC_SCAN", raising=False)
        else:
            monkeypatch.setenv("VIX_TC_SCAN", tc)
        prefix_property(lambda kk: P.idx.batch_search(q, kk, nprobe=8), 1500)


# ------------------------------------------------------------------------------------------------ 3. IVF-PQ against range search
PQ_CASES = {"fast16": (16, 256, "fast G 1"), "fast48": (48, 256, "fast G 3"), "generic12": (12, 256, "generic"),
            "ks16_m16": (16, 16, "generic")}


@gpu
@pytest.mark.parametrize("metric", [0, 1], ids=["l2", "ip"])
@pytest.mark.parametrize("name", list(PQ_CASES))
def test_ivfpq_range_and_oracle(oracle, monkeypatch, capfd, name, metric):
    """Each row is the start of a range search whose radius is its own k-th distance, bit for bit; the oracle agrees
    outside a band of relative width RTOL around that distance."""
    m, ks, kernel = PQ_CASES[name]
    rng = np.random.default_rng(zlib.crc32(f"pq/{name}/{metric}".encode()))
    kc, nq, nprobe, k = 12, 6, 6, 1000
    P = random_pq(oracle, rng, m, 2, rng.integers(300, 500, kc), ks=ks, metric=metric)
    q = queries_near(rng, P, rng.integers(0, kc, nq))
    (gd, gi), lines = knn(monkeypatch, capfd, lambda: P.idx.batch_search(q, k, nprobe=nprobe))
    assert lines[0]["kind"] == "ivfpq" and lines[0]["kernel"] == kernel
    od, oi, _ = P.oracle(oracle, q, nprobe, int(P.off[-1]))
    scale = float(np.nanmax(np.abs(od[oi >= 0])))
    for r in range(nq):
        radius = gd[r, k - 1]
        (lims, dist, ids), route = ranged(monkeypatch, capfd, lambda: P.idx.range_search(q[r:r + 1], radius, nprobe=nprobe))
        assert route["kernel"] == kernel
        assert np.array_equal(ids[:k], gi[r]) and np.array_equal(bits(dist[:k]), bits(gd[r]))
        band = RTOL * max(abs(float(radius)), scale if metric == 1 else 0.0)
        sel = oi[r] >= 0
        want = set(oi[r][sel & (od[r] < radius - band)].tolist())
        assert want <= set(gi[r].tolist())
        assert set(gi[r][gd[r] < radius - band].tolist()) <= set(oi[r][sel & (od[r] <= radius + band)].tolist())


# ------------------------------------------------------------------------------------------------ 4. fewer candidates than k
@gpu
def test_fewer_candidates_than_k(oracle, monkeypatch, capfd):
    """nprobe 1 on IVF-PQ and IVF-Flat, and a flat index of fewer rows than k: the range search with radius +inf, then
    padding"""
    from vectorindex_b200.index import FlatIndex, IVFIndex
    rng = np.random.default_rng(41)
    P = random_pq(oracle, rng, 16, 2, rng.integers(100, 300, 10))
    q = queries_near(rng, P, rng.integers(0, 10, 5))
    xb = rng.standard_normal((700, 32)).astype(np.float32)
    fl = FlatIndex(32)
    fl.batch_insert(xb)
    ivf = IVFIndex(32, nlist=8, nprobe=1)
    ivf.set_coarse(np.ascontiguousarray(xb[:8]))
    ivf.batch_insert(xb)
    qf = rng.standard_normal((5, 32)).astype(np.float32)
    for search, rs, k in ((lambda k: P.idx.batch_search(q, k, nprobe=1), lambda: P.idx.range_search(q, np.inf, nprobe=1), 600),
                          (lambda k: ivf.batch_search(qf, k), lambda: ivf.range_search(qf, np.inf), 800),
                          (lambda k: fl.batch_search(qf, k), lambda: fl.range_search(qf, np.inf), 1000)):
        (gd, gi), lines = knn(monkeypatch, capfd, lambda: search(k))
        lims, dist, ids = rs()
        for r in range(gd.shape[0]):
            c = int(lims[r + 1] - lims[r])
            assert c < k
            assert np.array_equal(gi[r, :c], ids[lims[r]:lims[r + 1]])
            assert np.array_equal(bits(gd[r, :c]), bits(dist[lims[r]:lims[r + 1]]))
            padded(gd[r:r + 1], gi[r:r + 1], c)
        assert lines[0]["total"] == int(lims[-1])


# ------------------------------------------------------------------------------------------------ 5. ties
@gpu
@pytest.mark.parametrize("name", ["fast48", "generic12"])
def test_ties_across_the_kth(oracle, monkeypatch, capfd, name):
    """3000 copies of one code in one list (grid-valued: every sum exact), one id stored twice; k = 1000 cuts through the
    tie: the smallest ids, the twice-stored one twice.  The same list probed twice: every entry comes back twice."""
    m = 48 if name == "fast48" else 12
    dsub = 2
    rng = np.random.default_rng(500 + m)
    kc, ntied, k = 8, 3000, 1000
    g = lambda a: (np.round(np.asarray(a) / TIE_STEP) * TIE_STEP).astype(np.float32)
    coarse = g(3.0 * rng.standard_normal((kc, m * dsub)))
    cb = g(0.5 * rng.standard_normal((m, 256, dsub)))
    code = rng.integers(0, 256, (1, m), dtype=np.uint8)
    tied = rng.permutation(ntied).astype(np.int64) * 7 + 1_000_000
    dup = int(tied.min())
    other = rng.integers(100, 200, kc - 1)
    assign = np.concatenate([np.zeros(ntied + 1, np.int32), np.repeat(np.arange(1, kc, dtype=np.int32), other)])
    codes = np.concatenate([np.repeat(code, ntied + 1, 0), rng.integers(0, 256, (int(other.sum()), m), dtype=np.uint8)])
    ids = np.concatenate([tied, [dup], np.arange(int(other.sum()), dtype=np.int64)])
    P = PQ(oracle, coarse, cb, assign, codes, ids)
    q = g(coarse[0] + decode(cb, code) + 0.05 * rng.standard_normal((4, m * dsub)))
    probes = np.concatenate([np.zeros((4, 1), np.int32), 1 + rng.permutation(kc - 1)[None, :3].repeat(4, 0).astype(np.int32)], 1)
    (gd, gi), _ = knn(monkeypatch, capfd, lambda: P.idx.search_with_probes(q, k, probes))
    assert (gi == np.sort(np.concatenate([tied, [dup]]))[:k]).all()
    assert (bits(gd) == bits(gd[:, :1])).all()
    same((gd, gi), P.idx.search_with_probes(q, 512, probes), cols=512)
    twice = np.concatenate([probes[:, 1:2], probes[:, 1:2]], 1)
    c = 2 * int(P.lens[probes[0, 1]])
    (td, ti), _ = knn(monkeypatch, capfd, lambda: P.idx.search_with_probes(q, c + 600, twice))
    assert np.array_equal(ti[:, :c:2], ti[:, 1:c:2]) and (np.diff(ti[:, :c:2], axis=1) != 0).all()
    padded(td, ti, c)


@gpu
def test_flat_duplicate_rows(oracle, monkeypatch, capfd):
    """A flat index of duplicated vectors (each row stored twice, ids reversed): ties go to the smaller row, both copies
    come back, the oracle's bits"""
    from vectorindex_b200.index import FlatIndex
    rng = np.random.default_rng(51)
    base = rng.standard_normal((2000, 16)).astype(np.float32)
    xb = np.concatenate([base, base])
    ids = np.arange(4000, dtype=np.int64)[::-1].copy()
    q = rng.standard_normal((4, 16)).astype(np.float32)
    idx = FlatIndex(16)
    idx.batch_insert(xb, ids)
    for k in (601, 1000):
        od, oi, _ = oracle.flat_search(q, xb, k, 0)
        (gd, gi), _ = knn(monkeypatch, capfd, lambda: idx.batch_search(q, k))
        same((gd, gi), (od, oracle_ids(oi, ids)))
        assert (bits(gd[:, 0:k - 1:2]) == bits(gd[:, 1:k:2])).all()


# ------------------------------------------------------------------------------------------------ 6. NaN query component
@gpu
def test_nan_query_component(oracle, monkeypatch, capfd):
    """A query with a NaN component: every distance is NaN, the row is the k smallest candidates by id (flat: rows), as the
    fused route returns at k = 512"""
    from vectorindex_b200.index import FlatIndex, IVFIndex
    rng = np.random.default_rng(61)
    xb = rng.standard_normal((3000, 24)).astype(np.float32)
    q = rng.standard_normal((3, 24)).astype(np.float32)
    q[1, 5] = np.nan
    fl = FlatIndex(24)
    fl.batch_insert(xb)
    gd, gi = prefix_property(lambda k: fl.batch_search(q, k), 900)
    assert np.array_equal(gi[1], np.arange(900)) and np.isnan(gd[1]).all()
    ivf = IVFIndex(24, nlist=8, nprobe=8)
    ivf.set_coarse(np.ascontiguousarray(xb[:8]))
    ivf.batch_insert(xb, np.arange(3000, dtype=np.int64)[::-1].copy())
    prefix_property(lambda k: ivf.batch_search(q, k), 900)
    P = random_pq(oracle, rng, 16, 2, rng.integers(300, 500, 8))
    qp = queries_near(rng, P, rng.integers(0, 8, 3))
    qp[2, 0] = np.nan
    prefix_property(lambda k: P.idx.batch_search(qp, k, nprobe=8), 900)


# ------------------------------------------------------------------------------------------------ 7. loose seeds
@gpu
def test_loose_seed_flat(oracle, monkeypatch, capfd):
    """Rows added cluster by cluster, the queries at the first cluster: one seed block holds the whole top k, the bound is
    loose (T >> k) and the first capacity too small (two passes; the next call one), the answer still the oracle's"""
    from vectorindex_b200.index import FlatIndex
    rng = np.random.default_rng(71)
    n, d, nq, k = 16384, 16, 32, 1000                    # (the collect outgrows the first capacity, 64 k entries)
    centers = np.zeros((4, d), np.float32)
    centers[:, 0] = [0.0, 40.0, 80.0, 120.0]
    xb = (np.repeat(centers, n // 4, 0) + rng.standard_normal((n, d))).astype(np.float32)
    q = (rng.standard_normal((nq, d)) * 0.1).astype(np.float32)
    idx = FlatIndex(d)
    idx.batch_insert(xb)
    od, oi, _ = oracle.flat_search(q, xb, k, 0)
    first, l1 = knn(monkeypatch, capfd, lambda: idx.batch_search(q, k))
    assert l1[0]["total"] > 4 * k * nq and l1[0]["passes"] == 2
    same(first, (od, oi))
    second, l2 = knn(monkeypatch, capfd, lambda: idx.batch_search(q, k))
    assert l2[0]["passes"] == 1
    same(second, first)


@gpu
@pytest.mark.parametrize("name", ["fast16", "generic12", "ivfflat"])
def test_loose_seed_far_first_probe(oracle, monkeypatch, capfd, name):
    """The first probed list is far from the query and holds more than 2 k vectors: the seed's bound comes from it alone,
    the collect keeps the whole near list (1500) and k of the far one; the answer is the one with the near list first"""
    from vectorindex_b200.index import IVFIndex
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    k, nq = 600, 4
    if name == "ivfflat":
        d, kc = 16, 6
        coarse = np.zeros((kc, d), np.float32)
        coarse[:, 0] = 30.0 * np.arange(kc)
        sizes = [2000, 300, 300, 300, 300, 1500]
        xb = (np.repeat(coarse, sizes, 0) + rng.standard_normal((sum(sizes), d))).astype(np.float32)
        idx = IVFIndex(d, nlist=kc, nprobe=4)
        idx.set_coarse(coarse)
        idx.batch_insert(xb)
        q = (coarse[5] + 0.1 * rng.standard_normal((nq, d))).astype(np.float32)
        from vectorindex_b200.index import IVFPQIndex      # (search_with_probes drives any trained IVF handle)
        run = lambda kk, pr: IVFPQIndex.search_with_probes(idx, q, kk, pr)
    else:
        m = 16 if name == "fast16" else 12
        P = random_pq(oracle, rng, m, 2, np.array([2000, 300, 300, 300, 300, 1500]), spread=5.0)
        q = queries_near(rng, P, np.full(nq, 5))
        run = lambda kk, pr: P.idx.search_with_probes(q, kk, pr)
    far = np.tile(np.array([[0, 5, 4, 3]], np.int32), (nq, 1))
    near = np.tile(np.array([[5, 4, 3, 0]], np.int32), (nq, 1))
    (gd, gi), lines = knn(monkeypatch, capfd, lambda: run(k, far))
    assert lines[0]["seed"] >= 2000 * nq and lines[0]["total"] >= 3 * k * nq
    want, _ = knn(monkeypatch, capfd, lambda: run(k, near))
    same((gd, gi), want)
    same((gd, gi), run(512, far), cols=512)


# ------------------------------------------------------------------------------------------------ 8. filters
@gpu
@pytest.mark.parametrize("fname", ["allow", "deny"])
@pytest.mark.parametrize("kind", ["flat", "ivfflat", "ivfpq"])
def test_filters_against_oracle(oracle, monkeypatch, capfd, kind, fname):
    """k = 1000 with an allow and a deny list: the oracle's full ranking with the filter cut (IVF-PQ: outside the RTOL band,
    distances to RTOL)"""
    from vectorindex_b200.index import FlatIndex, IVFIndex
    rng = np.random.default_rng(zlib.crc32(f"filt/{kind}/{fname}".encode()))
    k, nq = 1000, 6
    if kind == "ivfpq":
        P = random_pq(oracle, rng, 16, 2, rng.integers(400, 700, 10))
        q = queries_near(rng, P, rng.integers(0, 10, nq))
        filt = filters(int(P.lids.max()) + 1, rng)[fname]
        (gd, gi), lines = knn(monkeypatch, capfd, lambda: P.idx.batch_search(q, k, nprobe=6, filter=filt))
        od, oi, _ = P.oracle(oracle, q, 6, int(P.off[-1]))
        wd, wi = filtered_top(od, oi, k, filt.test)
        scale = float(np.nanmax(np.abs(od[oi >= 0])))
        for r in range(nq):
            ok = gi[r] >= 0
            assert np.array_equal(ok, wi[r] >= 0)
            kth = float(gd[r][ok][-1])
            band = RTOL * max(abs(kth), 1.0)
            assert set(wi[r][wd[r] < kth - band].tolist()) <= set(gi[r].tolist())
            common, ia, ib = np.intersect1d(gi[r][ok], wi[r][wi[r] >= 0], return_indices=True)
            np.testing.assert_allclose(gd[r][ok][ia], wd[r][ib], rtol=RTOL, atol=RTOL)
    else:
        n, d = 7000, 24
        xb = rng.standard_normal((n, d)).astype(np.float32)
        q = rng.standard_normal((nq, d)).astype(np.float32)
        ids = rng.permutation(n).astype(np.int64) * 2 + 1
        filt = filters(int(ids.max()) + 1, rng)[fname]
        if kind == "flat":
            idx = FlatIndex(d)
            idx.batch_insert(xb, ids)
            od, oi, _ = oracle.flat_search(q, xb, n, 0)
            oi = oracle_ids(oi, ids)
        else:
            coarse = np.ascontiguousarray(xb[rng.choice(n, 12, replace=False)])
            idx = IVFIndex(d, nlist=12, nprobe=6)
            idx.set_coarse(coarse)
            idx.batch_insert(xb, ids)
            asg = oracle.assign(xb, coarse)[0]
            off, order = oracle.build_lists(asg, 12)
            od, oi = oracle.ivfflat_search(q, coarse, off, xb[order], ids[order], 6, n, 0)
        (gd, gi), lines = knn(monkeypatch, capfd, lambda: idx.batch_search(q, k, filter=filt))
        same((gd, gi), filtered_top(od, oi, k, filt.test))
    assert lines[0]["filter"] == 1


# ------------------------------------------------------------------------------------------------ 9. rerank
@gpu
@pytest.mark.parametrize("metric", [0, 1], ids=["l2", "ip"])
def test_rerank_wide_shortlist(oracle, metric):
    """rerank_r in {1024, 4096}: the exact re-rank of the search(rerank_r) candidates, and the oracle's composition (its
    IVF-PQ top-rerank_r, re-scored exactly)"""
    from vectorindex_b200 import kernels
    rng = np.random.default_rng(90 + metric)
    m, kc, nq, k = 16, 16, 8, 50
    sizes = rng.integers(400, 700, kc)
    n = int(sizes.sum())
    P = random_pq(oracle, rng, m, 2, sizes, metric=metric, ids=np.arange(n, dtype=np.int64))
    xb = rng.standard_normal((n, 2 * m)).astype(np.float32)
    q = queries_near(rng, P, rng.integers(0, kc, nq))
    for r in (1024, 4096):
        sc, si = P.idx.batch_search_rerank(q, k, xb, r, nprobe=8)
        cd, ci = P.idx.batch_search(q, r, nprobe=8)
        same((sc, si), kernels.rerank_exact_topk(q, ci, xb, k, metric))
        od, oi, _ = P.oracle(oracle, q, 8, r)
        wd, wi = kernels.rerank_exact_topk(q, oi, xb, k, metric)
        for row in range(nq):
            assert len(set(si[row].tolist()) & set(wi[row].tolist())) >= k - 2


# ------------------------------------------------------------------------------------------------ 10. edges
@gpu
def test_limits_pointers_async_stats(oracle, monkeypatch, capfd):
    """k = VIX_MAX_K_LARGE accepted, one more refused; host and device pointers and asynchronous mode give the same bits;
    stats mark the route; k <= 512 prints no [vix knn] line"""
    import torch
    from vectorindex_b200.index import FlatIndex, IVFPQIndex
    assert _lib.MAX_K_LARGE == 16384 and _lib.MAX_K == 512
    rng = np.random.default_rng(101)
    P = random_pq(oracle, rng, 16, 2, rng.integers(1500, 2500, 12))
    q = queries_near(rng, P, rng.integers(0, 12, 5))
    (gd, gi), lines = knn(monkeypatch, capfd, lambda: P.idx.batch_search(q, _lib.MAX_K_LARGE, nprobe=12))
    assert lines[0]["k"] == _lib.MAX_K_LARGE
    n = int(P.off[-1])
    padded(gd, gi, min(n, _lib.MAX_K_LARGE))
    with pytest.raises(_lib.VectorIndexError) as e:
        P.idx.batch_search(q, _lib.MAX_K_LARGE + 1, nprobe=12)
    assert e.value.status == ERR_INVALID_K
    fl = FlatIndex(16)
    fl.batch_insert(rng.standard_normal((3000, 16)).astype(np.float32))
    with pytest.raises(_lib.VectorIndexError) as e:
        fl.batch_search(q[:, :16], _lib.MAX_K_LARGE + 1)
    assert e.value.status == ERR_INVALID_K
    # host vs device pointers, asynchronous mode
    k = 2000
    host = P.idx.batch_search(q, k, nprobe=6)
    dq = torch.from_numpy(q).cuda()
    dev = P.idx.batch_search(dq, k, nprobe=6)
    same((dev[0].cpu().numpy(), dev[1].cpu().numpy()), host)
    L = _lib.lib()
    was = L.vix_get_async()
    L.vix_set_async(1)
    try:
        asy = P.idx.batch_search(dq, k, nprobe=6)
        torch.cuda.synchronize()
    finally:
        L.vix_set_async(was)
    same((asy[0].cpu().numpy(), asy[1].cpu().numpy()), host)
    # stats and probes
    gd, gi, gp, st = P.idx.batch_search(q, k, nprobe=6, return_probes=True, stats=True)
    same((gd, gi), host)
    assert np.array_equal(gp, P.probes(q, 6))
    assert st.scan_path == 2 and st.merge_candidates >= nq_min(k, P, gp) and st.ms_total > 0 and st.cycles_scan == 0
    wd, wi, wst = P.idx.search_with_probes(q, k, gp, stats=True)
    same((wd, wi), host)
    assert wst.scan_path == 2
    # k <= 512: the fused route, no [vix knn] line
    capfd.readouterr()
    monkeypatch.setenv("VIX_SCAN_DEBUG", "1")
    P.idx.batch_search(q, 512, nprobe=6)
    fl.batch_search(q[:, :16], 512)
    monkeypatch.delenv("VIX_SCAN_DEBUG")
    assert "[vix knn]" not in capfd.readouterr().err


def nq_min(k, P, probes):
    """sum over queries of min(k, candidates of its probes)"""
    return sum(min(k, int(P.lens[np.unique(row[row >= 0])].sum())) for row in probes)
