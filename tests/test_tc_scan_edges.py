"""Edges of the list-major tensor-core IVF-PQ scan (vix_ivfpq_tc.cu), each with the route it must take proven.

Every case builds its lists directly (set_coarse / set_codebooks / add_encoded, no training) and, where the probes matter,
sets them too (search_with_probes), so the route of every query is known before the search runs.  A case then checks:
  - the route: vix_scan_tc_launches() tells whether the list-major scan ran; the line launch_ivfpq_scan_tc prints under
    VIX_TC_SCAN_DEBUG=1 gives the queries handed back to the query-major scan, the finalists (most per query) and the log
    capacity, and that no pipeline wait timed out;
  - bit equality with the query-major scan (vix_ivfpq_scan.cu), which the rest of the suite pins to the oracle;
  - a float64 reference of ||q - c_l - r^||^2 that shares no code with either scan or the oracle (pq_ref64.ref64).
"""
import re

import numpy as np
import pytest

from pq_ref64 import RTOL, assert_ref64, ref64
from test_gpu_parity import _make_ivfpq_problem, assert_topk_close, bits
from vectorindex_b200 import _lib

pytestmark = pytest.mark.gpu

TINY = float(np.finfo(np.float32).tiny)
LOG_CAP = 4096            # records of one filter warp's log at small batches (launch_ivfpq_scan_tc: at least 4096)
ROUTE = re.compile(r"\[vix tc scan\] nq (\d+), handed back (\d+), candidates (\d+) \(max (\d+) per query; (\d+) per log\), "
                   r"error (\d+)")


# ------------------------------------------------------------------------------------------------ building blocks
class Lists:
    """An IVF-PQ index (L2, ks = 256, dsub = 2) whose lists are given: coarse [kc x d], codebooks [m x 256 x 2], and per
    stored vector its list, code and id.  Keeps the exported list layout for the float64 reference."""

    def __init__(self, oracle, coarse, cb, assign, codes, ids, metric="euclidean", nprobe=8):
        from vectorindex_b200.index import IVFPQIndex
        self.coarse, self.cb = np.ascontiguousarray(coarse, np.float32), np.ascontiguousarray(cb, np.float32)
        self.kc, self.d = self.coarse.shape
        self.m = self.cb.shape[0]
        self.norms = oracle.pq_centroid_sq(self.cb, self.m, 256, 2)
        self.idx = IVFPQIndex(self.d, metric, nlist=self.kc, nprobe=nprobe, m=self.m)
        self.idx.set_coarse(self.coarse)
        self.idx.set_codebooks(self.cb, self.norms)
        self.rows = (np.zeros(0, np.int32), np.zeros((0, self.m), np.uint8), np.zeros(0, np.int64))
        self.add(assign, codes, ids)

    def add(self, assign, codes, ids):
        add = (np.asarray(assign, np.int32), np.asarray(codes, np.uint8), np.asarray(ids, np.int64))
        self.idx.add_encoded(*add)
        self.rows = tuple(np.concatenate([a, b]) for a, b in zip(self.rows, add))
        self.off, self.codes, self.lids, _ = self.idx.export_lists()
        self.lens = np.diff(self.off)

    def like(self, oracle, cb=None, metric="euclidean"):
        """the same lists (assignments, codes, ids) under other codebooks or another metric"""
        return Lists(oracle, self.coarse, self.cb if cb is None else cb, *self.rows, metric=metric)

    def search(self, q, k, probes=None):
        return (lambda: self.idx.search_with_probes(q, k, probes)) if probes is not None else (lambda: self.idx.batch_search(q, k))

    def ref64(self, q, probes, k):
        return ref64(q, self.coarse, self.cb, probes, self.off, self.codes, self.lids, k)

    def oracle(self, oracle, q, nprobe, k):
        return oracle.ivfpq_search(q, self.coarse, self.cb, self.norms, self.off, self.codes, self.lids, self.m, 256, nprobe, k, 0)

    def first_list(self, probes):
        """per query the list the seed scans: the first probe position whose list holds vectors (-1: none)"""
        out = np.full(len(probes), -1)
        for r, row in enumerate(probes):
            for l in row:
                if 0 <= l < self.kc and self.lens[l] > 0:
                    out[r] = l
                    break
        return out

    def flagged(self, probes, k):
        """per query whether the list-major scan hands it to the query-major one: its seed list holds fewer than k vectors
        (or there is none).  Its pairs never reach tc_scan_kernel."""
        f = self.first_list(probes)
        return (f < 0) | (self.lens[np.maximum(f, 0)] < k)

    def handed_back(self, probes, k):
        return int(self.flagged(probes, k).sum())


def tc_launches():
    return int(_lib.lib().vix_scan_tc_launches())


def route(mp, capfd, fn):
    """fn() once with VIX_TC_SCAN_DEBUG=1 -> (its result, (H, T, M, C, E)): queries handed back, finalists, most finalists
    of one query, records per log, error flag -- from the line launch_ivfpq_scan_tc prints to stderr.  E must be 0."""
    capfd.readouterr()
    mp.setenv("VIX_TC_SCAN_DEBUG", "1")
    try:
        out = fn()
    finally:
        mp.delenv("VIX_TC_SCAN_DEBUG")
    lines = ROUTE.findall(capfd.readouterr().err)
    assert len(lines) == 1, f"{len(lines)} list-major launches reported"
    h, t, mx, c, e = (int(v) for v in lines[0][1:])
    assert e == 0, "a pipeline wait of tc_scan_kernel timed out"
    return out, (h, t, mx, c, e)


def both_paths(mp, capfd, search, tc=True):
    """search() through the query-major scan (VIX_TC_SCAN=0), then with the list-major one forced (=1).  The launch counter
    shows that only the second run took it (none, tc=False); ids and distance bits of the two runs are equal.
    Returns (dist, ids, route of the second run or None)."""
    mp.setenv("VIX_TC_SCAN", "0")
    n0 = tc_launches()
    d0, i0 = search()
    assert tc_launches() == n0
    mp.setenv("VIX_TC_SCAN", "1")
    if tc:
        (d1, i1), r = route(mp, capfd, search)
    else:
        (d1, i1), r = search(), None
    assert tc_launches() == n0 + (1 if tc else 0), "list-major scan taken" if not tc else "list-major scan not taken"
    assert np.array_equal(i0, i1), "ids differ from the query-major scan"
    assert np.array_equal(bits(d0), bits(d1)), "distance bits differ from the query-major scan"
    return d1, i1, r


def decoded(cb, codes):
    m = cb.shape[0]
    return cb[np.arange(m), np.asarray(codes, np.intp)].reshape(len(codes), -1)


def on_grid(a, step):
    return (np.round(np.asarray(a, np.float64) / step) * step).astype(np.float32)


def random_lists(oracle, rng, m, sizes, spread=1.0, res=0.5, ids=None, step=None):
    """lists of random codes around Gaussian centroids (coordinates ~ N(0, spread^2)), residual codebooks ~ N(0, res^2);
    step: every centroid and codebook value a multiple of it"""
    kc, d = len(sizes), 2 * m
    coarse = (rng.standard_normal((kc, d)) * spread).astype(np.float32)
    cb = (rng.standard_normal((m, 256, 2)) * res).astype(np.float32)
    if step:
        coarse, cb = on_grid(coarse, step), on_grid(cb, step)
    assign = np.repeat(np.arange(kc, dtype=np.int32), sizes)
    codes = rng.integers(0, 256, (assign.size, m), dtype=np.uint8)
    if ids is None:
        ids = rng.permutation(assign.size).astype(np.int64) * 3 + 5                 # not monotone in the list order
    return Lists(oracle, coarse, cb, assign, codes, ids)


def queries_near(rng, L, home, noise=0.2):
    """one query per entry of home: the centroid plus a decoded random code plus noise"""
    r = decoded(L.cb, rng.integers(0, 256, (len(home), L.m)))
    return (L.coarse[home] + r + noise * rng.standard_normal(r.shape)).astype(np.float32)


def nearest_probes(q, coarse, nprobe, lists=None):
    """per query the nprobe nearest of `lists` (default all), nearest first"""
    lists = np.arange(len(coarse)) if lists is None else np.asarray(lists)
    dd = ((q.astype(np.float64)[:, None, :] - coarse[lists].astype(np.float64)[None]) ** 2).sum(-1)
    return lists[np.argsort(dd, axis=1, kind="stable")[:, :nprobe]].astype(np.int32)


# ------------------------------------------------------------------------------------------------ 1. scale invariance
def _grid_problem(rng, m, kc, n, nq, step):
    """every value a multiple of step = 2^-7 with 2 <= max |x| < 4: each product, sum and distance of the scans is a
    multiple of step^2 = 2^-14 (or 0), so scaling all inputs by 2^s scales every fp32 intermediate exactly as long as
    step^2 2^2s is normal"""
    g = lambda a, sd: np.clip(np.round(a * sd / step) * step, -3.0, 3.0).astype(np.float32)
    coarse = g(rng.standard_normal((kc, 2 * m)), 1.0)
    cb = g(rng.standard_normal((m, 256, 2)), 0.5)
    cb[0, 0, 0] = 3.0
    assign = rng.integers(0, kc, n).astype(np.int32)
    codes = rng.integers(0, 256, (n, m), dtype=np.uint8)
    home = rng.integers(0, kc, nq)
    q = g(coarse[home] + decoded(cb, rng.integers(0, 256, (nq, m))) + 0.3 * rng.standard_normal((nq, 2 * m)), 1.0)
    q[0, 0] = 3.0
    return coarse, cb, assign, codes, q


@pytest.mark.parametrize("s", [-56, -52, -40, -24, 0, 24, 40])
def test_power_of_two_scale_invariance(oracle, monkeypatch, capfd, s):
    """Queries, centroids and codebooks times 2^s, the same codes: ids equal to s = 0 and distance bits those of
    ldexp(d0, 2 s), on both scans and the oracle.  The tensor-core filter works in units of s_q s_c (the fp16 scales of
    queries and codebooks, 2^(10 - e) each): at s = -56 both are 2^64, whose product is not an fp32 number."""
    m, kc, n, nq, k, nprobe = 48, 32, 6000, 300, 10, 6
    step = 2.0 ** -7
    coarse, cb, assign, codes, q = _grid_problem(np.random.default_rng(11), m, kc, n, nq, step)
    ids = np.random.default_rng(12).permutation(n).astype(np.int64)
    for a in (q, coarse, cb):
        assert (np.ldexp(a.astype(np.float64), 7) % 1 == 0).all() and 2.0 <= np.abs(a).max() < 4.0
    L0 = Lists(oracle, coarse, cb, assign, codes, ids)
    _, _, probes = L0.idx.batch_search(q, k, nprobe=nprobe, return_probes=True)
    od0, oi0, op = L0.oracle(oracle, q, nprobe, k)
    assert np.array_equal(probes, op)
    assert L0.handed_back(probes, k) == 0
    d0, i0, r0 = both_paths(monkeypatch, capfd, L0.search(q, k, probes))
    assert r0[0] == 0
    assert_topk_close(d0, i0, od0, oi0)
    ref = L0.ref64(q, probes, k)
    assert_ref64(d0, i0, ref)
    # the smallest and largest fp32 intermediates at this s: LUT entries -2 <q_j, cb_j[c]> and the distances
    q64 = q.astype(np.float64).reshape(nq, m, 2)
    lut = np.abs(-2.0 * np.einsum("qjx,jcx->qjc", q64, cb.astype(np.float64)))
    dist = np.concatenate([c[0] for c in ref[2]])
    lo = min(lut[lut > 0].min(), dist[dist > 0].min())
    assert lo >= step * step and np.ldexp(lo, 2 * s) >= TINY, "an intermediate would be subnormal at this scale"
    assert np.ldexp(max(lut.max(), dist.max()) * 4 * m, 2 * s) < float(np.finfo(np.float32).max)
    if s == 0:
        return
    sc = lambda a: np.ldexp(a, s).astype(np.float32)
    Ls = Lists(oracle, sc(coarse), sc(cb), assign, codes, ids)
    qs = sc(q)
    ds, is_, rs = both_paths(monkeypatch, capfd, Ls.search(qs, k, probes))
    assert rs[0] == 0, "queries handed back"
    assert np.array_equal(is_, i0)
    assert np.array_equal(bits(ds), bits(np.ldexp(d0, 2 * s).astype(np.float32)))
    ods, ois, ops = Ls.oracle(oracle, qs, nprobe, k)
    assert np.array_equal(ops, op) and np.array_equal(ois, oi0)
    assert np.array_equal(bits(ods), bits(np.ldexp(od0, 2 * s).astype(np.float32)))


# ------------------------------------------------------------------------------------------------ 2. the eps bound on hard data
@pytest.mark.parametrize("kind", ["query_norms", "small_subquantisers", "near_ties"])
def test_error_bound_on_hard_data(oracle, monkeypatch, capfd, kind):
    """eps_q bounds |fp16 tensor-core score - the look-up-table scan's fp32 sum|; where it does not, a vector at the k-th
    distance is filtered out and the ids differ from the query-major scan.
      query_norms          one batch, ||q|| from 1e-4 to 1e3 (the fp16 query scale s_q is the batch's)
      small_subquantisers  half the sub-quantisers 2^25 smaller than the others: their fp16 table entries are subnormal
                           (the codebook scale s_c is global)
      near_ties            every codeword of sub-quantiser 0 has a twin one ulp away; each query's k-th vector gets a copy
                           with the twin codeword"""
    rng = np.random.default_rng({"query_norms": 1, "small_subquantisers": 2, "near_ties": 3}[kind])
    m, kc, nq, k, nprobe = 32, 24, 128, 10, 4
    sizes = rng.integers(150, 400, kc)
    L = random_lists(oracle, rng, m, sizes)
    if kind == "small_subquantisers":
        cb = L.cb.copy()
        cb[1::2] *= np.float32(2.0 ** -25)
        L = L.like(oracle, cb)
        e = np.frexp(np.abs(cb).max())[1]
        assert (np.abs(cb[1::2]) * 2.0 ** (10 - e) < 2.0 ** -14).all(), "fp16 table entries of the small ones are not subnormal"
    if kind == "near_ties":
        cb = L.cb.copy()
        cb[0, 1::2, 0] = np.nextafter(cb[0, 0::2, 0], np.float32(np.inf))
        cb[0, 1::2, 1] = cb[0, 0::2, 1]
        L = L.like(oracle, cb)
    q = queries_near(rng, L, rng.integers(0, kc, nq))
    if kind == "query_norms":
        q = (q / np.linalg.norm(q, axis=1, keepdims=True) * rng.permutation(np.logspace(-4, 3, nq))[:, None]).astype(np.float32)
    _, _, probes = L.idx.batch_search(q, k, nprobe=nprobe, return_probes=True)
    if kind == "near_ties":
        # the k-th vector of every query, again, with code 0 moved to its one-ulp twin (same list, new id)
        _, _, cand = L.ref64(q, probes, k)
        rows = set()
        for r, (d64, idr, tol, o) in enumerate(cand):
            rows.add(int(np.nonzero(L.lids == idr[o[k - 1]])[0][0]))
        rows = np.array(sorted(rows))
        lst = np.searchsorted(L.off, rows, side="right") - 1
        tw = L.codes[rows].copy()
        tw[:, 0] ^= 1
        L.add(lst, tw, L.lids.max() + 1 + np.arange(len(rows)))
    gd, gi, r = both_paths(monkeypatch, capfd, L.search(q, k, probes))
    assert r[0] == 0
    assert_ref64(gd, gi, L.ref64(q, probes, k))
    od, oi, op = L.oracle(oracle, q, nprobe, k)
    assert np.array_equal(op, probes)
    assert_topk_close(gd, gi, od, oi, atol=RTOL * float(np.nanmax(np.abs(od))))


# ------------------------------------------------------------------------------------------------ 3. / 4. many finalists
TIE_STEP = 2.0 ** -5


def _tied_list(oracle, rng, m, ntied, kc, other):
    """list 0: ntied copies of one code (distinct, shuffled ids); lists 1.. random.  Centroids, codebooks (and the queries)
    are multiples of TIE_STEP, so every sum of the scans is exact: the copies tie exactly although each slot adds the
    sub-quantisers in its own rotated order."""
    L = random_lists(oracle, rng, m, [0] + [other] * (kc - 1), spread=3.0, step=TIE_STEP)
    code = rng.integers(0, 256, (1, m), dtype=np.uint8)
    tied_ids = rng.permutation(ntied).astype(np.int64) * 7 + 1_000_000
    L.add(np.zeros(ntied, np.int32), np.repeat(code, ntied, axis=0), tied_ids)
    return L, code, tied_ids


def test_long_selection_of_tied_finalists(oracle, monkeypatch, capfd):
    """A few queries whose nearest list holds 3000 copies of one code: every copy is a finalist (> 512: select_long_kernel),
    the k returned are the k smallest ids among them, on both scans and in float64, and twice the same bits."""
    m, kc, k, ntied, nlong, nother = 32, 16, 64, 3000, 4, 60
    rng = np.random.default_rng(21)
    L, code, tied_ids = _tied_list(oracle, rng, m, ntied, kc, 200)
    # sizing: a filter warp logs at most (tiles / 2) 32 records per query of an item; only the nlong queries probe list 0
    assert (-(-ntied // 128) + 1) // 2 * 32 * nlong < LOG_CAP // 2
    ql = on_grid(L.coarse[0] + decoded(L.cb, code) + 0.05 * rng.standard_normal((nlong, L.d)), TIE_STEP)
    qo = on_grid(queries_near(rng, L, rng.integers(1, kc, nother)), TIE_STEP)
    q = np.concatenate([ql, qo])
    probes = np.concatenate([np.concatenate([np.zeros((nlong, 1), np.int32), nearest_probes(ql, L.coarse, 3, np.arange(1, kc))], 1),
                             nearest_probes(qo, L.coarse, 4, np.arange(1, kc))])
    gd, gi, r = both_paths(monkeypatch, capfd, L.search(q, k, probes))
    h, t, mx, c, e = r
    assert h == 0 and mx >= ntied > 512, f"route {r}"
    want = np.sort(tied_ids)[:k]
    assert (gi[:nlong] == want).all()
    ref = L.ref64(q, probes, k)
    assert (ref[1][:nlong] == want).all()
    assert_ref64(gd, gi, ref)
    # determinism: the keys reach their runs through atomics (key_scatter_kernel); the selection hides the order
    monkeypatch.setenv("VIX_TC_SCAN", "1")
    d2, i2 = L.search(q, k, probes)()
    assert np.array_equal(i2, gi) and np.array_equal(bits(d2), bits(gd))


def test_log_overflow_hands_back_every_query(oracle, monkeypatch, capfd):
    """4096 copies of one code, the first probe of 64 queries: a filter warp logs 16 tiles x 32 rows x 64 queries records,
    more than its log holds.  log_key_kernel flags the overflow and every query goes to the query-major scan."""
    m, kc, k, ntied, nq = 16, 8, 10, 4096, 64
    rng = np.random.default_rng(31)
    L, code, tied_ids = _tied_list(oracle, rng, m, ntied, kc, 300)
    assert (ntied // 128) // 2 * 32 * nq > LOG_CAP
    q = on_grid(L.coarse[0] + decoded(L.cb, code) + 0.05 * rng.standard_normal((nq, L.d)), TIE_STEP)
    probes = np.concatenate([np.zeros((nq, 1), np.int32), nearest_probes(q, L.coarse, 2, np.arange(1, kc))], 1)
    gd, gi, r = both_paths(monkeypatch, capfd, L.search(q, k, probes))
    h, t, mx, c, e = r
    assert c == LOG_CAP and h == nq, f"route {r}"
    assert (gi == np.sort(tied_ids)[:k]).all()
    assert_ref64(gd, gi, L.ref64(q, probes, k))


# ------------------------------------------------------------------------------------------------ 5. hand-back mix, probes
def test_hand_back_mix_and_probe_hygiene(oracle, monkeypatch, capfd):
    """One batch through search_with_probes: ordinary queries; queries whose first list with vectors holds fewer than k
    (handed back); queries whose first probes are empty lists, -1, >= kc or < -1 (the seed walks past them); queries
    with both; one query with no valid probe (ids -1, distances NaN).  Handed back = exactly the predicted queries."""
    m, kc, k, nprobe = 48, 40, 10, 8
    rng = np.random.default_rng(41)
    sizes = np.concatenate([[0] * 4, rng.integers(3, k, 4), rng.integers(150, 300, kc - 8)])
    L = random_lists(oracle, rng, m, sizes, spread=2.0)
    empty, tiny, normal = np.arange(4), np.arange(4, 8), np.arange(8, kc)
    nq = 256
    q = queries_near(rng, L, rng.choice(normal, nq))
    probes = nearest_probes(q, L.coarse, nprobe, normal)
    junk = [lambda: int(rng.choice(empty)), lambda: -1, lambda: kc + int(rng.integers(0, 3)), lambda: -int(rng.integers(2, 9)),
            lambda: 2 ** 30]
    kind = rng.integers(0, 4, nq)               # 0 ordinary, 1 tiny list first, 2 junk first, 3 junk then a tiny list
    for r in range(nq):
        lead = []
        if kind[r] in (2, 3):
            lead = [junk[j]() for j in rng.permutation(len(junk))[:int(rng.integers(1, 4))]]
            lead = [v for i, v in enumerate(lead) if v == -1 or v not in lead[:i]]
        if kind[r] in (1, 3):
            lead.append(int(rng.choice(tiny)))
        probes[r] = np.array(lead + list(probes[r]), np.int32)[:nprobe]
    probes[-1] = [-1, int(empty[0]), kc, -3, -1, 2 ** 30, int(empty[1]), -1]
    want_h = L.handed_back(probes, k)
    assert 0 < want_h < nq and (kind == 2).any() and (kind == 0).any()
    gd, gi, r = both_paths(monkeypatch, capfd, L.search(q, k, probes))
    assert r[0] == want_h, f"route {r}, {want_h} queries expected back"
    assert (gi[-1] == -1).all() and np.isnan(gd[-1]).all()
    assert_ref64(gd, gi, L.ref64(q, probes, k))


# ------------------------------------------------------------------------------------------------ 6. boundaries
@pytest.fixture(scope="module")
def k_problems(oracle):
    """one index per M for the k sweep, freed with the module"""
    cache = {}

    def get(m):
        if m not in cache:
            rng = np.random.default_rng(50 + m)
            kc, nq = 32, 300
            L = random_lists(oracle, rng, m, rng.integers(100, 400, kc))
            cache[m] = (L, queries_near(rng, L, rng.integers(0, kc, nq)))
        return cache[m]
    yield get
    cache.clear()


@pytest.mark.parametrize("k", [1, 16, 33, 63, 64, 65])
@pytest.mark.parametrize("m", [16, 32, 48, 64])
def test_k_boundaries(oracle, k_problems, monkeypatch, capfd, m, k):
    """k up to 64 takes the list-major scan (k = 64: the seed's k-th of 256 keys, P = 512 in select_long_kernel);
    k = 65 does not, and still answers correctly."""
    L, q = k_problems(m)
    nprobe = 6
    _, _, probes = L.idx.batch_search(q, k, nprobe=nprobe, return_probes=True)
    gd, gi, r = both_paths(monkeypatch, capfd, L.search(q, k, probes), tc=k <= 64)
    if k <= 64:
        assert r[0] == L.handed_back(probes, k) == 0, f"route {r}"
    assert_ref64(gd, gi, L.ref64(q, probes, k))
    od, oi, op = L.oracle(oracle, q, nprobe, k)
    assert np.array_equal(op, probes)
    assert_topk_close(gd, gi, od, oi)


@pytest.mark.parametrize("m", [16, 32, 48, 64])
def test_list_length_and_queries_per_list_boundaries(oracle, monkeypatch, capfd, m):
    """List lengths 1, 31, 32, 33 (the 32-vector chunk), 127, 128, 129 (the 128-row tile), 4097; lists probed by exactly 1,
    63, 64, 65, 128 and 129 queries of the list-major scan (64 query columns per item: a list probed by more is visited
    again); -1 padding.  A query handed back contributes no pair, so the counts hold among the queries that stay: each of
    them has a list of at least k vectors as its first probe.  The queries handed back (first probe a list of 3 vectors)
    also probe the boundary lists."""
    lengths = [1, 31, 32, 33, 127, 128, 129, 4097]
    counts = [129, 128, 65, 64, 63, 1, 129, 63]
    k, nq, nback = 8, 160, 6
    rng = np.random.default_rng(60 + m)
    L = random_lists(oracle, rng, m, lengths + [3], spread=2.0)
    nl, tiny = len(lengths), len(lengths)
    long_ = np.array(lengths) >= k
    while True:                                             # every query a member of at least one list of >= k vectors
        member = np.zeros((nq, nl), bool)
        for l, c in enumerate(counts):
            member[rng.choice(nq, c, replace=False), l] = True
        if (member & long_).any(1).all():
            break
    home = np.array([rng.choice(np.nonzero(row & long_)[0]) for row in member])
    back = rng.integers(0, nl, (nback, 3))
    q = queries_near(rng, L, np.concatenate([home, np.full(nback, tiny)]))
    order = nearest_probes(q, L.coarse, nl, np.arange(nl))
    nprobe = max(int(member.sum(1).max()), 4)
    probes = np.full((nq + nback, nprobe), -1, np.int32)
    for r in range(nq):
        mine = [home[r]] + [l for l in order[r] if member[r, l] and l != home[r]]
        probes[r, :len(mine)] = mine
    for r in range(nback):
        probes[nq + r, :4] = [tiny] + list(dict.fromkeys(back[r].tolist())) + [-1] * (3 - len(set(back[r].tolist())))
    flag = L.flagged(probes, k)
    assert not flag[:nq].any() and flag[nq:].all()
    stay = probes[~flag]
    assert (np.bincount(stay[stay >= 0], minlength=nl + 1)[:nl] == counts).all()
    gd, gi, r = both_paths(monkeypatch, capfd, L.search(q, k, probes))
    assert r[0] == nback, f"route {r}, {nback} queries expected back"
    assert_ref64(gd, gi, L.ref64(q, probes, k))


# ------------------------------------------------------------------------------------------------ 7. ids
def test_large_and_repeated_ids(oracle, monkeypatch, capfd):
    """External ids up to 2^32 - 2 in no particular order (the key keeps 32 bits of the id); an id stored twice comes back
    twice, in the order of the query-major scan (the two copies sit in slots that add the sub-quantisers in different
    orders: their distances may differ in the last bit)."""
    m, kc, k, nq, nprobe = 16, 16, 10, 200, 4
    rng = np.random.default_rng(71)
    sizes = rng.integers(200, 300, kc)
    n = int(sizes.sum())
    ids = np.unique(rng.integers(0, 2 ** 32 - 1, 2 * n))
    ids = rng.permutation(ids[(ids != 2 ** 32 - 2) & (ids != 2 ** 31)])[:n]
    ids[:2] = [2 ** 32 - 2, 2 ** 31]
    ids = rng.permutation(ids)
    L = random_lists(oracle, rng, m, sizes, ids=ids)
    big = int(np.nonzero(L.lids == 2 ** 32 - 2)[0][0])
    lst = int(np.searchsorted(L.off, big, side="right") - 1)
    L.add([lst], L.codes[big:big + 1], [2 ** 32 - 2])                                 # the same vector, the same id, again
    q = queries_near(rng, L, rng.integers(0, kc, nq))
    q[0] = L.coarse[lst] + decoded(L.cb, L.codes[big:big + 1])[0]                      # its nearest vector: both copies
    probes = nearest_probes(q, L.coarse, nprobe)
    gd, gi, r = both_paths(monkeypatch, capfd, L.search(q, k, probes))
    assert r[0] == 0
    assert (gi[0, :2] == 2 ** 32 - 2).all()
    assert (gi >= 2 ** 31).any()
    assert_ref64(gd, gi, L.ref64(q, probes, k))


# ------------------------------------------------------------------------------------------------ 8. default dispatch
def test_default_dispatch(oracle, monkeypatch):
    """Without VIX_TC_SCAN: L2, dsub = 2, ks = 256, k <= 64 batches of nq x nprobe >= 32768 pairs take the list-major scan
    (32768 does, 32767 does not).  Inner product, a filter, phase statistics, dsub = 4 and ks = 16 never take it (nor when
    it is forced)."""
    from vectorindex_b200.index import IDFilter, IVFPQIndex
    m, kc, k = 16, 64, 10
    rng = np.random.default_rng(81)
    sizes = rng.integers(250, 350, kc)
    L = random_lists(oracle, rng, m, sizes, ids=np.arange(int(sizes.sum()), dtype=np.int64))
    q = queries_near(rng, L, rng.integers(0, kc, 4681))

    def takes(search):
        monkeypatch.delenv("VIX_TC_SCAN", raising=False)
        n0 = tc_launches()
        d1, i1 = search()[:2]
        took = tc_launches() - n0
        monkeypatch.setenv("VIX_TC_SCAN", "0")
        d0, i0 = search()[:2]
        assert np.array_equal(i0, i1) and np.array_equal(bits(d0), bits(d1))
        return took, d1, i1

    for nq, nprobe, want in ((4096, 8, 1), (4681, 7, 0)):
        assert (nq * nprobe >= 32768) == bool(want)
        probes = nearest_probes(q[:nq], L.coarse, nprobe)
        took, gd, gi = takes(L.search(q[:nq], k, probes))
        assert took == want, f"nq {nq} x nprobe {nprobe}: {took} list-major launches"
        sub = slice(0, nq, 16)
        assert_ref64(gd[sub], gi[sub], L.ref64(q[sub], probes[sub], k))
    q8 = q[:4096]
    probes = nearest_probes(q8, L.coarse, 8)
    flt = IDFilter(int(sizes.sum()), "allow")
    flt.set(np.arange(0, int(sizes.sum()), 2))
    ip = L.like(oracle, metric="dotProduct")
    x = rng.standard_normal((5000, 2 * m)).astype(np.float32)
    dsub4 = IVFPQIndex(2 * m, "euclidean", nlist=kc, nprobe=8, m=m // 2)
    dsub4.set_coarse(L.coarse)
    dsub4.set_codebooks(rng.standard_normal((m // 2, 256, 4)).astype(np.float32))
    dsub4.batch_insert(x)
    ks16 = IVFPQIndex(2 * m, "euclidean", nlist=kc, nprobe=8, m=m, ks=16)
    ks16.set_coarse(L.coarse)
    ks16.set_codebooks(rng.standard_normal((m, 16, 2)).astype(np.float32))
    ks16.batch_insert(x)
    never = {
        "inner product": lambda: ip.idx.search_with_probes(q8, k, probes),
        "filter": lambda: L.idx.batch_search(q8, k, filter=flt),
        "stats": lambda: L.idx.search_with_probes(q8, k, probes, stats=True),
        "dsub 4": lambda: dsub4.search_with_probes(q8, k, probes),
        "ks 16": lambda: ks16.search_with_probes(q8, k, probes),
    }
    for name, search in never.items():
        for env in (None, "1"):
            if env is None:
                monkeypatch.delenv("VIX_TC_SCAN", raising=False)
            else:
                monkeypatch.setenv("VIX_TC_SCAN", env)
            n0 = tc_launches()
            search()
            assert tc_launches() == n0, f"{name} (VIX_TC_SCAN={env}) took the list-major scan"


# ------------------------------------------------------------------------------------------------ 9. determinism
def test_repeated_calls_are_bit_identical(oracle, monkeypatch, capfd):
    """C5-shaped (d = 96, M = 48), trained codebooks: three list-major launches, identical ids and bits, equal to the
    query-major scan and to the oracle."""
    from vectorindex_b200.index import IVFPQIndex
    n, d, m, kc, nq, nprobe, k = 40000, 96, 48, 64, 2000, 12, 10
    xb, q, coarse, cb, norms = _make_ivfpq_problem(oracle, n, d, m, kc, nq, seed=91, unit=True)
    idx = IVFPQIndex(d, "euclidean", nlist=kc, nprobe=nprobe, m=m)
    idx.set_coarse(coarse)
    idx.set_codebooks(cb, norms)
    idx.batch_insert(xb)
    gd, gi, r = both_paths(monkeypatch, capfd, lambda: idx.batch_search(q, k))
    for _ in range(2):
        d2, i2 = idx.batch_search(q, k)
        assert np.array_equal(i2, gi) and np.array_equal(bits(d2), bits(gd))
    off, codes, lids, _ = idx.export_lists()
    od, oi, _ = oracle.ivfpq_search(q, coarse, cb, norms, off, codes, lids, m, 256, nprobe, k, 0)
    assert_topk_close(gd, gi, od, oi)
