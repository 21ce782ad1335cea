"""Edges of the query-major IVF-PQ scan (vix_ivfpq_scan.cu), each with the route it must take proven.

The query-major scan serves inner product, dsub != 2, ks = 16, filtered searches, searches with statistics, k > 64, small
batches and the queries the list-major scan hands back.  Every case builds its lists directly (set_coarse / set_codebooks /
add_encoded) and, where the probes matter, sets them too (search_with_probes).  A case then checks:
  - the route: the line launch_ivfpq_scan_classic prints under VIX_SCAN_DEBUG=1 (kernel, filter / stats instantiation,
    warps, Pw, table and bias source, locality order, work items);
  - a float64 reference that shares no code with the scan or the oracle (pq_ref64), and oracle.ivfpq_search where the
    probes are the oracle's own (ids, distances to 1e-5);
  - bit-exact invariants: an allow-everything filter, stats=True and a repeated call give the same bits; within one route
    the first k1 results at k2 > k1 are the k1 result.
Searches run with VIX_TC_SCAN=0 unless a case is about the list-major scan.
"""
import re
import zlib

import numpy as np
import pytest

from pq_ref64 import RTOL, assert_ref64, decode, ref64
from test_gpu_parity import assert_topk_close, bits
from vectorindex_b200 import _lib

gpu = pytest.mark.gpu
ROUTE = re.compile(r"\[vix scan\] kernel (fast G (\d)|generic), filter (\d), stats (\d), warps (\d+), Pw (\d+), P2 (\d+), "
                   r"table (\w+), bias (\w+), order (\w+), items (\w+)")
METRICS = {0: "euclidean", 1: "dotProduct"}
ERR_INVALID_K, ERR_UNSUPPORTED = -2, -9


# ------------------------------------------------------------------------------------------------ building blocks
class PQ:
    """An IVF-PQ index whose lists are given: coarse [kc x d], codebooks [m x ks x dsub], per stored vector its list, code
    ([m] bytes, or [m / 2] nibble pairs at ks = 16) and id."""

    def __init__(self, oracle, coarse, cb, assign, codes, ids, metric=0):
        from vectorindex_b200.index import IVFPQIndex
        self.coarse, self.cb = np.ascontiguousarray(coarse, np.float32), np.ascontiguousarray(cb, np.float32)
        self.kc, self.d = self.coarse.shape
        self.m, self.ks, self.dsub = self.cb.shape
        self.metric = metric
        self.norms = oracle.pq_centroid_sq(self.cb, self.m, self.ks, self.dsub)
        self.idx = IVFPQIndex(self.d, METRICS[metric], nlist=self.kc, nprobe=8, m=self.m, ks=self.ks)
        self.idx.set_coarse(self.coarse)
        self.idx.set_codebooks(self.cb, self.norms)
        self.rows = (np.asarray(assign, np.int32), np.asarray(codes, np.uint8), np.asarray(ids, np.int64))
        self.idx.add_encoded(*self.rows)
        self.off, self.codes, self.lids, _ = self.idx.export_lists()
        self.lens = np.diff(self.off)

    def probes(self, q, nprobe):
        """the index's own probe selection (= the oracle's, asserted where the oracle is compared)"""
        return self.idx.batch_search(q, 1, nprobe=nprobe, return_probes=True)[2]

    def ref(self, q, probes, k):
        return ref64(q, self.coarse, self.cb, probes, self.off, self.codes, self.lids, k, self.metric)

    def oracle(self, oracle, q, nprobe, k):
        return oracle.ivfpq_search(q, self.coarse, self.cb, self.norms, self.off, self.codes, self.lids, self.m, self.ks,
                                   nprobe, k, self.metric)


def random_pq(oracle, rng, m, dsub, sizes, ks=256, metric=0, spread=1.0, res=0.5, ids=None):
    kc, d = len(sizes), m * dsub
    coarse = (rng.standard_normal((kc, d)) * spread).astype(np.float32)
    cb = (rng.standard_normal((m, ks, dsub)) * res).astype(np.float32)
    assign = np.repeat(np.arange(kc, dtype=np.int32), sizes)
    codes = rng.integers(0, 256, (assign.size, m if ks == 256 else m // 2), dtype=np.uint8)
    if ids is None:
        ids = rng.permutation(assign.size).astype(np.int64) * 3 + 5
    return PQ(oracle, coarse, cb, assign, codes, ids, metric)


def queries_near(rng, P, home, noise=0.2):
    r = decode(P.cb, rng.integers(0, 256, (len(home), P.m if P.ks == 256 else P.m // 2)).astype(np.uint8))
    return (P.coarse[home] + r + noise * rng.standard_normal(r.shape)).astype(np.float32)


def scan(mp, capfd, fn, tc="0"):
    """fn() with VIX_SCAN_DEBUG=1 (and VIX_TC_SCAN=tc) -> (its result, [route dicts of the query-major launches])"""
    capfd.readouterr()
    mp.setenv("VIX_TC_SCAN", tc)
    mp.setenv("VIX_SCAN_DEBUG", "1")
    try:
        out = fn()
    finally:
        mp.delenv("VIX_SCAN_DEBUG")
    routes = []
    for g in ROUTE.findall(capfd.readouterr().err):
        routes.append(dict(kernel=("fast" if g[1] else "generic"), G=int(g[1]) if g[1] else 0, filter=int(g[2]),
                           stats=int(g[3]), warps=int(g[4]), Pw=int(g[5]), P2=int(g[6]), table=g[7], bias=g[8],
                           order=g[9], items=g[10]))
    return out, routes


def one(mp, capfd, fn, **want):
    """fn() through exactly one query-major launch whose route has the fields of `want`"""
    out, routes = scan(mp, capfd, fn)
    assert len(routes) == 1, f"{len(routes)} query-major launches"
    for key, v in want.items():
        assert routes[0][key] == v, f"route {routes[0]}: {key} != {v}"
    return out, routes[0]


def same_bits(a, b):
    assert np.array_equal(a[1], b[1]), "ids differ"
    assert np.array_equal(bits(a[0]), bits(b[0])), "distance bits differ"


def check_oracle(oracle, P, q, probes, k, gd, gi):
    nprobe = probes.shape[1]
    od, oi, op = P.oracle(oracle, q, nprobe, k)
    assert np.array_equal(op, probes), "probes differ from the oracle's"
    atol = RTOL * float(np.nanmax(np.abs(od))) if P.metric == 1 else 0.0
    assert_topk_close(gd, gi, od, oi, atol=atol)


# ------------------------------------------------------------------------------------------------ 0. the reference itself
@pytest.mark.parametrize("metric,ks,dsub", [(0, 256, 3), (1, 256, 3), (0, 16, 2), (1, 16, 5)])
def test_ref64_matches_oracle(oracle, metric, ks, dsub):
    """CPU: the float64 reference agrees with the oracle's fp32 ADC search (L2 and IP, any dsub, packed nibbles)."""
    rng = np.random.default_rng(1 + metric + ks + dsub)
    m, kc, nprobe, k = 8, 12, 4, 20
    sizes = rng.integers(30, 80, kc)
    kc_, d = kc, m * dsub
    coarse = rng.standard_normal((kc_, d)).astype(np.float32)
    cb = (0.5 * rng.standard_normal((m, ks, dsub))).astype(np.float32)
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    codes = rng.integers(0, 256, (int(off[-1]), m if ks == 256 else m // 2), dtype=np.uint8)
    lids = rng.permutation(int(off[-1])).astype(np.int64)
    norms = oracle.pq_centroid_sq(cb, m, ks, dsub)
    q = (coarse[rng.integers(0, kc, 30)] + rng.standard_normal((30, d))).astype(np.float32)
    od, oi, op = oracle.ivfpq_search(q, coarse, cb, norms, off, codes, lids, m, ks, nprobe, k, metric)
    ref = ref64(q, coarse, cb, op, off, codes, lids, k, metric)
    assert_ref64(od, oi, ref)


# ------------------------------------------------------------------------------------------------ 1. route matrix
CONFIGS = {                       # name: (m, dsub, ks, expected kernel, G)
    "fast16": (16, 2, 256, "fast", 1), "fast32": (32, 2, 256, "fast", 2), "fast48": (48, 2, 256, "fast", 3),
    "fast64": (64, 2, 256, "fast", 4), "generic12": (12, 2, 256, "generic", 0), "generic80": (80, 2, 256, "generic", 0),
    "ks16_m16": (16, 2, 16, "generic", 0), "ks16_m10": (10, 2, 16, "generic", 0),
}


@pytest.fixture(scope="module")
def problems(oracle):
    cache = {}

    def get(name, metric):
        if (name, metric) not in cache:
            m, dsub, ks, _, _ = CONFIGS[name]
            rng = np.random.default_rng(zlib.crc32(f"{name}/{metric}".encode()))
            kc, nq = 16, 48
            P = random_pq(oracle, rng, m, dsub, rng.integers(150, 350, kc), ks=ks, metric=metric)
            cache[(name, metric)] = (P, queries_near(rng, P, rng.integers(0, kc, nq)))
        return cache[(name, metric)]
    yield get
    cache.clear()


@gpu
@pytest.mark.parametrize("metric", [0, 1], ids=["l2", "ip"])
@pytest.mark.parametrize("name", list(CONFIGS))
def test_route_matrix(oracle, problems, monkeypatch, capfd, name, metric):
    """Each kernel at L2 and IP, against float64 and the oracle; the fast kernels also through their FILTER and STATS
    instantiations: an allow-everything filter and stats=True give the bits of the plain search, as does a repeat."""
    from vectorindex_b200.index import IDFilter
    P, q = problems(name, metric)
    _, _, _, kern, G = CONFIGS[name]
    k, nprobe = 10, 6
    probes = P.probes(q, nprobe)
    base, r = one(monkeypatch, capfd, lambda: P.idx.search_with_probes(q, k, probes), kernel=kern, G=G, filter=0, stats=0,
                  table="kernel", bias="kernel", order="no", items=str(len(q)))
    gd, gi = base
    assert_ref64(gd, gi, P.ref(q, probes, k))
    check_oracle(oracle, P, q, probes, k, gd, gi)
    same_bits(one(monkeypatch, capfd, lambda: P.idx.search_with_probes(q, k, probes))[0], base)
    flt = IDFilter(int(P.lids.max()) + 1, "allow")
    flt.set(P.lids)
    got, _ = one(monkeypatch, capfd, lambda: P.idx.batch_search(q, k, nprobe=nprobe, filter=flt), kernel=kern, filter=1, stats=0)
    same_bits(got, base)
    got, _ = one(monkeypatch, capfd, lambda: P.idx.search_with_probes(q, k, probes, stats=True), kernel=kern, filter=0, stats=1)
    same_bits(got[:2], base)


# ------------------------------------------------------------------------------------------------ 2. table and bias routes
@gpu
@pytest.mark.parametrize("dsub", [2, 3, 4, 8, 12, 24])
def test_in_kernel_tables(oracle, monkeypatch, capfd, dsub):
    """build_lut's three branches (dsub = 2, dsub <= 16 with and without float4 reads, dsub > 16) at m = 16."""
    rng = np.random.default_rng(200 + dsub)
    P = random_pq(oracle, rng, 16, dsub, rng.integers(100, 300, 12), metric=dsub % 2)
    q = queries_near(rng, P, rng.integers(0, 12, 40))
    k, probes = 10, P.probes(q, 5)
    (gd, gi), _ = one(monkeypatch, capfd, lambda: P.idx.search_with_probes(q, k, probes), kernel="fast", table="kernel")
    assert_ref64(gd, gi, P.ref(q, probes, k))
    check_oracle(oracle, P, q, probes, k, gd, gi)


@gpu
@pytest.mark.parametrize("m,dsub,metric", [(64, 8, 0), (64, 10, 0), (64, 12, 1), (32, 16, 0), (48, 12, 1), (32, 16, 1)])
def test_batchwide_tables(oracle, monkeypatch, capfd, m, dsub, metric):
    """512 KB of codebooks or more: lut_image_kernel builds the tables; bit-equal to VIX_DISABLE_LUT_IMAGE=1."""
    rng = np.random.default_rng(300 + m + dsub + metric)
    P = random_pq(oracle, rng, m, dsub, rng.integers(100, 250, 10), metric=metric)
    q = queries_near(rng, P, rng.integers(0, 10, 40))
    k, probes = 10, P.probes(q, 4)
    img, _ = one(monkeypatch, capfd, lambda: P.idx.search_with_probes(q, k, probes), kernel="fast", G=m // 16, table="image")
    assert_ref64(*img, P.ref(q, probes, k))
    check_oracle(oracle, P, q, probes, k, *img)
    monkeypatch.setenv("VIX_DISABLE_LUT_IMAGE", "1")
    own, _ = one(monkeypatch, capfd, lambda: P.idx.search_with_probes(q, k, probes), kernel="fast", table="kernel")
    same_bits(own, img)


@gpu
@pytest.mark.parametrize("m,dsub,n0,n1,want", [(64, 8, 6, 17, "rows"), (16, 8, 40, 65, "rows"), (64, 26, 4, 5, "pairs")])
def test_bias_routes(oracle, monkeypatch, capfd, m, dsub, n0, n1, want):
    """The per-probe term in the scan (d x nprobe <= 8192), in probe_bias_rows_kernel (d <= 1536) or probe_bias_kernel
    (d > 1536).  Appending -1 probe columns switches the route and changes neither the probes scanned nor the bits."""
    rng = np.random.default_rng(400 + m + dsub)
    kc = 48
    P = random_pq(oracle, rng, m, dsub, rng.integers(20, 60, kc))
    d = m * dsub
    assert d * n0 <= 8192 < d * n1 and (want == "pairs") == (d > 1536)
    q = queries_near(rng, P, rng.integers(0, kc, 24))
    k, probes = 10, P.probes(q, n0)
    base, _ = one(monkeypatch, capfd, lambda: P.idx.search_with_probes(q, k, probes), kernel="fast", bias="kernel")
    assert_ref64(*base, P.ref(q, probes, k))
    check_oracle(oracle, P, q, probes, k, *base)
    wide = np.concatenate([probes, np.full((len(q), n1 - n0), -1, np.int32)], 1)
    got, _ = one(monkeypatch, capfd, lambda: P.idx.search_with_probes(q, k, wide), kernel="fast", bias=want)
    same_bits(got, base)


# ------------------------------------------------------------------------------------------------ 3. locality order
@gpu
def test_locality_order(oracle, monkeypatch, capfd):
    """Batches of more than 2 SMs queries are handed out sorted by their first probed list; the same queries in a batch of
    2 SMs (no order) give the same bits."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    rng = np.random.default_rng(500)
    kc = 64
    P = random_pq(oracle, rng, 16, 4, rng.integers(50, 150, kc), metric=0)
    q = queries_near(rng, P, rng.integers(0, kc, 2 * sms + 37))
    k, probes = 20, P.probes(q, 6)
    small, _ = one(monkeypatch, capfd, lambda: P.idx.search_with_probes(q[:2 * sms], k, probes[:2 * sms]), order="no")
    big, _ = one(monkeypatch, capfd, lambda: P.idx.search_with_probes(q, k, probes), order="yes", items=str(len(q)))
    same_bits((big[0][:2 * sms], big[1][:2 * sms]), small)
    assert_ref64(*big, P.ref(q, probes, k))
    check_oracle(oracle, P, q, probes, k, *big)


# ------------------------------------------------------------------------------------------------ 4. k sweep
KS = [1, 32, 33, 64, 65, 192, 193, 448, 449, 512]


@gpu
@pytest.mark.parametrize("metric", [0, 1], ids=["l2", "ip"])
@pytest.mark.parametrize("name", ["fast16", "fast48", "fast64", "generic12", "ks16_m16"])
def test_k_sweep(oracle, problems, monkeypatch, capfd, name, metric):
    """Every k from 1 to VIX_MAX_K at the boundaries of Pw, the k <= 32 chunk seed and the 512 registers of
    select_and_write; m = 48 / 64 with k > 448 run on two warps.  The last query probes one list of fewer than 512
    vectors (padded with -1 / NaN).  Within the route the first k1 results at k2 > k1 are the k1 result, bit for bit."""
    P, q = problems(name, metric)
    _, _, _, kern, G = CONFIGS[name]
    nprobe = 6
    probes = P.probes(q, nprobe)
    probes[-1] = [int(np.argmin(P.lens))] + [-1] * (nprobe - 1)
    assert P.lens.min() < 512
    prev = None
    for k in KS:
        (gd, gi), r = one(monkeypatch, capfd, lambda: P.idx.search_with_probes(q, k, probes), kernel=kern, G=G)
        if kern == "fast" and G >= 3 and k > 448:
            assert r["warps"] == 2, f"route {r}"
        assert_ref64(gd, gi, P.ref(q, probes, k))
        check_oracle(oracle, P, q[:-1], probes[:-1], k, gd[:-1], gi[:-1])
        if prev is not None:
            k1 = prev[0].shape[1]
            same_bits((gd[:, :k1], gi[:, :k1]), prev)
        prev = (gd, gi)


@gpu
def test_rerank_512_at_m48(oracle, monkeypatch, capfd):
    """vix_index_search_rerank with rerank_r = 512 at m = 48 (the C5 shape): the ADC candidates come from the fast kernel,
    the result is the exact top k among them."""
    rng = np.random.default_rng(600)
    kc, d, k, r = 12, 96, 10, 512
    P = random_pq(oracle, rng, 48, 2, rng.integers(200, 400, kc), ids=None)
    n = int(P.lids.max()) + 1
    xb = rng.standard_normal((n, d)).astype(np.float32)
    q = queries_near(rng, P, rng.integers(0, kc, 20))
    (cd, ci), _ = one(monkeypatch, capfd, lambda: P.idx.batch_search(q, r, nprobe=4), kernel="fast", G=3, warps=2)
    (sc, ids), _ = one(monkeypatch, capfd, lambda: P.idx.batch_search_rerank(q, k, xb, r, nprobe=4), kernel="fast", warps=2)
    for row in range(len(q)):
        cand = ci[row][ci[row] >= 0]
        ex = ((xb[cand].astype(np.float64) - q[row].astype(np.float64)) ** 2).sum(1)
        o = np.lexsort((cand, ex))[:k]
        np.testing.assert_allclose(sc[row], ex[o], rtol=1e-5)
        assert set(ids[row].tolist()) <= set(cand.tolist())


# ------------------------------------------------------------------------------------------------ 5. ties
TIE_STEP = 2.0 ** -5


@gpu
@pytest.mark.parametrize("k", [64, 512])
@pytest.mark.parametrize("name", ["fast48", "generic12"])
def test_tied_copies(oracle, monkeypatch, capfd, name, k):
    """3000 copies of one code in the nearest list (grid-valued data: every sum exact, so they tie whatever the order of
    the sub-quantisers), one id of them stored twice: the k smallest ids, the twice-stored one twice, through the long
    walk of select_and_write (more than 512 candidates published)."""
    m, dsub, _, kern, G = CONFIGS[name]
    rng = np.random.default_rng(700 + m + k)
    kc, ntied = 8, 3000
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
    q = g(coarse[0] + decode(cb, code) + 0.05 * rng.standard_normal((6, m * dsub)))
    probes = np.concatenate([np.zeros((6, 1), np.int32), 1 + rng.permutation(kc - 1)[None, :3].repeat(6, 0).astype(np.int32)], 1)
    (gd, gi), _ = one(monkeypatch, capfd, lambda: P.idx.search_with_probes(q, k, probes), kernel=kern, G=G)
    want = np.sort(np.concatenate([tied, [dup]]))[:k]
    assert (gi == want).all()
    assert (bits(gd) == bits(gd[:, :1])).all(), "tied copies with different distance bits"
    assert_ref64(gd, gi, P.ref(q, probes, k))
    again, _ = one(monkeypatch, capfd, lambda: P.idx.search_with_probes(q, k, probes))
    same_bits(again, (gd, gi))


# ------------------------------------------------------------------------------------------------ 6. nprobe
@gpu
@pytest.mark.parametrize("name", ["fast16", "fast48", "generic12"])
def test_nprobe_sweep(oracle, monkeypatch, capfd, name):
    """nprobe from 1 to VIX_MAX_K (the probe table takes blocks of 256; the generic kernel's probe setup loops), and
    nprobe above kc (probes padded with -1); nprobe = VIX_MAX_K + 1 is refused before any kernel runs."""
    from vectorindex_b200._lib import VectorIndexError
    m, dsub, ks, kern, G = CONFIGS[name]
    rng = np.random.default_rng(800 + m)
    kc = 520
    P = random_pq(oracle, rng, m, dsub, rng.integers(0, 12, kc))
    q = queries_near(rng, P, rng.integers(0, kc, 24))
    k = 20
    for nprobe in [1, 32, 33, 255, 256, 257, 512]:
        probes = P.probes(q, nprobe)
        (gd, gi), _ = one(monkeypatch, capfd, lambda: P.idx.search_with_probes(q, k, probes), kernel=kern, G=G)
        assert_ref64(gd, gi, P.ref(q, probes, k))
        check_oracle(oracle, P, q, probes, k, gd, gi)
    with pytest.raises(VectorIndexError) as e:
        P.idx.batch_search(q, k, nprobe=513)
    assert e.value.status == ERR_INVALID_K
    small = random_pq(oracle, rng, m, dsub, rng.integers(5, 30, 40))
    q2 = queries_near(rng, small, rng.integers(0, 40, 16))
    probes = small.probes(q2, 100)
    assert (probes[:, 40:] == -1).all()
    (gd, gi), _ = one(monkeypatch, capfd, lambda: small.idx.search_with_probes(q2, k, probes), kernel=kern)
    assert_ref64(gd, gi, small.ref(q2, probes, k))
    check_oracle(oracle, small, q2, probes, k, gd, gi)


@gpu
def test_list_major_hand_back_at_nprobe_300(oracle, monkeypatch, capfd):
    """The list-major scan forced at nprobe = 300, m = 48: the queries whose first list holds fewer than k vectors go to
    the query-major scan (work items on the device), bit-equal to the query-major scan alone."""
    rng = np.random.default_rng(900)
    kc, k = 400, 10
    P = random_pq(oracle, rng, 48, 2, rng.integers(2, 30, kc))
    q = queries_near(rng, P, rng.integers(0, kc, 64))
    probes = P.probes(q, 300)
    n0 = int(_lib.lib().vix_scan_tc_launches())
    (td, ti), routes = scan(monkeypatch, capfd, lambda: P.idx.search_with_probes(q, k, probes), tc="1")
    assert int(_lib.lib().vix_scan_tc_launches()) == n0 + 1, "list-major scan not taken"
    assert len(routes) == 1 and routes[0]["items"] == "device" and routes[0]["bias"] == "given", routes
    base, _ = one(monkeypatch, capfd, lambda: P.idx.search_with_probes(q, k, probes), kernel="fast", G=3)
    same_bits((td, ti), base)
    assert_ref64(td, ti, P.ref(q, probes, k))


@gpu
@pytest.mark.parametrize("name,metric", [("generic12", 0), ("generic12", 1), ("fast32", 1)])
def test_probe_hygiene(oracle, monkeypatch, capfd, name, metric):
    """-1, >= kc, < -1, empty lists, a row without a valid probe and a list probed twice (its vectors come back twice, both
    copies with the same bits)."""
    m, dsub, ks, kern, G = CONFIGS[name]
    rng = np.random.default_rng(1000 + m + metric)
    kc, k, nprobe = 24, 30, 8
    sizes = rng.integers(40, 120, kc)
    sizes[:3] = 0
    P = random_pq(oracle, rng, m, dsub, sizes, metric=metric)
    q = queries_near(rng, P, rng.integers(3, kc, 40))
    probes = P.probes(q, nprobe)
    junk = [-1, kc, kc + 7, -2, -(2 ** 31), 2 ** 31 - 1, 0, 1, 2]
    for r in range(0, 30):
        probes[r, rng.integers(0, nprobe, 3)] = rng.choice(junk, 3)
    for r in range(30, 39):
        probes[r, 1] = probes[r, 0]                                   # the nearest list twice
    probes[39] = [-1, 0, kc, -5, 1, -1, 2, kc + 1]
    (gd, gi), _ = one(monkeypatch, capfd, lambda: P.idx.search_with_probes(q, k, probes), kernel=kern)
    assert (gi[39] == -1).all() and np.isnan(gd[39]).all()
    assert_ref64(gd, gi, P.ref(q, probes, k))
    for r in range(30, 39):
        twice = set(P.lids[P.off[probes[r, 0]]:P.off[probes[r, 0] + 1]].tolist())
        for i in set(gi[r, :k - 1].tolist()) & twice:                  # (the last place may hold a first copy alone)
            sel = gi[r] == i
            assert sel.sum() == 2, f"row {r} id {i}: {sel.sum()} copies of a vector of the list probed twice"
            assert len(set(bits(gd[r][sel]).tolist())) == 1, f"row {r} id {i}: the two scans differ"


@gpu
def test_bookkeeping_limit(oracle, monkeypatch, capfd):
    """Two tables (m = 48 / 64) with k > 448 run on two warps while 4 nprobe + d <= 1912; beyond, the search is refused
    with VIX_ERR_UNSUPPORTED before any kernel of the scan runs (no route line is printed)."""
    from vectorindex_b200._lib import VectorIndexError
    rng = np.random.default_rng(1050)
    P = random_pq(oracle, rng, 64, 2, rng.integers(2, 6, 480))
    q = queries_near(rng, P, rng.integers(0, 480, 8))
    assert 4 * 446 + P.d <= 1912 < 4 * 447 + P.d
    probes = P.probes(q, 447)
    (gd, gi), _ = one(monkeypatch, capfd, lambda: P.idx.search_with_probes(q, 512, probes[:, :446]), kernel="fast", warps=2)
    assert_ref64(gd, gi, P.ref(q, probes[:, :446], 512))

    def refused():
        with pytest.raises(VectorIndexError) as e:
            P.idx.search_with_probes(q, 449, probes)
        return e.value.status
    status, routes = scan(monkeypatch, capfd, refused)
    assert status == ERR_UNSUPPORTED and routes == []
    (gd, gi), r = one(monkeypatch, capfd, lambda: P.idx.search_with_probes(q, 448, probes), kernel="fast", Pw=512)
    assert r["warps"] >= 3
    assert_ref64(gd, gi, P.ref(q, probes, 448))


# ------------------------------------------------------------------------------------------------ 7. filters
@gpu
@pytest.mark.parametrize("mode", ["allow", "deny"])
@pytest.mark.parametrize("name", ["fast16", "fast64", "ks16_m16"])
def test_filters(oracle, monkeypatch, capfd, name, mode):
    """Allow / deny bitsets: ids at capacity - 1 pass or not by the bit, ids at and above capacity never; a filter passing
    fewer than k vectors; k <= 32 (the chunk seed counts only entries that pass) and k = 512."""
    from vectorindex_b200.index import IDFilter
    m, dsub, ks, kern, G = CONFIGS[name]
    rng = np.random.default_rng(1100 + m + ks + (mode == "deny"))
    kc, nprobe = 12, 5
    sizes = rng.integers(100, 300, kc)
    n = int(sizes.sum())
    P = random_pq(oracle, rng, m, dsub, sizes, ks=ks, ids=rng.permutation(n).astype(np.int64))
    q = queries_near(rng, P, rng.integers(0, kc, 32))
    probes = P.probes(q, nprobe)
    cap = n - 3                                                   # ids n - 3 .. n - 1 are beyond the bitset
    for chosen, ks_ in ((rng.choice(cap, cap // 3, replace=False), (10, 32, 33, 512)),
                        (rng.choice(cap, 7, replace=False), (10, 32)),
                        (np.array([cap - 1, 5, 9]), (10,))):
        flt = IDFilter(cap, mode)
        flt.set(chosen)
        sel = np.isin(P.lids, chosen)
        keep = (sel if mode == "allow" else ~sel) & (P.lids < cap)
        rows = np.nonzero(keep)[0]
        lst = np.searchsorted(P.off, rows, side="right") - 1
        off = np.concatenate([[0], np.cumsum(np.bincount(lst, minlength=P.kc))])
        for k in ks_:
            (gd, gi), _ = one(monkeypatch, capfd, lambda: P.idx.batch_search(q, k, nprobe=nprobe, filter=flt), kernel=kern,
                              filter=1)
            assert_ref64(gd, gi, ref64(q, P.coarse, P.cb, probes, off, P.codes[rows], P.lids[rows], k, P.metric))
            assert not np.isin(gi[gi >= 0], np.nonzero(~np.isin(np.arange(n), P.lids[rows]))[0]).any()


# ------------------------------------------------------------------------------------------------ 8. values
@gpu
@pytest.mark.parametrize("metric", [0, 1], ids=["l2", "ip"])
@pytest.mark.parametrize("dsub", [4, 8])
def test_power_of_two_scaling(oracle, monkeypatch, capfd, dsub, metric):
    """Queries, centroids and codebooks times 2^s scale every fp32 intermediate exactly (grid-valued data keeps them
    normal): the same ids, distance bits those of ldexp(d0, 2 s)."""
    rng = np.random.default_rng(1200 + dsub + metric)
    m, kc, k, step = 16, 10, 16, 2.0 ** -7
    g = lambda a: np.clip(np.round(a / step) * step, -3, 3).astype(np.float32)
    coarse, cb = g(rng.standard_normal((kc, m * dsub))), g(0.5 * rng.standard_normal((m, 256, dsub)))
    assign = rng.integers(0, kc, 3000).astype(np.int32)
    codes = rng.integers(0, 256, (3000, m), dtype=np.uint8)
    ids = rng.permutation(3000).astype(np.int64)
    q = g(coarse[rng.integers(0, kc, 32)] + 0.3 * rng.standard_normal((32, m * dsub)))
    P0 = PQ(oracle, coarse, cb, assign, codes, ids, metric)
    probes = P0.probes(q, 4)
    d0, _ = one(monkeypatch, capfd, lambda: P0.idx.search_with_probes(q, k, probes), kernel="fast")
    assert_ref64(*d0, P0.ref(q, probes, k))
    check_oracle(oracle, P0, q, probes, k, *d0)
    for s in (-20, 24):
        sc = lambda a: np.ldexp(a, s).astype(np.float32)
        Ps = PQ(oracle, sc(coarse), sc(cb), assign, codes, ids, metric)
        ds, _ = one(monkeypatch, capfd, lambda: Ps.idx.search_with_probes(sc(q), k, probes), kernel="fast")
        assert np.array_equal(ds[1], d0[1])
        assert np.array_equal(bits(ds[0]), bits(np.ldexp(d0[0], 2 * s).astype(np.float32)))


@gpu
@pytest.mark.parametrize("name", ["fast16", "generic12"])
def test_zero_query_inner_product(oracle, problems, monkeypatch, capfd, name):
    """A zero query under IP: every score is 0; the distance -0 carries the oracle's sign, bit for bit."""
    P, _ = problems(name, 1)
    z = np.zeros((2, P.d), np.float32)
    k, probes = 10, P.probes(z, 4)
    (gd, gi), _ = one(monkeypatch, capfd, lambda: P.idx.search_with_probes(z, k, probes))
    od, oi, op = P.oracle(oracle, z, 4, k)
    assert np.array_equal(op, probes)
    assert (gd == 0).all()
    assert np.array_equal(bits(gd), bits(od)), f"{gd[0, :3]} vs oracle {od[0, :3]}"
    # every score ties: the k smallest probed ids (the oracle keeps its scan order among equal distances)
    for r in range(2):
        want = np.sort(np.concatenate([P.lids[P.off[l]:P.off[l + 1]] for l in probes[r] if l >= 0]))[:k]
        assert np.array_equal(gi[r], want)
    assert_ref64(gd, gi, P.ref(z, probes, k))


@gpu
@pytest.mark.parametrize("metric", [0, 1], ids=["l2", "ip"])
@pytest.mark.parametrize("name", ["fast16", "generic12"])
def test_non_finite_queries(oracle, problems, monkeypatch, capfd, name, metric):
    """Non-finite values, as vindex_cuda.h states them: results rank by (distance, id) with NaN after every number.
      NaN component     every probed vector scores NaN: the row is the k smallest probed ids, distances NaN (the oracle
                        also returns NaN, with its ids in scan order);
      +inf component    distances are +-inf or NaN (the decomposition can add +inf and -inf), never finite, still ranked
                        by (distance, id);
      huge query (L2)   every distance overflows to +inf (as in the oracle): the k smallest probed ids;
      huge query (IP)   finite scores: the oracle's ids and distances."""
    P, q = problems(name, metric)
    k, nprobe = 10, 4
    bad = q[:3].copy()
    bad[0, 0] = np.nan
    bad[1, 1] = np.inf
    bad[2] *= np.float32(1e30)
    od, oi, op = P.oracle(oracle, bad, nprobe, k)
    (gd, gi), _ = one(monkeypatch, capfd, lambda: P.idx.search_with_probes(bad, k, op))
    probed = [np.sort(np.concatenate([P.lids[P.off[l]:P.off[l + 1]] for l in row if l >= 0]))[:k] for row in op]

    def ranked(r):                       # (distance, id) ascending, NaN last, equal distance bits by id
        key = [(1, 0.0, i) if np.isnan(v) else (0, float(v), i) for v, i in zip(gd[r].tolist(), gi[r].tolist())]
        assert key == sorted(key), f"row {r}: {gd[r]} / {gi[r]} not ranked by (distance, id)"
    assert np.isnan(gd[0]).all() and np.isnan(od[0]).all()
    assert np.array_equal(gi[0], probed[0])
    assert not np.isfinite(gd[1]).any() and (gi[1] >= 0).all()
    for r in range(3):
        ranked(r)
    if metric == 0:
        assert (gd[2] == np.inf).all() and (od[2] == np.inf).all()
        assert np.array_equal(gi[2], probed[2])
    else:
        assert np.isfinite(od[2]).all()
        assert_topk_close(gd[2:], gi[2:], od[2:], oi[2:], atol=RTOL * float(np.abs(od[2]).max()))
