"""Edges of the tensor-core shortlist of the GEMM-shaped stages (vix_gemm.cu): coarse probe selection, flat search and IVF
list assignment, and the scale range of the tensor-core PQ encoder (vix_pq_tc.cu).

The shortlist keeps every column with S~ <= T_q = (k-th smallest group minimum) + 2 eps_q and rescores it exactly, so it
is exact only while eps_q bounds |S~ - S| for the score S the reference evaluates in fp32.  Every case here checks:
  - ids and distance / score bits equal the oracle's (oracle/, the reference restated in C);
  - they equal the exact CUDA-core route (VIX_DISABLE_TC=1) bit for bit;
  - vix_tc_shortlist_calls / vix_tc_shortlist_exact_rows show which route ran: the shortlist or not, and for flat search
    and assignment how many rows the exact kernel computed because their shortlist overflowed or was empty.
Where the oracle and the exact route differ on a NaN query (the reference orders NaN scores in its own way), the two routes
must still agree; the difference is reported as a warning.
"""
import ctypes as C
import warnings

import numpy as np
import pytest

from vectorindex_b200 import _lib

pytestmark = pytest.mark.gpu

PROBE, FLAT, ASSIGN = 0, 1, 2          # vix_shortlist_kind
SCALES = [2.0 ** e for e in (0, -6, -12, -20, -30)]


# ------------------------------------------------------------------------------------------------ building blocks
def unit_rows(rng, n, d):
    x = rng.standard_normal((n, d)).astype(np.float32)
    return (x / np.linalg.norm(x, axis=1, keepdims=True)).astype(np.float32)


def canon(a):
    """float32 bits with every NaN as the one quiet NaN (the payload of a NaN is not part of the result)"""
    a = np.array(a, dtype=np.float32)
    a[np.isnan(a)] = np.float32("nan")
    return a.view(np.uint32)


def counters(kind):
    L = _lib.lib()
    return int(L.vix_tc_shortlist_calls(kind)), int(L.vix_tc_shortlist_exact_rows(kind))


def margin(d, metric):
    """shortlist_margin of vix_gemm.cu: eps_q = rel ||q|| max||c|| + rel2 (||q||^2 + max||c||^2)"""
    l2 = metric == 0
    rel = np.float32((2.0 if l2 else 1.0) * 1.25 * (2.0 / 1024 + d / 2097152.0))
    rel2 = np.float32(1.25 * (d + 3) / 4194304.0) if l2 else np.float32(0)
    return float(rel), float(rel2)


def flat_call(vk, q, xb, k, metric):
    return lambda: vk.flat_search_f32(q, xb, k, metric)


def probe_call(vk, q, c, nprobe, metric):
    return lambda: vk.ivf_select_nprobe_batch_f32(q, c, nprobe, metric)


def assign_call(vk, x, c):
    return lambda: vk.ivf_assign_f32(x, c, return_dist=True)


def oracle_of(oracle, kind, a, b, k, metric):
    """(ids, scores) of the oracle for the call above"""
    if kind == FLAT:
        dist, ids, _ = oracle.flat_search(a, b, k, metric)
        return ids, dist
    if kind == PROBE:
        return oracle.probe_select_batch(a, b, k, metric)
    return oracle.assign(a, b)


def split(kind, out):
    """(ids, scores) of a product call"""
    if kind == FLAT:
        dist, ids = out
        return ids, dist
    return out


def check(mp, oracle, vk, kind, a, b, k=1, metric=0, tc=True, exact_rows=None, nan_rows_may_differ=False):
    """One call through the product's default route, compared with the oracle, then with VIX_DISABLE_TC=1.
    tc: whether the default route must take the shortlist; exact_rows: rows the exact kernel must have computed inside the
    shortlisted call (flat / assignment; None: not pinned).  Returns (ids, scores, exact rows taken)."""
    fn = {FLAT: flat_call(vk, a, b, k, metric), PROBE: probe_call(vk, a, b, k, metric), ASSIGN: assign_call(vk, a, b)}[kind]
    c0, e0 = counters(kind)
    gi, gs = split(kind, fn())
    c1, e1 = counters(kind)
    oi, os_ = oracle_of(oracle, kind, a, b, k, metric)
    bad = np.flatnonzero([not (np.array_equal(np.ravel(gi[r]), np.ravel(oi[r])) and
                               np.array_equal(canon(np.ravel(gs[r])), canon(np.ravel(os_[r])))) for r in range(len(gi))])
    if nan_rows_may_differ:
        nanrow = np.isnan(a).any(1)
        if bad.size and nanrow[bad].all():
            warnings.warn(f"kind {kind}: rows {bad.tolist()} with a NaN query differ from the oracle: "
                          f"ids {np.asarray(gi)[bad].tolist()} vs {np.asarray(oi)[bad].tolist()}")
            bad = bad[~nanrow[bad]]
    assert bad.size == 0, f"kind {kind}: rows {bad[:8].tolist()} differ from the oracle: " \
                          f"{np.asarray(gi)[bad[:2]].tolist()} vs {np.asarray(oi)[bad[:2]].tolist()}"
    mp.setenv("VIX_DISABLE_TC", "1")
    try:
        xi, xs = split(kind, fn())
    finally:
        mp.delenv("VIX_DISABLE_TC")
    assert counters(kind) == (c1, e1), "VIX_DISABLE_TC=1 took the shortlist"
    assert np.array_equal(gi, xi), f"kind {kind}: ids differ from the exact route"
    assert np.array_equal(canon(gs), canon(xs)), f"kind {kind}: score bits differ from the exact route"
    assert c1 - c0 == (1 if tc else 0), "shortlist not taken" if tc else "shortlist taken"
    if exact_rows is not None:
        assert e1 - e0 == exact_rows, f"kind {kind}: {e1 - e0} rows computed by the exact kernel, expected {exact_rows}"
    return gi, gs, e1 - e0


# ------------------------------------------------------------------------------------------------ zero rows
@pytest.mark.parametrize("d,kc", [(96, 1024), (128, 2048), (768, 1024)])
def test_zero_rows_assign_against_unit_centroids(oracle, vk, monkeypatch, d, kc):
    """A zero row against unit-norm centroids: S~ is exactly ||c||^2 as row_norms rounds it, and the dot-product margin is
    0, so a margin without the squared-norm term keeps only the centroids of the smallest ROUNDED norm -- while the
    reference's Km12 distance puts its minimum on another centroid.  The row must go to the exact kernel."""
    c = unit_rows(np.random.default_rng(0), kc, d)
    cn = oracle.centroid_norms(c)
    x = np.zeros((1024, d), np.float32)
    want, _ = oracle.assign(x[:1], c)
    assert cn[want[0]] > cn.min(), "not the adversarial case: the oracle's centroid has the smallest rounded norm"
    check(monkeypatch, oracle, vk, ASSIGN, x, c, exact_rows=1024)


def test_zero_rows_through_index_insert(oracle, monkeypatch):
    """the same case through IVFPQIndex.batch_insert: the exported list assignment equals the oracle's and the exact route's"""
    from vectorindex_b200.index import IVFPQIndex
    d, kc, m = 96, 1024, 48
    rng = np.random.default_rng(0)
    c = unit_rows(rng, kc, d)
    cb = rng.standard_normal((m, 256, 2)).astype(np.float32)
    x = rng.standard_normal((1536, d)).astype(np.float32)
    x[::3] = 0.0
    want, _ = oracle.assign(x, c)

    def insert():
        idx = IVFPQIndex(d, "euclidean", nlist=kc, nprobe=8, m=m)
        idx.set_coarse(c)
        idx.set_codebooks(cb, oracle.pq_centroid_sq(cb, m, 256, 2))
        idx.batch_insert(x)
        return idx.export_lists()

    c0, e0 = counters(ASSIGN)
    got = insert()
    c1, e1 = counters(ASSIGN)
    assert np.array_equal(got[3], want), f"{int((got[3] != want).sum())} rows assigned differently from the oracle"
    monkeypatch.setenv("VIX_DISABLE_TC", "1")
    try:
        exact = insert()
    finally:
        monkeypatch.delenv("VIX_DISABLE_TC")
    assert all(np.array_equal(u, v) for u, v in zip(got, exact)), "lists differ from the exact route's"
    assert counters(ASSIGN)[0] == c1, "VIX_DISABLE_TC=1 took the shortlist"
    assert c1 - c0 == 1, "shortlist not taken"
    assert e1 - e0 >= 512, f"{e1 - e0} rows computed by the exact kernel: fewer than the 512 zero rows"


@pytest.mark.parametrize("kind,metric", [(FLAT, 0), (FLAT, 1), (PROBE, 0), (PROBE, 1)])
def test_zero_queries_against_unit_rows(oracle, vk, monkeypatch, kind, metric):
    rng = np.random.default_rng(1)
    d = 96
    b = unit_rows(rng, 8192 if kind == FLAT else 2048, d)
    q = rng.standard_normal((32, d)).astype(np.float32)
    q[::2] = 0.0
    check(monkeypatch, oracle, vk, kind, q, b, k=10 if kind == FLAT else 16, metric=metric)


# ------------------------------------------------------------------------------------------------ scale separation
CONFIGS = [("flat-l2-d96", FLAT, 0, 96), ("flat-l2-d256", FLAT, 0, 256), ("flat-ip", FLAT, 1, 96),
           ("probe-l2", PROBE, 0, 96), ("probe-ip", PROBE, 1, 128), ("assign", ASSIGN, 0, 96)]


def scaled_problem(kind, d, s, reverse, seed):
    """queries (rows to assign) at s times the data, or (reverse) the data at s times the queries; the data rows have unit
    norm, so that their rounded norms tie within a few ulps"""
    rng = np.random.default_rng(seed)
    nb = 4096 if kind == FLAT else 1024
    na = 1024 if kind == ASSIGN else 32
    b = unit_rows(rng, nb, d)
    a = rng.standard_normal((na, d)).astype(np.float32)
    if reverse:
        a = (a / np.linalg.norm(a, axis=1, keepdims=True)).astype(np.float32)
        b = (rng.standard_normal((nb, d)) * s).astype(np.float32)
    else:
        a = (a * s).astype(np.float32)
    return a, b


@pytest.mark.parametrize("reverse", [False, True], ids=["queries-scaled", "data-scaled"])
@pytest.mark.parametrize("name,kind,metric,d", CONFIGS, ids=[c[0] for c in CONFIGS])
def test_scale_separation(oracle, vk, monkeypatch, name, kind, metric, d, reverse):
    """||q|| << max||c|| (and the reverse): the squared-norm share of eps_q carries the selection.  At equal scales the
    shortlist does the work: no row reaches the exact kernel."""
    for i, s in enumerate(SCALES):
        a, b = scaled_problem(kind, d, s, reverse, seed=100 * i + d)
        _, _, ex = check(monkeypatch, oracle, vk, kind, a, b, k={FLAT: 10, PROBE: 16, ASSIGN: 1}[kind], metric=metric)
        if s == 1.0 and kind != PROBE:
            assert ex == 0, f"{name}: {ex} rows went to the exact kernel at equal scales"


@pytest.mark.parametrize("name,kind,metric,d", CONFIGS, ids=[c[0] for c in CONFIGS])
def test_tensor_core_scores_within_margin(oracle, monkeypatch, name, kind, metric, d):
    """The premise of the shortlist, at every scale above: |S~ + const_q - S_ref| <= eps_q, S~ the raw tcgen05 scores
    (vix_debug_tc_scores_f32), S_ref the oracle's fp32 score of the consumer (the flat scan's includes ||q||^2, which S~
    leaves out: const_q = ||q||^2 in float64), eps_q = shortlist_margin with the fp32 row norms the kernels use."""
    import torch
    rel, rel2 = margin(d, metric)
    worst = 0.0
    for reverse in (False, True):
        for i, s in enumerate(SCALES):
            a, b = scaled_problem(kind, d, s, reverse, seed=100 * i + d)
            a = a[:64]
            bn = oracle.centroid_norms(b)
            an = oracle.centroid_norms(a).astype(np.float64)
            ta, tb, tn = (torch.from_numpy(v).cuda() for v in (a, b, bn))
            out = torch.empty((a.shape[0], b.shape[0]), dtype=torch.float32, device="cuda")
            _lib.check(_lib.lib().vix_debug_tc_scores_f32(_lib.ptr(ta), C.c_int64(a.shape[0]), _lib.ptr(tb), C.c_int(b.shape[0]),
                                                          C.c_int(d), C.c_int(metric), _lib.ptr(tn) if metric == 0 else None,
                                                          _lib.ptr(out)))
            st = out.cpu().numpy().astype(np.float64)
            if kind == PROBE:
                ref = oracle.centroid_batch_score(a, b, metric).astype(np.float64)
            elif kind == FLAT and metric == 1:
                ref = -np.stack([oracle.ip_block(r, b) for r in a]).astype(np.float64)
            elif kind == FLAT:
                ref = np.stack([oracle.l2sqr_block(r, b) for r in a]).astype(np.float64)
                st = st + (a.astype(np.float64) ** 2).sum(1)[:, None]
            else:
                ref = np.array([[oracle.km12_l2sq(r, c) for c in b[:256]] for r in a[:16]], np.float64)
                st = st[:16, :256] + (a[:16].astype(np.float64) ** 2).sum(1)[:, None]
                an = an[:16]
            bmax = float(np.float32(np.sqrt(bn.max())))
            eps = rel * np.sqrt(an) * bmax + rel2 * (an + bmax * bmax)
            err = np.abs(st - ref)
            assert np.all(err <= eps[:, None]), f"{name} s={s} reverse={reverse}: |S~ - S| / eps up to {np.max(err / eps[:, None])}"
            worst = max(worst, float(np.max(err / eps[:, None])))
    assert worst > 1e-4, "the scores are not the TF32 path's"


# ------------------------------------------------------------------------------------------------ other data
@pytest.mark.parametrize("kind,metric", [(FLAT, 0), (FLAT, 1), (PROBE, 0), (PROBE, 1), (ASSIGN, 0)])
def test_large_common_offset(oracle, vk, monkeypatch, kind, metric):
    """data far from the origin: scores are large, their differences small (cancellation in ||c||^2 - 2 <q, c>)"""
    rng = np.random.default_rng(7)
    d = 64
    nb, na = (4096, 32) if kind == FLAT else (1024, 1024 if kind == ASSIGN else 32)
    off = rng.standard_normal(d).astype(np.float32) * 256
    b = (rng.standard_normal((nb, d)) + off).astype(np.float32)
    a = (rng.standard_normal((na, d)) + off).astype(np.float32)
    check(monkeypatch, oracle, vk, kind, a, b, k={FLAT: 10, PROBE: 16, ASSIGN: 1}[kind], metric=metric)


@pytest.mark.parametrize("kind,metric", [(FLAT, 0), (FLAT, 1), (PROBE, 0), (PROBE, 1), (ASSIGN, 0)])
def test_near_ties_permuted_rows(oracle, vk, monkeypatch, kind, metric):
    """rows that are coordinate permutations of one vector, spread over the groups: equal norms in exact arithmetic, a few
    ulps apart in every fp32 evaluation order; queries near that vector, at it, and at zero"""
    rng = np.random.default_rng(11)
    d = 96
    nb, na = (8192, 32) if kind == FLAT else (2048, 1024 if kind == ASSIGN else 32)
    b = rng.standard_normal((nb, d)).astype(np.float32) * 2
    v = rng.standard_normal(d).astype(np.float32)
    pos = rng.choice(nb, 96, replace=False)
    for p in pos:
        b[p] = v[rng.permutation(d)]
    a = (v + rng.standard_normal((na, d)) * 1e-3).astype(np.float32)
    a[1] = v
    a[2] = 0.0
    a[3] = b[pos[5]]
    check(monkeypatch, oracle, vk, kind, a, b, k={FLAT: 10, PROBE: 16, ASSIGN: 1}[kind], metric=metric)


NONFINITE = [("query-nan", "a", np.nan), ("query-inf", "a", np.inf), ("data-nan", "b", np.nan), ("data-inf", "b", np.inf)]


@pytest.mark.parametrize("where,side,val", NONFINITE, ids=[n[0] for n in NONFINITE])
@pytest.mark.parametrize("kind,metric", [(FLAT, 0), (FLAT, 1), (PROBE, 0), (PROBE, 1), (ASSIGN, 0)])
def test_non_finite_values(oracle, vk, monkeypatch, kind, metric, where, side, val):
    """a NaN or +inf component in a query (row to assign) or in a base row / centroid.  A NaN query makes T_q NaN: its
    shortlist is empty and the row must go to the exact kernel, not come back as -1.  An infinite base row makes every
    margin infinite: every row of the call goes to the exact kernel."""
    rng = np.random.default_rng(13)
    d = 96
    nb, na = (4096, 32) if kind == FLAT else (1024, 1024 if kind == ASSIGN else 32)
    b = rng.standard_normal((nb, d)).astype(np.float32)
    a = rng.standard_normal((na, d)).astype(np.float32)
    if side == "a":
        a[3, 5] = val
        a[17, 90] = val
    else:
        b[100, 2] = val
    rows = None
    if kind != PROBE:
        rows = 2 if side == "a" else (na if val == np.inf else 0)
    check(monkeypatch, oracle, vk, kind, a, b, k={FLAT: 10, PROBE: 16, ASSIGN: 1}[kind], metric=metric, exact_rows=rows,
          nan_rows_may_differ=(where == "query-nan"))


# ------------------------------------------------------------------------------------------------ gates
GATES = [
    # name, kind, metric, na, nb, d, k, takes the shortlist
    ("probe-kc1023", PROBE, 0, 32, 1023, 64, 16, False), ("probe-kc1024", PROBE, 0, 32, 1024, 64, 16, True),
    ("assign-kc1023", ASSIGN, 0, 1024, 1023, 64, 1, False), ("assign-kc1024", ASSIGN, 0, 1024, 1024, 64, 1, True),
    ("assign-n1023", ASSIGN, 0, 1023, 1024, 64, 1, False),
    ("flat-n4095", FLAT, 0, 32, 4095, 64, 10, False), ("flat-n4096", FLAT, 0, 32, 4096, 64, 10, True),
    ("flat-nq15", FLAT, 0, 15, 4096, 64, 10, False), ("flat-nq16", FLAT, 0, 16, 4096, 64, 10, True),
    ("probe-nq15", PROBE, 1, 15, 1024, 64, 16, False), ("probe-nq16", PROBE, 1, 16, 1024, 64, 16, True),
    ("flat-d98", FLAT, 0, 32, 4096, 98, 10, False), ("probe-d98", PROBE, 0, 32, 1024, 98, 16, False),
    ("assign-d98", ASSIGN, 0, 1024, 1024, 98, 1, False),
    # (d 4096 / 4100 on probe selection: the exact flat-search kernel has no shared-memory tile for rows that long)
    ("probe-d4096", PROBE, 0, 16, 1024, 4096, 8, True), ("probe-d4100", PROBE, 0, 16, 1024, 4100, 8, False),
    ("flat-k256", FLAT, 0, 16, 65536, 32, 256, True), ("flat-k257", FLAT, 0, 16, 65536, 32, 257, False),
    ("probe-k256", PROBE, 1, 16, 16384, 32, 256, True), ("probe-k257", PROBE, 1, 16, 16384, 32, 257, False),
    ("flat-groups128-k64", FLAT, 0, 32, 4096, 64, 64, True), ("flat-groups128-k65", FLAT, 0, 32, 4096, 64, 65, False),
    ("probe-groups32-k16", PROBE, 0, 32, 1024, 64, 16, True), ("probe-groups32-k17", PROBE, 0, 32, 1024, 64, 17, False),
    # k >= n (flat search serves k <= VIX_MAX_K = 512, so n stays below the n >= 4096 gate as well)
    ("flat-k-eq-n", FLAT, 1, 16, 512, 32, 512, False), ("flat-k-gt-n", FLAT, 0, 16, 500, 32, 512, False),
]


@pytest.mark.parametrize("name,kind,metric,na,nb,d,k,tc", GATES, ids=[g[0] for g in GATES])
def test_gates(oracle, vk, monkeypatch, name, kind, metric, na, nb, d, k, tc):
    """each side of every condition that selects the shortlist: both sides give the oracle's answer, and the counter shows
    the side taken"""
    rng = np.random.default_rng(na + nb + d + k)
    b = rng.standard_normal((nb, d)).astype(np.float32)
    a = rng.standard_normal((na, d)).astype(np.float32)
    check(monkeypatch, oracle, vk, kind, a, b, k=k, metric=metric, tc=tc, exact_rows=0 if (tc and kind != PROBE) else None)


# ------------------------------------------------------------------------------------------------ overflow
@pytest.mark.parametrize("kind,metric,k,cap", [(FLAT, 0, 10, 168), (FLAT, 1, 10, 168), (PROBE, 0, 8, 160), (PROBE, 1, 8, 160),
                                               (ASSIGN, 0, 1, 32)])
def test_overflow_duplicates(oracle, vk, monkeypatch, kind, metric, k, cap):
    """cap + 1 exact duplicates of the best row (cap = 4 k + 128 for probe selection and flat search, 32 for assignment):
    the row's shortlist overflows and the exact kernel must return the duplicates in id order"""
    rng = np.random.default_rng(17)
    d = 64
    nb, na = (4096, 32) if kind == FLAT else (1024, 1024 if kind == ASSIGN else 32)
    b = rng.standard_normal((nb, d)).astype(np.float32)
    a = rng.standard_normal((na, d)).astype(np.float32)
    dup = rng.choice(nb, cap + 1, replace=False)
    b[dup] = a[0]
    gi, _, ex = check(monkeypatch, oracle, vk, kind, a, b, k=k, metric=metric)
    assert np.array_equal(np.ravel(gi[0])[:k], np.sort(dup)[:k])
    if kind != PROBE:
        assert ex >= 1, "the overflowing row did not reach the exact kernel"


# ------------------------------------------------------------------------------------------------ PQ encoder
@pytest.mark.parametrize("dsub", [8, 16])
def test_pq_encode_scale_sweep(oracle, vk, monkeypatch, dsub):
    """rows at 2^-30 .. 2^20 of the codewords through the tensor-core encoder (n >= 4096, dsub 8 / 16): the codes equal
    the oracle's and the CUDA-core kernel's (VIX_DISABLE_PQ_TC=1), with centroid norms (CSQ) and without (DOT), plain and
    residual"""
    rng = np.random.default_rng(dsub)
    n, m, ks, kc = 4096, 4, 256, 16
    d = m * dsub
    cb = rng.standard_normal((m, ks, dsub)).astype(np.float32).reshape(-1)
    csq = oracle.pq_centroid_sq(cb, m, ks, dsub, swift=False)
    coarse = rng.standard_normal((kc, d)).astype(np.float32)
    assign = rng.integers(0, kc, n).astype(np.int32)
    s = (2.0 ** rng.integers(-30, 21, n)).astype(np.float32)[:, None]
    r = (rng.standard_normal((n, d)) * s).astype(np.float32)
    x = r
    xr = (coarse[assign] + r).astype(np.float32)         # residuals down to zero (r below the rounding of coarse + r)
    want = {
        "dot": oracle.pq_encode_u8(x, cb, m, ks),
        "csq": oracle.pq_encode_u8(x, cb, m, ks, centroid_sq=csq),
        "res-csq": oracle.pq_encode_u8(xr, cb, m, ks, centroid_sq=csq, coarse=coarse, assign_=assign),
        "res-dot": oracle.pq_encode_u8(xr, cb, m, ks, coarse=coarse, assign_=assign),
    }
    for disable in (None, "1"):
        if disable:
            monkeypatch.setenv("VIX_DISABLE_PQ_TC", disable)
        got = {
            "dot": vk.pq_encode_u8_f32(x, cb, m),
            "csq": vk.pq_encode_u8_f32_withCSQ(x, cb, csq, m),
            "res-csq": vk.pq_encode_residual_u8_f32_withCSQ(xr, cb, csq, coarse, assign, m),
            "res-dot": vk.pq_encode_residual_u8_f32(xr, cb, coarse, assign, m),
        }
        for mode in want:
            bad = np.flatnonzero((got[mode] != want[mode]).any(1))
            assert bad.size == 0, f"{mode} (VIX_DISABLE_PQ_TC={disable}): rows {bad[:8].tolist()} at scales " \
                                  f"{s[bad[:8], 0].tolist()} differ from the oracle"
