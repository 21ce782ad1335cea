"""GPU parity: every call goes through the C ABI of libvindex_b200.so and is compared with the CPU oracle
on the same seeded inputs.  Bars (BASELINE.json north_star): PQ codes and IVF list assignments bit-exact;
distances within 1e-5 relative; top-k id sets equal except at ties inside that tolerance.  Where the GPU
kernel restates the reference's summation order (flat scan, probe scores, LUT, materialising ADC) the
comparison is bit-exact as well."""
import os
import re

import numpy as np
import pytest

import golden_inputs as gi
from conftest import parity_fixture
from vectorindex_b200 import _lib

pytestmark = pytest.mark.gpu

RTOL = 1e-5   # north_star: fp32 relative tolerance for distances


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def assert_topk_close(gd, gi, od, oi, rtol=RTOL, atol=0.0):
    """id sets equal except at ties within tolerance; distances within tolerance."""
    assert gd.shape == od.shape
    for r in range(gd.shape[0]):
        ov = oi[r] >= 0
        gv = gi[r] >= 0
        assert ov.sum() == gv.sum(), f"row {r}: {gv.sum()} results vs oracle {ov.sum()}"
        if ov.sum() == 0:
            continue
        np.testing.assert_allclose(gd[r][gv], od[r][ov], rtol=rtol, atol=atol, err_msg=f"row {r} distances")
        omap = dict(zip(oi[r][ov].tolist(), od[r][ov].tolist()))
        kth = od[r][ov][-1]
        for i, dist in zip(gi[r][gv].tolist(), gd[r][gv].tolist()):
            if i in omap:
                assert abs(dist - omap[i]) <= rtol * abs(omap[i]) + atol, f"row {r} id {i}: {dist} vs {omap[i]}"
            else:   # boundary tie inside the tolerance
                assert abs(dist - kth) <= 4 * rtol * abs(kth) + atol, f"row {r}: id {i} not in oracle set ({dist} vs kth {kth})"


# ------------------------------------------------------------------------------------------------ PQ encode
ENC_SHAPES = [(1000, 64, 8), (777, 48, 6), (300, 40, 4), (513, 96, 48), (260, 128, 16), (100, 24, 24)]


@pytest.mark.parametrize("n,d,m", ENC_SHAPES)
def test_pq_encode_bit_exact_all_entry_points(oracle, vk, n, d, m):
    rng = np.random.default_rng(n + d)
    ks, kc, dsub = 256, 7, d // m
    x = rng.standard_normal((n, d)).astype(np.float32)
    cb = (rng.standard_normal(m * ks * dsub) * 0.7).astype(np.float32)
    coarse = (rng.standard_normal((kc, d)) * 0.5).astype(np.float32)
    assign = rng.integers(0, kc, n).astype(np.int32)
    csq = oracle.pq_centroid_sq(cb, m, ks, dsub, swift=True)
    nodot = _lib.PQEncodeOpts(0, False, False, 8, 0, 0, 0)
    assert np.array_equal(vk.pq_encode_u8_f32(x, cb, m), oracle.pq_encode_u8(x, cb, m, ks, use_dot=True))
    assert np.array_equal(vk.pq_encode_u8_f32(x, cb, m, opts=nodot), oracle.pq_encode_u8(x, cb, m, ks, use_dot=False))
    assert np.array_equal(vk.pq_encode_u8_f32_withCSQ(x, cb, csq, m), oracle.pq_encode_u8(x, cb, m, ks, centroid_sq=csq))
    assert np.array_equal(vk.pq_encode_residual_u8_f32(x, cb, coarse, assign, m),
                          oracle.pq_encode_u8(x, cb, m, ks, coarse=coarse, assign_=assign, use_dot=True))
    assert np.array_equal(vk.pq_encode_residual_u8_f32(x, cb, coarse, assign, m, opts=nodot),
                          oracle.pq_encode_u8(x, cb, m, ks, coarse=coarse, assign_=assign, use_dot=False))
    assert np.array_equal(vk.pq_encode_residual_u8_f32_withCSQ(x, cb, csq, coarse, assign, m),
                          oracle.pq_encode_u8(x, cb, m, ks, centroid_sq=csq, coarse=coarse, assign_=assign))
    if m % 2 == 0:
        cb4 = (rng.standard_normal(m * 16 * dsub) * 0.7).astype(np.float32)
        assert np.array_equal(vk.pq_encode_u4_f32(x, cb4, m), oracle.pq_encode_u4(x, cb4, m, 16))
        assert np.array_equal(vk.pq_encode_residual_u4_f32(x, cb4, coarse, assign, m),
                              oracle.pq_encode_u4(x, cb4, m, 16, coarse=coarse, assign_=assign))


@pytest.mark.parametrize("n,d,m", [(700, 1024, 8), (300, 1536, 8), (130, 600, 4)])
def test_pq_encode_long_subvectors(oracle, vk, n, d, m):
    """d / m = 128 (ResidualKernelTests.swift:126-200: fused residual codes == codes of the materialised residuals), 192
    and 150: the staged [dsub x rows] tiles of the residual variants need the 64-row CTAs."""
    rng = np.random.default_rng(d + m)
    ks, kc, dsub = 256, 9, d // m
    x = rng.uniform(-1, 1, (n, d)).astype(np.float32)
    cb = rng.uniform(-1, 1, m * ks * dsub).astype(np.float32)
    coarse = rng.uniform(-1, 1, (kc, d)).astype(np.float32)
    assign = rng.integers(0, kc, n).astype(np.int32)
    nodot = _lib.PQEncodeOpts(0, False, False, 8, 0, 0, 0)
    fused = vk.pq_encode_residual_u8_f32(x, cb, coarse, assign, m)
    assert np.array_equal(fused, oracle.pq_encode_u8(x, cb, m, ks, coarse=coarse, assign_=assign, use_dot=True))
    assert np.array_equal(vk.pq_encode_residual_u8_f32(x, cb, coarse, assign, m, opts=nodot),
                          oracle.pq_encode_u8(x, cb, m, ks, coarse=coarse, assign_=assign, use_dot=False))
    assert np.array_equal(vk.pq_encode_u8_f32(x, cb, m), oracle.pq_encode_u8(x, cb, m, ks, use_dot=True))
    assert np.array_equal(fused, vk.pq_encode_u8_f32((x - coarse[assign]).astype(np.float32), cb, m))


@pytest.mark.parametrize("n,d,m", [(20000, 128, 16), (9000, 64, 4), (12345, 48, 6), (5000, 512, 64)])
def test_pq_encode_tensor_core_shortlist_is_exact(oracle, vk, n, d, m, monkeypatch):
    """n >= 4096 with d / m in {8, 16} takes the tcgen05 shortlist (vix_pq_tc.cu): one TF32 MMA per (row tile, sub-space),
    finalists re-evaluated in the reference's arithmetic.  The codes must equal the oracle's restatement of pq_encode.c and
    the CUDA-core kernel's (VIX_DISABLE_PQ_TC=1) bit for bit -- with and without centroid norms, plain and residual --
    including duplicated codewords (tie -> smaller k), rows that ARE codewords, zero rows, rows of large magnitude (the
    error bound scales with ||x_j||) and near-ties (codewords 1 ulp apart)."""
    rng = np.random.default_rng(n + d)
    ks, dsub, kc = 256, d // m, 7
    x = rng.uniform(-1, 1, (n, d)).astype(np.float32)
    cb = rng.uniform(-1, 1, (m, ks, dsub)).astype(np.float32)
    cb[:, 200] = cb[:, 17]                                                  # exact duplicates: the smaller index must win
    cb[:, 201] = np.nextafter(cb[:, 18], np.float32(2))                     # near-ties, one ulp apart
    x[:m * 8:8] = np.concatenate([cb[j, 17] for j in range(m)])            # rows that are codeword 17 in every sub-space
    x[1] = 0.0
    x[2] *= 1000.0
    x[3] *= 1e-4
    cbf = cb.reshape(-1)
    csq = oracle.pq_centroid_sq(cbf, m, ks, dsub, swift=False)
    coarse = rng.uniform(-1, 1, (kc, d)).astype(np.float32)
    assign = rng.integers(0, kc, n).astype(np.int32)
    want = oracle.pq_encode_u8(x, cbf, m, ks)
    want_csq = oracle.pq_encode_u8(x, cbf, m, ks, centroid_sq=csq)
    want_res = oracle.pq_encode_u8(x, cbf, m, ks, centroid_sq=csq, coarse=coarse, assign_=assign)
    want_res_dot = oracle.pq_encode_u8(x, cbf, m, ks, coarse=coarse, assign_=assign)
    for disable in (None, "1"):                                             # tensor-core path, then the CUDA-core kernel
        if disable:
            monkeypatch.setenv("VIX_DISABLE_PQ_TC", disable)
        assert np.array_equal(vk.pq_encode_u8_f32(x, cbf, m), want)
        assert np.array_equal(vk.pq_encode_u8_f32_withCSQ(x, cbf, csq, m), want_csq)
        assert np.array_equal(vk.pq_encode_residual_u8_f32_withCSQ(x, cbf, csq, coarse, assign, m), want_res)
        assert np.array_equal(vk.pq_encode_residual_u8_f32(x, cbf, coarse, assign, m), want_res_dot)
    assert (want[:m * 8:8] == 17).all()


def test_pq_encode_reference_fixture_and_layouts(oracle, vk):
    """fixture of PQEncodeParity_AoS_C_vs_Swift_Tests.swift:5-31 against the reference encoder's stored outputs
    (tests/golden/cpq_encode_reference_fixtures.npz), including the SoA-blocked and interleaved output layouts
    (pq_encode.c:260-276)."""
    x, cb, coarse, assign = parity_fixture(n=70)
    csq = oracle.pq_centroid_sq(cb, 8, 256, 4, swift=False)
    got = vk.pq_encode_u8_f32_withCSQ(x, cb, csq, 8)
    assert got[0].tolist() == [212, 186, 160, 117, 255, 154, 186, 249]
    gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cpq_encode_reference_fixtures.npz"))
    assert np.array_equal(got, gold["parity70.u8_csq"])
    m = 8
    for name, layout, B, g in gi.LAYOUTS:
        o = _lib.PQEncodeOpts(layout, True, False, 8, 0, B, g)
        ours = np.asarray(vk.pq_encode_u8_f32(x, cb, m, opts=o)).reshape(-1)
        ref = gold[f"layout.{name}"]
        assert np.array_equal(ours[:ref.size], ref), f"layout {layout} B={B} g={g}"


def test_pq_encode_empty_and_device_pointers(oracle, vk):
    import torch
    rng = np.random.default_rng(3)
    d, m = 32, 4
    cb = rng.standard_normal(m * 256 * 8).astype(np.float32)
    assert vk.pq_encode_u8_f32(np.zeros((0, d), np.float32), cb, m).shape == (0, m)
    x = rng.standard_normal((500, d)).astype(np.float32)
    want = oracle.pq_encode_u8(x, cb, m, 256, use_dot=True)
    got = vk.pq_encode_u8_f32(torch.from_numpy(x).cuda(), torch.from_numpy(cb).cuda(), m)
    assert got.is_cuda and np.array_equal(got.cpu().numpy(), want)


# ------------------------------------------------------------------------------------------------ assignment
@pytest.mark.parametrize("n,kc,d", [(3000, 100, 128), (2500, 257, 96), (1000, 33, 37), (700, 5, 8), (300, 70, 768)])
def test_ivf_assign_bit_exact(oracle, vk, n, kc, d):
    rng = np.random.default_rng(n + kc)
    x = rng.standard_normal((n, d)).astype(np.float32)
    c = x[rng.choice(n, kc, replace=False)] + (rng.standard_normal((kc, d)) * 0.1).astype(np.float32)
    oa, od = oracle.assign(x, c)
    ga, gd = vk.ivf_assign_f32(x, c, return_dist=True)
    assert np.array_equal(ga, oa)
    assert np.array_equal(bits(gd), bits(od))


@pytest.mark.parametrize("n,kc,d,kind", [(6000, 2048, 96, "gauss"), (5000, 1500, 128, "sift"), (3000, 4096, 100, "gauss"),
                                         (2000, 1024, 768, "gauss")])
def test_ivf_assign_tensor_core_shortlist_is_exact(oracle, vk, n, kc, d, kind):
    """kc >= 1024 takes the tcgen05 shortlist + exact rescoring path: same assignment and distance bits as the
    oracle, including duplicated centroids (tie -> lower index) and integer-valued data."""
    from vectorindex_b200 import datagen
    rng = np.random.default_rng(n + kc + d)
    if kind == "sift":
        x = datagen.sift_like(n + kc, d, 64, 11)
        c = np.ascontiguousarray(x[n:])
        x = np.ascontiguousarray(x[:n])
    else:
        x = rng.standard_normal((n, d)).astype(np.float32)
        c = (x[rng.integers(0, n, kc)] + rng.standard_normal((kc, d)).astype(np.float32) * 0.3).astype(np.float32)
    c[kc - 1] = c[7]
    c[kc // 2] = c[7]                                               # three identical centroids
    x[:5] = c[[7, 8, 9, kc - 1, kc // 2]]                           # points sitting exactly on centroids
    oa, od = oracle.assign(x, c)
    ga, gd = vk.ivf_assign_f32(x, c, return_dist=True)
    assert np.array_equal(ga, oa)
    assert np.array_equal(bits(gd), bits(od))
    assert ga[0] == 7 and ga[3] == 7 and ga[4] == 7


def test_ivf_assign_ties_go_to_lower_index(oracle, vk):
    """heavy ties: integer-valued SIFT-like data and duplicated centroids (KMeansMiniBatchKernel.swift:352)."""
    from vectorindex_b200 import datagen
    x = datagen.sift_like(4000, 32, 50, 77)
    c = np.concatenate([x[:40], x[:40], x[100:120]]).astype(np.float32)   # centroids 40..79 duplicate 0..39
    oa, _ = oracle.assign(x, c)
    ga = vk.ivf_assign_f32(x, c)
    assert np.array_equal(ga, oa)
    assert (ga[:40] == np.arange(40)).all()


@pytest.mark.parametrize("metric", [0, 1])
def test_ivf_assign_metric(oracle, vk, metric):
    rng = np.random.default_rng(5)
    x = rng.standard_normal((1500, 64)).astype(np.float32)
    c = rng.standard_normal((90, 64)).astype(np.float32)
    assert np.array_equal(vk.ivf_assign_metric_f32(x, c, metric), oracle.assign_metric(x, c, metric))


# ------------------------------------------------------------------------------------------------ flat scan
@pytest.mark.parametrize("n,d,nq,k,metric", [(5000, 128, 70, 10, 0), (3000, 256, 33, 10, 0), (4000, 100, 17, 5, 1),
                                            (2000, 768, 20, 10, 1), (900, 37, 9, 32, 0), (20, 16, 4, 50, 0)])
def test_flat_search_matches_reference_kernels(oracle, vk, n, d, nq, k, metric):
    rng = np.random.default_rng(n + d + k)
    xb = rng.standard_normal((n, d)).astype(np.float32)
    q = rng.standard_normal((nq, d)).astype(np.float32)
    od, oi, _ = oracle.flat_search(q, xb, k, metric)
    gd, gi = vk.flat_search_f32(q, xb, k, metric)
    assert np.array_equal(gi, oi)
    assert np.array_equal(bits(gd), bits(od))


def test_flat_search_bench_fixture_and_ties(oracle, vk):
    """reference benchmark recipe (unit-norm LCG vectors, seeds 123/321) + duplicated rows (ties -> smaller id)."""
    from vectorindex_b200 import datagen
    xb = datagen.bench_vectors(3000, 128, 123)
    xb = np.concatenate([xb, xb[:500]])            # rows 3000.. duplicate rows 0..499
    q = datagen.bench_vectors(40, 128, 321)
    q[:5] = xb[:5]
    od, oi, _ = oracle.flat_search(q, xb, 10, 0)
    gd, gi = vk.flat_search_f32(q, xb, 10, 0)
    assert np.array_equal(gi, oi) and np.array_equal(bits(gd), bits(od))
    assert gi[0, 0] == 0 and gi[0, 1] == 3000


@pytest.mark.parametrize("n,d,nq,k,metric", [(100000, 128, 200, 10, 0), (20000, 96, 64, 32, 1), (9000, 768, 40, 5, 0),
                                             (12000, 100, 33, 20, 0)])
def test_flat_search_tensor_core_shortlist_is_exact(oracle, vk, n, d, nq, k, metric):
    """n >= 4096 takes the tcgen05 shortlist + exact rescoring path (C1-shaped first case): ids and distance bits equal
    the oracle's restatement of the reference kernels, including duplicated base rows (tie -> smaller id)."""
    from vectorindex_b200 import datagen
    xb = datagen.bench_vectors(n, d, 123) if metric == 0 else np.random.default_rng(n).standard_normal((n, d)).astype(np.float32)
    q = datagen.bench_vectors(nq, d, 321)
    xb[n // 2] = xb[17]
    xb[n - 1] = xb[17]
    q[0] = xb[17]
    od, oi, _ = oracle.flat_search(q, xb, k, metric)
    gd, gi = vk.flat_search_f32(q, xb, k, metric)
    assert np.array_equal(gi, oi)
    assert np.array_equal(bits(gd), bits(od))
    assert gi[0, 0] == 17 and set(gi[0, :3]) == {17, n // 2, n - 1}


@pytest.mark.parametrize("n,d,nq,k", [(3000, 48, 40, 10), (9000, 768, 24, 7), (500, 130, 9, 500)])
def test_flat_cosine_matches_reference_two_pass(oracle, vk, n, d, nq, k):
    """Cosine.run without cached norms (Cosine.swift:94-119): InnerProduct.run, (dot * qInv) * inv, clamp, .max selection,
    API distance 1 - similarity (FlatIndexOptimized.swift:468-470) -- ids and distance bits equal the oracle's, through
    the kernel-level entry point and through a FLAT index with external ids; a zero row scores 0 (distance 1)."""
    from vectorindex_b200.index import FlatIndex
    rng = np.random.default_rng(n + d)
    xb = rng.standard_normal((n, d)).astype(np.float32) * rng.uniform(0.1, 5.0, (n, 1)).astype(np.float32)
    xb[7] = 0.0
    xb[11] = xb[3] * np.float32(2.0)                                  # same direction as row 3: ties broken by the id
    q = rng.standard_normal((nq, d)).astype(np.float32)
    q[0] = xb[3]
    od, oi, _ = oracle.flat_search(q, xb, k, 2)
    gd, gi = vk.flat_search_f32(q, xb, k, 2)
    assert np.array_equal(gi, oi) and np.array_equal(bits(gd), bits(od))
    assert gd.min() >= 0.0 and gd.max() <= 2.0
    ids = np.arange(n, dtype=np.int64) * 3 + 2
    idx = FlatIndex(d, "cosine")
    idx.batch_insert(xb, ids)
    fd, fi = idx.batch_search(q, k)
    assert np.array_equal(fi, ids[oi]) and np.array_equal(bits(fd), bits(od))


def test_cosine_is_flat_only():
    from vectorindex_b200 import VectorIndexError
    from vectorindex_b200.index import IVFPQIndex
    with pytest.raises(VectorIndexError):
        IVFPQIndex(32, "cosine", nlist=4, nprobe=2, m=4)


def test_flat_search_edge_cases(vk):
    q = np.zeros((3, 8), dtype=np.float32)
    d, i = vk.flat_search_f32(q, np.zeros((0, 8), np.float32), 4)
    assert (i == -1).all() and np.isnan(d).all()
    d, i = vk.flat_search_f32(q, np.ones((5, 8), np.float32), 0)
    assert d.shape == (3, 0)
    from vectorindex_b200 import VectorIndexError
    with pytest.raises(VectorIndexError):
        vk.flat_search_f32(q, np.ones((5, 9), np.float32), 2)


def test_block_scores_and_norms(oracle, vk):
    rng = np.random.default_rng(11)
    for d in (16, 100, 128, 256, 300):
        xb = rng.standard_normal((700, d)).astype(np.float32)
        q = rng.standard_normal(d).astype(np.float32)
        assert np.array_equal(bits(vk.l2sqr_f32_block(q, xb)), bits(oracle.l2sqr_block(q, xb)))
        assert np.array_equal(bits(vk.ip_f32_block(q, xb)), bits(oracle.ip_block(q, xb)))
        xn = oracle.centroid_norms(xb)
        assert np.array_equal(bits(vk.row_norms_f32(xb)), bits(xn))
        assert np.array_equal(bits(vk.l2sqr_f32_block(q, xb, xb_norm=xn)), bits(oracle.l2sqr_block(q, xb, xb_norm=xn)))


# ------------------------------------------------------------------------------------------------ selection
def test_select_and_merge_topk(oracle, vk):
    rng = np.random.default_rng(2)
    s = np.round(rng.standard_normal(50000) * 50).astype(np.float32)       # many ties
    for k, order in ((10, 0), (100, 1), (1, 0)):
        os_, oi = oracle.select_topk(s, k, order)
        gs, gi = vk.selectTopK(s, k, order)
        assert np.array_equal(gi, oi) and np.array_equal(bits(gs), bits(os_))
    gs, gi = vk.selectTopK(np.array([5, 3, 8, 1, 9], np.float32), 3, 1, ids=np.arange(10, 15, dtype=np.int32))
    assert gs.tolist() == [9, 8, 5] and gi.tolist() == [14, 12, 10]          # TelemetryRecorderTests.swift:229-241
    # merge of 3 sorted lists per row
    batch, nl, st, k = 6, 3, 8, 10
    sc = np.sort(np.round(rng.standard_normal((batch, nl, st)) * 3), axis=2).astype(np.float32)
    ids = rng.permutation(batch * nl * st).reshape(batch, nl, st).astype(np.int64)
    lens = rng.integers(0, st + 1, (batch, nl)).astype(np.int32)
    gs, gi = vk.mergeTopK(sc, ids, k, 0, lens)
    for b in range(batch):
        lists = []
        for l in range(nl):
            n_ = lens[b, l]
            o = np.lexsort((ids[b, l, :n_], sc[b, l, :n_]))
            lists.append((sc[b, l, :n_][o], ids[b, l, :n_][o].astype(np.int32)))
        ms, mi = oracle.merge_topk(lists, k, 0)
        assert gi[b, :mi.size].tolist() == mi.tolist() and (gi[b, mi.size:] == -1).all()
        assert np.array_equal(bits(gs[b, :ms.size]), bits(ms + np.float32(0)))   # keys canonicalise -0 to +0


# ------------------------------------------------------------------------------------------------ exact re-rank (Kernel #40)
@pytest.mark.parametrize("d,metric,norms", [(96, 0, False), (128, 0, True), (320, 0, False), (64, 1, False)])
def test_rerank_exact_topk(oracle, vk, d, metric, norms):
    """rerank_exact_topk with the DenseArray reader: reference kernel scores of the candidate rows (oracle restatement
    of L2Sqr.run / InnerProduct.run), missing ids skipped, ties -> smaller id, padded with the sentinel."""
    rng = np.random.default_rng(d + metric)
    n, nq, c, k = 5000, 20, 200, 12
    xb = np.round(rng.standard_normal((n, d)) * 2).astype(np.float32)          # integer-valued: ties
    q = np.round(rng.standard_normal((nq, d)) * 2).astype(np.float32)
    cand = rng.integers(0, n, (nq, c)).astype(np.int64)
    cand[:, 5] = -1                                                            # missing
    cand[:, 9] = n + 3                                                         # out of range -> missing
    cand[3, 20:] = -1                                                          # fewer than k present
    cand[3, 12:20] = -1
    xn = (xb.astype(np.float64) ** 2).sum(1).astype(np.float32) if norms else None     # caller-supplied ||x||^2
    gs, gi = vk.rerank_exact_topk(q, cand, xb, k, metric, xn)
    for r in range(nq):
        ids = np.array([v for v in cand[r] if 0 <= v < n], dtype=np.int64)
        rows = xb[ids]
        if metric == 1:
            sc = oracle.ip_block(q[r], rows)
        elif norms:
            qn = np.float32(0)
            for v in q[r]:
                qn = np.float32(qn + np.float32(v * v))                        # norm2: sequential sum (ExactRerank.swift:243)
            sc = oracle.l2sqr_block(q[r], rows, xn[ids], float(qn))
        else:
            sc = oracle.l2sqr_block(q[r], rows)
        order = np.lexsort((ids, -sc if metric == 1 else sc))[:k]
        want_i = np.full(k, -1, np.int64); want_s = np.full(k, -np.inf if metric == 1 else np.inf, np.float32)
        want_i[:order.size] = ids[order]; want_s[:order.size] = sc[order]
        assert np.array_equal(gi[r], want_i), r
        assert np.array_equal(bits(gs[r]), bits(want_s)), r


# ------------------------------------------------------------------------------------------------ tensor-core shortlist
@pytest.mark.parametrize("nq,kc,d,metric", [(300, 2048, 96, 0), (257, 1500, 128, 1), (130, 4096, 100, 0), (64, 1024, 768, 1)])
def test_tensor_core_scores_within_tf32_bound(vk, nq, kc, d, metric):
    """raw tcgen05 (kind::tf32) scores of the shortlist pass: |S~ - S| <= the bound the threshold uses."""
    import ctypes as C
    import torch
    from vectorindex_b200 import _lib
    rng = np.random.default_rng(nq + kc)
    q = rng.standard_normal((nq, d)).astype(np.float32)
    c = rng.standard_normal((kc, d)).astype(np.float32) * 2
    cn = (c.astype(np.float64) ** 2).sum(1).astype(np.float32)
    tq, tc_, tn = torch.from_numpy(q).cuda(), torch.from_numpy(c).cuda(), torch.from_numpy(cn).cuda()
    out = torch.empty((nq, kc), dtype=torch.float32, device="cuda")
    _lib.check(_lib.lib().vix_debug_tc_scores_f32(_lib.ptr(tq), C.c_int64(nq), _lib.ptr(tc_), C.c_int(kc), C.c_int(d),
                                                  C.c_int(metric), _lib.ptr(tn) if metric == 0 else None, _lib.ptr(out)))
    got = out.cpu().numpy().astype(np.float64)
    dot = q.astype(np.float64) @ c.astype(np.float64).T
    want = cn[None, :].astype(np.float64) - 2 * dot if metric == 0 else -dot
    rel = (2.0 if metric == 0 else 1.0) * 1.25 * (2.0 / 1024 + d / 4194304.0)
    bound = rel * np.linalg.norm(q, axis=1)[:, None] * np.linalg.norm(c, axis=1).max()
    assert np.all(np.abs(got - want) <= bound), float(np.max(np.abs(got - want) / bound))
    assert np.max(np.abs(got - want) / bound) > 1e-4          # and it really is the TF32 path, not fp32


@pytest.mark.parametrize("nq,kc,d,nprobe,metric", [(500, 4096, 96, 32, 0), (333, 2048, 128, 16, 1), (200, 8192, 64, 64, 0),
                                                   (150, 3000, 100, 8, 0)])
def test_tensor_core_probe_selection_is_exact(oracle, vk, nq, kc, d, nprobe, metric):
    """probe lists through the tensor-core shortlist + exact rescoring == the oracle's, bit for bit (ids and scores),
    including heavy ties (integer-valued data)."""
    rng = np.random.default_rng(kc + d)
    c = np.round(rng.standard_normal((kc, d)) * 3).astype(np.float32)
    q = np.round(rng.standard_normal((nq, d)) * 3).astype(np.float32)
    c[kc // 2] = c[kc // 3]                                      # exact duplicate centroids: tie -> lower index
    oi, os_ = oracle.probe_select_batch(q, c, nprobe, metric)
    gi, gs = vk.ivf_select_nprobe_batch_f32(q, c, nprobe, metric)
    assert np.array_equal(gi, oi)
    assert np.array_equal(bits(gs), bits(os_))


# ------------------------------------------------------------------------------------------------ coarse probing
@pytest.mark.parametrize("metric", [0, 1])
def test_centroid_scores_and_probe_selection(oracle, vk, metric):
    rng = np.random.default_rng(9)
    q = rng.standard_normal((150, 96)).astype(np.float32)
    c = rng.standard_normal((300, 96)).astype(np.float32)
    c[200:230] = c[10:40]                                                  # duplicated centroids => score ties
    assert np.array_equal(bits(vk.centroid_batch_score(q, c, metric)), bits(oracle.centroid_batch_score(q, c, metric)))
    oi, os_ = oracle.probe_select_batch(q, c, 32, metric)
    gi, gs = vk.ivf_select_nprobe_batch_f32(q, c, 32, metric)
    assert np.array_equal(gi, oi) and np.array_equal(bits(gs), bits(os_))


def test_centroid_scores_cosine_guarded(oracle, vk):
    """CentroidBatchScore.swift:70-84: 1 - <q, c> qInv cInv with the near-zero-norm guard, bit for bit (zero centroid, zero
    query and a tiny-norm centroid under the guard => exactly 1)."""
    rng = np.random.default_rng(21)
    q = rng.standard_normal((70, 96)).astype(np.float32)
    c = (rng.standard_normal((300, 96)) * rng.uniform(0.1, 3.0, (300, 1))).astype(np.float32)
    c[7] = 0.0
    c[9] = 1e-6 * c[9]
    c[11] = 1e-9
    q[3] = 0.0
    got = vk.centroid_batch_score(q, c, 2)
    want = oracle.centroid_batch_score(q, c, 2)
    assert np.array_equal(bits(got), bits(want))
    assert (got[:, 7] == 1.0).all() and (got[3] == 1.0).all()
    cn = oracle.centroid_norms(c)
    assert np.array_equal(bits(vk.centroid_batch_score(q, c, 2, cn)), bits(want))
    # IVFCosineCentroidEdgeCaseTests.swift:27-62: the tiny-norm centroid scores exactly 1, the identical direction ~0
    c3 = np.zeros((3, 8), np.float32)
    c3[0, :2] = 1.0; c3[1, 0] = 1.0; c3[2, 0] = 1e-8
    q3 = np.zeros((1, 8), np.float32)
    q3[0, :2] = 1.0
    s3 = vk.centroid_batch_score(q3, c3, 2)[0]
    assert s3[2] == np.float32(1.0) and abs(float(s3[0])) <= 1e-6 and s3[1] < s3[2]


@pytest.mark.parametrize("metric", [0, 1])
def test_probe_selection_long_rows(oracle, vk, metric):
    """IVFSelectTests.swift:578-609: d = 2048, 100 centroids, nprobe = 10 -- one thread per pair + selection on the
    materialised block; scores and lists bit for bit, also with disabled lists."""
    rng = np.random.default_rng(2048 + metric)
    q = rng.uniform(-1, 1, (21, 2048)).astype(np.float32)
    c = rng.uniform(-1, 1, (100, 2048)).astype(np.float32)
    c[40:45] = c[3:8]                                                      # score ties
    assert np.array_equal(bits(vk.centroid_batch_score(q, c, metric)), bits(oracle.centroid_batch_score(q, c, metric)))
    oi, os_ = oracle.probe_select_batch(q, c, 10, metric)
    gi, gs = vk.ivf_select_nprobe_batch_f32(q, c, 10, metric)
    assert np.array_equal(gi, oi) and np.array_equal(bits(gs), bits(os_))
    gi1, _ = vk.ivf_select_nprobe_batch_f32(q[:1], c, 10, metric)           # the reference test's single query
    assert np.array_equal(gi1, oi[:1])
    mask = np.zeros(2, dtype=np.uint64)
    mask[0] = np.uint64((1 << 3) | (1 << 40) | (1 << 63))
    mask[1] = np.uint64(1 << 5)                                            # list 69
    gm, _ = vk.ivf_select_nprobe_batch_f32(q, c, 10, metric, disabled_lists=mask)
    full = oracle.centroid_batch_score(q, c, metric)
    keep = np.array([i for i in range(100) if i not in (3, 40, 63, 69)])
    for r in range(q.shape[0]):
        order = keep[np.lexsort((keep, full[r][keep]))[:10]]
        assert gm[r].tolist() == order.tolist()


def test_probe_selection_pins_and_padding(oracle, vk):
    cents = np.ones((50, 8), dtype=np.float32)                              # IVFSelectTests.swift:305-347
    gi, _ = vk.ivf_select_nprobe_batch_f32(np.zeros((2, 8), np.float32), cents, 20)
    assert gi[0].tolist() == list(range(20))
    gi, gs = vk.ivf_select_nprobe_batch_f32(np.zeros((2, 8), np.float32), cents[:5], 8)   # nprobe > kc
    assert gi[1].tolist() == [0, 1, 2, 3, 4, -1, -1, -1] and np.isnan(gs[1, 5:]).all()
    mask = np.array([0b10110], dtype=np.uint64)                            # lists 1, 2, 4 disabled
    gi, _ = vk.ivf_select_nprobe_batch_f32(np.zeros((1, 8), np.float32), cents[:6], 3, disabled_lists=mask)
    assert gi[0].tolist() == [0, 3, 5]


# ------------------------------------------------------------------------------------------------ a16 seam
def test_accel_rank_candidates_reference_fixture(vk):
    """AccelerableIndexTests.swift:14-66: the reference test's three stored vectors and query [2, 3, 4], euclidean, k = 2:
    getCandidates hands over all three rows; the accelerated side answers with indices INTO that block, best first, and
    API distances (the shape of AcceleratedResults; the test itself feeds example numbers to finalizeResults).  Rows 0 and 1
    are the nearest, at sqrt(3) and sqrt(12)."""
    cand = np.array([[1, 2, 3], [4, 5, 6], [7, 8, 9]], dtype=np.float32)
    idx, dist = vk.accel_rank_candidates(np.array([[2, 3, 4]], dtype=np.float32), cand, 2)
    assert idx.tolist() == [[0, 1]]
    np.testing.assert_allclose(dist[0], [3 ** 0.5, 12 ** 0.5], rtol=1e-6)
    assert dist.dtype == np.float32 and idx.dtype == np.int32


@pytest.mark.parametrize("metric", [0, 1, 2])
@pytest.mark.parametrize("c,d,nq,k", [(700, 64, 9, 10), (5000, 128, 40, 10), (3, 16, 2, 10), (257, 96, 1, 1)])
def test_accel_rank_candidates_equals_flat_search(oracle, vk, metric, c, d, nq, k):
    """The AccelerableIndex seam (AccelerableIndex.swift:15-127, 130-194): candidates [c x d] row-major in, per query the
    best-first (indices into the candidate block, API distances) out == the reference's flat scoring + selectTopK over that
    block (FlatIndexOptimized.swift:390-477), bit for bit, incl. duplicate candidates (tie -> smaller index) and c < k."""
    rng = np.random.default_rng(1000 * metric + c)
    cand = rng.standard_normal((c, d)).astype(np.float32)
    if c > 20:
        cand[c // 2:c // 2 + 6] = cand[3:9]                                # exact ties
    q = rng.standard_normal((nq, d)).astype(np.float32)
    q[0] = cand[min(5, c - 1)]
    od, oi, _ = oracle.flat_search(q, cand, k, metric)
    gi, gd = vk.accel_rank_candidates(q, cand, k, metric)
    assert np.array_equal(gi.astype(np.int64), oi.astype(np.int64))
    valid = oi >= 0
    assert np.array_equal(bits(gd)[valid], bits(od)[valid])
    assert np.isnan(gd[~valid]).all()
    # nothing to rank: k <= 0 and an empty candidate block
    assert vk.accel_rank_candidates(q, cand, 0, metric)[0].shape == (nq, 0)
    ei, ed = vk.accel_rank_candidates(q, np.zeros((0, d), np.float32), 3, metric)
    assert (ei == -1).all() and np.isnan(ed).all()


# ------------------------------------------------------------------------------------------------ LUT + ADC
def test_pq_query_subnorms(oracle, vk):
    """pq_query_subnorms_f32 (PQLUT.swift:174-187): ||q_j||^2 in the LUT kernels' reduction order, bit for bit; feeding them
    to the oracle's pq_lut_l2 (its qSubNorms argument) reproduces the table the CUDA library builds on its own."""
    rng = np.random.default_rng(174)
    for d, m in ((128, 16), (96, 48), (768, 64), (40, 4)):
        q = rng.standard_normal((7, d)).astype(np.float32)
        got = vk.pq_query_subnorms_f32(q, m)
        dsub = d // m
        want = np.array([[oracle.lut_dot(q[i, j * dsub:(j + 1) * dsub], q[i, j * dsub:(j + 1) * dsub]) for j in range(m)]
                         for i in range(q.shape[0])], dtype=np.float32)
        assert np.array_equal(bits(got), bits(want))
        cb = rng.standard_normal(m * 256 * dsub).astype(np.float32)
        cn = oracle.pq_centroid_sq(cb, m, 256, dsub, swift=False)
        lut = vk.pq_lut_batch_l2_f32(q, cb, m, 256, cn)
        for i in range(q.shape[0]):
            assert np.array_equal(bits(lut[i]), bits(oracle.pq_lut_l2(q[i], cb, m, 256, cn, q_sub_norms=got[i])))


def test_fused_residual_lut_equals_lut_of_materialised_residual(oracle, vk):
    """ResidualKernelTests.swift:208-270: pq_lut_residual_l2_f32(q, c) == pq_lut_l2_f32(q - c) -- on the CUDA library, and
    both equal to the oracle's tables bit for bit (reference shape d 512, m 8, ks 256, plus a batch of residual shapes)."""
    rng = np.random.default_rng(208)
    for d, m in ((512, 8), (96, 48), (128, 16)):
        ks, nq, kc = 256, 6, 4
        q = rng.uniform(-1, 1, (nq, d)).astype(np.float32)
        coarse = rng.uniform(-1, 1, (kc, d)).astype(np.float32)
        cids = rng.integers(0, kc, nq).astype(np.int32)
        cb = rng.uniform(-1, 1, m * ks * (d // m)).astype(np.float32)
        fused = vk.pq_lut_residual_l2_f32(q, cids, coarse, cb, m, ks)
        plain = vk.pq_lut_batch_l2_f32((q - coarse[cids]).astype(np.float32), cb, m, ks)
        assert np.array_equal(bits(fused), bits(plain))
        for i in range(nq):
            assert np.array_equal(bits(fused[i]), bits(oracle.pq_lut_residual_l2(q[i], coarse[cids[i]], cb, m, ks)))
        cn = oracle.pq_centroid_sq(cb, m, ks, d // m, swift=False)
        fn = vk.pq_lut_residual_l2_f32(q, cids, coarse, cb, m, ks, cn)
        pn = vk.pq_lut_batch_l2_f32((q - coarse[cids]).astype(np.float32), cb, m, ks, cn)
        assert np.max(np.abs(fn - pn)) < 1e-4                              # the reference test's own accuracy


@pytest.mark.parametrize("d,m", [(128, 16), (96, 48), (768, 64), (40, 4)])
def test_pq_lut_bit_exact(oracle, vk, d, m):
    rng = np.random.default_rng(d)
    ks, dsub, nq, kc = 256, d // m, 5, 9
    q = rng.standard_normal((nq, d)).astype(np.float32)
    cb = rng.standard_normal(m * ks * dsub).astype(np.float32)
    coarse = rng.standard_normal((kc, d)).astype(np.float32)
    cids = rng.integers(0, kc, nq).astype(np.int32)
    cn = oracle.pq_centroid_sq(cb, m, ks, dsub, swift=False)
    for norms, use_dot, incq, strict in ((None, -1, True, False), (cn, -1, True, False), (cn, 1, False, False),
                                         (cn, 0, True, False), (None, -1, True, True), (cn, -1, True, True)):
        o = _lib.PQLutOpts(use_dot, incq, strict)
        g = vk.pq_lut_batch_l2_f32(q, cb, m, ks, norms, o)
        gr = vk.pq_lut_residual_l2_f32(q, cids, coarse, cb, m, ks, norms, o)
        for i in range(nq):
            want = oracle.pq_lut_l2(q[i], cb, m, ks, norms, use_dot, incq, strict)
            assert np.array_equal(bits(g[i]), bits(want)), (use_dot, incq, strict)
            wr = oracle.pq_lut_residual_l2(q[i], coarse[cids[i]], cb, m, ks, norms, use_dot, incq, strict)
            assert np.array_equal(bits(gr[i]), bits(wr)), ("res", use_dot, incq, strict)


def test_adc_scan_bit_exact(oracle, vk):
    rng = np.random.default_rng(4)
    for m in (16, 18, 64):
        n = 3000
        codes = rng.integers(0, 256, (n, m)).astype(np.uint8)
        lut = rng.random((m, 256)).astype(np.float32)
        assert np.array_equal(bits(vk.adc_scan_u8(codes, lut, m)), bits(oracle.adc_scan_u8(codes, lut, m)))
        o = _lib.ADCScanOpts(0, 0, 0, 0.375, True)
        assert np.array_equal(bits(vk.adc_scan_u8(codes, lut, m, opts=o)),
                              bits(oracle.adc_scan_u8(codes, lut, m, bias=0.375, strict_fp=True)))
        pad = np.zeros((n, m + 5), dtype=np.uint8)
        pad[:, :m] = codes
        o = _lib.ADCScanOpts(0, 0, m + 5, 0.0, False)
        assert np.array_equal(bits(vk.adc_scan_u8(pad, lut, m, opts=o)), bits(oracle.adc_scan_u8(codes, lut, m)))
        # u4
        c4 = rng.integers(0, 256, (n, m // 2)).astype(np.uint8)
        lut4 = rng.random((m, 16)).astype(np.float32)
        assert np.array_equal(bits(vk.adc_scan_u4(c4, lut4, m)), bits(oracle.adc_scan_u4(c4, lut4, m)))
        o = _lib.ADCScanOpts(0, 0, 0, 1.5, True)
        assert np.array_equal(bits(vk.adc_scan_u4(c4, lut4, m, opts=o)),
                              bits(oracle.adc_scan_u4(c4, lut4, m, bias=1.5, strict_fp=True)))
    # interleavedBlock (ADCScan.swift:288-379): one sequential accumulator per vector
    n, m, g = 103, 16, 8
    codes = rng.integers(0, 256, (n, m)).astype(np.uint8)
    lut = rng.random((m, 256)).astype(np.float32)
    inter = np.zeros(((n + g - 1) // g) * m * g, dtype=np.uint8)
    for i in range(n):
        for j in range(m):
            inter[(i // g) * m * g + j * g + i % g] = codes[i, j]
    want = np.zeros(n, dtype=np.float32)
    for j in range(m):
        want = (want + lut[j, codes[:, j]]).astype(np.float32)
    got = vk.adc_scan_u8(inter, lut, m, opts=_lib.ADCScanOpts(1, g, 0, 0.0, False), n=n)
    assert np.array_equal(bits(got), bits(want))
    assert vk.adc_scan_u8(np.zeros((0, 16), np.uint8), lut, 16).shape == (0,)


# ------------------------------------------------------------------------------------------------ indexes
def _make_ivfpq_problem(oracle, n, d, m, kc, nq, seed, sift=False, unit=False):
    from vectorindex_b200 import datagen
    rng = np.random.default_rng(seed)
    if sift:
        x = datagen.sift_like(n + nq, d, max(kc // 2, 4), seed)
    else:
        x = datagen.clustered_unit(n + nq, d, max(kc // 2, 4), seed) if unit else \
            (rng.standard_normal((n + nq, d)) + 3 * rng.standard_normal((max(kc // 2, 4), d))[rng.integers(0, max(kc // 2, 4), n + nq)]).astype(np.float32)
    xb, q = np.ascontiguousarray(x[:n]), np.ascontiguousarray(x[n:])
    coarse = np.ascontiguousarray(xb[rng.choice(n, kc, replace=False)])
    asg, _ = oracle.assign(xb, coarse)
    rc, cb, norms, _ = oracle.pq_train(xb[:2000], m, 256, coarse=coarse, assign_=asg[:2000], max_iters=4, sample_n=0)
    assert rc == 0
    return xb, q, coarse, cb, norms


# the route each row takes in the query-major scan (VIX_SCAN_DEBUG=1): "fast G table bias" or "generic"
STAGEWISE_ROUTE = {
    (20000, 128, 16): "fast 1 kernel kernel",
    (12000, 96, 48): "fast 3 kernel kernel",
    (8000, 64, 8): "generic",
    (6000, 48, 12): "generic",
    (6000, 160, 80): "generic",
    (6000, 192, 96): "generic",
    (5000, 256, 128): "generic",
    (8000, 128, 32): "fast 2 kernel kernel",
    (9000, 128, 64): "fast 4 kernel kernel",
    (6000, 512, 64): "fast 4 image kernel",
    (5000, 768, 64): "fast 4 image kernel",
    (4000, 640, 64): "fast 4 image kernel",
    (3000, 1664, 64): "fast 4 kernel kernel",
}


@pytest.mark.parametrize("n,d,m,kc,nprobe,metric,kind", [
    (20000, 128, 16, 64, 8, 0, "sift"),            # C3-shaped, fast kernel m=16
    (12000, 96, 48, 50, 6, 0, "unit"),             # C5-shaped, m=48 (dsub=2)
    (8000, 64, 8, 30, 5, 0, "gauss"),              # m=8: generic kernel (the fast one takes m = 16, 32, 48, 64)
    (6000, 48, 12, 20, 5, 0, "gauss"),             # m=12: generic kernel
    (6000, 160, 80, 24, 5, 0, "gauss"),            # m=80: generic kernel, 80 KB table
    (6000, 192, 96, 24, 5, 1, "unit"),             # m=96 inner product: generic kernel
    (5000, 256, 128, 16, 4, 0, "gauss"),           # m=128: generic kernel, largest table (128 KB)
    (8000, 128, 32, 40, 40, 0, "gauss"),           # nprobe == kc: exhaustive
    (9000, 128, 64, 32, 6, 1, "unit"),             # C4-shaped inner product, m=64
    (6000, 512, 64, 24, 5, 0, "gauss"),            # 512 KB of codebooks: tables built batch-wide (lut_image_kernel), dsub=8
    (5000, 768, 64, 16, 4, 1, "unit"),             # C4's d / m: dsub=12, inner product, batch-wide tables (d x nprobe = 3072: bias in the scan)
    (4000, 640, 64, 16, 4, 0, "gauss"),            # dsub=10: scalar codebook reads in the batch-wide table build
    (3000, 1664, 64, 12, 4, 0, "gauss"),           # d=1664 (near the exact engine's limit): staged queries still leave room for 16 warps; dsub=26 (tables in the scan)
])
def test_ivfpq_index_stagewise_parity(oracle, monkeypatch, capfd, n, d, m, kc, nprobe, metric, kind):
    from vectorindex_b200.index import IVFPQIndex
    nq, k = 64, 10
    xb, q, coarse, cb, norms = _make_ivfpq_problem(oracle, n, d, m, kc, nq, seed=n + m, sift=(kind == "sift"),
                                                   unit=(kind == "unit"))
    idx = IVFPQIndex(d, metric, nlist=kc, nprobe=nprobe, m=m)
    idx.set_coarse(coarse)
    idx.set_codebooks(cb, norms)
    ids = (np.arange(n, dtype=np.int64) * 3 + 7)                       # non-trivial external ids, ascending
    idx.batch_insert(xb[: n // 2], ids[: n // 2])
    idx.batch_insert(xb[n // 2:], ids[n // 2:])                        # two adds: lists must merge
    assert idx.count == n
    off, codes, lids, asg = idx.export_lists()
    # list assignment + codes: bit-exact
    oasg = oracle.assign(xb, coarse)[0] if metric == 0 else oracle.assign_metric(xb, coarse, metric)
    assert np.array_equal(asg, oasg)
    ocodes = oracle.pq_encode_u8(xb, cb, m, 256, centroid_sq=norms.reshape(-1), coarse=coarse, assign_=oasg)
    ooff, order = oracle.build_lists(oasg, kc)
    assert np.array_equal(off, ooff)
    assert np.array_equal(lids, ids[order])
    assert np.array_equal(codes, ocodes[order])
    assert np.array_equal(idx.list_sizes(), np.diff(ooff))
    # the route of the search (VIX_SCAN_DEBUG line of the query-major scan): kernel, G, table source, bias source
    od, oi, op = oracle.ivfpq_search(q, coarse, cb, norms, off, codes, lids, m, 256, nprobe, k, metric)
    capfd.readouterr()
    monkeypatch.setenv("VIX_SCAN_DEBUG", "1")
    gd, gi, gp = idx.batch_search(q, k, return_probes=True)
    monkeypatch.delenv("VIX_SCAN_DEBUG")
    lines = re.findall(r"\[vix scan\] kernel (fast G (\d)|generic),.*table (\w+), bias (\w+)", capfd.readouterr().err)
    assert len(lines) == 1, lines
    got = "generic" if lines[0][0] == "generic" else f"fast {lines[0][1]} {lines[0][2]} {lines[0][3]}"
    assert got == STAGEWISE_ROUTE[(n, d, m)]
    # search: probes exact, distances 1e-5, id sets up to ties
    assert np.array_equal(gp, op)
    scale = float(np.nanmax(np.abs(od)))
    assert_topk_close(gd, gi, od, oi, rtol=RTOL, atol=RTOL * scale * (1.0 if metric == 1 else 0.0))
    # import path: a second index fed the exported lists answers identically
    idx2 = IVFPQIndex(d, metric, nlist=kc, nprobe=nprobe, m=m)
    idx2.set_coarse(coarse)
    idx2.set_codebooks(cb, norms)
    idx2.import_lists(off, codes, lids)
    gd2, gi2 = idx2.batch_search(q, k)
    assert np.array_equal(gi2, gi) and np.array_equal(bits(gd2), bits(gd))


@pytest.mark.parametrize("d,metric", [(512, "euclidean"), (640, "euclidean"), (768, "dotProduct")])
def test_batchwide_tables_equal_in_kernel_tables(oracle, monkeypatch, d, metric):
    """lut_image_kernel + copy and build_lut inside the scan use the same operation order: identical bits."""
    from vectorindex_b200.index import IVFPQIndex
    n, m, kc, nq, k, nprobe = 4000, 64, 20, 48, 10, 5
    xb, q, coarse, cb, norms = _make_ivfpq_problem(oracle, n, d, m, kc, nq, seed=31)
    idx = IVFPQIndex(d, metric, nlist=kc, nprobe=nprobe, m=m)
    idx.set_coarse(coarse); idx.set_codebooks(cb, norms)
    idx.batch_insert(xb)
    d1, i1 = idx.batch_search(q, k)                                   # 512 KB of codebooks or more: batch-wide tables
    monkeypatch.setenv("VIX_DISABLE_LUT_IMAGE", "1")
    d2, i2 = idx.batch_search(q, k)
    assert np.array_equal(i1, i2) and np.array_equal(bits(d1), bits(d2))


@pytest.mark.parametrize("d,m,n,kc,nq,nprobe,k,kind", [
    (96, 48, 60000, 64, 600, 12, 10, "unit"),      # C5-shaped: three groups of 16 sub-quantisers (the last one read through its replica)
    (32, 16, 30000, 40, 300, 8, 10, "gauss"),      # one group
    (64, 32, 30000, 48, 257, 10, 5, "gauss"),      # two groups
    (128, 64, 30000, 32, 300, 6, 32, "gauss"),     # four groups, two K-atoms, k = 32
    (96, 48, 3000, 200, 300, 40, 10, "gauss"),     # tiny lists (many below k vectors: their queries are handed back), 15 per list
    (96, 48, 40000, 24, 1500, 24, 10, "unit"),     # nprobe == kc and > 64 queries per list: several column groups per list
    (96, 48, 20000, 32, 200, 8, 1, "sift"),        # k = 1, integer-valued data with heavy ties
])
def test_list_major_tensor_core_scan_equals_query_major_scan(oracle, monkeypatch, d, m, n, kc, nq, nprobe, k, kind):
    """vix_ivfpq_tc.cu (decode once per list, fp16 tensor-core shortlist, finalists in the look-up-table scan's arithmetic)
    returns the ids AND the distance bits of vix_ivfpq_scan.cu, which the other tests pin to the oracle at 1e-5."""
    from vectorindex_b200 import _lib
    from vectorindex_b200.index import IVFPQIndex
    xb, q, coarse, cb, norms = _make_ivfpq_problem(oracle, n, d, m, kc, nq, seed=d + m + k + n, sift=kind == "sift", unit=kind == "unit")
    idx = IVFPQIndex(d, "euclidean", nlist=kc, nprobe=nprobe, m=m)
    idx.set_coarse(coarse); idx.set_codebooks(cb, norms)
    idx.batch_insert(xb)
    monkeypatch.setenv("VIX_TC_SCAN", "0")
    before = _lib.lib().vix_scan_tc_launches()
    d1, i1 = idx.batch_search(q, k)
    assert _lib.lib().vix_scan_tc_launches() == before
    monkeypatch.setenv("VIX_TC_SCAN", "1")
    d2, i2 = idx.batch_search(q, k)
    assert _lib.lib().vix_scan_tc_launches() == before + 1
    assert np.array_equal(i1, i2)
    assert np.array_equal(bits(d1), bits(d2))
    # and the oracle (the reference's composition) on the first queries, as for the query-major scan
    off, codes, lids, _ = idx.export_lists()
    od, oi, _ = oracle.ivfpq_search(q[:48], coarse, cb, norms, off, codes, lids, m, 256, nprobe, k, 0)
    assert_topk_close(d2[:48], i2[:48], od, oi, rtol=RTOL, atol=0.0)


def test_sharded_pieces_emulated_on_one_gpu(oracle):
    """Two list-block shards built and searched in ONE process (the ranks emulated sequentially, the collectives
    replaced by concatenation): probe_range + merge == the single index's probe lists, search_with_probes + merge
    == the single index's result, and encode/add_encoded build the same lists as batch_insert."""
    from vectorindex_b200 import kernels as vk
    from vectorindex_b200.index import IVFPQIndex, list_block, list_owner
    n, d, m, kc, nq, k, nprobe, world = 9000, 64, 16, 40, 50, 10, 6, 2
    xb, q, coarse, cb, norms = _make_ivfpq_problem(oracle, n, d, m, kc, nq, seed=99)
    ids = np.arange(n, dtype=np.int64) * 5 + 3
    single = IVFPQIndex(d, "euclidean", nlist=kc, nprobe=nprobe, m=m)
    single.set_coarse(coarse); single.set_codebooks(cb, norms)
    single.batch_insert(xb, ids)
    sd, si, sp = single.batch_search(q, k, return_probes=True)
    shards = []
    for r in range(world):
        ix = IVFPQIndex(d, "euclidean", nlist=kc, nprobe=nprobe, m=m)
        ix.set_coarse(coarse); ix.set_codebooks(cb, norms)
        shards.append(ix)
    asg, codes = shards[0].encode(xb)                                  # any rank may encode
    owner = list_owner(asg.astype(np.int64), kc, world)
    for r in range(world):
        sel = owner == r
        shards[r].add_encoded(asg[sel], codes[sel], ids[sel])
    assert sum(s_.count for s_ in shards) == n
    # stage 1: local top-nprobe per centroid block -> merged global probe lists
    pid, psc = zip(*[shards[r].probe_range(q, nprobe, *list_block(kc, r, world)) for r in range(world)])
    sc = np.ascontiguousarray(np.stack(psc, 1))                         # [nq x world x nprobe]
    idm = np.ascontiguousarray(np.stack(pid, 1).astype(np.int64))
    _, gp = vk.mergeTopK(sc, idm, nprobe, 0)
    assert np.array_equal(gp.astype(np.int32), sp)
    # stage 2: every shard scans the probed lists it owns -> merged top-k
    res = [shards[r].search_with_probes(q, k, gp.astype(np.int32)) for r in range(world)]
    dd = np.ascontiguousarray(np.stack([r_[0] for r_ in res], 1))
    ii = np.ascontiguousarray(np.stack([r_[1] for r_ in res], 1))
    md, mi = vk.mergeTopK(dd, ii, k, 0)
    assert np.array_equal(mi, si)
    assert np.array_equal(bits(md), bits(sd))


@pytest.mark.parametrize("mode", ["allow", "deny"])
@pytest.mark.parametrize("m", [16, 12])          # fused fast kernel / generic kernel
def test_ivfpq_filtered_search_is_prefilter(oracle, mode, m):
    """IDFilter semantics (IDFilter.swift:115-135) as a PRE-filter (IVFIndex.swift:813, 1034): the filtered search
    equals the oracle's search over an index from which the failing vectors were removed; ids outside the bitset's
    domain never pass."""
    from vectorindex_b200.index import IDFilter, IVFPQIndex
    n, d, kc, nq, k, nprobe = 6000, 48, 32, 40, 10, 6
    xb, q, coarse, cb, norms = _make_ivfpq_problem(oracle, n, d, m, kc, nq, seed=5)
    ids = np.arange(n, dtype=np.int64) * 2 + 1                         # odd ids up to 2n
    idx = IVFPQIndex(d, "euclidean", nlist=kc, nprobe=nprobe, m=m)
    idx.set_coarse(coarse); idx.set_codebooks(cb, norms)
    idx.batch_insert(xb, ids)
    rng = np.random.default_rng(3)
    cap = int(ids.max() * 0.8)                                         # the largest ids lie outside the domain
    f = IDFilter(cap, mode)
    f.set(rng.choice(cap, cap // 3, replace=False))
    keep = f.test(ids)
    assert 0 < keep.sum() < n and not keep[ids >= cap].any()
    gd, gi = idx.batch_search(q, k, filter=f)
    off, codes, lids, asg = idx.export_lists()
    kept = f.test(lids)
    lens = np.bincount(np.repeat(np.arange(kc), np.diff(off))[kept], minlength=kc)
    off2 = np.concatenate([[0], np.cumsum(lens)])
    od, oi, _ = oracle.ivfpq_search(q, coarse, cb, norms, off2, codes[kept], lids[kept], m, 256, nprobe, k, 0)
    np.testing.assert_allclose(gd, od, rtol=1e-5, equal_nan=True)
    same = np.mean([len(set(gi[r]) & set(oi[r])) / k for r in range(nq)])
    assert same > 0.995
    assert f.test(gi[gi >= 0]).all()
    # a filter nothing passes -> empty results (id -1, NaN)
    none = IDFilter(cap, "allow")
    ed, ei = idx.batch_search(q, k, filter=none)
    assert (ei == -1).all() and np.isnan(ed).all()


@pytest.mark.parametrize("kind", ["flat", "ivfflat"])
def test_flat_and_ivfflat_filtered_search(oracle, kind):
    from vectorindex_b200.index import FlatIndex, IDFilter, IVFIndex
    rng = np.random.default_rng(11)
    n, d, nq, k = 5000, 32, 30, 10
    xb = rng.standard_normal((n, d)).astype(np.float32)
    q = rng.standard_normal((nq, d)).astype(np.float32)
    ids = rng.permutation(3 * n)[:n].astype(np.int64)
    f = IDFilter(3 * n, "deny").set(rng.choice(3 * n, n, replace=False))
    keep = f.test(ids)
    if kind == "flat":
        idx = FlatIndex(d, "euclidean")
    else:
        idx = IVFIndex(d, "euclidean", nlist=8, nprobe=8)              # every list probed: same answer as flat
        idx.set_coarse(xb[:8].copy())
    idx.batch_insert(xb, ids)
    gd, gi = idx.batch_search(q, k, filter=f)
    od, oi, _ = oracle.flat_search(q, xb[keep], k, 0)
    assert np.array_equal(gi, ids[keep][oi])
    assert np.array_equal(bits(gd), bits(od))


@pytest.mark.parametrize("metric,d,m", [("euclidean", 64, 16), ("dotProduct", 96, 48), ("euclidean", 40, 10)])
def test_ivfpq_index_with_u4_codes(oracle, vk, metric, d, m):
    """ks = 16 inside the index handles (the reference's 4-bit API: cpq_encode_residual_u4_f32, pq_encode.c:692-739;
    adc_scan_u4 with packed nibbles, ADCScan.swift:384-456): list assignment and packed codes bit-exact with the oracle's
    restatement of the C encoder, the fused search within 1e-5 of pq_lut_residual_l2 -> adc_scan_u4 -> selectTopK ->
    mergeTopK, lists exported / imported in the packed format, and a GPU-trained ks = 16 index answers queries."""
    from vectorindex_b200.index import IVFPQIndex
    n, kc, nq, k, nprobe, ks = 7000, 20, 41, 10, 5, 16
    mi = 1 if metric == "dotProduct" else 0
    rng = np.random.default_rng(d + m)
    centres = 3 * rng.standard_normal((kc // 2, d))
    x = (rng.standard_normal((n + nq, d)) + centres[rng.integers(0, kc // 2, n + nq)]).astype(np.float32)
    xb, q = np.ascontiguousarray(x[:n]), np.ascontiguousarray(x[n:])
    coarse = np.ascontiguousarray(xb[rng.choice(n, kc, replace=False)])
    cb = (0.8 * rng.standard_normal((m, ks, d // m))).astype(np.float32)
    idx = IVFPQIndex(d, metric, nlist=kc, nprobe=nprobe, m=m, ks=ks)
    idx.set_coarse(coarse)
    idx.set_codebooks(cb)
    ids = np.arange(n, dtype=np.int64) * 2 + 1
    idx.batch_insert(xb, ids)
    off, codes, lids, asg = idx.export_lists()
    assert codes.shape == (n, m // 2)
    oasg = oracle.assign(xb, coarse)[0] if mi == 0 else oracle.assign_metric(xb, coarse, 1)
    assert np.array_equal(asg, oasg)
    ocodes = oracle.pq_encode_u4(xb, cb, m, ks, coarse=coarse, assign_=oasg)
    _, order = oracle.build_lists(oasg, kc)
    assert np.array_equal(codes, ocodes[order]) and np.array_equal(lids, ids[order])
    _, norms = idx.get_codebooks()
    gd, gi = idx.batch_search(q, k)
    od, oi, _ = oracle.ivfpq_search(q, coarse, cb, norms, off, codes, lids, m, ks, nprobe, k, mi)
    assert_topk_close(gd, gi, od, oi, atol=1e-5)
    # the packed lists travel: import into a fresh handle == same answers; encode() returns the packed codes
    other = IVFPQIndex(d, metric, nlist=kc, nprobe=nprobe, m=m, ks=ks)
    other.set_coarse(coarse)
    other.set_codebooks(cb, norms)
    other.import_lists(off, codes, lids)
    d2, i2 = other.batch_search(q, k)
    assert np.array_equal(i2, gi) and np.array_equal(bits(d2), bits(gd))
    a3, c3 = idx.encode(xb[:100])
    assert np.array_equal(a3, oasg[:100]) and np.array_equal(c3, ocodes[:100])
    # trained on the GPU
    tr = IVFPQIndex(d, metric, nlist=kc, nprobe=kc, m=m, ks=ks)
    tr.optimize(xb)
    tr.batch_insert(xb)
    td, ti = tr.batch_search(xb[:20], 5)
    assert (ti >= 0).all() and tr.get_codebooks()[0].shape == (m, ks, d // m)


@pytest.mark.parametrize("metric", ["euclidean", "dotProduct"])
def test_ivfpq_search_with_exact_rerank(oracle, vk, metric):
    """Step 7 of the IVF-PQ query (DONE_22_adc_scan.md:873-878): ADC top-R, then Kernel #40 over the original vectors.
    Equal to the composition the oracle runs -- ivfpq_search(k = R) -> rerank_exact_topk (ExactRerank.swift:698-814): ids and
    exact score bits (the candidate SETS agree unless an ADC tie inside the 1e-5 tolerance straddles rank R; such rows are
    compared on the candidates both sides hold).  The re-rank recovers recall the codes lost."""
    from vectorindex_b200.index import IVFPQIndex
    n, d, m, kc, nq, k, R, nprobe = 6000, 64, 16, 24, 60, 10, 50, 6
    xb, q, coarse, cb, norms = _make_ivfpq_problem(oracle, n, d, m, kc, nq, seed=77)
    mi = 1 if metric == "dotProduct" else 0
    idx = IVFPQIndex(d, metric, nlist=kc, nprobe=nprobe, m=m)
    idx.set_coarse(coarse)
    idx.set_codebooks(cb, norms)
    idx.batch_insert(xb)                                                    # ids = rows
    gs, gi = idx.batch_search_rerank(q, k, xb, R)
    off, codes, lids, _ = idx.export_lists()
    od, oi, _ = oracle.ivfpq_search(q, coarse, cb, norms, off, codes, lids, m, 256, nprobe, R, mi)
    ad, ai = idx.batch_search(q, R)
    exact_d, exact_i, _ = oracle.flat_search(q, xb, k, mi)
    hit_adc = hit_rr = 0
    for r in range(nq):
        cand = oi[r][oi[r] >= 0]
        rows = xb[cand]
        sc = oracle.ip_block(q[r], rows) if mi else oracle.l2sqr_block(q[r], rows)
        order = np.lexsort((cand, -sc if mi else sc))[:k]
        if set(ai[r].tolist()) == set(oi[r].tolist()):                      # same candidate set: bit-exact outcome
            assert np.array_equal(gi[r], cand[order]), r
            assert np.array_equal(bits(gs[r]), bits(sc[order])), r
        else:                                                               # boundary tie of the ADC stage
            assert len(set(gi[r].tolist()) & set(cand[order].tolist())) >= k - 1
        hit_adc += len(set(ai[r][:k].tolist()) & set(exact_i[r].tolist()))
        hit_rr += len(set(gi[r].tolist()) & set(exact_i[r].tolist()))
    assert hit_rr >= hit_adc and hit_rr > 0
    from vectorindex_b200 import VectorIndexError
    with pytest.raises(VectorIndexError):
        idx.batch_search_rerank(q, 10, xb, 5)                               # K <= C (ExactRerank.swift:730)
    s2, i2 = idx.batch_search_rerank(q[:3], 4, xb[:100], 40)                # candidates beyond the reader's rows are missing
    assert ((i2 < 100) & (i2 >= -1)).all()


def test_ivfpq_edge_cases(oracle):
    from vectorindex_b200.index import IVFPQIndex
    from vectorindex_b200 import VectorIndexError
    d, m, kc = 32, 16, 8
    xb, q, coarse, cb, norms = _make_ivfpq_problem(oracle, 3000, d, m, kc, 5, seed=1)
    idx = IVFPQIndex(d, "euclidean", nlist=kc, nprobe=3, m=m)
    with pytest.raises(VectorIndexError) as e:
        idx.batch_insert(xb)
    assert e.value.kind == "notTrained"
    idx.set_coarse(coarse)
    idx.set_codebooks(cb, norms)
    gd, gi = idx.batch_search(q, 4)                                    # empty index
    assert (gi == -1).all() and np.isnan(gd).all()
    idx.batch_insert(xb[:6])                                           # fewer vectors than k, ragged lists
    gd, gi = idx.batch_search(q, 10, nprobe=kc)
    assert ((gi >= 0).sum(axis=1) == 6).all()
    assert idx.batch_search(q, 0)[0].shape == (5, 0)                   # k <= 0 => [] (IVFIndex.swift:866)
    gd, gi = idx.batch_search(q, 3, nprobe=20)                         # nprobe > kc is clamped by padding
    assert (gi >= 0).all()
    with pytest.raises(VectorIndexError):
        idx.batch_search(np.zeros((2, d + 1), np.float32), 3)          # dimension mismatch throws
    with pytest.raises(VectorIndexError):
        idx.batch_insert(xb[:2], np.array([-1, 5], dtype=np.int64))    # ids must fit the reference's id type
    assert idx.search(q[0], 2)[0][0] >= 0


def test_invalid_list_ids_device_ids_and_duplicates(oracle):
    """Contract edges of the handles (include/vindex_cuda.h conventions): list assignments outside [0, kc) are rejected,
    probe ids outside [0, kc) are skipped like the -1 padding, DEVICE-resident ids are range-checked like host ids, an id
    stored twice comes back twice (append, not replace), and a NaN row is refused by an IVF-PQ add / left without a list
    by an IVF-Flat one (IVFIndex.swift:376-435: "guard best >= 0 else continue")."""
    import torch
    from vectorindex_b200.index import IVFIndex, IVFPQIndex
    from vectorindex_b200 import VectorIndexError
    d, m, kc = 32, 16, 8
    xb, q, coarse, cb, norms = _make_ivfpq_problem(oracle, 2000, d, m, kc, 6, seed=5)
    idx = IVFPQIndex(d, "euclidean", nlist=kc, nprobe=3, m=m)
    idx.set_coarse(coarse)
    idx.set_codebooks(cb, norms)
    asg, codes = idx.encode(xb)
    ids = np.arange(2000, dtype=np.int64)
    bad = asg.copy()
    bad[17] = kc
    with pytest.raises(VectorIndexError):
        idx.add_encoded(bad, codes, ids)
    bad[17] = -1
    with pytest.raises(VectorIndexError):
        idx.add_encoded(torch.from_numpy(bad).cuda(), torch.from_numpy(codes).cuda(), torch.from_numpy(ids).cuda())
    dev_ids = torch.from_numpy(ids).cuda()
    dev_ids[3] = -7
    with pytest.raises(VectorIndexError):
        idx.add_encoded(torch.from_numpy(asg).cuda(), torch.from_numpy(codes).cuda(), dev_ids)
    dev_ids[3] = 0xFFFFFFFF
    with pytest.raises(VectorIndexError):
        idx.batch_insert(torch.from_numpy(xb).cuda(), dev_ids)
    assert idx.count == 0
    nanrow = xb[:4].copy()
    nanrow[2] = np.nan
    # euclidean: no distance of a NaN row is "< best", so _vi_km12_assignAOS leaves it in list 0
    # (KMeansMiniBatchKernel.swift:341-359); dot product: the row has no minimum and no list -- the add is refused
    assert idx.encode(nanrow)[0].tolist() == oracle.assign(nanrow, coarse)[0].tolist() and idx.encode(nanrow)[0][2] == 0
    ipx = IVFPQIndex(d, "dotProduct", nlist=kc, nprobe=3, m=m)
    ipx.set_coarse(coarse)
    ipx.set_codebooks(cb, norms)
    assert oracle.assign_metric(nanrow, coarse, 1)[2] == -1
    with pytest.raises(VectorIndexError):
        ipx.batch_insert(nanrow)
    with pytest.raises(VectorIndexError):
        ipx.encode(nanrow)
    assert ipx.count == 0 and idx.count == 0
    idx.add_encoded(torch.from_numpy(asg).cuda(), torch.from_numpy(codes).cuda(),
                    torch.from_numpy(ids).to(torch.int32).cuda())          # a tensor of another width is cast, not reinterpreted
    # probes: ids >= kc / < -1 behave like the -1 padding
    gd, gi, probes = idx.batch_search(q, 5, return_probes=True)
    wide = np.concatenate([probes, np.full((6, 1), -1, np.int32)], axis=1)
    junk = wide.copy()
    junk[:, -1] = [kc, kc + 100, -5, 2 ** 30, -1, kc]
    d1, i1 = idx.search_with_probes(q, 5, wide)
    d2, i2 = idx.search_with_probes(q, 5, junk)
    assert np.array_equal(i1, gi) and np.array_equal(i2, gi) and np.array_equal(bits(d2), bits(gd))
    # the same id stored twice: both rows are results of their own (identical code => identical distance)
    row = int(gi[0, 0])
    idx.add_encoded(asg[row:row + 1], codes[row:row + 1], np.array([row], dtype=np.int64))
    d3, i3 = idx.batch_search(q[:1], 5)
    assert i3[0, 0] == row and i3[0, 1] == row and bits(d3)[0, 0] == bits(d3)[0, 1]
    assert np.array_equal(i3[0, 2:], gi[0, 1:4])
    # IVF-Flat, cosine: the guarded CentroidBatchScore row of a NaN vector is all 1 (CentroidBatchScore.swift:70-84), so
    # it lands in list 0 as in the reference; its candidate distance is NaN and it is never returned
    flat = IVFIndex(d, "cosine", nlist=kc, nprobe=kc)
    flat.set_coarse(coarse)
    xs = xb[:300].copy()
    xs[5] = np.nan
    flat.batch_insert(xs)
    fd, fi = flat.batch_search(q, 10)
    assert 5 not in fi and (fi >= 0).all() and flat.count == 300
    want = oracle.assign_metric(xs, coarse, 2, oracle.centroid_norms(coarse))
    assert want[5] == 0 and flat.list_sizes().tolist() == np.bincount(want[want >= 0], minlength=kc).tolist()


@pytest.mark.parametrize("metric", [0, 1])
def test_ivfflat_and_flat_index(oracle, metric):
    from vectorindex_b200.index import FlatIndex, IVFIndex
    rng = np.random.default_rng(8)
    n, d, kc, nq, k, nprobe = 6000, 48, 40, 30, 10, 6
    xb = rng.standard_normal((n, d)).astype(np.float32)
    q = rng.standard_normal((nq, d)).astype(np.float32)
    coarse = np.ascontiguousarray(xb[rng.choice(n, kc, replace=False)])
    ids = np.arange(n, dtype=np.int64) + 100
    ivf = IVFIndex(d, metric, nlist=kc, nprobe=nprobe)
    ivf.set_coarse(coarse)
    ivf.batch_insert(xb, ids)
    asg = oracle.assign(xb, coarse)[0] if metric == 0 else oracle.assign_metric(xb, coarse, metric)
    off, order = oracle.build_lists(asg, kc)
    od, oi = oracle.ivfflat_search(q, coarse, off, xb[order], ids[order], nprobe, k, metric)
    gd, gi = ivf.batch_search(q, k)
    assert np.array_equal(gi, oi) and np.array_equal(bits(gd), bits(od))
    flat = FlatIndex(d, metric)
    flat.batch_insert(xb, ids)
    fd, fi = flat.batch_search(q, k)
    od, oi, _ = oracle.flat_search(q, xb, k, metric)
    assert np.array_equal(fi, oi + 100) and np.array_equal(bits(fd), bits(od))


def test_ivfflat_cosine_index(oracle):
    """IVFIndex with the cosine metric: lists by the first minimum of the guarded CentroidBatchScore row
    (IVFIndex.swift:376-435), probes by (score, list id) (:905-927), candidate distances 1 - clamp(dot / sqrt(|q|^2 |x|^2))
    (DistanceUtils.swift:22-38); a zero vector sits at distance exactly 1."""
    from vectorindex_b200.index import IVFIndex
    rng = np.random.default_rng(18)
    n, d, kc, nq, k, nprobe = 6000, 48, 40, 30, 10, 6
    xb = (rng.standard_normal((n, d)) * rng.uniform(0.2, 3.0, (n, 1))).astype(np.float32)
    xb[17] = 0.0
    q = rng.standard_normal((nq, d)).astype(np.float32)
    coarse = np.ascontiguousarray(xb[rng.choice(n, kc, replace=False)])
    coarse[3] = 0.0                                                     # degenerate centroid: score exactly 1
    ids = np.arange(n, dtype=np.int64) + 100
    ivf = IVFIndex(d, "cosine", nlist=kc, nprobe=nprobe)
    ivf.set_coarse(coarse)
    ivf.batch_insert(xb, ids)
    asg = oracle.assign_metric(xb, coarse, 2)
    assert np.array_equal(ivf.list_sizes(), np.bincount(asg, minlength=kc))
    off, order = oracle.build_lists(asg, kc)
    od, oi = oracle.ivfflat_search(q, coarse, off, xb[order], ids[order], nprobe, k, 2)
    gd, gi, gp = ivf.batch_search(q, k, return_probes=True)
    assert np.array_equal(gp, oracle.probe_select_batch(q, coarse, nprobe, 2)[0])
    assert_topk_close(gd, gi, od, oi, rtol=RTOL, atol=1e-6)


def test_ivfflat_insert_then_optimize(oracle):
    """IVFMoreTests.swift:5-15 (linear scan before optimize) and the reference's build order: vectors first, then
    optimize() over the stored vectors, which files them into their lists; set_coarse on a filled index does the same."""
    from vectorindex_b200.index import IVFIndex
    rng = np.random.default_rng(28)
    n, d, kc, nq, k, nprobe = 5000, 32, 24, 25, 10, 5
    xb = rng.standard_normal((n, d)).astype(np.float32)
    q = rng.standard_normal((nq, d)).astype(np.float32)
    ids = np.arange(n, dtype=np.int64) + 7
    ivf = IVFIndex(d, "euclidean", nlist=kc, nprobe=nprobe)
    ivf.batch_insert(xb[:3000], ids[:3000])
    ivf.batch_insert(xb[3000:], ids[3000:])
    fd, fi, _ = oracle.flat_search(q, xb, k, 0)
    gd, gi = ivf.batch_search(q, k)                                     # not optimised yet: exact linear scan
    assert np.array_equal(gi, fi + 7) and np.array_equal(bits(gd), bits(fd))
    ivf.optimize()                                                      # k-means over the stored vectors
    coarse = ivf.get_coarse()
    asg = oracle.assign(xb, coarse)[0]
    assert np.array_equal(ivf.list_sizes(), np.bincount(asg, minlength=coarse.shape[0]))
    off, order = oracle.build_lists(asg, coarse.shape[0])
    od, oi = oracle.ivfflat_search(q, coarse, off, xb[order], ids[order], nprobe, k, 0)
    gd, gi = ivf.batch_search(q, k)
    assert np.array_equal(gi, oi) and np.array_equal(bits(gd), bits(od))
    # the same through set_coarse on an index that already holds its vectors, then more vectors
    ivf2 = IVFIndex(d, "euclidean", nlist=kc, nprobe=nprobe)
    ivf2.batch_insert(xb[:4000], ids[:4000])
    ivf2.set_coarse(coarse)
    ivf2.batch_insert(xb[4000:], ids[4000:])
    gd2, gi2 = ivf2.batch_search(q, k)
    assert np.array_equal(gi2, oi) and np.array_equal(bits(gd2), bits(od))


def test_device_resident_search_equals_host_path(oracle):
    import torch
    from vectorindex_b200.index import IVFPQIndex
    d, m, kc = 64, 16, 16
    xb, q, coarse, cb, norms = _make_ivfpq_problem(oracle, 5000, d, m, kc, 40, seed=21)
    idx = IVFPQIndex(d, "euclidean", nlist=kc, nprobe=4, m=m)
    idx.set_coarse(coarse)
    idx.set_codebooks(cb, norms)
    idx.batch_insert(torch.from_numpy(xb).cuda())
    hd, hi = idx.batch_search(q, 10)
    dd, di = idx.batch_search(torch.from_numpy(q).cuda(), 10)
    assert dd.is_cuda and np.array_equal(di.cpu().numpy(), hi) and np.array_equal(bits(dd.cpu().numpy()), bits(hd))


# ------------------------------------------------------------------------------------------------ reference-parity trainers
def test_kmeanspp_seed_parity(oracle, vk):
    """kmeansPlusPlusSeed (KMeansSeeding.swift:167-409): same LCG stream, same chosen rows, same centroids."""
    rng = np.random.default_rng(4)
    x = (rng.standard_normal((3000, 24)) + 3 * rng.standard_normal((9, 24))[rng.integers(0, 9, 3000)]).astype(np.float32)
    for seed, stream, k in ((42, 0, 37), (7, 3, 64)):
        oc, och = oracle.kmeanspp_seed(x, k, seed, stream)
        gc, gch = vk.kmeansPlusPlusSeed(x, k, seed, stream)
        assert np.array_equal(gch, och)
        assert np.array_equal(bits(gc), bits(oc))


def test_kmeanspp_seed_edge_cases(oracle, vk):
    """KMeansPPSeedingTests.swift:182-296 (k = 1, k = n, duplicated points): the same chosen rows as the oracle."""
    from test_oracle_pins import _kmeanspp_edge_cases
    for data, k, seed in _kmeanspp_edge_cases():
        oc, och = oracle.kmeanspp_seed(data, k, seed, 0)
        gc, gch = vk.kmeansPlusPlusSeed(data, k, seed, 0)
        assert np.array_equal(gch, och) and np.array_equal(bits(gc), bits(oc))


def test_kmeans_minibatch_edge_cases(oracle, vk):
    """KMeansMiniBatchTests.swift:405-487, 616-646 (one centroid, batch larger than n, identical points): bit-identical
    to the oracle in reference-parity mode."""
    from test_oracle_pins import _kmeans_minibatch_edge_cases
    for x, kc, init, batch, epochs in _kmeans_minibatch_edge_cases():
        rc, oc, _, _ = oracle.kmeans_minibatch(x, kc, init, batch, epochs, 1e-4, 0, 0)
        assert rc == 0
        st, gc, _ = vk.kmeans_minibatch_f32(x, kc, init, vk.kmeans_cfg(batch, epochs, 1e-4, 0, 0, False, 0))
        assert np.array_equal(bits(gc), bits(oc))


@pytest.mark.parametrize("n,d,kc,batch,epochs", [(5000, 16, 64, 1024, 5), (1500, 33, 20, 256, 3), (900, 8, 300, 128, 2)])
def test_kmeans_minibatch_parity(oracle, vk, n, d, kc, batch, epochs):
    """kmeans_minibatch_f32 in reference-parity mode: batches drawn with replacement from the LCG, batch-mean
    replacement, the 'empties' repair quirk, reservoir-sampled inertia and the early stop -- centroids and final
    assignments bit-identical to the oracle (KMeansMiniBatchKernel.swift:401-724)."""
    rng = np.random.default_rng(n + kc)
    x = (rng.standard_normal((n, d)) + 2 * rng.standard_normal((11, d))[rng.integers(0, 11, n)]).astype(np.float32)
    rc, oc, oa, info = oracle.kmeans_minibatch(x, kc, None, batch, epochs, 1e-4, 42, 0, compute_assignments=True)
    assert rc == 0
    st, gc, ga = vk.kmeans_minibatch_f32(x, kc, None, vk.kmeans_cfg(batch, epochs, 1e-4, 42, 0, True, 0), compute_assignments=True)
    assert np.array_equal(bits(gc), bits(oc))
    assert np.array_equal(ga, oa)
    # explicit initial centroids take the same path minus the seeding
    init = np.ascontiguousarray(x[:kc])
    rc, oc2, _, _ = oracle.kmeans_minibatch(x, kc, init, batch, 2, 1e-4, 5, 1)
    _, gc2, _ = vk.kmeans_minibatch_f32(x, kc, init, vk.kmeans_cfg(batch, 2, 1e-4, 5, 1, False, 0))
    assert np.array_equal(bits(gc2), bits(oc2))


@pytest.mark.parametrize("n,d,m,ks,algo,policy,residual,sample_n", [
    (3000, 32, 4, 256, 0, 0, False, 0),      # Lloyd, subset seeding (n > 4 ks), .split
    (3000, 32, 4, 256, 0, 1, True, 0),       # Lloyd on residuals, .reseed
    (700, 24, 3, 256, 0, 0, True, 0),        # n <= 4 ks: strided seeding; empty clusters guaranteed -> .split repair
    (2500, 16, 2, 64, 0, 2, False, 1200),    # sampled training set, .ignore
    (3000, 32, 4, 256, 1, 0, True, 0),       # mini-batch (forces sample_n = 2000 and .reseed, PQTrain.swift:144-149)
    (1800, 16, 2, 128, 1, 0, False, 900),    # mini-batch with an explicit sample
])
def test_pq_train_parity(oracle, vk, n, d, m, ks, algo, policy, residual, sample_n):
    """pq_train_f32 in reference-parity mode: Xoroshiro128** streams per sub-space, selection sampling, k-means++
    seeding, Lloyd / mini-batch with the reference's repair policies -- codebooks and norms bit-identical to the
    oracle (PQTrain.swift:83-388, 856-1442)."""
    rng = np.random.default_rng(n + ks + algo)
    x = (rng.standard_normal((n, d)) + 2 * rng.standard_normal((7, d))[rng.integers(0, 7, n)]).astype(np.float32)
    coarse = asg = None
    if residual:
        coarse = np.ascontiguousarray(x[rng.choice(n, 9, replace=False)])
        asg, _ = oracle.assign(x, coarse)
    rc, ocb, onorm, _ = oracle.pq_train(x, m, ks, coarse=coarse, assign_=asg, algorithm=algo, max_iters=4, batch_size=512,
                                        empty_policy=policy, sample_n=sample_n, seed=42, stream_id=2)
    assert rc == 0
    cfg = vk.pq_train_cfg(algorithm=algo, max_iters=4, tol=1e-4, batch_size=512, sample_n=sample_n, seed=42, stream_id=2,
                          empty_policy=policy, mode=0)
    gcb, gnorm = vk.pq_train_f32(x, m, ks, coarse, asg, cfg)
    assert np.array_equal(bits(gcb), bits(ocb))
    assert np.array_equal(bits(gnorm), bits(onorm))


def test_pq_train_streaming_reference_golden_bits(oracle, vk):
    """pq_train_streaming_f32 on the GPU reproduces the reference's OWN golden vector (PQTrainTests.swift:724-817: ks 16,
    d 16, m 2, 40 LCG rows in two chunks, seed 42, mini-batch, 10 passes, batch 512 => the bit patterns of codebooks[0..3])
    and the oracle's codebooks bit for bit -- from host chunks and from device chunks."""
    import torch
    from vectorindex_b200 import datagen
    ks, d, m, n = 16, 16, 2, 40
    full = datagen.lcg24_floats(0x5773_7EA1_1234_5678, n * d)[0].reshape(n, d)
    chunks = [np.ascontiguousarray(full[:20]), np.ascontiguousarray(full[20:])]
    cfg = vk.pq_train_cfg(algorithm=1, max_iters=10, batch_size=512, seed=42, mode=0)
    cb, norms = vk.pq_train_streaming_f32(chunks, m, ks, cfg)
    want = np.array([0.7648039, -0.5310464, -0.7147653, 0.30723625], dtype=np.float32)
    assert bits(cb.reshape(-1)[:4]).tolist() == bits(want).tolist()
    rc, ocb = oracle.pq_train_streaming(chunks, d, m, ks, seed=42, algorithm=1, max_iters=10, batch_size=512)
    assert rc == 0 and np.array_equal(bits(cb), bits(ocb))
    cb2, _ = vk.pq_train_streaming_f32([torch.from_numpy(c).cuda() for c in chunks], m, ks, cfg)
    assert np.array_equal(bits(cb2), bits(cb))
    seq = np.zeros((m, ks), dtype=np.float32)                              # centroid norms: sequential sum of squares (PQTrain.swift:299-307)
    for u in range(d // m):
        seq = (seq + cb[:, :, u] * cb[:, :, u]).astype(np.float32)
    assert np.array_equal(bits(norms), bits(seq))


@pytest.mark.parametrize("sizes,d,m,ks,iters,batch,sample_n", [
    ((700, 0, 1300, 450), 32, 4, 64, 3, 256, 0),       # more rows than 2000: Bernoulli sampling (sample_n forced to 2000), subset seeding
    ((300, 260), 24, 3, 256, 3, 128, 0),               # fewer rows than 4 ks: streaming seeding; empty clusters -> pass-level repair
    ((900, 900, 900), 16, 2, 32, 2, 8192, 1000),       # explicit sample, default batch (one batch per chunk)
])
def test_pq_train_streaming_parity(oracle, vk, sizes, d, m, ks, iters, batch, sample_n):
    """Streaming trainer against the oracle on ragged chunk lists (one of them empty): per-chunk permutations, row sampling,
    blend, repair -- codebooks bit-identical (PQTrain.swift:391-706, 1444-1575)."""
    rng = np.random.default_rng(sum(sizes) + ks)
    chunks = [(rng.standard_normal((n, d)) + 2 * rng.standard_normal((5, d))[rng.integers(0, 5, n)]).astype(np.float32) for n in sizes]
    rc, ocb = oracle.pq_train_streaming(chunks, d, m, ks, seed=7, stream_id=3, algorithm=1, max_iters=iters, batch_size=batch,
                                        sample_n=sample_n)
    assert rc == 0
    cfg = vk.pq_train_cfg(algorithm=1, max_iters=iters, batch_size=batch, sample_n=sample_n, seed=7, stream_id=3, mode=0)
    gcb, gnorm = vk.pq_train_streaming_f32(chunks, m, ks, cfg)
    assert np.array_equal(bits(gcb), bits(ocb))
    from vectorindex_b200 import VectorIndexError
    with pytest.raises(VectorIndexError):
        vk.pq_train_streaming_f32([chunks[0][:ks - 1]], m, ks, cfg)      # fewer rows than centroids (PQTrain.swift:127-135)


def test_gpu_training_builds_a_working_index(oracle):
    """mode-1 trainers (deterministic Lloyd): the trained IVF-PQ index reaches a sane recall and two
    trainings give bit-identical parameters (rank-to-rank reproducibility for the sharded build)."""
    from vectorindex_b200 import datagen
    from vectorindex_b200.index import IVFPQIndex
    n, d, m, kc, nq, k = 30000, 64, 16, 64, 100, 10
    x = datagen.clustered_unit(n + nq, d, 200, 5)
    xb, q = x[:n], x[n:]
    params = []
    for _ in range(2):
        idx = IVFPQIndex(d, "euclidean", nlist=kc, nprobe=16, m=m)
        idx.optimize(xb)
        params.append((idx.get_coarse(), idx.get_codebooks()[0]))
    assert np.array_equal(bits(params[0][0]), bits(params[1][0]))
    assert np.array_equal(bits(params[0][1]), bits(params[1][1]))
    idx.batch_insert(xb)
    sizes = idx.list_sizes()
    assert sizes.sum() == n and (sizes > 0).sum() >= kc * 0.9
    gd, gi = idx.batch_search(q, k)
    _, ti, _ = oracle.flat_search(q, xb, k, 0)
    recall = np.mean([len(set(gi[r]) & set(ti[r])) / k for r in range(nq)])
    assert recall > 0.3, recall                                        # PQ-limited (m=16 codes of 64-d vectors)
    # and the oracle, fed the same trained parameters and lists, agrees with the GPU search
    off, codes, lids, _ = idx.export_lists()
    cb, norms = idx.get_codebooks()
    od, oi, _ = oracle.ivfpq_search(q, idx.get_coarse(), cb, norms, off, codes, lids, m, 256, 16, k, 0)
    assert_topk_close(gd, gi, od, oi)
