"""The oracle pinned against everything the reference's own tests hold for this path (SURVEY.md 8c):

  E1  the reference's C encoder (its stored outputs, tests/golden/cpq_encode_reference.npz), on the fixture of
      Tests/VectorIndexTests/PQEncodeParity_AoS_C_vs_Swift_Tests.swift:5-31
  E2  the bit-level golden vector of Tests/VectorIndexTests/PQTrainTests.swift:724-817
  E3  the published IVF recall 0.9565000000000008 (.bench/post-phase3/ivf_search.json:54)
  +   tie-break pins: TelemetryRecorderTests.swift:229-241, IVFSelectTests.swift:305-347,
      IVFListVecsReaderRerankTests.swift:5-126 (tie -> smaller id)
  +   tolerance fixtures, at the reference tests' own accuracies: ScoreBlockTests.swift:24-131 (LCG block, L2^2 / dot /
      cosine, 1e-4), IVFBatchGEMMParityTests.swift:160-190 (CentroidBatchScore, 1e-3)
"""
import os

import numpy as np
import pytest

import golden_inputs as gi
from conftest import parity_fixture
from vectorindex_b200 import datagen

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _reference_fixtures():
    """outputs of the reference's pq_encode.c (compiled unmodified) on the inputs of tests/golden_inputs.py"""
    return np.load(os.path.join(GOLD, "cpq_encode_reference_fixtures.npz"))


def test_e1_reference_encoder_fixture(oracle):
    """The reference encoder's outputs on this fixture are stored in tests/golden/cpq_encode_reference.npz ("parity.*",
    written by scripts/make_golden.py from pq_encode.c compiled unmodified)."""
    x, cb, coarse, assign = parity_fixture()
    csq = oracle.pq_centroid_sq(cb, 8, 256, 4, swift=False)
    ours = oracle.pq_encode_u8(x, cb, 8, 256, centroid_sq=csq)
    assert ours[0].tolist() == [212, 186, 160, 117, 255, 154, 186, 249]
    gold = np.load(os.path.join(GOLD, "cpq_encode_reference.npz"))
    assert np.array_equal(csq.view(np.uint32), gold["parity.csq"].view(np.uint32))
    assert np.array_equal(gold["parity.u8_csq"], ours)
    # direct path == dot path on this fixture (PQEncodeParity...:61)
    assert np.array_equal(gold["parity.u8_nodot"], ours) and np.array_equal(gold["parity.u8"], ours)


@pytest.mark.parametrize("variant", gi.ENCODER_VARIANTS)
def test_oracle_encoder_equals_reference_encoder(oracle, variant):
    """our C restatement of pq_encode.c vs the reference encoder's stored outputs, every entry point, random data."""
    x, cb, coarse, assign, m, ks = gi.encoder_variant_problem(variant)
    csq = oracle.pq_centroid_sq(cb, m, ks, x.shape[1] // m, swift=True)
    res = dict(coarse=coarse, assign_=assign) if variant.startswith("res") else {}
    if variant.endswith("u4"):
        b = oracle.pq_encode_u4(x, cb, m, ks, **res)
    elif variant.endswith("csq"):
        b = oracle.pq_encode_u8(x, cb, m, ks, centroid_sq=csq, **res)
    else:
        b = oracle.pq_encode_u8(x, cb, m, ks, use_dot=not variant.endswith("nodot"), **res)
    assert np.array_equal(_reference_fixtures()[f"variant.{variant}"], b)


def test_e2_pq_streaming_train_golden_bits(oracle):
    """PQTrainTests.swift:724-817: ks=16, d=16, m=2, n=40 in two chunks, LCG fill, seed 42, minibatch,
    maxIters 10, batch 512 => codebooks[0..3] bit patterns."""
    ks, d, m, n = 16, 16, 2, 40
    full = datagen.lcg24_floats(0x5773_7EA1_1234_5678, n * d)[0].reshape(n, d)
    chunks = [full[:20], full[20:]]
    rc, cb = oracle.pq_train_streaming(chunks, d, m, ks, seed=42, algorithm=1, max_iters=10, batch_size=512)
    assert rc == 0
    got = cb.reshape(-1)[:4]
    want = np.array([0.7648039, -0.5310464, -0.7147653, 0.30723625], dtype=np.float32)
    assert got.view(np.uint32).tolist() == want.view(np.uint32).tolist()
    assert np.isfinite(cb).all()


def test_e3_ivf_end_to_end_recall(oracle):
    """bench recipe (main.swift:267-268,535-548): n=5000, d=384, nlist=64, nprobe=4, q=200, k=10, seeds
    123/321; IVFIndex.optimize (sorted String ids, k-means++ seed 42, mini-batch 1024 x 20 epochs) +
    search; published recallAvg = 0.9565000000000008 (.bench/post-phase3/ivf_search.json:54)."""
    n, d, nq, k, nlist, nprobe = 5000, 384, 200, 10, 64, 4
    base = datagen.bench_vectors(n, d, 123)
    qs = datagen.bench_vectors(nq, d, 321)
    order = sorted(range(n), key=lambda i: "id%d" % i)          # IVFIndex.swift:325
    xs = base[order]
    cents, _ = oracle.kmeanspp_seed(xs, nlist, seed=42)
    rc, cents, asg, info = oracle.kmeans_minibatch(xs, nlist, init=cents, batch_size=1024, epochs=20, tol=1e-4,
                                                   seed=42, compute_assignments=True)
    assert rc == 0 and info["epochs"] == 2
    assert info["empties"].tolist() == [0, 1, 11, 34, 46, 53, 54, 57, 58, 58]
    sizes = np.bincount(asg, minlength=nlist)
    assert sorted(sizes[sizes > 0].tolist(), reverse=True) == [1748, 1450, 1316, 301, 148, 36, 1]

    def seqdist(q, X):                                            # sequential fp32 sum (stands in for VectorCore)
        acc = np.zeros(X.shape[0], dtype=np.float32)
        for j in range(X.shape[1]):
            df = (q[j] - X[:, j]).astype(np.float32)
            acc = (acc + df * df).astype(np.float32)
        return acc

    rec, ncand = [], []
    for qi in range(nq):
        q = qs[qi]
        sc = oracle.l2sqr_block(q, cents)                         # single-query path: L2Sqr dot-trick (d >= 256)
        probes = sorted(range(nlist), key=lambda c: (sc[c], c))[:nprobe]      # IVFIndex.swift:593-595
        idx = np.nonzero(np.isin(asg, probes))[0]
        ncand.append(idx.size)
        dd = seqdist(q, xs[idx])
        top = idx[np.lexsort((idx, dd))[:k]]
        bf = seqdist(q, xs)
        gt = np.lexsort((np.arange(n), bf))[:k]
        rec.append(len(set(top.tolist()) & set(gt.tolist())) / k)
    s = 0.0
    for r in rec:
        s += r
    assert repr(s / nq) == "0.9565000000000008"
    assert abs(np.mean(ncand) - 4680.8) < 0.05


def test_topk_max_tie_pin(oracle):
    """TelemetryRecorderTests.swift:229-241: top-3 .max of [5,3,8,1,9] with ids 10..14."""
    s, i = oracle.select_topk(np.array([5, 3, 8, 1, 9], dtype=np.float32), 3, oracle.ORDER_MAX,
                              ids=np.arange(10, 15, dtype=np.int32))
    assert s.tolist() == [9, 8, 5] and i.tolist() == [14, 12, 10]


def test_probe_identical_centroids_pin(oracle):
    """IVFSelectTests.swift:305-347: 50 identical centroids => ids 0..19 in order."""
    cents = np.ones((50, 8), dtype=np.float32)
    q = np.zeros((1, 8), dtype=np.float32)
    idx, _ = oracle.probe_select_batch(q, cents, 20)
    assert idx[0].tolist() == list(range(20))


def test_topk_min_tie_smaller_id(oracle):
    s, i = oracle.select_topk(np.array([1, 0, 0, 0, 2], dtype=np.float32), 2, oracle.ORDER_MIN)
    assert i.tolist() == [1, 2]
    ms, mi = oracle.merge_topk([(np.array([0.0, 1.0], np.float32), np.array([7, 1], np.int32)),
                                (np.array([0.0, 0.5], np.float32), np.array([3, 9], np.int32))], 3)
    assert mi.tolist() == [3, 7, 9]


# ------------------------------------------------------------------------------------------ tolerance fixtures
_M64 = (1 << 64) - 1


def _lcg_stream(seed):
    """The LCG every reference fixture uses: s = 2862933555777941757 s + 3037000493 (mod 2^64)."""
    s = seed & _M64
    while True:
        s = (2862933555777941757 * s + 3037000493) & _M64
        yield s


def _seq(fn, a, b):
    """Scalar float32 loop of the reference's test-side references (`expected += ...` in row order)."""
    acc = np.float32(0)
    for x, y in zip(a, b):
        acc = np.float32(acc + fn(np.float32(x), np.float32(y)))
    return acc


def test_scoreblock_lcg_fixture(oracle):
    """ScoreBlockTests.swift:24-131: n = 32, d = 16 blocks from the LCG (u = Float(s >> 40) / 2^24, value 2u - 1; seeds
    0x9E3779B97F4A7C15 / 0xD1B54A32D192ED03); L2^2, dot and cosine of ScoreBlock.run against the scalar loops of the test,
    at the test's own accuracy 1e-4."""
    def seeded(count, seed):
        g = _lcg_stream(seed)
        return np.array([np.float32(np.float32(next(g) >> 40) / np.float32(1 << 24)) * np.float32(2) - np.float32(1)
                         for _ in range(count)], dtype=np.float32)
    n, d = 32, 16
    q = seeded(d, 0x9E3779B97F4A7C15)
    xb = seeded(n * d, 0xD1B54A32D192ED03).reshape(n, d)
    assert q.min() >= -1 and q.max() < 1 and abs(float(xb.mean())) < 0.2
    l2 = oracle.l2sqr_block(q, xb)
    ip = oracle.ip_block(q, xb)
    cd, ci, _ = oracle.flat_search(q[None, :], xb, n, 2)                     # cosine: API distance 1 - similarity
    cos = np.empty(n, np.float32)
    cos[ci[0]] = np.float32(1) - cd[0]
    eps = np.float32(1e-12)
    q_inv = np.float32(1) / (np.sqrt(_seq(lambda a, b: a * b, q, q)) + eps)
    for i in range(n):
        assert abs(l2[i] - _seq(lambda a, b: (a - b) * (a - b), q, xb[i])) <= 1e-4, i
        dot = _seq(lambda a, b: a * b, q, xb[i])
        assert abs(ip[i] - dot) <= 1e-4, i
        x_inv = np.float32(1) / (np.sqrt(_seq(lambda a, b: a * b, xb[i], xb[i])) + eps)
        want = max(np.float32(-1), min(np.float32(1), np.float32(np.float32(dot * q_inv) * x_inv)))
        assert abs(cos[i] - want) <= 1e-4, i


@pytest.mark.parametrize("metric,seed", [(0, 99), (1, 123)])
def test_centroid_batch_score_lcg_fixture(oracle, metric, seed):
    """IVFBatchGEMMParityTests.swift:160-190: d = 12, kc = 7, nq = 5 from LCG(state) with nextInRange(-1...1) =
    -1 + 2 * Float(s >> 11) / 2^53; CentroidBatchScore against `cNormSq - 2 dot` / `-dot` at the test's accuracy 1e-3."""
    g = _lcg_stream(seed)

    def nxt():
        return np.float32(-1) + np.float32(2) * np.float32(np.float32(next(g) >> 11) / np.float32(1 << 53))
    d, kc, nq = 12, 7, 5
    queries = np.array([[nxt() for _ in range(d)] for _ in range(nq)], dtype=np.float32)
    cents = np.array([[nxt() for _ in range(d)] for _ in range(kc)], dtype=np.float32)
    got = oracle.centroid_batch_score(queries, cents, metric)
    for qi in range(nq):
        for c in range(kc):
            dot = _seq(lambda a, b: a * b, queries[qi], cents[c])
            want = (_seq(lambda a, b: a * b, cents[c], cents[c]) - np.float32(2) * dot) if metric == 0 else -dot
            assert abs(got[qi, c] - want) <= 1e-3, (qi, c)


def test_rerank_reader_fixtures(oracle):
    """IVFListVecsReaderRerankTests.swift:5-126: rows (0,0) (1,0) (0,1) (1,1); the nearest two of q = (0.95, 0.06) are ids
    1, 3; for q = (0.95, 0.05) ids 0 and 3 tie for second place and the smaller id wins (L2Sqr.run scores + the
    (score, id) order of the selection)."""
    rows = np.array([[0, 0], [1, 0], [0, 1], [1, 1]], dtype=np.float32)
    s = oracle.l2sqr_block(np.array([0.95, 0.06], np.float32), rows)
    _, ids = oracle.select_topk(s, 2, oracle.ORDER_MIN)
    assert ids.tolist() == [1, 3]
    s = oracle.l2sqr_block(np.array([0.95, 0.05], np.float32), rows)
    assert s[0] == s[3]
    _, ids = oracle.select_topk(s, 2, oracle.ORDER_MIN)
    assert ids.tolist() == [1, 0]


def test_centroid_batch_score_cosine_degenerate_centroid_fixture(oracle):
    """IVFBatchGEMMParityTests.swift:192-214: LCG(456), d = 12, kc = 6, nq = 5, centroid 2 all zero; cosine scores
    1 - dot qInv cInv at the test's accuracy 1e-3, and the degenerate centroid forced to exactly 1."""
    g = _lcg_stream(456)

    def nxt():
        return np.float32(-1) + np.float32(2) * np.float32(np.float32(next(g) >> 11) / np.float32(1 << 53))
    d, kc, nq = 12, 6, 5
    queries = np.array([[nxt() for _ in range(d)] for _ in range(nq)], dtype=np.float32)
    cents = np.array([[nxt() for _ in range(d)] for _ in range(kc)], dtype=np.float32)
    cents[2] = 0.0
    got = oracle.centroid_batch_score(queries, cents, 2)
    eps = np.float32(1e-12)
    for qi in range(nq):
        qn = _seq(lambda a, b: a * b, queries[qi], queries[qi])
        for c in range(kc):
            cn = _seq(lambda a, b: a * b, cents[c], cents[c])
            dot = _seq(lambda a, b: a * b, queries[qi], cents[c])
            if np.sqrt(np.float32(qn * cn)) > np.finfo(np.float32).eps:
                want = np.float32(1) - dot * (np.float32(1) / (np.sqrt(qn) + eps)) * (np.float32(1) / (np.sqrt(cn) + eps))
            else:
                want = np.float32(1)
            assert abs(got[qi, c] - want) <= 1e-3, (qi, c)
        assert got[qi, 2] == np.float32(1)
    # probe order and list assignment under cosine follow the same scores (IVFIndex.swift:376-435, 905-927)
    pid, psc = oracle.probe_select_batch(queries, cents, 3, 2)
    for qi in range(nq):
        order = np.lexsort((np.arange(kc), got[qi]))[:3]
        assert pid[qi].tolist() == order.tolist() and np.array_equal(psc[qi], got[qi][order])
    assert np.array_equal(oracle.assign_metric(queries, cents, 2), np.argmin(got, axis=1))


def test_fused_residual_encode_equals_materialised(oracle):
    """ResidualKernelTests.swift:126-200 (n = 2000, d = 1024, m = 8, ks = 256, kc = 100, uniform [-1, 1)): the fused
    residual encoder and the plain encoder on materialised residuals give the same codes -- for the restatement and for
    the reference's own compiled C encoder (its stored outputs), which also agree with each other."""
    x, cent, asg, cb, m, ks = gi.long_subvector_residual_problem()
    r = (x - cent[asg]).astype(np.float32)
    plain = oracle.pq_encode_u8(r, cb, m, ks)
    fused = oracle.pq_encode_u8(x, cb, m, ks, coarse=cent, assign_=asg)
    assert np.array_equal(plain, fused)
    gold = _reference_fixtures()
    assert np.array_equal(gold["long_residual.plain"], plain)
    assert np.array_equal(gold["long_residual.fused"], fused)


def test_cosine_zero_norm_and_clamp_pins(oracle):
    """CosineKernelTests.swift:124-160: an all-zero row has similarity 0 (API distance 1), and two identical vectors of
    1000s give a similarity that the clamp keeps at <= 1 (distance >= 0)."""
    rng = np.random.default_rng(4)
    q = rng.uniform(-1, 1, (1, 16)).astype(np.float32)
    xb = rng.uniform(-1, 1, (4, 16)).astype(np.float32)
    xb[0] = 0.0
    d, i, _ = oracle.flat_search(q, xb, 4, 2)
    assert abs(float(d[0][i[0] == 0][0]) - 1.0) <= 1e-6
    big = np.full((1, 8), 1000.0, np.float32)
    d, _, _ = oracle.flat_search(big, big, 1, 2)
    assert 0.0 <= float(d[0, 0]) <= 1e-6


def _kmeanspp_edge_cases():
    """KMeansPPSeedingTests.swift:182-296: (data, k, seed) of testKEqualsOne / testKEqualsN / testDuplicateData."""
    return [
        (np.arange(60, dtype=np.float32).reshape(20, 3), 1, 999),
        (np.arange(20, dtype=np.float32).reshape(10, 2), 10, 42),
        (np.array([[0, 0, 0]] * 5 + [[1, 1, 1]] * 5, dtype=np.float32), 3, 555),
    ]


def test_kmeanspp_edge_case_pins(oracle):
    """k = 1: one valid index; k = n: every point chosen once; duplicated points: still k distinct indices (the zero-total
    fallback of the D^2 sampler, KMeansSeeding.swift:368-409)."""
    for data, k, seed in _kmeanspp_edge_cases():
        cents, chosen = oracle.kmeanspp_seed(data, k, seed, 0)
        assert len(set(chosen.tolist())) == k and chosen.min() >= 0 and chosen.max() < data.shape[0]
        assert np.array_equal(cents, data[chosen])


def _kmeans_minibatch_edge_cases():
    """KMeansMiniBatchTests.swift:405-487, 616-646: (x, kc, init, batch, epochs) of testSingleCentroid (seeded stand-in for
    its random data), testBatchSizeLargerThanN (its own deterministic fixture) and testIdenticalData."""
    rng = np.random.default_rng(0)
    n, d, k = 30, 4, 3
    data = (np.arange(n * d) % 20 / 5.0).astype(np.float32).reshape(n, d)
    init = (np.arange(k * d) % 15 / 5.0).astype(np.float32).reshape(k, d)
    return [
        (rng.uniform(-5, 5, (50, 3)).astype(np.float32), 1, None, 10, 5),
        (data, k, init, 100, 10),
        (np.ones((50, 4), np.float32), 3, None, 10, 5),
    ]


def test_kmeans_minibatch_edge_case_pins(oracle):
    (x1, k1, i1, b1, e1), (x2, k2, i2, b2, e2), (x3, k3, i3, b3, e3) = _kmeans_minibatch_edge_cases()
    rc, c, _, _ = oracle.kmeans_minibatch(x1, k1, i1, b1, e1, 1e-4, 0, 0)
    assert rc == 0 and np.linalg.norm(c[0] - x1.mean(0)) < 3.0            # "single centroid should be near data mean"
    rc, c, _, _ = oracle.kmeans_minibatch(x2, k2, i2, b2, e2, 1e-4, 0, 0)
    assert rc == 0 and np.isfinite(c).all()                                # batchSize > n is handled
    rc, c, _, _ = oracle.kmeans_minibatch(x3, k3, i3, b3, e3, 1e-4, 0, 0)
    assert rc == 0 and np.abs(c - 1.0).max() <= 0.1                        # identical data: every centroid on the point


def test_pq_train_data_requirements(oracle):
    """PQTrainTests.swift:574-625: n == ks is the minimum viable training set; n < ks is .emptyInput (status -4)."""
    rng = np.random.default_rng(0)
    rc, cb, _, _ = oracle.pq_train(rng.uniform(-1, 1, (64, 128)).astype(np.float32), 4, 64)
    assert rc == 0 and cb.shape == (4, 64, 32) and np.isfinite(cb).all()
    assert oracle.pq_train(np.zeros((50, 128), np.float32), 4, 100)[0] == -4


def test_encode_with_csq_equals_default_fixture(oracle):
    """PQEncodeParity_SwiftOnly_Tests.swift:41-106 (n = 12, d = 24, m = 6, ks = 256 on the sin / cos fixture, sequential
    centroid norms): the with-CSQ encoders give the codes of the default ones, plain and residual -- for the restatement and,
    where oracle/_ref is built, for the reference's compiled C encoder (its codes on this fixture are not stored: no test
    has pinned the restatement to them here, so nothing records what they are)."""
    n, d, m, ks, kc = 12, 24, 6, 256, 4
    dsub = d // m
    i = np.arange(n * d, dtype=np.int64)
    x = (np.sin((i * 131 % 1024).astype(np.float64)) * 0.25 + np.cos((i * 17 % 997).astype(np.float64)) * 0.125).astype(np.float32).reshape(n, d)
    j = np.arange(m * ks * dsub, dtype=np.int64)
    cb = (np.sin((j * 313 % 2048).astype(np.float64)) * 0.2 + np.cos((j * 23 % 1237).astype(np.float64)) * 0.15).astype(np.float32)
    g = np.arange(kc * d, dtype=np.int64)
    coarse = (np.cos((g * 19 % 4096).astype(np.float64)) * 0.33).astype(np.float32).reshape(kc, d)
    asg = (np.arange(n) % kc).astype(np.int32)
    csq = oracle.pq_centroid_sq(cb, m, ks, dsub, swift=True)             # s += v * v, in order
    assert np.array_equal(oracle.pq_encode_u8(x, cb, m, ks, centroid_sq=csq), oracle.pq_encode_u8(x, cb, m, ks))
    assert np.array_equal(oracle.pq_encode_u8(x, cb, m, ks, centroid_sq=csq, coarse=coarse, assign_=asg),
                          oracle.pq_encode_u8(x, cb, m, ks, coarse=coarse, assign_=asg))
    if oracle.ref_lib() is not None:
        assert np.array_equal(oracle.ref_encode("cpq_encode_u8_f32_with_csq", x, cb, m, ks, centroid_sq=csq),
                              oracle.ref_encode("cpq_encode_u8_f32", x, cb, m, ks))
        assert np.array_equal(oracle.ref_encode("cpq_encode_residual_u8_f32_with_csq", x, cb, m, ks, centroid_sq=csq,
                                                coarse=coarse, assign_=asg),
                              oracle.ref_encode("cpq_encode_residual_u8_f32", x, cb, m, ks, coarse=coarse, assign_=asg))


def test_cosine_degenerate_centroid_fixtures(oracle):
    """IVFCosineCentroidEdgeCaseTests.swift:27-134: centroids (1,1,0..), (1,0,0..), (1e-8,0,..) and the query (1,1,0..):
    the tiny-norm centroid scores EXACTLY 1 (the guard, not an approximation), the identical direction ~0, both
    well-formed centroids sort before it, so nprobe = 2 of 3 never probes its list while nprobe = 3 reaches it; all-NaN
    centroid scores assign nothing (-1)."""
    c = np.zeros((3, 8), np.float32)
    c[0, :2] = 1.0
    c[1, 0] = 1.0
    c[2, 0] = 1e-8
    q = np.zeros((1, 8), np.float32)
    q[0, :2] = 1.0
    s = oracle.centroid_batch_score(q, c, 2)[0]
    assert s[2] == np.float32(1.0) and s[0] < s[2] and s[1] < s[2] and abs(float(s[0])) <= 1e-6
    assert oracle.probe_select_batch(q, c, 2, 2)[0][0].tolist() == [0, 1]
    assert oracle.probe_select_batch(q, c, 3, 2)[0][0].tolist() == [0, 1, 2]
    # one vector in list 0, one that only a probe of the degenerate centroid's list can surface
    vecs = np.stack([q[0], q[0]])
    off = np.array([0, 1, 1, 2], dtype=np.int64)
    ids = np.array([10, 20], dtype=np.int64)
    _, i2 = oracle.ivfflat_search(q, c, off, vecs, ids, 2, 5, 2)
    _, i3 = oracle.ivfflat_search(q, c, off, vecs, ids, 3, 5, 2)
    assert set(i2[0][i2[0] >= 0].tolist()) == {10} and set(i3[0][i3[0] >= 0].tolist()) == {10, 20}
    nan_c = np.array([[np.nan, 0, 0, 0], [np.nan, 1, 1, 1]], dtype=np.float32)
    assert oracle.assign_metric(np.zeros((1, 4), np.float32), nan_c, 0).tolist() == [-1]


def test_recall_improves_with_nprobe_fixture(oracle):
    """IVFProbeMonotonicTests.swift:18-44: n = 300, d = 32, nlist = 32, 20 queries, k = 5, LCG seeds 17 / 19, the actor's
    optimize() (sorted String ids, k-means++ seed 42, mini-batch min(1024, n) x 20 epochs): recall with nprobe = 8 is at
    least the recall with nprobe = 1."""
    n, d, nq, k, nlist = 300, 32, 20, 5, 32
    base = datagen.bench_vectors(n, d, 17)
    qs = datagen.bench_vectors(nq, d, 19)
    order = sorted(range(n), key=lambda i: "id%d" % i)          # IVFIndex.swift:325
    xs = base[order]
    cents, _ = oracle.kmeanspp_seed(xs, nlist, seed=42)
    rc, cents, asg, _ = oracle.kmeans_minibatch(xs, nlist, init=cents, batch_size=min(1024, n), epochs=20, tol=1e-4,
                                                seed=42, compute_assignments=True)
    assert rc == 0
    off, lorder = oracle.build_lists(asg, nlist)
    ids = np.arange(n, dtype=np.int64)
    truth = oracle.flat_search(qs, xs, k, 0)[1]
    avg = []
    for nprobe in (1, 8):
        _, got = oracle.ivfflat_search(qs, cents, off, xs[lorder], ids[lorder], nprobe, k, 0)
        avg.append(np.mean([len(set(truth[r].tolist()) & set(got[r][got[r] >= 0].tolist())) / k for r in range(nq)]))
    assert avg[1] >= avg[0] and avg[1] > 0.5


def test_fused_residual_lut_equals_lut_of_materialised_residual(oracle):
    """ResidualKernelTests.swift:208-270 (disabled there over an alignment precondition of the LUT kernel, the property
    itself is the contract of pq_lut_residual_l2_f32, PQLUT.swift:266-386): the fused residual LUT equals the plain LUT of
    the materialised residual q - c.  Both restatements subtract first and walk the same accumulators (PQLUT.swift:293-341
    against :197-240), so with the reference test's shape (d 512, m 8, ks 256) and without centroid norms the two tables are
    bit-identical -- far inside the reference's own 1e-4; with norms + dot trick the reference's tolerance applies."""
    rng = np.random.default_rng(208)
    d, m, ks = 512, 8, 256
    q = rng.uniform(-1, 1, d).astype(np.float32)
    c = rng.uniform(-1, 1, d).astype(np.float32)
    cb = rng.uniform(-1, 1, m * ks * (d // m)).astype(np.float32)
    fused = oracle.pq_lut_residual_l2(q, c, cb, m, ks)
    plain = oracle.pq_lut_l2((q - c).astype(np.float32), cb, m, ks)
    assert np.array_equal(fused.view(np.uint32), plain.view(np.uint32))
    cn = oracle.pq_centroid_sq(cb, m, ks, d // m, swift=False)
    fused_n = oracle.pq_lut_residual_l2(q, c, cb, m, ks, cn)
    plain_n = oracle.pq_lut_l2((q - c).astype(np.float32), cb, m, ks, cn)
    assert np.max(np.abs(fused_n - plain_n)) < 1e-4 and np.max(np.abs(fused_n - plain)) < 1e-3
