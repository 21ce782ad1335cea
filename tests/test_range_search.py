"""Range search (vix_index_range_search): every stored vector within a radius, per query sorted by (distance, id).

The reference answer of a case is the oracle's own k-NN search with k = every candidate (flat: every row; IVF: every row of
the probed lists, the oracle's probe selection), cut at the radius and sorted by (distance, id): the per-candidate
arithmetic of vo_flat_search / vo_ivfflat_search / vo_ivfpq_search, with no new code in the oracle.  A case checks
  - flat and IVF-Flat (L2, IP): the same CSR as that reference, ids equal, distance bits equal;
  - IVF-Flat cosine (whose oracle is tolerance parity): the oracle to 1e-5, and the library's own k-NN search bit for bit;
  - IVF-PQ: the route taken (the "[vix range]" line of VIX_SCAN_DEBUG=1), the oracle outside a band of relative width RTOL
    around the radius, and the library's k-NN search on the query-major scan (VIX_TC_SCAN=0, same probes): the k-NN
    entries within the radius are the first entries of the range row, bit for bit;
  - the output path: rows of more than a million entries (merged in global memory), a first capacity that is too small
    (two passes, then one), repeated calls give the same bits.
"""
import re
import zlib

import numpy as np
import pytest

from pq_ref64 import RTOL
from test_gpu_parity import bits
from test_scan_edges import queries_near, random_pq
from vectorindex_b200 import _lib

gpu = pytest.mark.gpu
RANGE = re.compile(r"\[vix range\] kind (\w+), kernel (fast G \d|generic|ivfflat|flat), filter (\d), passes (\d), "
                   r"total (\d+), max_row (\d+), sorted_long (\d+)")
METRICS = {0: "euclidean", 1: "dotProduct", 2: "cosine"}
ERR_INVALID_K, ERR_INVALID_PARAM = -2, -5


# ------------------------------------------------------------------------------------------------ building blocks
def cut(od, oi, radius, keep=None):
    """CSR of the entries of sorted k-NN rows (padded with id -1) within the radius (and passing `keep`), by (distance, id)"""
    lims, dist, ids = [0], [], []
    for r in range(od.shape[0]):
        d, i = od[r], oi[r]
        sel = (i >= 0) & (d <= np.float32(radius))
        if keep is not None:
            sel &= keep(i)
        d, i = d[sel], i[sel]
        o = np.lexsort((i, d))
        dist.append(d[o]); ids.append(i[o])
        lims.append(lims[-1] + int(sel.sum()))
    return (np.array(lims, np.int64), np.concatenate(dist).astype(np.float32) if dist else np.zeros(0, np.float32),
            np.concatenate(ids).astype(np.int64) if ids else np.zeros(0, np.int64))


def same_csr(got, want):
    assert np.array_equal(got[0], want[0]), "row lengths differ"
    assert np.array_equal(got[2], want[2]), "ids differ"
    assert np.array_equal(bits(got[1]), bits(want[1])), "distance bits differ"


def knn_prefix(got, kd, ki, radius):
    """the k-NN entries within the radius are the first entries of each range row, bit for bit (the whole row when the
    k-NN row was not full)"""
    lims, dist, ids = got
    for r in range(len(lims) - 1):
        a, da = ids[lims[r]:lims[r + 1]], dist[lims[r]:lims[r + 1]]
        sel = (ki[r] >= 0) & (kd[r] <= radius)
        n = int(sel.sum())
        assert np.array_equal(a[:n], ki[r][sel]), f"row {r}: ids differ from k-NN"
        assert np.array_equal(bits(da[:n]), bits(kd[r][sel])), f"row {r}: distance bits differ from k-NN"
        if ki[r, -1] < 0:
            assert a.size == n, f"row {r}: {a.size} entries, k-NN found {n}"


def ranged(mp, capfd, fn):
    """fn() under VIX_SCAN_DEBUG=1 -> (its result, the fields of its one [vix range] line)"""
    capfd.readouterr()
    mp.setenv("VIX_SCAN_DEBUG", "1")
    try:
        out = fn()
    finally:
        mp.delenv("VIX_SCAN_DEBUG")
    lines = RANGE.findall(capfd.readouterr().err)
    assert len(lines) == 1, f"{len(lines)} [vix range] lines"
    g = lines[0]
    return out, dict(kind=g[0], kernel=g[1], filter=int(g[2]), passes=int(g[3]), total=int(g[4]), max_row=int(g[5]),
                     sorted_long=int(g[6]))


def radii(od, oi):
    """quantiles of the candidate distances, one radius equal to a stored distance, one below every distance, +inf"""
    v = od[(oi >= 0) & np.isfinite(od)]
    qs = [np.float32(x) for x in np.quantile(v.astype(np.float64), [0.002, 0.02, 0.2])]
    return qs + [np.float32(od[0, 3]), np.nextafter(np.float32(v.min()), np.float32(-np.inf)), np.float32(np.inf)]


def filters(capacity, rng):
    from vectorindex_b200.index import IDFilter
    allow = IDFilter(capacity, "allow")
    allow.set(rng.choice(capacity, capacity // 3, replace=False))
    deny = IDFilter(capacity, "deny")
    deny.set(rng.choice(capacity, capacity // 4, replace=False))
    return {"none": None, "allow": allow, "deny": deny}


# ------------------------------------------------------------------------------------------------ CPU: the reference cut
def test_cut_matches_float64_brute_force(oracle):
    """CPU: the oracle's full flat ranking cut at a radius equals a float64 brute force, outside a band around the radius."""
    rng = np.random.default_rng(3)
    xb = rng.standard_normal((500, 24)).astype(np.float32)
    q = rng.standard_normal((6, 24)).astype(np.float32)
    ids = np.arange(500, dtype=np.int64)
    for metric in (0, 1):
        od, oi, _ = oracle.flat_search(q, xb, 500, metric)
        d64 = (np.sqrt(((q[:, None, :].astype(np.float64) - xb[None]) ** 2).sum(-1)) if metric == 0
               else -(q.astype(np.float64) @ xb.T.astype(np.float64)))
        for radius in np.quantile(d64, [0.01, 0.1, 0.5]):
            lims, dist, got = cut(od, oi, radius)
            for r in range(len(q)):
                row = set(got[lims[r]:lims[r + 1]].tolist())
                band = RTOL * max(1.0, abs(radius))
                assert set(ids[d64[r] < radius - band].tolist()) <= row
                assert row <= set(ids[d64[r] <= radius + band].tolist())
                np.testing.assert_allclose(dist[lims[r]:lims[r + 1]], d64[r][got[lims[r]:lims[r + 1]]], rtol=1e-5, atol=1e-5)


# ------------------------------------------------------------------------------------------------ flat
@gpu
@pytest.mark.parametrize("metric,d", [(0, 40), (0, 300), (1, 40), (2, 36)], ids=["l2", "l2_dot", "ip", "cosine"])
def test_flat(oracle, monkeypatch, capfd, metric, d):
    """Direct16 below d = 256, the dot form with norms from d = 256, Ip4, cosine: the oracle's CSR and bits."""
    from vectorindex_b200.index import FlatIndex
    rng = np.random.default_rng(10 + d + metric)
    n, nq = 2500, 12
    xb = rng.standard_normal((n, d)).astype(np.float32)
    q = rng.standard_normal((nq, d)).astype(np.float32)
    ids = rng.permutation(n).astype(np.int64) * 2 + 7
    idx = FlatIndex(d, METRICS[metric])
    idx.batch_insert(xb, ids)
    od, oi, _ = oracle.flat_search(q, xb, n, metric)
    oi = np.where(oi >= 0, ids[np.maximum(oi, 0)], -1)
    for radius in radii(od, oi):
        got, route = ranged(monkeypatch, capfd, lambda: idx.range_search(q, radius))
        assert route["kind"] == "flat" and route["kernel"] == "flat" and route["filter"] == 0
        same_csr(got, cut(od, oi, radius))
    # the radius equal to a stored distance keeps that entry; below every distance: empty; +inf: everything
    lims, dist, gi = idx.range_search(q, od[0, 3])
    assert oi[0, 3] in gi[lims[0]:lims[1]]
    v = od[(oi >= 0)]
    assert idx.range_search(q, np.nextafter(np.float32(v.min()), np.float32(-np.inf)))[0][-1] == 0
    assert idx.range_search(q, np.inf)[0][-1] == nq * n


# ------------------------------------------------------------------------------------------------ IVF-Flat
@gpu
@pytest.mark.parametrize("fname", ["none", "allow", "deny"])
@pytest.mark.parametrize("metric", [0, 1, 2], ids=["l2", "ip", "cosine"])
def test_ivfflat(oracle, monkeypatch, capfd, metric, fname):
    """Trained: the oracle's CSR and bits (cosine: to 1e-5, and the library's k-NN bit for bit); un-optimised: the linear
    scan through the flat engine, the oracle's flat CSR and bits.  With allow and deny filters."""
    from vectorindex_b200.index import IVFIndex
    rng = np.random.default_rng(20 + metric)
    n, d, kc, nq, nprobe = 1600, 32, 20, 16, 4
    xb = rng.standard_normal((n, d)).astype(np.float32)
    q = rng.standard_normal((nq, d)).astype(np.float32)
    coarse = np.ascontiguousarray(xb[rng.choice(n, kc, replace=False)])
    ids = np.arange(n, dtype=np.int64) * 3 + 1
    filt = filters(int(ids.max()) + 1, rng)[fname]
    keep = filt.test if filt is not None else None
    # un-optimised: a linear scan over every row
    lin = IVFIndex(d, METRICS[metric], nlist=kc, nprobe=nprobe)
    lin.batch_insert(xb, ids)
    od, oi, _ = oracle.flat_search(q, xb, n, metric)
    oi = np.where(oi >= 0, ids[np.maximum(oi, 0)], -1)
    for radius in radii(od, oi)[:3]:
        got, route = ranged(monkeypatch, capfd, lambda: lin.range_search(q, radius, filter=filt))
        assert route["kind"] == "ivfflat" and route["kernel"] == "flat" and route["filter"] == int(filt is not None)
        same_csr(got, cut(od, oi, radius, keep))
    # trained
    ivf = IVFIndex(d, METRICS[metric], nlist=kc, nprobe=nprobe)
    ivf.set_coarse(coarse)
    ivf.batch_insert(xb, ids)
    asg = oracle.assign(xb, coarse)[0] if metric == 0 else oracle.assign_metric(xb, coarse, metric)
    off, order = oracle.build_lists(asg, kc)
    od, oi = oracle.ivfflat_search(q, coarse, off, xb[order], ids[order], nprobe, n, metric)
    kd, ki = ivf.batch_search(q, 512, filter=filt)
    for radius in radii(od, oi)[:3] + [np.float32(np.inf)]:
        got, route = ranged(monkeypatch, capfd, lambda: ivf.range_search(q, radius, filter=filt))
        assert route["kind"] == "ivfflat" and route["kernel"] == "ivfflat" and route["filter"] == int(filt is not None)
        knn_prefix(got, kd, ki, radius)
        want = cut(od, oi, radius, keep)
        if metric != 2:
            same_csr(got, want)
        elif np.isfinite(radius):
            lims, dist, gi = got
            for r in range(nq):     # tolerance parity: the same ids away from the radius, distances to 1e-5
                a, b = gi[lims[r]:lims[r + 1]], want[2][want[0][r]:want[0][r + 1]]
                da, db = dist[lims[r]:lims[r + 1]], want[1][want[0][r]:want[0][r + 1]]
                assert set(a[da < radius - 1e-5]) <= set(b) and set(b[db < radius - 1e-5]) <= set(a)
        else:
            assert np.array_equal(got[0], want[0])


# ------------------------------------------------------------------------------------------------ IVF-PQ
PQ_CASES = {                       # name: (m, dsub, ks, kernel)
    "fast16": (16, 2, 256, "fast G 1"), "fast32": (32, 2, 256, "fast G 2"), "fast48": (48, 2, 256, "fast G 3"),
    "fast64": (64, 2, 256, "fast G 4"), "generic12": (12, 2, 256, "generic"), "ks16_m16": (16, 2, 16, "generic"),
}


@gpu
@pytest.mark.parametrize("filtered", [False, True], ids=["plain", "filter"])
@pytest.mark.parametrize("metric", [0, 1], ids=["l2", "ip"])
@pytest.mark.parametrize("name", list(PQ_CASES))
def test_ivfpq(oracle, monkeypatch, capfd, name, metric, filtered):
    from vectorindex_b200.index import IDFilter
    m, dsub, ks, kernel = PQ_CASES[name]
    rng = np.random.default_rng(zlib.crc32(f"{name}/{metric}/{filtered}".encode()))
    kc, nq, nprobe, k = 12, 40, 4, 64
    P = random_pq(oracle, rng, m, dsub, rng.integers(100, 250, kc), ks=ks, metric=metric)
    q = queries_near(rng, P, rng.integers(0, kc, nq))
    filt = None
    if filtered:
        filt = IDFilter(int(P.lids.max()) + 1, "allow")
        filt.set(rng.choice(P.lids, P.lids.size // 2, replace=False))
    n = int(P.off[-1])
    od, oi, op = P.oracle(oracle, q, nprobe, n)
    assert np.array_equal(op, P.probes(q, nprobe)), "probes differ from the oracle's"
    monkeypatch.setenv("VIX_TC_SCAN", "0")
    kd, ki = P.idx.batch_search(q, k, nprobe=nprobe, filter=filt)
    keep = filt.test if filt is not None else None
    scale = float(np.nanmax(np.abs(od[oi >= 0])))
    for radius in radii(od, oi)[:4] + [np.float32(np.nanmin(kd[:, k // 2]))]:
        got, route = ranged(monkeypatch, capfd, lambda: P.idx.range_search(q, radius, nprobe=nprobe, filter=filt))
        assert route["kind"] == "ivfpq" and route["kernel"] == kernel and route["filter"] == int(filtered)
        lims, dist, gi = got
        want = cut(od, oi, radius, keep)
        band = RTOL * max(abs(float(radius)), scale if metric == 1 else 0.0)
        for r in range(nq):
            a, da = gi[lims[r]:lims[r + 1]], dist[lims[r]:lims[r + 1]]
            b, db = want[2][want[0][r]:want[0][r + 1]], want[1][want[0][r]:want[0][r + 1]]
            assert (da <= radius).all() and (np.diff(da) >= 0).all()
            assert set(a[da < radius - band]) <= set(b) and set(b[db < radius - band]) <= set(a)
            common, ia, ib = np.intersect1d(a, b, return_indices=True)
            np.testing.assert_allclose(da[ia], db[ib], rtol=RTOL, atol=RTOL * scale if metric == 1 else 0.0)
        # the library's own k-NN: its entries within the radius open the range row, bit for bit
        knn_prefix(got, kd, ki, radius)


# ------------------------------------------------------------------------------------------------ output path
@gpu
def test_long_rows_and_two_passes(oracle, monkeypatch, capfd):
    """Rows of more than a million entries (runs merged in global memory); the first call outgrows its capacity and scans
    twice, the second takes one pass; both give the oracle's CSR and identical bits."""
    from vectorindex_b200.index import FlatIndex
    rng = np.random.default_rng(5)
    n, d, nq = 1_100_000, 8, 2
    xb = rng.standard_normal((n, d)).astype(np.float32)
    q = rng.standard_normal((nq, d)).astype(np.float32)
    idx = FlatIndex(d, "euclidean")
    idx.batch_insert(xb)
    od, oi, _ = oracle.flat_search(q, xb, n, 0)
    radius = np.float32(np.inf)
    first, r1 = ranged(monkeypatch, capfd, lambda: idx.range_search(q, radius))
    assert r1["passes"] == 2 and r1["sorted_long"] == nq and r1["max_row"] == n and r1["total"] == nq * n
    same_csr(first, cut(od, oi, radius))
    second, r2 = ranged(monkeypatch, capfd, lambda: idx.range_search(q, radius))
    assert r2["passes"] == 1
    same_csr(second, first)
    radius = np.float32(np.quantile(od[0], 0.6))
    got, r3 = ranged(monkeypatch, capfd, lambda: idx.range_search(q, radius))
    assert r3["passes"] == 1 and r3["sorted_long"] >= 1
    same_csr(got, cut(od, oi, radius))


@gpu
def test_batch_over_first_capacity(oracle, monkeypatch, capfd):
    """Many short rows whose total exceeds the first capacity: two passes, the oracle's CSR; then one pass, same bits."""
    from vectorindex_b200.index import FlatIndex
    rng = np.random.default_rng(6)
    n, d, nq = 3000, 16, 64
    xb = rng.standard_normal((n, d)).astype(np.float32)
    q = rng.standard_normal((nq, d)).astype(np.float32)
    idx = FlatIndex(d, "dotProduct")
    idx.batch_insert(xb)
    od, oi, _ = oracle.flat_search(q, xb, n, 1)
    radius = np.float32(np.quantile(od, 0.5))
    got, r1 = ranged(monkeypatch, capfd, lambda: idx.range_search(q, radius))
    assert r1["passes"] == 2 and r1["total"] > 65536 and r1["sorted_long"] == 0
    same_csr(got, cut(od, oi, radius))
    again, r2 = ranged(monkeypatch, capfd, lambda: idx.range_search(q, radius))
    assert r2["passes"] == 1
    same_csr(again, got)


# ------------------------------------------------------------------------------------------------ contract edges
@gpu
def test_contract_edges(oracle):
    import torch
    from vectorindex_b200.index import FlatIndex, IVFIndex
    rng = np.random.default_rng(7)
    n, d = 400, 16
    xb = rng.standard_normal((n, d)).astype(np.float32)
    q = rng.standard_normal((5, d)).astype(np.float32)
    idx = FlatIndex(d, "euclidean")
    # an empty index; nq = 0
    lims, dist, ids = idx.range_search(q, np.inf)
    assert lims.tolist() == [0] * 6 and dist.size == 0 and ids.size == 0
    idx.batch_insert(xb)
    lims, dist, ids = idx.range_search(np.zeros((0, d), np.float32), 1.0)
    assert lims.tolist() == [0] and dist.size == 0
    # NaN radius; negative L2 radius
    with pytest.raises(_lib.VectorIndexError) as e:
        idx.range_search(q, float("nan"))
    assert e.value.status == ERR_INVALID_PARAM
    assert idx.range_search(q, -0.5)[0][-1] == 0
    # duplicate ids come back twice; removed ids never
    idx.batch_insert(xb[:3], np.array([0, 1, 2], np.int64))
    lims, dist, ids = idx.range_search(xb[:1], 1e-3)
    assert sorted(ids.tolist()) == [0, 0]
    assert idx.batch_remove(np.arange(0, n, 2)) == n // 2 + 2
    lims, dist, ids = idx.range_search(q, np.inf)
    assert lims[-1] == 5 * (n // 2 + 1) and (ids % 2 == 1).all()    # (the second row of id 1 stays)
    # torch CUDA tensors in and out (the result copied into device pointers), equal to the host path
    tl, td, ti = idx.range_search(torch.from_numpy(q).cuda(), 4.0)
    assert tl.is_cuda and td.is_cuda and ti.is_cuda
    same_csr((tl.cpu().numpy(), td.cpu().numpy(), ti.cpu().numpy()), idx.range_search(q, 4.0))
    # range_query: one query as [(id, distance)], nearest first
    hits = idx.range_query(q[0], 4.0)
    lims, dist, ids = idx.range_search(q[:1], 4.0)
    assert hits == [(int(a), float(b)) for a, b in zip(ids, dist)]
    # nprobe > VIX_MAX_K
    ivf = IVFIndex(d, "euclidean", nlist=4, nprobe=2)
    ivf.set_coarse(xb[:4])
    ivf.batch_insert(xb)
    with pytest.raises(_lib.VectorIndexError) as e:
        ivf.range_search(q, 1.0, nprobe=513)
    assert e.value.status == ERR_INVALID_K
