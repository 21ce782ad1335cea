"""Float64 reference of the IVF-PQ list scans (query-major vix_ivfpq_scan.cu, list-major vix_ivfpq_tc.cu), shared by their
edge suites.  It shares no code with either scan or the oracle: it decodes every probed vector, x^ = c_l + r^, and ranks
by (distance, id) in float64.

  metric 0 (L2): distance ||q - c_l - r^||^2
  metric 1 (IP): score <q, c_l + r^>, distance -score
  any dsub; ks = 256 (one byte per sub-quantiser) or ks = 16 (packed nibbles, the low nibble the even sub-quantiser)
"""
import collections

import numpy as np

RTOL = 1e-5


def unpack(codes, m, ks):
    """[n x m] code indices of stored codes ([n x m] bytes, or [n x m / 2] nibble pairs at ks = 16)"""
    codes = np.asarray(codes)
    if ks != 16:
        return codes.astype(np.intp)
    c = np.empty((codes.shape[0], m), np.intp)
    c[:, 0::2] = codes & 15
    c[:, 1::2] = codes >> 4
    return c


def decode(cb, codes):
    """r^ [n x d] of stored codes under codebooks cb [m x ks x dsub], in float64"""
    cb64 = np.asarray(cb, np.float64)
    m, ks = cb64.shape[:2]
    c = unpack(codes, m, ks)
    return cb64[np.arange(m), c].reshape(len(c), -1)


def ref64(q, coarse, cb, probes, off, codes, lids, k, metric=0):
    """float64 top-k over the vectors of the probed lists (-1, probes outside [0, kc) and empty lists skipped; a list probed
    twice contributes its vectors twice), by (distance, id).  Returns (dist [nq x k], ids [nq x k], per query (d64, ids,
    tol, order) of every probed vector).  tol is what the fp32 decomposition of the scans may be off by:
      L2: 1e-5 (||q - c||^2 + |t_x| + 2 ||q|| ||r^||),  t_x = ||r^||^2 + 2 <c, r^>
      IP: 1e-5 (sum |q_e c_e| + sum |q_e r^_e|)"""
    q64, c64 = np.asarray(q, np.float64), np.asarray(coarse, np.float64)
    kc = c64.shape[0]
    rhat = decode(cb, codes)
    lens = np.diff(off)
    nq = q64.shape[0]
    dist, ids, cand = np.full((nq, k), np.nan), np.full((nq, k), -1, np.int64), []
    for r in range(nq):
        ls = [int(l) for l in probes[r] if 0 <= l < kc and lens[l] > 0]
        rows = np.concatenate([np.arange(off[l], off[l + 1]) for l in ls]) if ls else np.zeros(0, np.intp)
        cl = c64[np.repeat(np.array(ls, np.intp), lens[ls])] if ls else np.zeros((0, c64.shape[1]))
        rr = rhat[rows]
        if metric == 1:
            d64 = -(cl @ q64[r] + rr @ q64[r])
            tol = RTOL * (np.abs(cl * q64[r]).sum(1) + np.abs(rr * q64[r]).sum(1))
        else:
            qc = q64[r] - cl
            d64 = ((qc - rr) ** 2).sum(1)
            tx = (rr * rr).sum(1) + 2.0 * (cl * rr).sum(1)
            tol = RTOL * ((qc * qc).sum(1) + np.abs(tx) + 2.0 * np.linalg.norm(q64[r]) * np.linalg.norm(rr, axis=1))
        idr = lids[rows]
        o = np.lexsort((idr, d64))[:k]
        dist[r, :o.size], ids[r, :o.size] = d64[o], idr[o]
        cand.append((d64, idr, tol, o))
    return dist, ids, cand


def assert_ref64(gd, gi, ref):
    """as many results as min(k, vectors probed), each distance within tol of the float64 value of its id, the id set that
    of the reference except for ties at the k-th distance within tol (ids stored twice counted twice)"""
    _, _, cand = ref
    k = gd.shape[1]
    for r, (d64, idr, tol, o) in enumerate(cand):
        nv = min(k, d64.size)
        assert (gi[r, :nv] >= 0).all() and (gi[r, nv:] == -1).all() and np.isnan(gd[r, nv:]).all(), \
            f"row {r}: {(gi[r] >= 0).sum()} results, {d64.size} vectors probed, k {k}"
        if nv == 0:
            continue
        assert (np.diff(gd[r, :nv]) >= 0).all(), f"row {r}: distances not ascending"
        kth, tk = d64[o[nv - 1]], tol[o[nv - 1]]
        for i, g in zip(gi[r, :nv].tolist(), gd[r, :nv].astype(np.float64).tolist()):
            sel = idr == i
            assert sel.any(), f"row {r}: id {i} is not in a probed list"
            assert (np.abs(d64[sel] - g) <= tol[sel]).any(), f"row {r} id {i}: {g} vs float64 {d64[sel].min()}"
            assert (d64[sel] - tol[sel] <= kth + tk).any(), f"row {r} id {i}: {g} beyond the k-th distance {kth}"
        got = collections.Counter(gi[r, :nv].tolist())
        for i, c in collections.Counter(idr[d64 + tol < kth - tk].tolist()).items():
            assert got[i] >= c, f"row {r}: id {i} (clearly inside the top {k}) missing"
