"""The list-major scan's seed (seed_scan_kernel in vix_ivfpq_tc.cu), on its own through vix_debug_tc_seed.

Per query the seed is the k-th smallest exact key of the first 256 stored vectors of the query's first probed list that
holds vectors, +inf when that sample holds fewer than k.  The filter of the list-major scan drops every vector above it, so
it must be an upper bound of the k-th best distance in the look-up-table scan's own arithmetic: here it is checked bit for
bit against the distances the query-major scan (vix_ivfpq_scan.cu) returns for the same vectors, at every m the list-major
scan takes and at k = 1, 10 and 64.
"""
import ctypes as C

import numpy as np
import pytest

from test_tc_scan_edges import Lists
from vectorindex_b200 import _lib

pytestmark = pytest.mark.gpu

SAMPLE = 256                                                        # vectors of the first list the seed looks at
LENS = [0, 7, 40, 64, 256, 300, 97, 0, 180, 257]                    # list lengths: empty, below / at / above k and SAMPLE


def seed(lists, q, probes, k):
    thr = np.empty(len(q), np.float32)
    q = np.ascontiguousarray(q, np.float32)
    probes = np.ascontiguousarray(probes, np.int32)
    _lib.check(_lib.lib().vix_debug_tc_seed(lists.idx._h, _lib.ptr(q, np.float32), C.c_int64(len(q)), C.c_int(k),
                                            _lib.ptr(probes, np.int32), C.c_int(probes.shape[1]), _lib.ptr(thr, np.float32)))
    _lib.lib().vix_synchronize()
    return thr


@pytest.mark.parametrize("m", [16, 32, 48, 64])
def test_seed_is_the_kth_exact_key_of_its_sample(oracle, monkeypatch, m):
    monkeypatch.setenv("VIX_TC_SCAN", "0")                          # the reference keys come from the query-major scan
    rng = np.random.default_rng(1000 + m)
    d, kc = 2 * m, len(LENS)
    coarse = rng.standard_normal((kc, d)).astype(np.float32)
    cb = (0.3 * rng.standard_normal((m, 256, 2))).astype(np.float32)
    assign = np.repeat(np.arange(kc), LENS).astype(np.int32)
    codes = rng.integers(0, 256, (len(assign), m), dtype=np.uint8)
    lists = Lists(oracle, coarse, cb, assign, codes, np.arange(len(assign)) * 3 + 11)

    nq, nprobe = 96, 4
    q = (coarse[rng.integers(0, kc, nq)] + 0.5 * rng.standard_normal((nq, d))).astype(np.float32)
    probes = np.stack([rng.permutation(kc)[:nprobe] for _ in range(nq)]).astype(np.int32)
    probes[::7, 0] = 0                                              # an empty list first: the seed takes the next one
    probes[::11, 0] = -1                                            # padding first
    probes[::13] = [0, 7, -1, 0]                                    # no list with vectors: +inf
    first = lists.first_list(probes)

    # every distance of every vector of the query's first list, from the query-major scan, keyed by id
    rows = np.where(first >= 0, first, 0)[:, None].astype(np.int32)
    full = int(lists.lens.max())
    dist, ids = lists.idx.search_with_probes(q, full, rows)
    for k in (1, 10, 64):
        thr = seed(lists, q, probes, k)
        for r in range(nq):
            l = first[r]
            if l < 0 or min(lists.lens[l], SAMPLE) < k:
                assert np.isposinf(thr[r]), (m, k, r)
                continue
            sample = set(lists.lids[lists.off[l]:lists.off[l] + SAMPLE].tolist())
            keep = np.array([i in sample for i in ids[r]])
            want = np.sort(dist[r][keep])[k - 1]
            assert thr[r].view(np.uint32) == want.view(np.uint32), (m, k, r, thr[r], want)
