"""The decode layout of the list-major tensor-core scan (vix_scan.cuh, vix_ivfpq_tc.cu): a second copy of an IVF-PQ index's
codes that only tc_scan_kernel's decoders read.

  - byte for byte what the stated mapping makes of the stored codes, for every m the path serves and lists of 1, 31, 32, 33
    and 4097 vectors (partial, full and several chunks), also after rows are added to an index that was already searched;
  - kept only by indexes the list-major path can serve;
  - code patterns that put every thread of a decoding warp on the same code or on a different one per slot: the list-major
    scan still returns the ids and distance bits of the query-major scan.
"""
import ctypes as C

import numpy as np
import pytest

from test_tc_scan_edges import Lists, both_paths, queries_near
from vectorindex_b200 import _lib

pytestmark = pytest.mark.gpu

SIZES = [1, 31, 32, 33, 4097]


def tc_codes(idx):
    """the index's decode layout (vix_debug_tc_codes), empty when it keeps none"""
    L = _lib.lib()
    n = C.c_int64(0)
    _lib.check(L.vix_debug_tc_codes(idx._h, C.c_void_p(0), C.c_int64(0), C.byref(n)))
    buf = np.zeros(n.value, np.uint8)
    if n.value:
        _lib.check(L.vix_debug_tc_codes(idx._h, _lib.ptr(buf), C.c_int64(buf.size), C.byref(n)))
        _lib.lib().vix_synchronize()
    return buf


def expected_tc_codes(off, codes, m):
    """the layout from the exported lists: list l starts at slot sum_{l' < l} roundup(len_l', 32) (padding slots hold code
    0); in the 512-byte block of chunk ch and group grp, thread t = 4 r + c owns bytes [16 t, 16 t + 16) and byte 4 v + s
    holds the code of slot r + 8 v, sub-quantiser 16 grp + 4 (s ^ (r & 3)) + c"""
    lens = np.diff(off)
    starts = np.concatenate([[0], np.cumsum((lens + 31) // 32 * 32)])
    slots = np.zeros((int(starts[-1]), m), np.uint8)
    for l, n in enumerate(lens):
        slots[starts[l]:starts[l] + n] = codes[off[l]:off[l + 1]]
    grp, t, v, s = np.meshgrid(np.arange(m // 16), np.arange(32), np.arange(4), np.arange(4), indexing="ij")
    r, c = t // 4, t % 4
    pos = (grp * 512 + 16 * t + 4 * v + s).ravel()
    slot = (r + 8 * v).ravel()
    sq = (16 * grp + 4 * (s ^ (r & 3)) + c).ravel()
    nch = slots.shape[0] // 32
    out = np.zeros((nch, 32 * m), np.uint8)
    out[:, pos] = slots.reshape(nch, 32, m)[:, slot, sq]
    return out.ravel()


def _lists(oracle, rng, m, sizes, codes=None):
    kc = len(sizes)
    coarse = (rng.standard_normal((kc, 2 * m)) * 2.0).astype(np.float32)
    cb = (rng.standard_normal((m, 256, 2)) * 0.5).astype(np.float32)
    assign = np.repeat(np.arange(kc, dtype=np.int32), sizes)
    if codes is None:
        codes = rng.integers(0, 256, (assign.size, m), dtype=np.uint8)
    ids = rng.permutation(assign.size).astype(np.int64) * 7 + 1
    return Lists(oracle, coarse, cb, assign, codes, ids, nprobe=2)


@pytest.mark.parametrize("m", [16, 32, 48, 64])
def test_decode_layout_equals_stored_codes(oracle, monkeypatch, capfd, m):
    """the layout of lists of 1, 31, 32, 33 and 4097 vectors; then a search through the list-major scan, rows added to
    every list (one list grows from 31 to 32, one from 32 to 33), and the layout and the search again"""
    rng = np.random.default_rng(m)
    L = _lists(oracle, rng, m, SIZES)
    got = tc_codes(L.idx)
    assert got.size == int(np.sum((np.array(SIZES) + 31) // 32 * 32)) * m
    assert np.array_equal(got, expected_tc_codes(L.off, L.codes, m))
    q = queries_near(rng, L, rng.integers(0, len(SIZES), 200))
    both_paths(monkeypatch, capfd, L.search(q, 10))
    add = np.array([3, 1, 1, 40, 5])
    assign = np.repeat(np.arange(len(SIZES), dtype=np.int32), add)
    L.add(assign, rng.integers(0, 256, (assign.size, m), dtype=np.uint8), 10 ** 6 + np.arange(assign.size))
    got = tc_codes(L.idx)
    assert got.size == int(np.sum((np.array(SIZES) + add + 31) // 32 * 32)) * m
    assert np.array_equal(got, expected_tc_codes(L.off, L.codes, m))
    both_paths(monkeypatch, capfd, L.search(q, 10))


@pytest.mark.parametrize("case", ["ip", "dsub4", "u4"])
def test_no_decode_layout_off_the_list_major_path(case):
    """inner product, four dimensions per sub-quantiser, 16 codes per sub-quantiser: the list-major scan never serves these
    indexes, and they keep no second copy of their codes"""
    from vectorindex_b200.index import IVFPQIndex
    rng = np.random.default_rng(5)
    m, kc, n = 16, 4, 300
    d = 4 * m if case == "dsub4" else 2 * m
    ks = 16 if case == "u4" else 256
    idx = IVFPQIndex(d, "ip" if case == "ip" else "euclidean", nlist=kc, nprobe=2, m=m, ks=ks)
    idx.set_coarse(rng.standard_normal((kc, d)).astype(np.float32))
    cb = rng.standard_normal((m, ks, d // m)).astype(np.float32)
    idx.set_codebooks(cb, (cb.astype(np.float64) ** 2).sum(-1).astype(np.float32))
    idx.batch_insert(rng.standard_normal((n, d)).astype(np.float32))
    assert tc_codes(idx).size == 0


@pytest.mark.parametrize("pattern", ["all_equal", "code_is_slot"])
@pytest.mark.parametrize("m", [16, 48, 64])
def test_adversarial_codes_equal_query_major_scan(oracle, monkeypatch, capfd, pattern, m):
    """all_equal: every stored code the same byte, so the 32 threads of a decoder warp look up one code and only the
    table slot (replica, sub-quantiser) tells them apart; code_is_slot: every code of a vector is its slot number within the
    list (mod 256), so each TMEM lane gets different rows.  Ids and distance bits equal those of the query-major scan, and
    every query whose seed list holds k vectors went through tc_scan_kernel.  (all_equal keeps the lists short: every vector
    of a list ties with the seed's k-th, so all of them are finalists.)"""
    rng = np.random.default_rng(100 + m)
    k = 10
    sizes, nq = ([1, 31, 32, 33, 97], 64) if pattern == "all_equal" else ([1, 31, 32, 33, 700, 4097], 256)
    n = int(np.sum(sizes))
    if pattern == "all_equal":
        codes = np.full((n, m), 173, np.uint8)
    else:
        codes = np.repeat(np.concatenate([np.arange(s) % 256 for s in sizes]).astype(np.uint8)[:, None], m, axis=1)
    L = _lists(oracle, rng, m, sizes, codes)
    assert np.array_equal(tc_codes(L.idx), expected_tc_codes(L.off, L.codes, m))
    q = queries_near(rng, L, rng.integers(0, len(sizes), nq))
    _, _, probes = L.idx.batch_search(q, k, nprobe=2, return_probes=True)
    _, _, r = both_paths(monkeypatch, capfd, L.search(q, k, probes))
    assert r[0] == L.handed_back(probes, k) < nq, "queries handed back beyond those with a short seed list"
    assert r[1] > 0, "no finalists"
