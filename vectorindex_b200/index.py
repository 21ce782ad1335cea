"""Index API -- the host-side mirror of the reference's ``VectorIndexProtocol``
(/root/reference/Sources/VectorIndex/IndexProtocols.swift:50-103) for the three index kinds on the hot
path, over device-resident handles of ``libvindex_b200.so``:

  FlatIndex     FlatIndex / FlatIndexOptimized  (FlatIndex.swift, FlatIndexOptimized.swift:390-477)
  IVFIndex      IVF-Flat actor                  (IVFIndex.swift:279-451 optimize, :865-985 batchSearch)
  IVFPQIndex    the IVF-PQ composition the reference only writes down as a spec
                (docs/kernel-specs/DONE_22_adc_scan.md:831-881)

Semantics kept: ``k <= 0`` returns empty results (IVFIndex.swift:787,866); dimension mismatch raises
(:788-790); results ascend by API distance (L2: sqrt of L2^2 for Flat/IVF-Flat, ADC L2^2 for IVF-PQ as in
the composition; dot product: -dot, DistanceUtils.swift:40-46); an un-optimised IVF index answers by
linear scan (:820-832); ``nlist`` is clamped to the number of training vectors (:320); ties go to the
smaller id (TopK.swift:8-31).  Ids are integers in [0, 2^32 - 1) (the reference's TopK id type is Int32).
The metadata filter of the reference is a host closure and cannot run on the device; the only filter the
kernels honour is the list-disable bitmask of ivf_select_nprobe (IVFSelect.swift:366-395).

Multi-GPU: ``ShardedIVFPQIndex`` partitions the inverted lists over the ranks of a ``torch.distributed``
process group; queries are replicated, every rank scores its block of centroids and scans the probed lists
it owns, and probe lists / per-rank top-k lists are merged with an all-gather + the mergeTopK kernel.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import (INDEX_FLAT, INDEX_IVF_FLAT, INDEX_IVF_PQ, IndexParams, KMeansCfg, METRIC_IP, METRIC_L2, PQTrainCfg,
                   SearchStats, VectorIndexError, as_input, check, empty_like_input, lib, ptr)

_METRICS = {"euclidean": METRIC_L2, "l2": METRIC_L2, METRIC_L2: METRIC_L2,
            "dotProduct": METRIC_IP, "dot": METRIC_IP, "ip": METRIC_IP, METRIC_IP: METRIC_IP,
            "cosine": 2, 2: 2}                                       # cosine: FlatIndex and IVFIndex (not IVF-PQ)


def _metric(m):
    if m not in _METRICS:
        raise VectorIndexError(-5, f"unsupported metric {m!r}: the GPU hot path serves euclidean and dotProduct")
    return _METRICS[m]


class IDFilter:
    """IDFilterBitset + FilterMode of Operations/Filtering/IDFilter.swift:13-112: ceil(capacity / 64) 64-bit words over
    the dense id domain [0, capacity).  ``allow``: bit 1 = keep; ``deny``: bit 1 = drop; ids outside the domain never pass."""
    ALLOW, DENY = 0, 1

    def __init__(self, capacity: int, mode="allow", initial_bit=False):
        self.capacity = int(capacity)
        self.mode = {"allow": 0, "allowlist": 0, "deny": 1, "denylist": 1}[mode] if isinstance(mode, str) else int(mode)
        self.words = np.full((self.capacity + 63) >> 6, np.uint64(0xFFFFFFFFFFFFFFFF) if initial_bit else np.uint64(0),
                             dtype=np.uint64)

    def set(self, ids, value=True):
        ids = np.asarray(ids, dtype=np.int64).reshape(-1)
        ids = ids[(ids >= 0) & (ids < self.capacity)]
        bit = np.uint64(1) << (ids & 63).astype(np.uint64)
        if value:
            np.bitwise_or.at(self.words, ids >> 6, bit)
        else:
            np.bitwise_and.at(self.words, ids >> 6, ~bit)
        return self

    def test(self, ids):
        """idFilterPass for an array of ids"""
        ids = np.asarray(ids, dtype=np.int64)
        inside = (ids >= 0) & (ids < self.capacity)
        if self.words.size == 0:
            return np.zeros(ids.shape, dtype=bool)
        safe = np.where(inside, ids, 0)
        bit = ((self.words[safe >> 6] >> (safe & 63).astype(np.uint64)) & np.uint64(1)).astype(bool)
        return inside & (bit if self.mode == 0 else ~bit)


def compose_id_filters(allows=(), deny=None, capacity=None):
    """idFilterPassN (Operations/Filtering/IDFilter.swift:140-176): keep = allow0 AND allow1 AND ... AND NOT deny, ids
    outside [0, capacity) never pass -- folded on the host into ONE allowlist bitset, which is what the device takes.
    ``allows``: up to four allowlist IDFilters (the reference's limit), ``deny``: one denylist IDFilter; all over the same
    capacity (or pass ``capacity``).  With no allowlist every in-range id starts allowed."""
    allows = [a for a in allows if a is not None]
    if len(allows) > 4:
        raise ValueError("up to 4 allowlists + 1 denylist (IDFilter.swift:219)")
    parts = allows + ([deny] if deny is not None else [])
    if capacity is None:
        if not parts:
            raise ValueError("capacity is needed when no filter is given")
        capacity = parts[0].capacity
    if any(f.capacity != capacity for f in parts):
        raise ValueError("composed filters must cover the same id domain")
    if any(a.mode != IDFilter.ALLOW for a in allows) or (deny is not None and deny.mode != IDFilter.DENY):
        raise ValueError("allows must be allowlists and deny a denylist")
    out = IDFilter(capacity, "allow", initial_bit=True)
    for a in allows:
        out.words &= a.words
    if deny is not None:
        out.words &= ~deny.words
    if capacity & 63 and out.words.size:                             # bits past the domain stay clear
        out.words[-1] &= np.uint64((1 << (capacity & 63)) - 1)
    return out


class _Index:
    kind = INDEX_FLAT

    def __init__(self, dimension: int, metric="euclidean", nlist: int = 256, nprobe: int = 8, m: int = 16,
                 ks: int = 256):
        p = IndexParams()
        lib().vix_index_params_default(C.byref(p))
        p.kind, p.d, p.metric = self.kind, int(dimension), _metric(metric)
        p.nlist, p.nprobe, p.m, p.ks = int(nlist), int(nprobe), int(m), int(ks)
        self.params = p
        self.dimension = int(dimension)
        self.metric = p.metric
        self._h = C.c_void_p(0)
        check(lib().vix_index_create(C.byref(p), C.byref(self._h)))

    def __del__(self):
        try:
            if getattr(self, "_h", None) is not None and self._h:
                lib().vix_index_destroy(self._h)
                self._h = C.c_void_p(0)
        except Exception:
            pass

    close = __del__

    # ---- VectorIndexProtocol ----
    @property
    def count(self) -> int:
        return int(lib().vix_index_count(self._h))

    def _check_dim(self, a, what):
        if a.ndim != 2 or int(a.shape[1]) != self.dimension:
            raise VectorIndexError(-1, f"{what}: expected [n x {self.dimension}], got {tuple(a.shape)}")

    def batch_insert(self, vectors, ids=None):
        x = as_input(vectors, np.float32)
        self._check_dim(x, "batch_insert")
        idp = as_input(ids, np.int64)
        check(lib().vix_index_add(self._h, ptr(x, np.float32), ptr(idp), C.c_int64(int(x.shape[0]))))

    def insert(self, id_: int, vector):
        v = np.ascontiguousarray(vector, dtype=np.float32).reshape(1, -1)
        self.batch_insert(v, np.array([id_], dtype=np.int64))

    add = batch_insert

    def batch_remove(self, ids) -> int:
        """Removes every stored row whose id is in ``ids`` (numpy or torch, host or device; duplicates and ids that are not
        stored are allowed; a row stored twice is removed twice).  Returns the number of rows removed.  The index then
        answers exactly as one built from the remaining rows in their order."""
        i = as_input(ids, np.int64).reshape(-1)
        removed = C.c_int64(0)
        check(lib().vix_index_remove(self._h, ptr(i, np.int64), C.c_int64(int(i.shape[0])), C.byref(removed)))
        return int(removed.value)

    def remove(self, id_: int) -> int:
        return self.batch_remove(np.array([id_], dtype=np.int64))

    def clear(self):
        check(lib().vix_index_clear(self._h))

    def batch_search(self, queries, k: int, nprobe: int = 0, return_probes=False, stats=False, filter=None, out=None):
        """``filter``: an :class:`IDFilter` (allow / deny bitset over dense ids, applied before selection -- the
        device-expressible form of the reference's ``filter:`` closures, IVFIndex.swift:813, 1034).
        ``out``: optional (distances f32 [nq x k], ids int64 [nq x k]) buffers to write into (e.g. pinned host arrays)."""
        q = as_input(queries, np.float32)
        self._check_dim(q, "batch_search")
        nq = int(q.shape[0])
        kk = max(int(k), 0)
        if out is not None:
            dist, ids = out
            if tuple(dist.shape) != (nq, kk) or tuple(ids.shape) != (nq, kk):
                raise ValueError("out buffers must be [nq x k]")
        else:
            dist = empty_like_input(q, (nq, kk), np.float32)
            ids = empty_like_input(q, (nq, kk), np.int64)
        if kk == 0 or nq == 0:
            return (dist, ids)
        if filter is not None:
            if return_probes or stats:
                raise ValueError("filtered search returns (distances, ids) only")
            check(lib().vix_index_search_filtered(self._h, ptr(q, np.float32), C.c_int64(nq), C.c_int(k), C.c_int(nprobe),
                                                  ptr(filter.words, np.uint64), C.c_int64(filter.capacity),
                                                  C.c_int(filter.mode), ptr(dist, np.float32), ptr(ids, np.int64)))
            return (dist, ids)
        npb = nprobe if nprobe > 0 else self.params.nprobe
        probes = empty_like_input(q, (nq, npb), np.int32) if return_probes else None
        st = SearchStats() if stats else None
        check(lib().vix_index_search_ex(self._h, ptr(q, np.float32), C.c_int64(nq), C.c_int(k), C.c_int(nprobe),
                                        ptr(dist, np.float32), ptr(ids, np.int64), ptr(probes),
                                        C.byref(st) if st is not None else None))
        out = (dist, ids)
        if return_probes:
            out += (probes,)
        if stats:
            out += (st,)
        return out

    def search(self, query, k: int, nprobe: int = 0):
        q = np.ascontiguousarray(query, dtype=np.float32).reshape(1, -1)
        d, i = self.batch_search(q, k, nprobe)
        valid = i[0] >= 0
        return [(int(a), float(b)) for a, b in zip(i[0][valid], d[0][valid])]

    def range_search(self, queries, radius: float, nprobe: int = 0, filter=None):
        """Every stored vector whose distance to a query is at most ``radius`` (the distance k-NN search returns: L2
        sqrt(L2^2), or the ADC squared distance on an IVF-PQ index; IP -dot; cosine 1 - similarity), per query sorted by
        (distance, id).  Candidates, ``nprobe`` and ``filter`` (an :class:`IDFilter`) are those of :meth:`batch_search`.
        Returns CSR ``(lims int64 [nq + 1], distances f32 [total], ids int64 [total])``: row r is
        ``[lims[r], lims[r + 1])``; numpy for host queries, torch tensors on the queries' device for CUDA tensors."""
        q = as_input(queries, np.float32)
        self._check_dim(q, "range_search")
        nq = int(q.shape[0])
        res = C.c_void_p(0)
        try:
            words = filter.words if filter is not None else None
            check(lib().vix_index_range_search(self._h, ptr(q, np.float32), C.c_int64(nq), C.c_float(float(radius)),
                                               C.c_int(nprobe), ptr(words, np.uint64),
                                               C.c_int64(filter.capacity if filter is not None else 0),
                                               C.c_int(filter.mode if filter is not None else 0), C.byref(res)))
            total = int(lib().vix_range_result_total(res))
            lims = empty_like_input(q, (nq + 1,), np.int64)
            dist = empty_like_input(q, (total,), np.float32)
            ids = empty_like_input(q, (total,), np.int64)
            check(lib().vix_range_result_get(res, ptr(lims, np.int64), ptr(dist, np.float32) if total else None,
                                             ptr(ids, np.int64) if total else None))
            return lims, dist, ids
        finally:
            lib().vix_range_result_destroy(res)

    def range_query(self, query, radius: float, nprobe: int = 0):
        """:meth:`range_search` for one query: ``[(id, distance), ...]`` nearest first."""
        q = np.ascontiguousarray(query, dtype=np.float32).reshape(1, -1)
        _, d, i = self.range_search(q, radius, nprobe)
        return [(int(a), float(b)) for a, b in zip(i, d)]


class FlatIndex(_Index):
    kind = INDEX_FLAT

    def optimize(self):
        return None


class IVFIndex(_Index):
    """IVF-Flat.  ``optimize(training_vectors)`` trains the coarse quantiser (k-means).  Like the reference actor
    (insert -> optimize() -> search, IVFIndex.swift:279-451) the IVF-Flat kind also takes vectors BEFORE it is trained:
    searches are linear scans until then (:820-832) and ``optimize()`` without arguments trains on the stored vectors
    and files them into their lists.  The IVF-PQ kind keeps codes, not vectors: it is trained first (faiss-style)."""
    kind = INDEX_IVF_FLAT

    def optimize(self, training_vectors=None, kmeans_cfg: KMeansCfg | None = None, pq_cfg: PQTrainCfg | None = None):
        if kmeans_cfg is None:
            kmeans_cfg = KMeansCfg(1024, 10, 1e-4, 42, 0, False, 1)
        if pq_cfg is None:
            pq_cfg = PQTrainCfg(0, 25, 1e-4, 1024, 0, 42, 0, 0, 1)
        if training_vectors is None:                                  # the stored vectors (IVF-Flat only)
            check(lib().vix_index_train(self._h, None, C.c_int64(0), C.byref(kmeans_cfg), C.byref(pq_cfg)))
            return
        x = as_input(training_vectors, np.float32)
        self._check_dim(x, "optimize")
        check(lib().vix_index_train(self._h, ptr(x, np.float32), C.c_int64(int(x.shape[0])), C.byref(kmeans_cfg),
                                    C.byref(pq_cfg)))

    train = optimize

    def set_coarse(self, centroids):
        c = as_input(centroids, np.float32)
        self._check_dim(c, "set_coarse")
        check(lib().vix_index_set_coarse(self._h, ptr(c, np.float32), C.c_int(int(c.shape[0]))))

    def get_coarse(self):
        kc = C.c_int(0)
        check(lib().vix_index_get_coarse(self._h, None, C.byref(kc)))
        out = np.empty((kc.value, self.dimension), dtype=np.float32)
        check(lib().vix_index_get_coarse(self._h, ptr(out), C.byref(kc)))
        return out

    def list_sizes(self):
        kc = C.c_int(0)
        check(lib().vix_index_get_coarse(self._h, None, C.byref(kc)))
        out = np.empty(kc.value, dtype=np.int64)
        check(lib().vix_index_list_sizes(self._h, ptr(out)))
        return out


class IVFPQIndex(IVFIndex):
    kind = INDEX_IVF_PQ

    @property
    def code_bytes(self) -> int:
        """bytes of one stored code: m (ks = 256), m / 2 (ks = 16: two codes per byte, ADCScan.swift:384-456)"""
        return self.params.m // 2 if self.params.ks == 16 else self.params.m

    def set_codebooks(self, codebooks, centroid_norms=None):
        cb = as_input(codebooks, np.float32)
        cn = as_input(centroid_norms, np.float32)
        check(lib().vix_index_set_codebooks(self._h, ptr(cb, np.float32), ptr(cn)))

    def get_codebooks(self):
        m, ks, dsub = self.params.m, self.params.ks, self.dimension // self.params.m
        cb = np.empty((m, ks, dsub), dtype=np.float32)
        cn = np.empty((m, ks), dtype=np.float32)
        check(lib().vix_index_get_codebooks(self._h, ptr(cb), ptr(cn)))
        return cb, cn

    # ---- pieces of the sharded pipeline (ShardedIVFPQIndex)
    def probe_range(self, queries, nprobe, list_begin, list_count):
        """local top-nprobe over the centroid block [list_begin, list_begin + list_count): (global list ids, scores)"""
        q = as_input(queries, np.float32)
        self._check_dim(q, "probe_range")
        nq = int(q.shape[0])
        ids = empty_like_input(q, (nq, nprobe), np.int32)
        sc = empty_like_input(q, (nq, nprobe), np.float32)
        check(lib().vix_index_probe_range(self._h, ptr(q, np.float32), C.c_int64(nq), C.c_int(nprobe), C.c_int(list_begin),
                                          C.c_int(list_count), ptr(ids, np.int32), ptr(sc, np.float32)))
        return ids, sc

    def batch_search_rerank(self, queries, k: int, vectors, rerank_r: int, nprobe: int = 0, sq_norms=None):
        """The IVF-PQ query with the spec's optional step 7 (DONE_22_adc_scan.md:873-878): ADC top-``rerank_r`` candidates,
        then Kernel #40 exact re-rank against the original ``vectors`` (row = id).  Returns (raw exact scores, ids)."""
        q = as_input(queries, np.float32)
        self._check_dim(q, "batch_search_rerank")
        xb = as_input(vectors, np.float32)
        nq, kk = int(q.shape[0]), max(int(k), 0)
        sc = empty_like_input(q, (nq, kk), np.float32)
        ids = empty_like_input(q, (nq, kk), np.int64)
        if nq == 0 or kk == 0:
            return sc, ids
        nr = as_input(sq_norms, np.float32)
        check(lib().vix_index_search_rerank(self._h, ptr(q, np.float32), C.c_int64(nq), C.c_int(k), C.c_int(nprobe),
                                            C.c_int(int(rerank_r)), ptr(xb, np.float32), C.c_int64(int(xb.shape[0])), ptr(nr),
                                            ptr(sc, np.float32), ptr(ids, np.int64)))
        return sc, ids

    def search_with_probes(self, queries, k, probes, stats=False):
        q = as_input(queries, np.float32)
        self._check_dim(q, "search_with_probes")
        pr = as_input(probes, np.int32)
        nq, nprobe = int(q.shape[0]), int(pr.shape[1])
        dist = empty_like_input(q, (nq, k), np.float32)
        ids = empty_like_input(q, (nq, k), np.int64)
        if stats:
            st = _lib.SearchStats()
            check(lib().vix_index_search_with_probes_ex(self._h, ptr(q, np.float32), C.c_int64(nq), C.c_int(k),
                                                        ptr(pr, np.int32), C.c_int(nprobe), ptr(dist, np.float32),
                                                        ptr(ids, np.int64), C.byref(st)))
            return dist, ids, st
        check(lib().vix_index_search_with_probes(self._h, ptr(q, np.float32), C.c_int64(nq), C.c_int(k), ptr(pr, np.int32),
                                                 C.c_int(nprobe), ptr(dist, np.float32), ptr(ids, np.int64)))
        return dist, ids

    def encode(self, vectors):
        """(list assignment, PQ codes) of a batch without storing it (bit-exact, same kernels as batch_insert)"""
        x = as_input(vectors, np.float32)
        self._check_dim(x, "encode")
        n = int(x.shape[0])
        asg = empty_like_input(x, (n,), np.int32)
        codes = empty_like_input(x, (n, self.code_bytes), np.uint8)
        if n == 0:
            return asg, codes
        check(lib().vix_index_encode(self._h, ptr(x, np.float32), C.c_int64(n), ptr(asg, np.int32), ptr(codes, np.uint8)))
        return asg, codes

    def add_encoded(self, assign, codes, ids):
        a, c, i = as_input(assign, np.int32), as_input(codes, np.uint8), as_input(ids, np.int64)
        if int(a.shape[0]) == 0:
            return
        check(lib().vix_index_add_encoded(self._h, ptr(a, np.int32), ptr(c, np.uint8), ptr(i, np.int64),
                                          C.c_int64(int(a.shape[0]))))

    def import_lists(self, list_offsets, codes, ids):
        lo = np.ascontiguousarray(list_offsets, dtype=np.int64)
        codes = as_input(codes, np.uint8)
        ids = as_input(ids, np.int64)
        check(lib().vix_index_import_lists(self._h, ptr(lo), ptr(codes, np.uint8), ptr(ids, np.int64)))

    def export_lists(self):
        """CSR lists in the reference's AoS list format (Kernels/IVFAppend.swift:220-236) + assignments."""
        n = self.count
        kc = C.c_int(0)
        check(lib().vix_index_get_coarse(self._h, None, C.byref(kc)))
        off = np.empty(kc.value + 1, dtype=np.int64)
        codes = np.empty((n, self.code_bytes), dtype=np.uint8)
        ids = np.empty(n, dtype=np.int64)
        asg = np.empty(n, dtype=np.int32)
        check(lib().vix_index_export_lists(self._h, ptr(off), ptr(codes), ptr(ids), ptr(asg)))
        return off, codes, ids, asg


# ------------------------------------------------------------------------------------------------
# multi-GPU
# ------------------------------------------------------------------------------------------------
def list_block(kc: int, rank: int, world: int, bounds=None):
    """Contiguous block of inverted lists owned by ``rank``: (first list, number of lists).  Lists are disjoint
    (IVFIndex.swift:370-375), so they shard without any data-path dependency between ranks.  ``bounds`` ([world + 1]
    ascending list ids, see :func:`balanced_list_bounds`) replaces the default equal-count blocks."""
    if bounds is not None:
        return int(bounds[rank]), int(bounds[rank + 1]) - int(bounds[rank])
    per = (kc + world - 1) // world
    b = min(kc, rank * per)
    return b, min(kc, b + per) - b


def list_owner(assign, kc: int, world: int, bounds=None):
    """Rank owning each list id in ``assign`` (numpy or torch)."""
    if bounds is not None:
        if _lib._is_torch(assign):
            import torch
            inner = torch.as_tensor(np.asarray(bounds[1:-1], dtype=np.int64), device=assign.device)
            return torch.bucketize(assign, inner, right=True)
        return np.searchsorted(np.asarray(bounds[1:-1], dtype=np.int64), assign, side="right")
    per = (kc + world - 1) // world
    return assign // per


def balanced_list_bounds(list_sizes, world: int):
    """Block boundaries [world + 1] that equalise the expected scan work of the ranks.  A list of length L is probed in
    proportion to the share of queries that fall near it -- for queries drawn like the data, in proportion to L -- and
    costs L when it is, so its expected work is ~ L^2: boundaries are cut where the prefix sum of L^2 crosses
    multiples of total / world.  ``list_sizes`` may come from a sample (only ratios matter)."""
    w = np.asarray(list_sizes, dtype=np.float64) ** 2 + 1e-9
    cum = np.concatenate([[0.0], np.cumsum(w)])
    targets = cum[-1] * np.arange(1, world) / world
    inner = np.searchsorted(cum, targets, side="left")
    b = np.concatenate([[0], inner, [w.size]]).astype(np.int64)
    return np.maximum.accumulate(b)


def merge_shard_results(dist_all, ids_all, k, metric=METRIC_L2):
    """mergeTopK over per-rank results.  dist_all/ids_all: [world x nq x k] (numpy or torch).  API distances and
    probe scores both ascend ("smaller is better"), so the merge order is always .min with ties -> smaller id
    (TopKMerge.swift:66-71)."""
    from .kernels import mergeTopK
    if _lib._is_torch(dist_all):
        sc = dist_all.permute(1, 0, 2).contiguous()
        idm = ids_all.permute(1, 0, 2).contiguous()
    else:
        sc = np.ascontiguousarray(np.transpose(dist_all, (1, 0, 2)))
        idm = np.ascontiguousarray(np.transpose(ids_all, (1, 0, 2)))
    return mergeTopK(sc, idm, k, 0)


def merge_shard_results_host(dist_all, ids_all, k):
    """Host restatement of the shard merge (CPU-only ranks, gloo tests): k smallest of the union by
    (distance, id); NaN / id -1 entries are padding."""
    world, nq, kk = dist_all.shape
    d = np.transpose(dist_all, (1, 0, 2)).reshape(nq, world * kk)
    i = np.transpose(ids_all, (1, 0, 2)).reshape(nq, world * kk)
    out_d = np.full((nq, k), np.nan, dtype=np.float32)
    out_i = np.full((nq, k), -1, dtype=np.int64)
    for r in range(nq):
        valid = i[r] >= 0
        dv, iv = d[r][valid], i[r][valid]
        order = np.lexsort((iv, dv))[:k]
        out_d[r, :order.size] = dv[order]
        out_i[r, :order.size] = iv[order]
    return out_d, out_i


class Comm:
    """``vix_comm_t``: the library's own communicator of one process per GPU (NCCL, bound at run time, + peer-mapped
    exchange memory).  The 128-byte id of rank 0 reaches the other ranks by the host's own means -- here a
    ``torch.distributed`` broadcast, in a Swift host whatever it already uses to start its workers."""

    def __init__(self, rank: int, world: int, unique_id: bytes):
        self._c = C.c_void_p(0)
        buf = (C.c_char * len(unique_id)).from_buffer_copy(unique_id)
        check(lib().vix_comm_create(buf, C.c_size_t(len(unique_id)), C.c_int(rank), C.c_int(world), C.byref(self._c)))
        self.rank, self.world = int(rank), int(world)

    @staticmethod
    def unique_id() -> bytes:
        buf = (C.c_char * 128)()
        check(lib().vix_comm_unique_id(buf, C.c_size_t(128)))
        return bytes(buf)

    @classmethod
    def from_torch(cls, group=None):
        """One communicator per process of an initialised ``torch.distributed`` NCCL group (the id travels by broadcast)."""
        import torch
        import torch.distributed as dist
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        dev = torch.device("cuda", torch.cuda.current_device())
        idt = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(cls.unique_id()), dtype=torch.uint8))
        dist.broadcast(idt, 0, group=group)
        torch.cuda.synchronize()
        return cls(rank, world, bytes(idt.cpu().numpy().tobytes()))

    @property
    def uses_peer_memory(self) -> int:
        return int(lib().vix_comm_uses_peer_memory(self._c))

    def close(self):
        if getattr(self, "_c", None) is not None and self._c:
            lib().vix_comm_destroy(self._c)
            self._c = C.c_void_p(0)

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass


class ShardedIVFPQIndex:
    """IVF-PQ index partitioned over the ranks of a ``torch.distributed`` group by contiguous blocks of
    inverted lists (SURVEY.md 8e).  Every rank holds the coarse centroids and PQ codebooks and the codes of
    ITS lists only.

    build   any rank assigns + encodes whatever rows it is handed (``add``); rows travel to the rank that
            owns their list with one all-to-all and are appended there already encoded;
    search  each rank selects the probes of ITS block of queries against all centroids (the single-GPU code path:
            IVFIndex.swift:593-595 order by construction) -> all-gather of list ids = the global probe lists of
            the whole batch on every rank -> each rank scans the probed lists it owns -> all-gather + mergeTopK of
            the per-rank [nq x k] results (TopKMerge.swift:11-61).  (probe_range over a centroid BLOCK + merge of
            per-block candidates remains available for hosts that shard the centroids instead.)

    ``local`` may be any object with probe_range / search_with_probes / encode / add_encoded / set_coarse /
    set_codebooks (the gloo tests plug in an oracle-backed one, the product path an ``IVFPQIndex``)."""

    def __init__(self, dimension, metric="euclidean", nlist=256, nprobe=8, m=16, ks=256, group=None, local=None):
        import torch.distributed as dist
        self.group = group
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.local = local if local is not None else IVFPQIndex(dimension, metric, nlist, nprobe, m, ks)
        self.nprobe = int(nprobe)
        self.kc = int(nlist)
        self.bounds = None

    @classmethod
    def wrap(cls, local_index, kc, nprobe, group=None):
        """Sharded view over an already built per-rank index."""
        self = cls.__new__(cls)
        import torch.distributed as dist
        self.group = group
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.local, self.kc, self.nprobe = local_index, int(kc), int(nprobe)
        self.bounds = None
        return self

    def set_list_bounds(self, bounds):
        """Block boundaries of the list partition ([world + 1], identical on every rank; before the first ``add``).
        Default: equal-count blocks."""
        b = np.asarray(bounds, dtype=np.int64)
        if b.size != self.world + 1 or b[0] != 0 or b[-1] != self.kc or (np.diff(b) < 0).any():
            raise ValueError("bounds must be [world + 1] ascending list ids from 0 to nlist")
        self.bounds = b

    # ---- parameters
    def set_parameters(self, coarse, codebooks, centroid_norms=None):
        self.kc = int(coarse.shape[0])
        self.local.set_coarse(coarse)
        self.local.set_codebooks(codebooks, centroid_norms)

    def _nccl(self):
        import torch.distributed as dist
        return dist.get_backend(self.group) == "nccl"

    def _native(self):
        """The product path: the whole sharded step inside the library (vix_sharded_search / vix_sharded_add over a
        ``vix_comm_t``).  The Python exchange below remains for CPU ranks (gloo tests with an oracle-backed local index)."""
        if self.world <= 1 or not self._nccl() or not hasattr(self.local, "_h"):
            return None
        if self.__dict__.get("comm") is None:
            self.comm = Comm.from_torch(self.group)
        return self.comm

    def _pinned(self, tag, shape, dtype):
        import torch
        pins = self.__dict__.setdefault("_pins", {})
        key = (tag, dtype, tuple(shape))
        buf = pins.get(key)
        if buf is None:
            if len(pins) > 8:
                pins.clear()
            buf = pins[key] = torch.empty(shape, dtype=dtype, pin_memory=True)
        return buf

    def _to_comm(self, a):
        """array -> tensor on the device the process group communicates over"""
        import torch
        if not _lib._is_torch(a):
            a = torch.from_numpy(np.ascontiguousarray(a))
        if self._nccl() and not a.is_cuda:
            # stream-ordered copy: with a pinned source the host does not wait for it (everything that reads the tensor is
            # enqueued behind it on the same stream); pageable sources are staged by torch and stay safe
            a = a.to(torch.device("cuda", torch.cuda.current_device()), non_blocking=a.is_pinned())
        return a.contiguous()

    def _to_host(self, t):
        """device tensor -> numpy array through a pinned staging buffer kept with the index (one D2H at full PCIe rate,
        one wait), copied out so that the caller owns the result"""
        import torch
        pins = self.__dict__.setdefault("_pins", {})
        key = (t.dtype, tuple(t.shape))
        buf = pins.get(key)
        if buf is None:
            if len(pins) > 8:
                pins.clear()
            buf = pins[key] = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
        buf.copy_(t, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return buf.numpy().copy()

    def _comm_device(self):
        import torch
        return torch.device("cuda", torch.cuda.current_device()) if self._nccl() else torch.device("cpu")

    def _all_gather(self, t):
        import torch
        import torch.distributed as dist
        out = torch.empty((self.world * t.shape[0],) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
        dist.all_gather_into_tensor(out, t, group=self.group)                  # concatenated along dim 0
        return out.view((self.world,) + tuple(t.shape))

    # ---- build
    def add(self, vectors, ids):
        """Rows handed to THIS rank (any rows; ranks normally pass disjoint slices of the database)."""
        import torch
        import torch.distributed as dist
        comm = self._native()
        if comm is not None:
            x = as_input(vectors, np.float32)
            i = as_input(ids, np.int64)
            b = None if self.bounds is None else np.ascontiguousarray(self.bounds, dtype=np.int64)
            check(lib().vix_sharded_add(self.local._h, comm._c, ptr(b), ptr(x, np.float32), ptr(i, np.int64),
                                        C.c_int64(int(x.shape[0]))))
            return
        assign, codes = self.local.encode(vectors)
        if self.world == 1:
            self.local.add_encoded(assign, codes, ids)
            return
        assign, codes, ids = self._to_comm(assign), self._to_comm(codes), self._to_comm(ids)
        owner = list_owner(assign.to(torch.int64), self.kc, self.world, self.bounds)
        order = torch.argsort(owner, stable=True)
        send_cnt = torch.bincount(owner, minlength=self.world).to(torch.int64)
        recv_cnt = torch.empty_like(send_cnt)
        dist.all_to_all_single(recv_cnt, send_cnt, group=self.group)
        ssz, rsz = send_cnt.tolist(), recv_cnt.tolist()
        nrecv = int(sum(rsz))

        def exchange(t):
            t = t[order].contiguous()
            out = torch.empty((nrecv,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
            dist.all_to_all_single(out, t, output_split_sizes=rsz, input_split_sizes=ssz, group=self.group)
            return out

        r_assign, r_codes, r_ids = exchange(assign), exchange(codes), exchange(ids)
        if nrecv:
            if not self._nccl():
                r_assign, r_codes, r_ids = r_assign.numpy(), r_codes.numpy(), r_ids.numpy()
            self.local.add_encoded(r_assign, r_codes, r_ids)

    def remove(self, ids) -> int:
        """Collective: every rank passes the SAME ids (as for ``batch_search``) and removes the rows of them it holds;
        returns the number of rows removed on all ranks together."""
        n = self.local.batch_remove(ids)
        if self.world == 1:
            return n
        import torch
        import torch.distributed as dist
        t = torch.tensor([n], dtype=torch.int64, device=self._comm_device())
        dist.all_reduce(t, group=self.group)
        return int(t.item())

    # ---- search
    def query_block(self, nq: int):
        """Rows of the batch whose probe lists THIS rank computes: (first row, rows, rows per rank)."""
        per = (nq + self.world - 1) // self.world
        lo = min(nq, self.rank * per)
        return lo, min(nq, lo + per) - lo, per

    def global_probes(self, queries, nprobe=0):
        """The global probe lists [nq x nprobe] (int32), identical on every rank.  Probe selection is partitioned by
        QUERY: every rank holds all coarse centroids (25 MB at nlist = 65536), selects the probes of its 1/world of
        the batch against all of them -- the very code path of a single GPU, so the lists are identical to it by
        construction -- and one all-gather of int32 list ids (nq x nprobe x 4 bytes in total) hands every rank the
        lists of the whole batch.  No merge step, a sixteenth of the bytes of exchanging per-block candidates."""
        import torch
        nprobe = nprobe if nprobe > 0 else self.nprobe
        nq = int(queries.shape[0])
        if self.world == 1:
            return self.local.probe_range(queries, nprobe, 0, self.kc)[0]
        if nq == 0:                                                            # nothing to exchange (every rank sees nq)
            return torch.empty((0, nprobe), dtype=torch.int32, device=self._comm_device())
        lo, cnt, per = self.query_block(nq)
        if cnt > 0:
            ids = self._to_comm(self.local.probe_range(queries[lo:lo + cnt], nprobe, 0, self.kc)[0]).to(torch.int32)
        if cnt == per:
            buf = ids
        else:
            buf = torch.full((per, nprobe), -1, dtype=torch.int32, device=self._comm_device())
            if cnt > 0:
                buf[:cnt] = ids
        return self._all_gather(buf).view(self.world * per, nprobe)[:nq].contiguous()

    def batch_search(self, queries, k, nprobe=0, out=None, filter=None):
        """Replicated queries in, merged [nq x k] (distances, ids) out on every rank.  Host (numpy) queries are
        staged to the device once and only the merged result returns to the host.  ``out``: optional (distances f32,
        ids int64) host arrays the result is written into (pinned ones make the copy back asynchronous).  ``filter``: an
        :class:`IDFilter` (the same on every rank), applied before selection as in ``IVFPQIndex.batch_search``.  ``k`` goes
        up to ``VIX_MAX_K_LARGE`` (16384) through the library's exchange, as on one GPU: above 512 each rank runs the
        exact two-pass route with one bound per query shared by all ranks, the rows cut at k are exchanged and merged on
        the device, and the call synchronises.  (The Python exchange path of CPU / gloo ranks is not covered by this.)"""
        import torch
        if filter is not None:
            return self._filtered_search(queries, k, nprobe, filter, out)
        was_numpy = not _lib._is_torch(queries)
        if int(queries.shape[0]) == 0 or int(k) <= 0:                          # IVFIndex.swift:866: nothing to do
            kk = max(int(k), 0)
            if was_numpy:
                return np.empty((0 if int(queries.shape[0]) == 0 else int(queries.shape[0]), kk), np.float32), \
                    np.empty((int(queries.shape[0]), kk), np.int64)
            return (torch.empty((int(queries.shape[0]), kk), dtype=torch.float32, device=queries.device),
                    torch.empty((int(queries.shape[0]), kk), dtype=torch.int64, device=queries.device))
        nprobe = nprobe if nprobe > 0 else self.nprobe
        comm = self._native()
        if comm is not None:
            # one library call: probe selection of this rank's block, both exchanges over peer memory, fused scan, merge.
            # Host queries: the library moves only this rank's block across PCIe; results land in pinned memory.
            q = as_input(queries, np.float32)
            nq = int(q.shape[0])
            if was_numpy:
                if out is not None:
                    od, oi = out
                    check(lib().vix_sharded_search(self.local._h, comm._c, ptr(q, np.float32), C.c_int64(nq), C.c_int(k),
                                                   C.c_int(nprobe), ptr(od, np.float32), ptr(oi, np.int64)))
                    return od, oi
                pd, pi = self._pinned("d", (nq, k), torch.float32), self._pinned("i", (nq, k), torch.int64)
                check(lib().vix_sharded_search(self.local._h, comm._c, ptr(q, np.float32), C.c_int64(nq), C.c_int(k),
                                               C.c_int(nprobe), C.c_void_p(pd.data_ptr()), C.c_void_p(pi.data_ptr())))
                return pd.numpy().copy(), pi.numpy().copy()
            md = torch.empty((nq, k), dtype=torch.float32, device=q.device)
            mi = torch.empty((nq, k), dtype=torch.int64, device=q.device)
            check(lib().vix_sharded_search(self.local._h, comm._c, ptr(q, np.float32), C.c_int64(nq), C.c_int(k),
                                           C.c_int(nprobe), ptr(md, np.float32), ptr(mi, np.int64)))
            return md, mi
        if self.world > 1 and was_numpy and self._nccl():
            queries = self._to_comm(np.ascontiguousarray(queries, dtype=np.float32))
        probes = self.global_probes(queries, nprobe)
        if not self._nccl() and _lib._is_torch(probes):
            probes = probes.numpy()
        d_loc, i_loc = self.local.search_with_probes(queries, k, probes)
        if self.world == 1:
            return d_loc, i_loc
        d_all, i_all = self._all_gather(self._to_comm(d_loc)), self._all_gather(self._to_comm(i_loc))
        if d_all.is_cuda:
            md, mi = merge_shard_results(d_all, i_all, k)
        else:
            md, mi = merge_shard_results_host(d_all.numpy(), i_all.numpy(), k)
        if was_numpy and _lib._is_torch(md):
            md, mi = md.cpu().numpy(), mi.cpu().numpy()
        return md, mi

    def _filtered_search(self, queries, k, nprobe, filter, out):
        """batch_search with an id filter: vix_sharded_search_filtered (one rank: the local index's filtered search); k up to
        ``VIX_MAX_K_LARGE``, the filter applied on both passes of the large-k route on every rank"""
        nprobe = nprobe if nprobe > 0 else self.nprobe
        comm = self._native()
        if comm is None:
            if self.world == 1 and hasattr(self.local, "_h"):
                return self.local.batch_search(queries, k, nprobe=nprobe, filter=filter, out=out)
            raise NotImplementedError("a filtered sharded search needs the library's exchange (NCCL ranks over IVFPQIndex "
                                      "shards); the Python exchange path does not filter")
        q = as_input(queries, np.float32)
        nq, kk = int(q.shape[0]), max(int(k), 0)
        if out is not None:
            dist, ids = out
        else:
            dist, ids = empty_like_input(q, (nq, kk), np.float32), empty_like_input(q, (nq, kk), np.int64)
        if nq == 0 or kk == 0:
            return dist, ids
        check(lib().vix_sharded_search_filtered(self.local._h, comm._c, ptr(q, np.float32), C.c_int64(nq), C.c_int(k),
                                                C.c_int(nprobe), ptr(filter.words, np.uint64), C.c_int64(filter.capacity),
                                                C.c_int(filter.mode), ptr(dist, np.float32), ptr(ids, np.int64)))
        return dist, ids

    def range_search(self, queries, radius: float, nprobe: int = 0, filter=None):
        """Every stored vector within ``radius`` of each query, over all ranks' lists: ``IVFPQIndex.range_search`` on one
        GPU holding every row (vix_sharded_range_search: the probes of the whole batch, each rank's range scan of the lists
        it owns, the sorted rows exchanged and merged on the device).  Collective: every rank passes the same queries,
        radius, nprobe and ``filter`` (an :class:`IDFilter`) and receives the whole CSR ``(lims int64 [nq + 1], distances
        f32 [total], ids int64 [total])``: numpy for host queries, torch tensors on the queries' device for CUDA tensors."""
        nprobe = nprobe if nprobe > 0 else self.nprobe
        comm = self._native()
        if comm is None:
            if self.world == 1 and hasattr(self.local, "range_search"):
                return self.local.range_search(queries, radius, nprobe=nprobe, filter=filter)
            raise NotImplementedError("a sharded range search needs the library's exchange (NCCL ranks over IVFPQIndex "
                                      "shards); the Python exchange path has none")
        q = as_input(queries, np.float32)
        self.local._check_dim(q, "range_search")
        nq = int(q.shape[0])
        res = C.c_void_p(0)
        try:
            words = filter.words if filter is not None else None
            check(lib().vix_sharded_range_search(self.local._h, comm._c, ptr(q, np.float32), C.c_int64(nq),
                                                 C.c_float(float(radius)), C.c_int(nprobe), ptr(words, np.uint64),
                                                 C.c_int64(filter.capacity if filter is not None else 0),
                                                 C.c_int(filter.mode if filter is not None else 0), C.byref(res)))
            total = int(lib().vix_range_result_total(res))
            lims = empty_like_input(q, (nq + 1,), np.int64)
            dist = empty_like_input(q, (total,), np.float32)
            ids = empty_like_input(q, (total,), np.int64)
            check(lib().vix_range_result_get(res, ptr(lims, np.int64), ptr(dist, np.float32) if total else None,
                                             ptr(ids, np.int64) if total else None))
            return lims, dist, ids
        finally:
            lib().vix_range_result_destroy(res)


class ReplicatedIVFPQIndex(ShardedIVFPQIndex):
    """The other way to use several GPUs, for an index that fits ONE of them (BASELINE configs[4] is 12.5 GB of 180 GB):
    every rank holds ALL inverted lists and a batch is partitioned by QUERY.  Queries are independent units, so the data
    path has no exchange step at all -- a rank runs the single-GPU search (probe selection + fused scan + top-k, at the
    single-GPU efficiency: whole probe sets per query, the global k-th best as the threshold) on its 1/world of the batch;
    one all-gather of the finished [nq/world x k] blocks hands every rank the whole answer (callers that consume their
    own block skip it: ``gather=False``).  The list-sharded ``ShardedIVFPQIndex`` remains the layout for indexes larger
    than one GPU's memory (and the one `north_star` names).

    build   a rank assigns + encodes the rows it is handed (1/world of the encoding work); the encoded rows
            (assignment, codes, ids: m + 12 bytes each) are all-gathered and appended everywhere, rank by rank in
            the same order, so every replica holds identical lists;
    search  identical to ``IVFPQIndex.batch_search`` on the rank's query block: results are the single-GPU results by
            construction."""

    def set_list_bounds(self, bounds):
        raise ValueError("a replicated index has no list partition")

    def remove(self, ids) -> int:
        """Every replica removes the rows locally (no exchange); returns this replica's count, which is every replica's."""
        return self.local.batch_remove(ids)

    def add(self, vectors, ids):
        import torch
        import torch.distributed as dist
        assign, codes = self.local.encode(vectors)
        if self.world == 1:
            self.local.add_encoded(assign, codes, ids)
            return
        assign, codes, ids = self._to_comm(assign), self._to_comm(codes), self._to_comm(ids)
        n = int(assign.shape[0])
        cnt = torch.tensor([n], dtype=torch.int64, device=assign.device)
        counts = [int(v) for v in self._all_gather(cnt).view(-1).tolist()]
        cap = max(counts)
        if cap == 0:
            return

        def gathered(t):
            if n < cap:                                                   # ragged: pad to the largest contribution
                pad = torch.zeros((cap - n,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
                t = torch.cat([t, pad])
            return self._all_gather(t.contiguous())                       # [world][cap, ...]

        g_assign, g_codes, g_ids = gathered(assign.to(torch.int32)), gathered(codes), gathered(ids.to(torch.int64))
        for r in range(self.world):
            c = counts[r]
            if c == 0:
                continue
            a, co, i = g_assign[r, :c].contiguous(), g_codes[r, :c].contiguous(), g_ids[r, :c].contiguous()
            if not self._nccl():
                a, co, i = a.numpy(), co.numpy(), i.numpy()
            self.local.add_encoded(a, co, i)

    def range_search(self, queries, radius: float, nprobe: int = 0, filter=None):
        """Not available: every replica holds every list, so the sharded merge would return each row ``world`` times."""
        raise NotImplementedError("ReplicatedIVFPQIndex has no range search (ShardedIVFPQIndex.range_search merges list "
                                  "shards; a replica holds all lists)")

    def batch_search(self, queries, k, nprobe=0, gather=True, filter=None):
        """[nq x k] (distances, ids) of the whole batch on every rank (``gather=False``: this rank's block only, rows
        ``query_block(nq)``).  ``filter`` is not available on replicas."""
        import torch
        if filter is not None:
            raise NotImplementedError("ReplicatedIVFPQIndex has no filtered search")
        was_numpy = not _lib._is_torch(queries)
        nprobe = nprobe if nprobe > 0 else self.nprobe
        nq = int(queries.shape[0])
        lo, cnt, per = self.query_block(nq)
        qb = queries[lo:lo + cnt]
        if was_numpy and self.world > 1 and self._nccl():
            qb = self._to_comm(np.ascontiguousarray(qb, dtype=np.float32))      # only this rank's block crosses PCIe
        if hasattr(self.local, "batch_search"):
            d_loc, i_loc = self.local.batch_search(qb, k, nprobe)
        else:                                                                  # oracle-backed stand-in of the gloo tests
            probes = self.local.probe_range(qb, nprobe, 0, self.kc)[0]
            d_loc, i_loc = self.local.search_with_probes(qb, k, probes)
        if self.world == 1 or not gather:
            return d_loc, i_loc
        d_loc, i_loc = self._to_comm(d_loc), self._to_comm(i_loc)
        if cnt < per:                                                          # ragged last block: pad, gather, trim
            pad_d = torch.full((per - cnt, k), float("nan"), dtype=d_loc.dtype, device=d_loc.device)
            pad_i = torch.full((per - cnt, k), -1, dtype=i_loc.dtype, device=i_loc.device)
            d_loc, i_loc = torch.cat([d_loc, pad_d]), torch.cat([i_loc, pad_i])
        md = self._all_gather(d_loc.contiguous()).view(self.world * per, k)[:nq]
        mi = self._all_gather(i_loc.contiguous()).view(self.world * per, k)[:nq]
        if was_numpy:
            if md.is_cuda:
                return self._to_host(md.contiguous()), self._to_host(mi.contiguous())
            return md.numpy().copy(), mi.numpy().copy()
        return md.contiguous(), mi.contiguous()


class _ShardedExactIndex:
    """The sharded layout of the exact kinds (flat, IVF-Flat) over the ranks of a ``torch.distributed`` NCCL group: every
    call is one library call over a ``vix_comm_t`` (vix_sharded_add / vix_sharded_search_filtered /
    vix_sharded_range_search), bit for bit the one-GPU answer on an index holding every row in the slot the shards hold
    it in.  One rank is the local index.  There is no Python exchange for these kinds: a group whose backend is not NCCL
    raises ``NotImplementedError``."""

    def _setup(self, local, group):
        import torch.distributed as dist
        self.group = group
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.local = local
        self.bounds = None

    def _native(self):
        if self.world <= 1:
            return None
        import torch.distributed as dist
        if dist.get_backend(self.group) != "nccl":
            raise NotImplementedError(f"{type(self).__name__} needs the library's exchange (one NCCL rank per GPU); there "
                                      "is no Python exchange for the exact kinds")
        if self.__dict__.get("comm") is None:
            self.comm = Comm.from_torch(self.group)
        return self.comm

    def _pinned(self, tag, shape, dtype):
        return ShardedIVFPQIndex._pinned(self, tag, shape, dtype)

    @property
    def count(self) -> int:
        """rows THIS rank holds"""
        return self.local.count

    def add(self, vectors, ids):
        """Collective: the rows THIS rank contributes (any rows; n may be 0; explicit ids)."""
        comm = self._native()
        if comm is None:
            self.local.batch_insert(vectors, ids)
            return
        x = as_input(vectors, np.float32)
        self.local._check_dim(x, "add")
        i = as_input(ids, np.int64)
        b = None if self.bounds is None else np.ascontiguousarray(self.bounds, dtype=np.int64)
        check(lib().vix_sharded_add(self.local._h, comm._c, ptr(b), ptr(x, np.float32), ptr(i, np.int64),
                                    C.c_int64(int(x.shape[0]))))

    def remove(self, ids) -> int:
        """Collective: every rank passes the SAME ids and removes the rows of them it holds; returns the rows removed on all
        ranks together."""
        n = self.local.batch_remove(ids)
        if self.world == 1:
            return n
        import torch
        import torch.distributed as dist
        t = torch.tensor([n], dtype=torch.int64, device=torch.device("cuda", torch.cuda.current_device()))
        dist.all_reduce(t, group=self.group)
        return int(t.item())

    def batch_search(self, queries, k, nprobe=0, out=None, filter=None):
        """Collective: every rank passes the same queries, k (up to ``VIX_MAX_K_LARGE``), nprobe and ``filter`` (an
        :class:`IDFilter`) and receives the merged [nq x k] (distances, ids).  Host queries: over peer memory only this rank's
        block crosses PCIe (the library moves it to the peers), and the result lands in pinned memory; ``out``: optional
        (distances f32, ids int64) arrays to write into."""
        import torch
        comm = self._native()
        if comm is None:
            return self.local.batch_search(queries, k, nprobe, filter=filter, out=out)
        q = as_input(queries, np.float32)
        self.local._check_dim(q, "batch_search")
        nq, kk = int(q.shape[0]), max(int(k), 0)
        host = not _lib._is_torch(queries)
        if out is not None:
            dist_, ids = out
        elif host and nq and kk:
            dist_, ids = self._pinned("d", (nq, kk), torch.float32), self._pinned("i", (nq, kk), torch.int64)
        else:
            dist_, ids = empty_like_input(q, (nq, kk), np.float32), empty_like_input(q, (nq, kk), np.int64)
        if nq and kk:
            words = filter.words if filter is not None else None
            check(lib().vix_sharded_search_filtered(self.local._h, comm._c, ptr(q, np.float32), C.c_int64(nq), C.c_int(k),
                                                    C.c_int(nprobe), ptr(words, np.uint64),
                                                    C.c_int64(filter.capacity if filter is not None else 0),
                                                    C.c_int(filter.mode if filter is not None else 0),
                                                    ptr(dist_, np.float32), ptr(ids, np.int64)))
        if out is None and host and nq and kk:
            return dist_.numpy().copy(), ids.numpy().copy()
        return dist_, ids

    def range_search(self, queries, radius: float, nprobe: int = 0, filter=None):
        """Collective: every stored vector within ``radius`` of each query over all ranks, as the local index's
        ``range_search`` on one GPU holding every row: CSR ``(lims int64 [nq + 1], distances f32 [total], ids int64
        [total])``, numpy for host queries, torch tensors on the queries' device for CUDA tensors."""
        comm = self._native()
        if comm is None:
            return self.local.range_search(queries, radius, nprobe=nprobe, filter=filter)
        q = as_input(queries, np.float32)
        self.local._check_dim(q, "range_search")
        nq = int(q.shape[0])
        res = C.c_void_p(0)
        try:
            words = filter.words if filter is not None else None
            check(lib().vix_sharded_range_search(self.local._h, comm._c, ptr(q, np.float32), C.c_int64(nq),
                                                 C.c_float(float(radius)), C.c_int(nprobe), ptr(words, np.uint64),
                                                 C.c_int64(filter.capacity if filter is not None else 0),
                                                 C.c_int(filter.mode if filter is not None else 0), C.byref(res)))
            total = int(lib().vix_range_result_total(res))
            lims = empty_like_input(q, (nq + 1,), np.int64)
            dist_ = empty_like_input(q, (total,), np.float32)
            ids = empty_like_input(q, (total,), np.int64)
            check(lib().vix_range_result_get(res, ptr(lims, np.int64), ptr(dist_, np.float32) if total else None,
                                             ptr(ids, np.int64) if total else None))
            return lims, dist_, ids
        finally:
            lib().vix_range_result_destroy(res)


class ShardedFlatIndex(_ShardedExactIndex):
    """Flat index partitioned by rows: a row stays on the rank that adds it (no exchange at build time), every rank scans
    its rows and the per-rank results are merged on the device.  The answer equals ``FlatIndex`` on one GPU holding rank
    0's rows first, then rank 1's, and so on, each in add order: flat search breaks ties at an equal score by row."""

    def __init__(self, dimension, metric="euclidean", group=None):
        self._setup(FlatIndex(dimension, metric), group)


class ShardedIVFFlatIndex(_ShardedExactIndex):
    """IVF-Flat index partitioned by contiguous blocks of inverted lists, as ``ShardedIVFPQIndex``: every rank holds the
    coarse centroids (``set_coarse``, or ``optimize`` on the same sample on every rank) and the vectors of ITS lists; a row
    travels to the rank owning its list at ``add``.  Probes of the batch are selected once and exchanged; each rank scans
    the probed lists it owns; the answer equals ``IVFIndex`` on one GPU (its distances are exact per pair and its ties
    fall to the id, so the order the rows arrived in does not matter)."""

    def __init__(self, dimension, metric="euclidean", nlist=256, nprobe=8, group=None):
        self._setup(IVFIndex(dimension, metric, nlist, nprobe), group)
        self.kc = int(nlist)
        self.nprobe = int(nprobe)

    def set_list_bounds(self, bounds):
        """Block boundaries of the list partition ([world + 1], identical on every rank; before the first ``add``).
        Default: equal-count blocks."""
        b = np.asarray(bounds, dtype=np.int64)
        if b.size != self.world + 1 or b[0] != 0 or b[-1] != self.kc or (np.diff(b) < 0).any():
            raise ValueError("bounds must be [world + 1] ascending list ids from 0 to nlist")
        self.bounds = b

    def set_coarse(self, centroids):
        self.local.set_coarse(centroids)
        self.kc = int(self.local.get_coarse().shape[0])

    def optimize(self, training_vectors, kmeans_cfg: KMeansCfg | None = None):
        """Trains the coarse quantiser on ``training_vectors`` -- the same sample (and seed) on every rank, so every rank
        holds the same centroids.  Before the first ``add``."""
        if training_vectors is None:
            raise ValueError("a sharded IVF-Flat index trains on an explicit sample, the same on every rank")
        self.local.optimize(training_vectors, kmeans_cfg)
        self.kc = int(self.local.get_coarse().shape[0])

    train = optimize


class _ReplicatedIndex:
    """Replicas over the ranks of a ``torch.distributed`` NCCL group, behind the library's C ABI: every rank holds the WHOLE
    index and answers its block of each batch (``query_block``) with the one-GPU search; the blocks are assembled on the
    device (vix_replicated_add / vix_replicated_search_filtered / vix_replicated_range_search over a ``vix_comm_t``).  The
    answer on every rank is the local index's answer on one GPU holding the rows in the order the replicas append them (rank
    0's contributions first), bit for bit.  ``gather=False`` returns this rank's block only and skips the assembly (no
    exchange: the local index's search on the rows ``query_block(nq)``).  One rank is the local index."""

    def _setup(self, local, group):
        _ShardedExactIndex._setup(self, local, group)

    def _native(self):
        return _ShardedExactIndex._native(self)

    def _pinned(self, tag, shape, dtype):
        return ShardedIVFPQIndex._pinned(self, tag, shape, dtype)

    @property
    def count(self) -> int:
        """rows every replica holds"""
        return self.local.count

    def query_block(self, nq: int):
        """Rows of a batch of ``nq`` queries THIS rank answers: (first row, rows)."""
        first, cnt = C.c_int64(0), C.c_int64(0)
        check(lib().vix_sharded_query_block(C.c_int64(int(nq)), C.c_int(self.rank), C.c_int(self.world), C.byref(first),
                                            C.byref(cnt)))
        return int(first.value), int(cnt.value)

    def add(self, vectors, ids):
        """Collective: the rows THIS rank contributes (any rows; n may be 0; explicit ids).  Every replica appends every
        rank's rows, rank 0's first."""
        comm = self._native()
        if comm is None:
            self.local.batch_insert(vectors, ids)
            return
        x = as_input(vectors, np.float32)
        self.local._check_dim(x, "add")
        i = as_input(ids, np.int64)
        check(lib().vix_replicated_add(self.local._h, comm._c, ptr(x, np.float32), ptr(i, np.int64), C.c_int64(int(x.shape[0]))))

    def remove(self, ids) -> int:
        """Every replica passes the SAME ids and removes the rows locally (no exchange: the remaining rows keep their order,
        so the replicas stay identical); returns the rows removed, the same on every replica."""
        return self.local.batch_remove(ids)

    def batch_search(self, queries, k, nprobe=0, out=None, filter=None, gather=True):
        """Collective: every rank passes the same queries, k (up to ``VIX_MAX_K_LARGE``), nprobe and ``filter`` (an
        :class:`IDFilter`) and receives the whole [nq x k] (distances, ids).  Host queries: only this rank's block crosses
        PCIe, and the result lands in pinned memory; ``out``: optional (distances f32, ids int64) arrays to write into.
        ``gather=False``: this rank's block only (rows ``query_block(nq)``), with no exchange."""
        import torch
        q = as_input(queries, np.float32)
        self.local._check_dim(q, "batch_search")
        if not gather:
            lo, cnt = self.query_block(int(q.shape[0]))
            return self.local.batch_search(q[lo:lo + cnt], k, nprobe, filter=filter, out=out)
        comm = self._native()
        if comm is None:
            return self.local.batch_search(q, k, nprobe, filter=filter, out=out)
        nq, kk = int(q.shape[0]), max(int(k), 0)
        host = not _lib._is_torch(queries)
        if out is not None:
            dist_, ids = out
        elif host and nq and kk:
            dist_, ids = self._pinned("d", (nq, kk), torch.float32), self._pinned("i", (nq, kk), torch.int64)
        else:
            dist_, ids = empty_like_input(q, (nq, kk), np.float32), empty_like_input(q, (nq, kk), np.int64)
        if nq and kk:
            words = filter.words if filter is not None else None
            check(lib().vix_replicated_search_filtered(self.local._h, comm._c, ptr(q, np.float32), C.c_int64(nq), C.c_int(k),
                                                       C.c_int(nprobe), ptr(words, np.uint64),
                                                       C.c_int64(filter.capacity if filter is not None else 0),
                                                       C.c_int(filter.mode if filter is not None else 0),
                                                       ptr(dist_, np.float32), ptr(ids, np.int64)))
        if out is None and host and nq and kk:
            return dist_.numpy().copy(), ids.numpy().copy()
        return dist_, ids

    def range_search(self, queries, radius: float, nprobe: int = 0, filter=None, gather=True):
        """Collective: every stored vector within ``radius`` of each query, as the local index's ``range_search`` on one GPU:
        CSR ``(lims int64 [nq + 1], distances f32 [total], ids int64 [total])``, numpy for host queries, torch tensors on the
        queries' device for CUDA tensors.  ``gather=False``: this rank's block only, with no exchange."""
        q = as_input(queries, np.float32)
        self.local._check_dim(q, "range_search")
        if not gather:
            lo, cnt = self.query_block(int(q.shape[0]))
            return self.local.range_search(q[lo:lo + cnt], radius, nprobe=nprobe, filter=filter)
        comm = self._native()
        if comm is None:
            return self.local.range_search(q, radius, nprobe=nprobe, filter=filter)
        nq = int(q.shape[0])
        res = C.c_void_p(0)
        try:
            words = filter.words if filter is not None else None
            check(lib().vix_replicated_range_search(self.local._h, comm._c, ptr(q, np.float32), C.c_int64(nq),
                                                    C.c_float(float(radius)), C.c_int(nprobe), ptr(words, np.uint64),
                                                    C.c_int64(filter.capacity if filter is not None else 0),
                                                    C.c_int(filter.mode if filter is not None else 0), C.byref(res)))
            total = int(lib().vix_range_result_total(res))
            lims = empty_like_input(q, (nq + 1,), np.int64)
            dist_ = empty_like_input(q, (total,), np.float32)
            ids = empty_like_input(q, (total,), np.int64)
            check(lib().vix_range_result_get(res, ptr(lims, np.int64), ptr(dist_, np.float32) if total else None,
                                             ptr(ids, np.int64) if total else None))
            return lims, dist_, ids
        finally:
            lib().vix_range_result_destroy(res)


class ReplicatedFlatIndex(_ReplicatedIndex):
    """Flat index replicated on every rank (see :class:`_ReplicatedIndex`)."""

    def __init__(self, dimension, metric="euclidean", group=None):
        self._setup(FlatIndex(dimension, metric), group)


class ReplicatedIVFFlatIndex(_ReplicatedIndex):
    """IVF-Flat index replicated on every rank.  Every rank holds the same coarse centroids (``set_coarse``, or ``optimize``
    on the same sample on every rank) before the first ``add``."""

    def __init__(self, dimension, metric="euclidean", nlist=256, nprobe=8, group=None):
        self._setup(IVFIndex(dimension, metric, nlist, nprobe), group)

    def set_coarse(self, centroids):
        self.local.set_coarse(centroids)

    def optimize(self, training_vectors, kmeans_cfg: KMeansCfg | None = None):
        if training_vectors is None:
            raise ValueError("a replicated IVF-Flat index trains on an explicit sample, the same on every rank")
        self.local.optimize(training_vectors, kmeans_cfg)

    train = optimize


class ReplicatedNativeIVFPQIndex(_ReplicatedIndex):
    """IVF-PQ index replicated on every rank, entirely inside the library (``ReplicatedIVFPQIndex`` is the older layout whose
    add and final all-gather run through ``torch.distributed``, and which has no range search or filters).  Every rank holds
    the same coarse centroids and codebooks (``set_parameters``, or ``optimize`` on the same sample on every rank)."""

    def __init__(self, dimension, metric="euclidean", nlist=256, nprobe=8, m=16, ks=256, group=None):
        self._setup(IVFPQIndex(dimension, metric, nlist, nprobe, m, ks), group)

    def set_parameters(self, coarse, codebooks, centroid_norms=None):
        self.local.set_coarse(coarse)
        self.local.set_codebooks(codebooks, centroid_norms)

    def optimize(self, training_vectors, kmeans_cfg: KMeansCfg | None = None, pq_cfg: PQTrainCfg | None = None):
        self.local.optimize(training_vectors, kmeans_cfg, pq_cfg)

    train = optimize
