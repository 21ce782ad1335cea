// vix_range.cuh -- the output path of range search (vix_index_range_search): every candidate whose API distance is at most
// the radius, per query, sorted by (distance, id).
//
// The scan kernels (flat pair tiles, the IVF-Flat candidate scan, the query-major IVF-PQ scan) append each passing candidate
// as the library's 64-bit selection key (make_key over the API distance, ids < 2^32) together with its query index, into a
// buffer the call owns: one atomicAdd on a shared cursor per warp (warp-aggregated), and a per-query count kept by the
// kernel.  Entries past the capacity are counted but not written; the host reads the total once, and when it exceeds the
// capacity the scan runs once more with the exact capacity.  vix_range.cu then groups the entries by query (exclusive scan
// of the counts + counting-sort scatter) and sorts each query's keys: one CTA in shared memory up to kRangeSegment keys,
// runs of that size merged pass by pass in global memory above it.  No CUB on this path.
#pragma once

#include "vix_common.cuh"

#include <functional>

namespace vix {

// where a scan kernel writes what passes (device pointers)
struct RangeOut {
    u64* keys = nullptr;                       // [cap] make_key(api distance, id, 0)
    uint32_t* qry = nullptr;                   // [cap] query of the entry
    unsigned long long* cursor = nullptr;      // [1]   entries appended (may exceed cap)
    unsigned long long* counts = nullptr;      // [nq]  entries per query (written or added by the scan kernels)
    unsigned long long cap = 0;
    float radius = 0.0f;
    // k-NN search beyond VIX_MAX_K (vix_knn_large.cu): when set, an entry passes when the high word of its key is at most
    // bound[query] (the key space of make_key, so NaN distances pass a bound of 0xFFFFFFFF); radius is then not read.  The
    // key is then the one the kind's k-NN search selects on: the IVF scans' as in range search, the flat engine's the
    // score in the order of its metric (KnnDecode)
    const uint32_t* bound = nullptr;           // [nq]
};

#ifdef __CUDACC__
// warp-collective (all 32 lanes): append the entries of the lanes whose bit is set in `ball` (= ballot of `pass`)
__device__ __forceinline__ void range_append(const RangeOut& o, unsigned ball, bool pass, u64 key, uint32_t q) {
    const int lane = threadIdx.x & 31;
    unsigned long long base = 0;
    if (lane == 0) base = atomicAdd(o.cursor, (unsigned long long)__popc(ball));
    base = __shfl_sync(0xFFFFFFFFu, base, 0);
    if (pass) {
        const unsigned long long pos = base + (unsigned long long)__popc(ball & ((1u << lane) - 1u));
        if (pos < o.cap) { o.keys[pos] = key; o.qry[pos] = q; }
    }
}
#endif

}  // namespace vix

// the result object of vix_index_range_search (device memory owned by it)
struct vix_range_result {
    int64_t nq = 0, total = 0;
    int64_t* lims = nullptr;     // [nq + 1]
    float* dist = nullptr;       // [total]
    int64_t* ids = nullptr;      // [total]
};

namespace vix {

// What one range call reports for the [vix range] line of VIX_SCAN_DEBUG.
struct RangeInfo { int passes = 0; int64_t total = 0, max_row = 0, sorted_long = 0; };

// The grouped and sorted keys of one range call, before decoding (device buffers held by the caller): row q is
// sorted[lims[q] .. lims[q + 1]), ascending.
struct RangeKeys {
    Scratch<int64_t> lims;                     // [nq + 1]
    Scratch<u64> a, b;                         // sort buffers; `sorted` points into one of them
    u64* sorted = nullptr;
    int64_t total = 0;
};

// Runs `scan` (which appends into the RangeOut it is handed and fills the per-query counts) once, or twice when the first
// capacity (cap_hint, updated for the next call) is too small, then groups the entries by query and sorts each row.  The
// only host synchronisation is the read of the total.  bound: handed to the scan in RangeOut::bound.  flag_dev / flag_host:
// a device word the scan writes, read in the same synchronisation as the total (the value after the last pass).
int range_collect_keys(int64_t nq, float radius, size_t& cap_hint, const std::function<int(const RangeOut&)>& scan,
                       RangeKeys& keys, RangeInfo* info, const uint32_t* bound = nullptr,
                       const unsigned long long* flag_dev = nullptr, unsigned long long* flag_host = nullptr);

// sorted keys -> a new result object (lims copied from `lims`, device pointers).  neg_zero: the path reports a zero distance
// as -0 (inner product through the flat engine and the IVF-PQ scan, whose API distance is the negated score); the key
// keeps +0.
int range_decode(int64_t nq, const int64_t* lims, const u64* sorted, int64_t total, bool neg_zero, vix_range_result** out);

// range_collect_keys, then range_decode
int range_collect(int64_t nq, float radius, size_t& cap_hint, bool neg_zero, const std::function<int(const RangeOut&)>& scan,
                  vix_range_result** out, RangeInfo* info);

// the result object with its arrays allocated (freed again on failure), and its release
int range_alloc(int64_t nq, int64_t total, vix_range_result** out);
void range_free(vix_range_result* r);

#ifdef __CUDACC__
// one sorted key as the result reports it
__device__ __forceinline__ void range_decode_key(u64 key, int neg_zero, float* dist, int64_t* id) {
    float v = key_score(key, 0);
    if (neg_zero && v == 0.0f) v = -0.0f;
    *dist = v;
    *id = (int64_t)key_id(key);
}
#endif

// ---- k-NN search for VIX_MAX_K < k <= VIX_MAX_K_LARGE (vix_knn_large.cu) ----
constexpr int kKnnBeta = 2;                    // the seed covers about kKnnBeta * k candidates per query

// what one call reports for the [vix knn] line of VIX_SCAN_DEBUG and vix_search_stats
struct KnnInfo { int64_t seed = 0; RangeInfo collect; };

// the seed's probe prefix of every query (device [nq x nprobe]); seed_cap: the stored vectors of all prefixes,
// max_entries: those of all probes (synchronises the stream)
int knn_probe_prefix(const int32_t* probes, int64_t nq, int nprobe, const int32_t* list_len, int kc, int k, int32_t* prefix,
                     size_t* seed_cap, size_t* max_entries);

// how a collected key becomes the reported distance: key_score(key, order_max), then dist_mode as the fused flat search
// maps it (0 itself, 1 sqrt, 2 negated, 3 1 - score), and neg_zero as range_decode_key
struct KnnDecode { int order_max = 0, dist_mode = 0, neg_zero = 0; };

// seed (nullable: every candidate passes), collect with the per-query bound, cut -> out [nq x k] (device).  seed_cap: the
// seed's capacity; max_entries: an upper bound of the candidates; cap_hint: the collect's first capacity, updated on success.
int knn_large_run(int64_t nq, int k, KnnDecode dec, size_t seed_cap, const std::function<int(const RangeOut&)>* seed,
                  const std::function<int(const RangeOut&)>& collect, size_t max_entries, size_t& cap_hint, float* out_dist,
                  int64_t* out_ids, KnnInfo* info);

// The halves of knn_large_run.  knn_seed_bound: bound [nq] (device) <- the word of each row's k-th sorted seed key,
// 0xFFFFFFFF where the seed holds fewer than k or there is no seed (seed nullable); *seed_total: the seed's entries.
int knn_seed_bound(int64_t nq, int k, size_t seed_cap, const std::function<int(const RangeOut&)>* seed, uint32_t* bound,
                   int64_t* seed_total);
// knn_collect: the candidates within the bound, grouped and sorted (rk).  cap: in, the hint of the last call; out, the
// next call's.  short_rows (nullable): the queries whose row is shorter than k although their bound is finite.
int knn_collect(int64_t nq, int k, const uint32_t* bound, const std::function<int(const RangeOut&)>& collect,
                size_t max_entries, size_t& cap, RangeKeys& rk, RangeInfo* info, unsigned long long* short_rows);
// the first min(k, row length) keys of every sorted row of rk, compacted with new row starts (out.lims, device).  out.total
// is an upper bound (min(rk.total, nq k)); the exact total is out.lims[nq] on the device.
int knn_trim(int64_t nq, int k, const RangeKeys& rk, RangeKeys& out);

// lims = exclusive scan of counts [nq] (lims[nq] = total), info [3] = {total, longest row, rows longer than the in-shared-
// memory sort} (device pointers, one launch)
int range_lims(const unsigned long long* counts, int64_t nq, int64_t* lims, unsigned long long* info);

// the fused flat search's selection key and API mapping: the raw score, largest first for inner product and cosine, then
// sqrt (L2), -s (IP) or 1 - s (cosine); the zero of an IP distance is -0 by that mapping
inline KnnDecode flat_knn_decode(int metric) {
    KnnDecode dec;
    dec.order_max = metric != VIX_METRIC_L2;
    dec.dist_mode = metric == VIX_METRIC_L2 ? 1 : metric == VIX_METRIC_IP ? 2 : 3;
    return dec;
}

// The flat engine's two passes, apart (flat_knn_large_device runs them as knn_large_run; sharded search runs the seed on
// every rank, takes the minimum of the ranks' bounds, then the collect): seed over T row blocks (empty when every row fits
// the seed's budget), collect = the flat range kernel within the bound; both key (raw score word, row index).  The
// functions capture q, xb and the mask by value and the seed's buffers of the object, which must outlive them.
struct FlatKnnPass {
    KnnDecode dec;
    size_t seed_cap = 0, max_entries = 0;
    std::function<int(const RangeOut&)> seed, collect;
    Scratch<float> bd;
    Scratch<int64_t> bi;
};
int flat_knn_pass(const float* q, int64_t nq, const float* xb, int64_t n, int d, int metric, int k,
                  const uint64_t* disabled_rows, FlatKnnPass& p);

// the flat engine's route (ids = row indices; disabled_rows: bit r set => row r skipped)
int flat_knn_large_device(const float* q, int64_t nq, const float* xb, int64_t n, int d, int metric, int k,
                          const uint64_t* disabled_rows, size_t& cap_hint, float* out_dist, int64_t* out_rows, KnnInfo* info);

// an empty result of nq rows (lims all 0)
int range_empty(int64_t nq, vix_range_result** out);

// flat range scan over xb (pair-tile engine, vix_scoring.cu); ids[r] is the id of row r; disabled_rows: bit r set => skipped
int flat_range_device(const float* q, int64_t nq, const float* xb, int64_t n, int d, int metric, const int64_t* ids,
                      const uint64_t* disabled_rows, const RangeOut& out);

}  // namespace vix
