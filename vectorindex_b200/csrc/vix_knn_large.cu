// vix_knn_large.cu -- k-NN search for VIX_MAX_K < k <= VIX_MAX_K_LARGE: two passes over the range-search scans.
//
// Exactness.  Let S be any sub-multiset of a query's candidates with |S| >= k and tau the k-th smallest distance word
// (make_key(api distance, id, 0) >> 32) of S.  Then tau >= the k-th smallest word over all candidates, so the candidates
// whose word is <= tau hold the true top k together with every tie at the k-th distance; sorted by (distance, id) and cut
// at k they are exactly the k-NN answer.  With fewer than k entries in S, tau = 0xFFFFFFFF keeps every candidate, NaN
// included (make_key maps NaN to that word).
//
//   1. seed: S per query -- the range scan over a prefix of the probe list that holds about kKnnBeta * k stored vectors
//      (IVF), or the union of the fused top-min(512, rows) of contiguous row blocks (flat engine) -- grouped and sorted by
//      range_collect_keys; tau_q = the word of row key k - 1;
//      (the key is the one the kind's k-NN search selects on: the API distance for the IVF scans, the raw score in the
//      metric's order for the flat engine, whose API mapping -- sqrt, 1 - s -- can round two scores to one distance)
//   2. collect: the same range scan over every candidate with the per-query bound tau_q (RangeOut::bound);
//   3. cut: the first min(k, row length) keys of each sorted row, padded with id -1 / NaN.
//
// The two passes must agree on every distance (they run the same kernels on the same data): a row shorter than k whose
// bound is not 0xFFFFFFFF means they did not, and the call fails with VIX_ERR_CONTRACT.
//
// The halves are separate (knn_seed_bound, knn_collect) because sharded search (vix_sharded.cu) runs the seed on every rank,
// takes the minimum of the ranks' bounds between them, and exchanges each rank's collected rows cut at k (knn_trim).
#include "vix_common.cuh"
#include "vix_index.cuh"
#include "vix_range.cuh"

#include <math.h>

#include <algorithm>

namespace vix {

// The probe prefix of the seed: the probes of each query in order, with the scans' skip rules (ids outside [0, kc) and
// empty lists contribute nothing), up to and including the probe at which the running length reaches `target`; the rest
// of the row is -1.  total[0] += the stored vectors of the prefix (the seed's capacity), total[1] += those of every probe.
__global__ void knn_probe_prefix_kernel(const int32_t* __restrict__ probes, int64_t nq, int nprobe,
                                        const int32_t* __restrict__ list_len, int kc, int64_t target,
                                        int32_t* __restrict__ prefix, unsigned long long* __restrict__ total) {
    const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    const int32_t* pr = probes + q * nprobe;
    int32_t* out = prefix + q * nprobe;
    int64_t run = 0, all = 0;
    for (int p = 0; p < nprobe; ++p) {
        const int l = pr[p];
        const int64_t len = (unsigned)l < (unsigned)kc ? list_len[l] : 0;
        out[p] = run < target ? l : -1;
        if (run < target) run += len;
        all += len;
    }
    atomicAdd(total, (unsigned long long)run);
    atomicAdd(total + 1, (unsigned long long)all);
}

// The seed of the flat engine: one block's fused top-kb rows [nq x kb] (raw scores, block-local row indices, -1 padding)
// appended to the range output as selection keys with block-base row ids.  One CTA per query (warp-collective appends).
__global__ void __launch_bounds__(256)
knn_flat_seed_kernel(const float* __restrict__ score, const int64_t* __restrict__ rows, int64_t nq, int kb, int64_t base,
                     int order_max, RangeOut out) {
    __shared__ int s_cnt;
    for (int64_t q = blockIdx.x; q < nq; q += gridDim.x) {
        __syncthreads();
        if (threadIdx.x == 0) s_cnt = 0;
        __syncthreads();
        for (int j0 = 0; j0 < kb; j0 += blockDim.x) {
            const int j = j0 + threadIdx.x;
            const int64_t r = j < kb ? rows[q * kb + j] : -1;
            const bool pass = r >= 0;
            const u64 key = pass ? make_key(score[q * kb + j], (uint32_t)(r + base), order_max) : kEmptyKey;
            const unsigned ball = __ballot_sync(0xFFFFFFFFu, pass);
            if (ball) {
                range_append(out, ball, pass, key, (uint32_t)q);
                if ((threadIdx.x & 31) == 0) atomicAdd(&s_cnt, __popc(ball));
            }
        }
        __syncthreads();
        if (threadIdx.x == 0 && s_cnt) atomicAdd(out.counts + q, (unsigned long long)s_cnt);
    }
}

// bound[q] = the distance word of the k-th sorted seed key of row q, 0xFFFFFFFF when the row is shorter than k
__global__ void knn_bound_kernel(const u64* __restrict__ sorted, const int64_t* __restrict__ lims, int64_t nq, int k,
                                 uint32_t* __restrict__ bound) {
    const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    const int64_t lo = lims[q], len = lims[q + 1] - lo;
    bound[q] = len >= k ? (uint32_t)(sorted[lo + k - 1] >> 32) : 0xFFFFFFFFu;
}

// flag += queries whose collected row is shorter than k although their seed held k entries within the bound
__global__ void knn_short_kernel(const unsigned long long* __restrict__ counts, const uint32_t* __restrict__ bound,
                                 int64_t nq, int k, unsigned long long* __restrict__ flag) {
    const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    if (counts[q] < (unsigned long long)k && bound[q] != 0xFFFFFFFFu) atomicAdd(flag, 1ull);
}

// [nq x k] <- the first min(k, row length) keys of every sorted row, decoded (KnnDecode); padding id -1 / NaN
__global__ void knn_cut_kernel(const u64* __restrict__ sorted, const int64_t* __restrict__ lims, int64_t nq, int k,
                               KnnDecode dec, float* __restrict__ out_dist, int64_t* __restrict__ out_ids) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= nq * (int64_t)k) return;
    const int64_t q = e / k, i = e - q * k;
    const int64_t lo = lims[q], len = lims[q + 1] - lo;
    if (i < len) {
        const u64 key = sorted[lo + i];
        float v = key_score(key, dec.order_max);
        if (dec.dist_mode == 1) v = __fsqrt_rn(v);
        else if (dec.dist_mode == 2) v = -v;
        else if (dec.dist_mode == 3) v = __fsub_rn(1.0f, v);
        if (dec.neg_zero && v == 0.0f) v = -0.0f;
        out_dist[e] = v;
        out_ids[e] = (int64_t)key_id(key);
    } else { out_dist[e] = __int_as_float(0x7fc00000); out_ids[e] = -1; }
}

// counts[q] = min(k, row length): the keys of row q that can still belong to a top k
__global__ void knn_trim_counts_kernel(const int64_t* __restrict__ lims, int64_t nq, int k,
                                       unsigned long long* __restrict__ counts) {
    const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    const int64_t len = lims[q + 1] - lims[q];
    counts[q] = (unsigned long long)(len < k ? len : k);
}

// the first min(k, row length) keys of every sorted row, compacted at the new row starts out_lims (one CTA per row)
__global__ void __launch_bounds__(256)
knn_trim_kernel(const u64* __restrict__ sorted, const int64_t* __restrict__ lims, int64_t nq, int k,
                const int64_t* __restrict__ out_lims, u64* __restrict__ out) {
    for (int64_t q = blockIdx.x; q < nq; q += gridDim.x) {
        const int64_t lo = lims[q], olo = out_lims[q], n = out_lims[q + 1] - olo;
        for (int64_t i = threadIdx.x; i < n; i += blockDim.x) out[olo + i] = sorted[lo + i];
    }
}

int knn_probe_prefix(const int32_t* probes, int64_t nq, int nprobe, const int32_t* list_len, int kc, int k,
                     int32_t* prefix, size_t* seed_cap, size_t* max_entries) {
    cudaStream_t s = ctx().stream;
    Scratch<unsigned long long> total;
    VIX_TRY(total.alloc(2));
    VIX_CUDA(cudaMemsetAsync(total.ptr, 0, 16, s));
    knn_probe_prefix_kernel<<<(unsigned)((nq + 255) / 256), 256, 0, s>>>(probes, nq, nprobe, list_len, kc,
                                                                         (int64_t)kKnnBeta * k, prefix, total.ptr);
    VIX_LAUNCH_CHECK();
    unsigned long long h[2] = {0, 0};
    VIX_CUDA(cudaMemcpyAsync(h, total.ptr, 16, cudaMemcpyDeviceToHost, s));
    VIX_CUDA(cudaStreamSynchronize(s));
    *seed_cap = (size_t)h[0];
    *max_entries = (size_t)h[1];
    return VIX_OK;
}

int knn_seed_bound(int64_t nq, int k, size_t seed_cap, const std::function<int(const RangeOut&)>* seed, uint32_t* bound,
                   int64_t* seed_total) {
    cudaStream_t s = ctx().stream;
    VIX_CUDA(cudaMemsetAsync(bound, 0xFF, (size_t)nq * 4, s));           // every candidate passes (the seed's own bound)
    *seed_total = 0;
    if (!seed) return VIX_OK;
    RangeKeys srk;
    RangeInfo si;
    VIX_TRY(range_collect_keys(nq, INFINITY, seed_cap, *seed, srk, &si, bound));
    *seed_total = srk.total;
    if (srk.total > 0) {
        knn_bound_kernel<<<(unsigned)((nq + 255) / 256), 256, 0, s>>>(srk.sorted, srk.lims.ptr, nq, k, bound);
        VIX_LAUNCH_CHECK();
    }
    return VIX_OK;
}

int knn_collect(int64_t nq, int k, const uint32_t* bound, const std::function<int(const RangeOut&)>& collect,
                size_t max_entries, size_t& cap, RangeKeys& rk, RangeInfo* info, unsigned long long* short_rows) {
    cudaStream_t s = ctx().stream;
    // first capacity: the hint of the last call, at least kKnnBeta k per query, never more than the candidates
    const size_t floor_cap = std::min((size_t)kKnnBeta * (size_t)k * (size_t)nq, max_entries);
    if (cap < floor_cap) cap = floor_cap;
    if (!short_rows) return range_collect_keys(nq, INFINITY, cap, collect, rk, info, bound);
    Scratch<unsigned long long> flag;
    VIX_TRY(flag.alloc(1));
    auto checked = [&](const RangeOut& o) -> int {
        VIX_CUDA(cudaMemsetAsync(flag.ptr, 0, 8, s));
        VIX_TRY(collect(o));
        knn_short_kernel<<<(unsigned)((nq + 255) / 256), 256, 0, s>>>(o.counts, o.bound, nq, k, flag.ptr);
        VIX_LAUNCH_CHECK();
        return VIX_OK;
    };
    *short_rows = 0;
    return range_collect_keys(nq, INFINITY, cap, checked, rk, info, bound, flag.ptr, short_rows);
}

int knn_trim(int64_t nq, int k, const RangeKeys& rk, RangeKeys& out) {
    cudaStream_t s = ctx().stream;
    VIX_TRY(out.lims.alloc((size_t)nq + 1));
    Scratch<unsigned long long> cnt;                                     // [counts nq][scan info 3]
    VIX_TRY(cnt.alloc((size_t)nq + 3));
    knn_trim_counts_kernel<<<(unsigned)((nq + 255) / 256), 256, 0, s>>>(rk.lims.ptr, nq, k, cnt.ptr);
    VIX_LAUNCH_CHECK();
    VIX_TRY(range_lims(cnt.ptr, nq, out.lims.ptr, cnt.ptr + nq));
    // (the trimmed total stays on the device: the exchange of the row starts carries it)
    out.total = std::min<int64_t>(rk.total, nq * (int64_t)k);
    out.sorted = nullptr;
    if (out.total == 0) return VIX_OK;
    VIX_TRY(out.a.alloc((size_t)out.total));
    out.sorted = out.a.ptr;
    const unsigned grid = (unsigned)std::min<int64_t>((int64_t)num_sms() * 8, nq);
    knn_trim_kernel<<<grid, 256, 0, s>>>(rk.sorted, rk.lims.ptr, nq, k, out.lims.ptr, out.a.ptr);
    VIX_LAUNCH_CHECK();
    return VIX_OK;
}

int knn_large_run(int64_t nq, int k, KnnDecode dec, size_t seed_cap, const std::function<int(const RangeOut&)>* seed,
                  const std::function<int(const RangeOut&)>& collect, size_t max_entries, size_t& cap_hint, float* out_dist,
                  int64_t* out_ids, KnnInfo* info) {
    cudaStream_t s = ctx().stream;
    Scratch<uint32_t> bound;
    VIX_TRY(bound.alloc((size_t)nq));
    VIX_TRY(knn_seed_bound(nq, k, seed_cap, seed, bound.ptr, &info->seed));
    size_t cap = cap_hint;
    unsigned long long short_rows = 0;
    RangeKeys rk;
    VIX_TRY(knn_collect(nq, k, bound.ptr, collect, max_entries, cap, rk, &info->collect, &short_rows));
    VIX_REQUIRE(short_rows == 0, VIX_ERR_CONTRACT,
                "k-NN search (k = %d): %llu queries collected fewer than k entries within the bound their seed pass found",
                k, short_rows);
    knn_cut_kernel<<<(unsigned)((nq * (int64_t)k + 255) / 256), 256, 0, s>>>(rk.sorted, rk.lims.ptr, nq, k, dec, out_dist,
                                                                            out_ids);
    VIX_LAUNCH_CHECK();
    cap_hint = cap;
    return VIX_OK;
}

int flat_knn_pass(const float* q, int64_t nq, const float* xb, int64_t n, int d, int metric, int k,
                  const uint64_t* disabled_rows, FlatKnnPass& p) {
    // seed blocks: T = ceil(kKnnBeta k / VIX_MAX_K) contiguous blocks whose boundaries are multiples of 64 rows (the
    // filter's row mask is then offset by whole words); none when every row fits the seed's budget anyway
    // the fused flat search's selection: the score, largest first for inner product and cosine, then its API mapping
    p.dec = flat_knn_decode(metric);
    p.seed = nullptr;
    p.seed_cap = 0;
    p.max_entries = (size_t)(nq * n);
    if (n > (int64_t)kKnnBeta * k) {
        const int64_t T = ((int64_t)kKnnBeta * k + VIX_MAX_K - 1) / VIX_MAX_K;
        const int64_t nb = ((n + T - 1) / T + 63) / 64 * 64;
        for (int64_t base = 0; base < n; base += nb) p.seed_cap += (size_t)nq * (size_t)std::min<int64_t>(VIX_MAX_K, std::min(nb, n - base));
        const int64_t kb_max = std::min<int64_t>(VIX_MAX_K, nb);
        VIX_TRY(p.bd.alloc((size_t)(nq * kb_max)));
        VIX_TRY(p.bi.alloc((size_t)(nq * kb_max)));
        float* bd = p.bd.ptr;
        int64_t* bi = p.bi.ptr;
        const int order_max = p.dec.order_max;
        p.seed = [=](const RangeOut& o) -> int {
            for (int64_t base = 0; base < n; base += nb) {
                const int64_t rows = std::min(nb, n - base);
                const int kb = (int)std::min<int64_t>(VIX_MAX_K, rows);
                if (disabled_rows)
                    VIX_TRY(flat_search_masked_device(q, nq, xb + (size_t)base * d, rows, d, metric, kb, disabled_rows + base / 64,
                                                      bd, bi, true));
                else
                    VIX_TRY(flat_search_auto_device(q, nq, xb + (size_t)base * d, rows, d, metric, kb, nullptr, bd, bi, true));
                const unsigned grid = (unsigned)std::min<int64_t>((int64_t)num_sms() * 8, nq);
                knn_flat_seed_kernel<<<grid, 256, 0, ctx().stream>>>(bd, bi, nq, kb, base, order_max, o);
                VIX_LAUNCH_CHECK();
            }
            return VIX_OK;
        };
    }
    // (row indices as ids and the raw score as the key: the order of the fused flat search, ties to the smaller row)
    p.collect = [=](const RangeOut& o) { return flat_range_device(q, nq, xb, n, d, metric, nullptr, disabled_rows, o); };
    return VIX_OK;
}

int flat_knn_large_device(const float* q, int64_t nq, const float* xb, int64_t n, int d, int metric, int k,
                          const uint64_t* disabled_rows, size_t& cap_hint, float* out_dist, int64_t* out_rows, KnnInfo* info) {
    FlatKnnPass p;
    VIX_TRY(flat_knn_pass(q, nq, xb, n, d, metric, k, disabled_rows, p));
    return knn_large_run(nq, k, p.dec, p.seed_cap, p.seed ? &p.seed : nullptr, p.collect, p.max_entries, cap_hint, out_dist,
                         out_rows, info);
}

}  // namespace vix
