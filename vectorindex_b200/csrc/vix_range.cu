// vix_range.cu -- the output path of range search (see vix_range.cuh): capacity / second pass, grouping by query, the
// per-query sort and the result object of the C ABI.
#include "vix_common.cuh"
#include "vix_topk.cuh"
#include "vix_range.cuh"

#include <new>
#include <stdlib.h>

namespace vix {

constexpr int kRangeSegment = 2048;    // keys a CTA sorts in shared memory (16 KB); longer rows are merged in global memory

// single CTA: lims = exclusive scan of the counts (lims[nq] = total); info = {total, longest row, rows longer than a segment}
__global__ void __launch_bounds__(1024)
range_lims_kernel(const unsigned long long* __restrict__ counts, int64_t nq, int64_t* __restrict__ lims,
                  unsigned long long* __restrict__ info) {
    __shared__ unsigned long long s_sum[1024], s_max[1024], s_long[1024];
    const int64_t per = (nq + 1023) / 1024;
    const int64_t b = threadIdx.x * per, e = min(b + per, nq);
    unsigned long long sum = 0, mx = 0, nl = 0;
    for (int64_t i = b; i < e; ++i) {
        const unsigned long long c = counts[i];
        sum += c; mx = c > mx ? c : mx; nl += c > (unsigned long long)kRangeSegment ? 1 : 0;
    }
    s_sum[threadIdx.x] = sum; s_max[threadIdx.x] = mx; s_long[threadIdx.x] = nl;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {                      // inclusive scan of the sums
        const unsigned long long v = (int)threadIdx.x >= o ? s_sum[threadIdx.x - o] : 0;
        __syncthreads();
        s_sum[threadIdx.x] += v;
        __syncthreads();
    }
    unsigned long long run = s_sum[threadIdx.x] - sum;
    for (int64_t i = b; i < e; ++i) { lims[i] = (int64_t)run; run += counts[i]; }
    if (threadIdx.x == 1023) lims[nq] = (int64_t)s_sum[1023];
    for (int o = 512; o > 0; o >>= 1) {                       // max and count of long rows
        __syncthreads();
        if ((int)threadIdx.x < o) {
            s_max[threadIdx.x] = max(s_max[threadIdx.x], s_max[threadIdx.x + o]);
            s_long[threadIdx.x] += s_long[threadIdx.x + o];
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) { info[0] = s_sum[1023]; info[1] = s_max[0]; info[2] = s_long[0]; }
}

// counting-sort scatter: sorted[lims[q] + fill[q]++] = key (the order inside a row is fixed by the sort that follows).
// Lanes with the same query share one atomic (entries of a query arrive in runs).
__global__ void __launch_bounds__(256)
range_scatter_kernel(const u64* __restrict__ keys, const uint32_t* __restrict__ qry, int64_t total,
                     const int64_t* __restrict__ lims, unsigned long long* __restrict__ fill, u64* __restrict__ sorted) {
    const int lane = threadIdx.x & 31;
    for (int64_t base = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) & ~31LL; base < total;
         base += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = base + lane;
        const bool live = i < total;
        const uint32_t q = live ? qry[i] : 0xFFFFFFFFu;
        const unsigned peers = __match_any_sync(0xFFFFFFFFu, q);
        const int leader = __ffs(peers) - 1;
        unsigned long long pos = 0;
        if (lane == leader && live) pos = atomicAdd(fill + q, (unsigned long long)__popc(peers));
        pos = __shfl_sync(0xFFFFFFFFu, pos, leader);
        if (live) sorted[lims[q] + (int64_t)pos + __popc(peers & ((1u << lane) - 1u))] = keys[i];
    }
}

// one CTA per row: rows up to kRangeSegment keys are sorted whole; longer rows in runs of kRangeSegment (merged below)
__global__ void __launch_bounds__(512)
range_sort_rows_kernel(u64* __restrict__ keys, const int64_t* __restrict__ lims, int64_t nq) {
    __shared__ u64 s[kRangeSegment];
    for (int64_t q = blockIdx.x; q < nq; q += gridDim.x) {
        const int64_t lo = lims[q], len = lims[q + 1] - lo;
        if (len < 2) continue;
        for (int64_t r0 = 0; r0 < len; r0 += kRangeSegment) {
            const int n = (int)min((int64_t)kRangeSegment, len - r0);
            const int P = next_pow2(n);
            __syncthreads();
            for (int i = threadIdx.x; i < P; i += blockDim.x) s[i] = i < n ? keys[lo + r0 + i] : kEmptyKey;
            __syncthreads();
            bitonic_sort_keys<false>(s, P, threadIdx.x, blockDim.x);
            for (int i = threadIdx.x; i < n; i += blockDim.x) keys[lo + r0 + i] = s[i];
        }
    }
}

// One merge pass over every row: sorted runs of w keys are merged pairwise (src -> dst).  Element i of the left run goes to
// its index plus the number of right-run keys < it, an element of the right run to its index plus the number of left-run
// keys <= it (stable, and correct for equal keys).  Rows no longer than w are copied.
__global__ void __launch_bounds__(256)
range_merge_pass_kernel(const u64* __restrict__ src, u64* __restrict__ dst, const int64_t* __restrict__ lims, int64_t nq,
                        int64_t total, int64_t w) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        int64_t a = 0, b = nq;                                // row of i: last q with lims[q] <= i
        while (b - a > 1) { const int64_t mid = (a + b) >> 1; if (lims[mid] <= i) a = mid; else b = mid; }
        const int64_t lo = lims[a], len = lims[a + 1] - lo, r = i - lo;
        const u64 key = src[i];
        const int64_t pair = (r / (2 * w)) * (2 * w);
        const int64_t mid = pair + w, end = min(pair + 2 * w, len);
        if (len <= w || mid >= len) { dst[i] = key; continue; }
        int64_t pos;
        if (r < mid) {                                        // left run: count right keys < key
            int64_t x = mid, y = end;
            while (x < y) { const int64_t m = (x + y) >> 1; if (src[lo + m] < key) x = m + 1; else y = m; }
            pos = (r - pair) + (x - mid);
        } else {                                              // right run: count left keys <= key
            int64_t x = pair, y = mid;
            while (x < y) { const int64_t m = (x + y) >> 1; if (src[lo + m] <= key) x = m + 1; else y = m; }
            pos = (r - mid) + (x - pair);
        }
        dst[lo + pair + pos] = key;
    }
}

__global__ void range_decode_kernel(const u64* __restrict__ keys, int64_t total, int neg_zero, float* __restrict__ dist,
                                    int64_t* __restrict__ ids) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    range_decode_key(keys[i], neg_zero, dist + i, ids + i);
}

int range_lims(const unsigned long long* counts, int64_t nq, int64_t* lims, unsigned long long* info) {
    range_lims_kernel<<<1, 1024, 0, ctx().stream>>>(counts, nq, lims, info);
    VIX_LAUNCH_CHECK();
    return VIX_OK;
}

void range_free(vix_range_result* r) {
    if (!r) return;
    if (r->lims) cudaFree(r->lims);
    if (r->dist) cudaFree(r->dist);
    if (r->ids) cudaFree(r->ids);
    delete r;
}

int range_alloc(int64_t nq, int64_t total, vix_range_result** out) {
    vix_range_result* r = new (std::nothrow) vix_range_result();
    VIX_REQUIRE(r, VIX_ERR_OOM, "vix_index_range_search: out of host memory");
    r->nq = nq; r->total = total;
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&r->lims), (size_t)(nq + 1) * 8);
    if (e == cudaSuccess && total > 0) e = cudaMalloc(reinterpret_cast<void**>(&r->dist), (size_t)total * 4);
    if (e == cudaSuccess && total > 0) e = cudaMalloc(reinterpret_cast<void**>(&r->ids), (size_t)total * 8);
    if (e != cudaSuccess) { range_free(r); VIX_CUDA(e); }
    *out = r;
    return VIX_OK;
}

int range_empty(int64_t nq, vix_range_result** out) {
    vix_range_result* r = nullptr;
    VIX_TRY(range_alloc(nq, 0, &r));
    const cudaError_t e = cudaMemsetAsync(r->lims, 0, (size_t)(nq + 1) * 8, ctx().stream);
    if (e != cudaSuccess) { range_free(r); VIX_CUDA(e); }
    *out = r;
    return VIX_OK;
}

int range_collect_keys(int64_t nq, float radius, size_t& cap_hint, const std::function<int(const RangeOut&)>& scan,
                       RangeKeys& rk, RangeInfo* info, const uint32_t* bound, const unsigned long long* flag_dev,
                       unsigned long long* flag_host) {
    cudaStream_t s = ctx().stream;
    const size_t floor_cap = (size_t)(nq * 64 > 65536 ? nq * 64 : 65536);
    size_t cap = cap_hint > floor_cap ? cap_hint : floor_cap;
    Scratch<unsigned long long> ctr;                          // [cursor][counts nq][info 3]
    VIX_TRY(ctr.alloc((size_t)nq + 4));
    VIX_TRY(rk.lims.alloc((size_t)nq + 1));
    Scratch<u64> keys;
    Scratch<uint32_t> qry;
    unsigned long long h_info[3] = {0, 0, 0};
    int passes = 0;
    for (;;) {
        VIX_TRY(keys.alloc(cap));
        VIX_TRY(qry.alloc(cap));
        VIX_CUDA(cudaMemsetAsync(ctr.ptr, 0, ((size_t)nq + 1) * 8, s));
        RangeOut o;
        o.keys = keys.ptr; o.qry = qry.ptr; o.cursor = ctr.ptr; o.counts = ctr.ptr + 1; o.cap = cap; o.radius = radius;
        o.bound = bound;
        VIX_TRY(scan(o));
        ++passes;
        range_lims_kernel<<<1, 1024, 0, s>>>(o.counts, nq, rk.lims.ptr, ctr.ptr + 1 + nq);
        VIX_LAUNCH_CHECK();
        VIX_CUDA(cudaMemcpyAsync(h_info, ctr.ptr + 1 + nq, sizeof h_info, cudaMemcpyDeviceToHost, s));
        if (flag_dev) VIX_CUDA(cudaMemcpyAsync(flag_host, flag_dev, sizeof *flag_host, cudaMemcpyDeviceToHost, s));
        VIX_CUDA(cudaStreamSynchronize(s));                   // the one synchronisation: the size of the answer
        if (h_info[0] <= cap) break;
        VIX_REQUIRE(passes == 1, VIX_ERR_CONTRACT, "range search: the second pass found %llu entries after a first count of %zu",
                    h_info[0], cap);
        cap = (size_t)h_info[0];
        keys.release(); qry.release();
    }
    const int64_t total = (int64_t)h_info[0];
    cap_hint = (size_t)(total + total / 8);
    if (info) { info->passes = passes; info->total = total; info->max_row = (int64_t)h_info[1]; info->sorted_long = (int64_t)h_info[2]; }
    rk.total = total;
    rk.sorted = nullptr;
    if (total > 0) {
        VIX_TRY(rk.a.alloc((size_t)total));
        const int64_t max_row = (int64_t)h_info[1];
        if (max_row > kRangeSegment) VIX_TRY(rk.b.alloc((size_t)total));
        VIX_CUDA(cudaMemsetAsync(ctr.ptr + 1, 0, (size_t)nq * 8, s));   // the counts become the scatter's fill cursors
        const unsigned grid = (unsigned)min((int64_t)num_sms() * 8, (total + 255) / 256);
        range_scatter_kernel<<<grid, 256, 0, s>>>(keys.ptr, qry.ptr, total, rk.lims.ptr, ctr.ptr + 1, rk.a.ptr);
        const unsigned rows_grid = (unsigned)min((int64_t)num_sms() * 4, nq);
        range_sort_rows_kernel<<<rows_grid, 512, 0, s>>>(rk.a.ptr, rk.lims.ptr, nq);
        ctx().launches += 2;
        u64* cur = rk.a.ptr;
        u64* oth = rk.b.ptr;
        for (int64_t w = kRangeSegment; w < max_row; w *= 2) {
            range_merge_pass_kernel<<<grid, 256, 0, s>>>(cur, oth, rk.lims.ptr, nq, total, w);
            ctx().launches += 1;
            u64* t = cur; cur = oth; oth = t;
        }
        VIX_CUDA(cudaGetLastError());
        rk.sorted = cur;
    }
    return VIX_OK;
}

int range_decode(int64_t nq, const int64_t* lims, const u64* sorted, int64_t total, bool neg_zero, vix_range_result** out) {
    cudaStream_t s = ctx().stream;
    vix_range_result* r = nullptr;
    VIX_TRY(range_alloc(nq, total, &r));
    auto fail = [&](int rc) { range_free(r); return rc; };
    cudaError_t ce = cudaMemcpyAsync(r->lims, lims, (size_t)(nq + 1) * 8, cudaMemcpyDeviceToDevice, s);
    if (ce != cudaSuccess) return fail(cuda_fail(ce, "range lims copy", __FILE__, __LINE__));
    if (total > 0) {
        range_decode_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(sorted, total, neg_zero ? 1 : 0, r->dist, r->ids);
        ctx().launches += 1;
        ce = cudaGetLastError();
        if (ce != cudaSuccess) return fail(cuda_fail(ce, "range decode", __FILE__, __LINE__));
    }
    *out = r;
    return VIX_OK;
}

int range_collect(int64_t nq, float radius, size_t& cap_hint, bool neg_zero, const std::function<int(const RangeOut&)>& scan,
                  vix_range_result** out, RangeInfo* info) {
    RangeKeys rk;
    VIX_TRY(range_collect_keys(nq, radius, cap_hint, scan, rk, info));
    return range_decode(nq, rk.lims.ptr, rk.sorted, rk.total, neg_zero, out);
}

}  // namespace vix

using namespace vix;

extern "C" {

int64_t vix_range_result_nq(const vix_range_result_t* r) { return r ? r->nq : 0; }

int64_t vix_range_result_total(const vix_range_result_t* r) { return r ? r->total : 0; }

int vix_range_result_get(const vix_range_result_t* r, int64_t* lims, float* dist, int64_t* ids) {
    VIX_TRY(ensure_device());
    VIX_REQUIRE(r, VIX_ERR_NULL_PTR, "vix_range_result_get: null result");
    cudaStream_t s = ctx().stream;
    bool host = false;
    if (lims) {
        VIX_CUDA(cudaMemcpyAsync(lims, r->lims, (size_t)(r->nq + 1) * 8, cudaMemcpyDefault, s));
        host = host || !is_device_ptr(lims);
    }
    if (dist && r->total) {
        VIX_CUDA(cudaMemcpyAsync(dist, r->dist, (size_t)r->total * 4, cudaMemcpyDefault, s));
        host = host || !is_device_ptr(dist);
    }
    if (ids && r->total) {
        VIX_CUDA(cudaMemcpyAsync(ids, r->ids, (size_t)r->total * 8, cudaMemcpyDefault, s));
        host = host || !is_device_ptr(ids);
    }
    return finish(host);
}

void vix_range_result_destroy(vix_range_result_t* r) {
    if (!r) return;
    cudaStreamSynchronize(ctx().stream);
    range_free(r);
}

}  // extern "C"
