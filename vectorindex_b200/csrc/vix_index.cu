// vix_index.cu -- device-resident index handles (Flat, IVF-Flat, IVF-PQ) and the fused IVF-PQ search.
//
// Search pipeline of an IVF-PQ index (the composition of /root/reference/docs/kernel-specs/
// DONE_22_adc_scan.md:831-881: ivf_select_nprobe -> pq_lut_residual_l2 -> adc_scan_u8 -> selectTopK
// -> mergeTopK), restructured for B200:
//
//   1. probe selection   probe_select_device (vix_scoring.cu) / the tcgen05 path (vix_gemm.cu)
//   2. locality order    queries sorted by their first probed list (one small radix sort)
//   3. fused scan        vix_ivfpq_scan.cu: query-only LUT + ADC over the probed lists + top-k
//
// This file owns the device-resident state: rows in add order (AoS codes, the reference's interchange
// format) and the scan layout derived from them (lists padded to whole chunks of 32 slots, codes
// rotated inside each group of 16 sub-quantisers, per-vector term t_x = ||r^||^2 + 2 <c, r^>).
#include "vix_common.cuh"
#include "vix_topk.cuh"
#include "vix_exact.cuh"
#include "vix_scan.cuh"
#include "vix_index.cuh"
#include "vix_range.cuh"
#include "vix_group.cuh"

#include <algorithm>
#include <new>
#include <stdio.h>
#include <stdlib.h>

using namespace vix;

namespace vix {

// ------------------------------------------------------------------------------------------------
// list building
// ------------------------------------------------------------------------------------------------
// slot_row[off[l] + r] = sorted_rows[off_raw[l] + r]
// Rows without a list (assignment outside [0, kc): the -1 of an all-NaN / all-+inf score row, IVFIndex.swift:376-435
// "guard best >= 0 else continue") carry the sort key kc, so they sort behind every list and are not placed.
__global__ void place_rows_kernel(const int32_t* __restrict__ sorted_rows, const int32_t* __restrict__ sorted_lists,
                                  int64_t n, int kc, const int64_t* __restrict__ off, const int64_t* __restrict__ off_raw,
                                  int32_t* __restrict__ slot_row) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int l = sorted_lists[i];
    if ((unsigned)l >= (unsigned)kc) return;
    slot_row[off[l] + (i - off_raw[l])] = sorted_rows[i];
}

// flag[0] += number of assignments outside [0, kc)
__global__ void count_invalid_assign_kernel(const int32_t* __restrict__ assign, int64_t n, int kc,
                                            unsigned long long* __restrict__ flag) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool bad = i < n && (unsigned)assign[i] >= (unsigned)kc;
    const unsigned ball = __ballot_sync(0xFFFFFFFFu, bad);
    if (ball && (threadIdx.x & 31) == 0) atomicAdd(flag, (unsigned long long)__popc(ball));
}

__global__ void sanitise_assign_kernel(const int32_t* __restrict__ assign, int64_t n, int kc, int32_t* __restrict__ keys) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { const int a = assign[i]; keys[i] = (unsigned)a < (unsigned)kc ? a : kc; }
}

// flag[0] += ids outside [0, 2^32 - 1) (the id half of a selection key; 0xFFFFFFFF is the empty key)
__global__ void count_invalid_ids_kernel(const int64_t* __restrict__ ids, int64_t n, unsigned long long* __restrict__ flag) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool bad = i < n && (ids[i] < 0 || ids[i] >= 0xFFFFFFFFLL);
    const unsigned ball = __ballot_sync(0xFFFFFFFFu, bad);
    if (ball && (threadIdx.x & 31) == 0) atomicAdd(flag, (unsigned long long)__popc(ball));
}

// number of assignments outside [0, kc) in a device array (synchronises the stream)
int count_invalid_assign(const int32_t* assign, int64_t n, int kc, unsigned long long* out) {
    *out = 0;
    if (n <= 0) return VIX_OK;
    Scratch<unsigned long long> flag;
    VIX_TRY(flag.alloc(1));
    cudaStream_t s = ctx().stream;
    VIX_CUDA(cudaMemsetAsync(flag.ptr, 0, 8, s));
    count_invalid_assign_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(assign, n, kc, flag.ptr);
    VIX_LAUNCH_CHECK();
    VIX_CUDA(cudaMemcpyAsync(out, flag.ptr, 8, cudaMemcpyDeviceToHost, s));
    VIX_CUDA(cudaStreamSynchronize(s));
    return VIX_OK;
}

int count_invalid_rows_device(const int32_t* assign, const int64_t* ids, int64_t n, int kc, unsigned long long* count_dev) {
    if (n <= 0) return VIX_OK;
    cudaStream_t s = ctx().stream;
    const unsigned grid = (unsigned)((n + 255) / 256);
    count_invalid_assign_kernel<<<grid, 256, 0, s>>>(assign, n, kc, count_dev);
    VIX_LAUNCH_CHECK();
    count_invalid_ids_kernel<<<grid, 256, 0, s>>>(ids, n, count_dev);
    VIX_LAUNCH_CHECK();
    return VIX_OK;
}

// Fill one slot: codes in the scan layout (vix_scan.cuh), id, t_x.  One warp per slot (lanes split the
// sub-quantisers).  rotated != 0: byte b of slot g holds sub-quantiser (b & ~15) | ((b ^ g) & 15), chunk-blocked.
__global__ void __launch_bounds__(256)
fill_slots_pq_kernel(const int32_t* __restrict__ slot_row, int64_t nslots, const uint8_t* __restrict__ codes,
                     const int64_t* __restrict__ ids, const int32_t* __restrict__ assign,
                     const float* __restrict__ coarse, const float* __restrict__ codebooks, int d, int m, int ks,
                     int rotated, int metric, uint8_t* __restrict__ slot_codes, int64_t* __restrict__ slot_ids,
                     float* __restrict__ slot_tx) {
    // ks = 16: packed nibbles (m / 2 bytes per row, plain AoS slots; never rotated)
    const int cb_ = ks == 16 ? m / 2 : m;
    const int lane = threadIdx.x & 31;
    const int64_t g = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (g >= nslots) return;
    const int row = slot_row[g];
    const int dsub = d / m;
    // rotated (fast) layout is also chunk-blocked: byte b of slot g lives at chunk * 32 m + (b / 16) * 512 + (g % 32) * 16 + b % 16
    constexpr int PS = 16;                             // bytes of a slot stored contiguously: one 128-bit load per group
    uint8_t* dst = rotated ? slot_codes + (g >> 5) * (int64_t)(32 * m) + (g & 31) * PS : slot_codes + g * (int64_t)cb_;
    const int cstride = rotated ? 32 * PS - PS : 0;    // extra offset per piece
    if (row < 0) {
        for (int b = lane; b < cb_; b += 32) dst[b + (b / PS) * cstride] = 0;
        if (lane == 0) { slot_ids[g] = -1; slot_tx[g] = 0.0f; }
        return;
    }
    const uint8_t* src = codes + (int64_t)row * cb_;
    const float* c = coarse + (int64_t)assign[row] * d;
    double acc = 0.0;
    for (int b = lane; b < cb_; b += 32) {
        const int j = rotated ? ((b & ~15) | ((b ^ (int)(g & 15)) & 15)) : b;
        dst[b + (b / PS) * cstride] = src[j];
    }
    if (metric == VIX_METRIC_L2) {
        for (int j = lane; j < m; j += 32) {
            const int code = ks == 16 ? ((j & 1) ? (src[j >> 1] >> 4) : (src[j >> 1] & 15)) : src[j];
            const float* cw = codebooks + ((size_t)j * ks + code) * dsub;
            const float* cj = c + (size_t)j * dsub;
            for (int e = 0; e < dsub; ++e) {
                double r = (double)cw[e];
                acc += r * r + 2.0 * (double)cj[e] * r;
            }
        }
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xFFFFFFFFu, acc, o);
    }
    if (lane == 0) { slot_ids[g] = ids[row]; slot_tx[g] = (float)acc; }
}

// The decode layout (vix_scan.cuh) from the AoS rows: one thread per 16-byte piece (chunk, group, thread t = 4 r + c of the
// decoding warp), which gathers four bytes of each of the slots r + 8 v and writes them with one coalesced store.
__global__ void __launch_bounds__(256)
fill_tc_codes_kernel(const int32_t* __restrict__ slot_row, int64_t npieces, const uint8_t* __restrict__ codes, int m,
                     uint4* __restrict__ tc_codes) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npieces) return;
    const int64_t ch = i / (2 * m);
    const int rem = (int)(i - ch * 2 * m), grp = rem >> 5, r = (rem >> 2) & 7, c = rem & 3;
    uint32_t w[4];
#pragma unroll
    for (int v = 0; v < 4; ++v) {
        const int row = slot_row[ch * 32 + r + 8 * v];
        w[v] = 0;
        if (row >= 0) {
            const uint8_t* src = codes + (int64_t)row * m + 16 * grp + c;
#pragma unroll
            for (int s = 0; s < 4; ++s) w[v] |= (uint32_t)src[4 * (s ^ (r & 3))] << (8 * s);
        }
    }
    tc_codes[i] = make_uint4(w[0], w[1], w[2], w[3]);
}

__global__ void fill_slots_flat_kernel(const int32_t* __restrict__ slot_row, int64_t nslots,
                                       const float* __restrict__ vecs, const int64_t* __restrict__ ids, int d,
                                       float* __restrict__ slot_vecs, int64_t* __restrict__ slot_ids) {
    const int lane = threadIdx.x & 31;
    const int64_t g = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (g >= nslots) return;
    const int row = slot_row[g];
    for (int e = lane; e < d; e += 32) slot_vecs[g * (int64_t)d + e] = row >= 0 ? vecs[(int64_t)row * d + e] : 0.0f;
    if (lane == 0) slot_ids[g] = row >= 0 ? ids[row] : -1;
}

int build_lists(vix_index* h) {
    const int kc = h->kc;
    const int64_t n = h->n;
    cudaStream_t s = ctx().stream;
    VIX_TRY(h->list_len.resize((size_t)kc, false));
    VIX_TRY(h->list_off.resize((size_t)kc + 1, false));
    Scratch<int64_t> off_raw;
    VIX_TRY(off_raw.alloc((size_t)kc + 1));
    h->align = (h->p.kind == VIX_INDEX_IVF_PQ) ? scan_layout(h->p.m).align : 32;
    VIX_TRY(key_offsets(h->assign.ptr, n, kc, h->list_len.ptr, h->list_off.ptr, h->align, off_raw.ptr));
    int64_t nslots = 0;
    VIX_CUDA(cudaMemcpyAsync(&nslots, h->list_off.ptr + kc, 8, cudaMemcpyDeviceToHost, s));
    VIX_CUDA(cudaStreamSynchronize(s));
    VIX_REQUIRE(nslots < 0x7FFFFFFFLL, VIX_ERR_INVALID_PARAM, "index shard limited to 2^31 - 1 list slots (rows + list padding)");
    h->nslots = nslots;
    VIX_TRY(h->slot_row.resize((size_t)nslots, false));
    VIX_TRY(h->slot_ids.resize((size_t)nslots, false));
    if (nslots > 0) VIX_CUDA(cudaMemsetAsync(h->slot_row.ptr, 0xFF, (size_t)nslots * 4, s));
    if (n > 0) {
        // stable sort of rows by list: radix sort over the list-id bits.  Rows without a list (assignment outside
        // [0, kc)) get the key kc in a sanitised copy of the keys, made only when such rows exist.
        unsigned long long invalid = 0;
        VIX_TRY(count_invalid_assign(h->assign.ptr, n, kc, &invalid));
        Scratch<int32_t> keys;
        const int32_t* list_keys = h->assign.ptr;
        if (invalid) {
            VIX_TRY(keys.alloc((size_t)n));
            sanitise_assign_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(h->assign.ptr, n, kc, keys.ptr);
            VIX_LAUNCH_CHECK();
            list_keys = keys.ptr;
        }
        Scratch<int32_t> rows_out, lists_out;
        VIX_TRY(rows_out.alloc((size_t)n));
        VIX_TRY(lists_out.alloc((size_t)n));
        VIX_TRY(order_by_key(list_keys, n, kc + 1, rows_out.ptr, lists_out.ptr));   // keys 0 .. kc
        place_rows_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(rows_out.ptr, lists_out.ptr, n, kc, h->list_off.ptr,
                                                                     off_raw.ptr, h->slot_row.ptr);
        VIX_LAUNCH_CHECK();
    }
    if (h->p.kind == VIX_INDEX_IVF_PQ) {
        const int m = h->p.m;
        const int rotated = (scan_layout(m).fast && h->p.ks == 256) ? 1 : 0;
        VIX_TRY(h->slot_codes.resize((size_t)nslots * h->code_bytes() + 16, false));
        VIX_TRY(h->slot_tx.resize((size_t)nslots, false));
        const bool tc = tc_codes_shape(h->p.metric, m, h->p.ks, h->p.d / m);
        if (tc) VIX_TRY(h->tc_codes.resize((size_t)nslots * m, false));
        else h->tc_codes.free_all();
        if (nslots > 0) {
            int64_t threads = nslots * 32;
            fill_slots_pq_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, s>>>(
                h->slot_row.ptr, nslots, h->codes.ptr, h->ids.ptr, h->assign.ptr, h->coarse.ptr, h->codebooks.ptr,
                h->p.d, m, h->p.ks, rotated, h->p.metric, h->slot_codes.ptr, h->slot_ids.ptr, h->slot_tx.ptr);
            VIX_LAUNCH_CHECK();
            if (tc) {
                const int64_t npieces = nslots * m / 16;
                fill_tc_codes_kernel<<<(unsigned)((npieces + 255) / 256), 256, 0, s>>>(
                    h->slot_row.ptr, npieces, h->codes.ptr, m, reinterpret_cast<uint4*>(h->tc_codes.ptr));
                VIX_LAUNCH_CHECK();
            }
        }
    } else {
        VIX_TRY(h->slot_vecs.resize((size_t)nslots * h->p.d, false));
        if (nslots > 0) {
            int64_t threads = nslots * 32;
            fill_slots_flat_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, s>>>(
                h->slot_row.ptr, nslots, h->vecs.ptr, h->ids.ptr, h->p.d, h->slot_vecs.ptr, h->slot_ids.ptr);
            VIX_LAUNCH_CHECK();
        }
    }
    h->dirty = false;
    return VIX_OK;
}

// ------------------------------------------------------------------------------------------------
// query order for the scan: work item -> query, sorted by first probed list (L2 locality)
// ------------------------------------------------------------------------------------------------
// key of a query = the first probed list that holds vectors HERE (on a shard most probes belong to other ranks), kc if
// none does; one warp per query.  The keys are list ids, so the order is a COUNTING sort written here (histogram over
// the kc + 1 keys -> exclusive scan -> scatter), three small kernels, no library call on the search path.
__global__ void first_probe_kernel(const int32_t* __restrict__ probes, int64_t nq, int nprobe,
                                   const int32_t* __restrict__ list_len, int kc, int32_t* __restrict__ keys,
                                   int32_t* __restrict__ hist) {
    const int lane = threadIdx.x & 31;
    const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (i >= nq) return;
    int key = kc;
    for (int base = 0; base < nprobe; base += 32) {
        const int p = base + lane;
        const int l = p < nprobe ? __ldg(probes + i * nprobe + p) : -1;
        const bool here = (unsigned)l < (unsigned)kc && __ldg(list_len + l) > 0;
        const unsigned ball = __ballot_sync(0xFFFFFFFFu, here);
        if (ball) { key = __shfl_sync(0xFFFFFFFFu, l, __ffs(ball) - 1); break; }
    }
    if (lane == 0) { keys[i] = key; if (hist) atomicAdd(hist + key, 1); }
}

// single CTA: hist[0, n) -> exclusive prefix sums in place (each thread owns a contiguous run of bins)
__global__ void __launch_bounds__(1024)
exclusive_scan_kernel(int32_t* __restrict__ hist, int n) {
    __shared__ int s_part[1024];
    const int per = (n + 1023) / 1024;
    const int b = threadIdx.x * per, e = min(b + per, n);
    int sum = 0;
    for (int i = b; i < e; ++i) sum += hist[i];
    s_part[threadIdx.x] = sum;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {
        const int v = (int)threadIdx.x >= o ? s_part[threadIdx.x - o] : 0;
        __syncthreads();
        s_part[threadIdx.x] += v;
        __syncthreads();
    }
    int run = s_part[threadIdx.x] - sum;
    for (int i = b; i < e; ++i) { const int v = hist[i]; hist[i] = run; run += v; }
}

// order[cursor[key]++] = query (queries with the same key land next to each other; their mutual order is free)
__global__ void scatter_order_kernel(const int32_t* __restrict__ keys, int64_t nq, int32_t* __restrict__ cursor,
                                     int32_t* __restrict__ order) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nq) order[atomicAdd(cursor + keys[i], 1)] = (int32_t)i;
}

// Batches of up to 32 k queries: the position of query i in the order is its RANK -- the number of queries with a smaller
// key, or the same key and a smaller index -- counted directly (nq^2 comparisons through shared-memory tiles: 10^8 for 10 k
// queries, a few microseconds; stable and deterministic).  The histogram path below serves larger batches.
__global__ void __launch_bounds__(256)
rank_order_kernel(const int32_t* __restrict__ keys, int nq, int32_t* __restrict__ order) {
    __shared__ int32_t s_k[256];
    const int i = blockIdx.x * 256 + threadIdx.x;
    const int mine = i < nq ? keys[i] : 0x7FFFFFFF;
    int rank = 0;
    for (int base = 0; base < nq; base += 256) {
        const int j = base + threadIdx.x;
        __syncthreads();
        s_k[threadIdx.x] = j < nq ? keys[j] : 0x7FFFFFFF;
        __syncthreads();
        const int lim = min(256, nq - base);
#pragma unroll 8
        for (int t = 0; t < lim; ++t) {
            const int k = s_k[t];
            rank += (k < mine || (k == mine && base + t < i)) ? 1 : 0;
        }
    }
    if (i < nq) order[rank] = i;
}

static int query_order(const int32_t* probes, int64_t nq, int nprobe, const int32_t* list_len, int kc,
                       Scratch<int32_t>& order) {
    cudaStream_t s = ctx().stream;
    Scratch<int32_t> keys, hist;
    VIX_TRY(keys.alloc((size_t)nq));
    VIX_TRY(order.alloc((size_t)nq));
    if (nq <= 32768) {
        first_probe_kernel<<<(unsigned)((nq * 32 + 255) / 256), 256, 0, s>>>(probes, nq, nprobe, list_len, kc, keys.ptr, nullptr);
        VIX_LAUNCH_CHECK();
        rank_order_kernel<<<(unsigned)((nq + 255) / 256), 256, 0, s>>>(keys.ptr, (int)nq, order.ptr);
        VIX_LAUNCH_CHECK();
        return VIX_OK;
    }
    VIX_TRY(hist.alloc((size_t)kc + 1));
    VIX_CUDA(cudaMemsetAsync(hist.ptr, 0, ((size_t)kc + 1) * 4, s));
    first_probe_kernel<<<(unsigned)((nq * 32 + 255) / 256), 256, 0, s>>>(probes, nq, nprobe, list_len, kc, keys.ptr, hist.ptr);
    VIX_LAUNCH_CHECK();
    exclusive_scan_kernel<<<1, 1024, 0, s>>>(hist.ptr, kc + 1);
    VIX_LAUNCH_CHECK();
    scatter_order_kernel<<<(unsigned)((nq + 255) / 256), 256, 0, s>>>(keys.ptr, nq, hist.ptr, order.ptr);
    VIX_LAUNCH_CHECK();
    return VIX_OK;
}

// Cosine candidate distance of the IVF-Flat scan (DistanceUtils.swift:22-38): 1 - clamp(dot / sqrt(|a|^2 |b|^2)), and 1
// when the denominator is not above ulpOfOne.  The dot product and the sums of squares are VectorCore's there (source not
// in the reference tree): tolerance parity (1e-5), like the other candidate distances.
__device__ __forceinline__ float seq_sumsq(const float* v, int d) {
    float s = 0.0f;
    for (int e = 0; e < d; ++e) s = fadd(s, fmul(v[e], v[e]));
    return s;
}
__device__ __forceinline__ float cosine_distance(float dot, float amag2, float bmag2) {
    const float denom = __fsqrt_rn(fmul(amag2, bmag2));
    if (!(denom > 1.1920929e-07f)) return 1.0f;
    const float sim = fmaxf(-1.0f, fminf(1.0f, __fdiv_rn(dot, denom)));
    return fsub(1.0f, sim);
}

// Cosine list assignment and probe selection (IVFIndex.swift:376-435, 905-927): the guarded CentroidBatchScore block of a
// tile of rows, then per row the first minimum (strict <, ascending list id) / the nprobe best by (score, list id).
__global__ void __launch_bounds__(256)
row_argmin_kernel(const float* __restrict__ scores, int64_t rows, int kc, int32_t* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (r >= rows) return;
    const float* row = scores + r * (int64_t)kc;
    float bs = INFINITY;
    int bi = 0x7fffffff;
    for (int c = lane; c < kc; c += 32) {
        const float v = row[c];
        if (v < bs) { bs = v; bi = c; }
    }
    for (int o = 16; o > 0; o >>= 1) {
        const float os = __shfl_xor_sync(0xFFFFFFFFu, bs, o);
        const int oi = __shfl_xor_sync(0xFFFFFFFFu, bi, o);
        if (os < bs || (os == bs && oi < bi)) { bs = os; bi = oi; }
    }
    if (lane == 0) out[r] = bi == 0x7fffffff ? -1 : bi;
}

// rows per tile of the materialised score block: at most 64 M scores (256 MB)
static int64_t cosine_tile_rows(int64_t n, int kc) {
    int64_t t = (64LL << 20) / (kc > 0 ? kc : 1);
    if (t < 1) t = 1;
    if (t > 4096) t = 4096;                                     // the reference's tile (IVFIndex.swift:380)
    return t < n ? t : n;
}

static int assign_cosine_device(const float* x, int64_t n, int d, const float* coarse, int kc, const float* cnorm,
                                int32_t* assign) {
    if (n == 0) return VIX_OK;
    const int64_t tile = cosine_tile_rows(n, kc);
    Scratch<float> scores;
    VIX_TRY(scores.alloc((size_t)tile * kc));
    for (int64_t b = 0; b < n; b += tile) {
        const int64_t cnt = n - b < tile ? n - b : tile;
        VIX_TRY(centroid_batch_score_cosine_device(x + (size_t)b * d, cnt, coarse, kc, d, cnorm, scores.ptr));
        row_argmin_kernel<<<(unsigned)((cnt * 32 + 255) / 256), 256, 0, ctx().stream>>>(scores.ptr, cnt, kc, assign + b);
        VIX_LAUNCH_CHECK();
    }
    return VIX_OK;
}

static int probe_select_cosine_device(const float* q, int64_t nq, const float* coarse, int kc, int d, const float* cnorm,
                                      int nprobe, int32_t* out_idx) {
    if (nq == 0) return VIX_OK;
    const int64_t tile = cosine_tile_rows(nq, kc);
    Scratch<float> scores;
    VIX_TRY(scores.alloc((size_t)tile * kc));
    for (int64_t b = 0; b < nq; b += tile) {
        const int64_t cnt = nq - b < tile ? nq - b : tile;
        VIX_TRY(centroid_batch_score_cosine_device(q + (size_t)b * d, cnt, coarse, kc, d, cnorm, scores.ptr));
        VIX_TRY(row_select_device(scores.ptr, cnt, kc, nprobe, nullptr, out_idx + (size_t)b * nprobe, nullptr));
    }
    return VIX_OK;
}

// list assignment under the index's metric (the three callers below): euclidean => _vi_km12_assignAOS
// (IVFIndex.swift:362-375); dot product / cosine => first minimum of the CentroidBatchScore row (:376-435)
int assign_lists_device(vix_index_t* h, const float* x, int64_t n, int32_t* assign) {
    const int d = h->p.d;
    if (h->p.metric == VIX_METRIC_L2) return ivf_assign_auto_device(x, n, d, h->coarse.ptr, h->kc, assign, nullptr);
    if (h->p.metric == VIX_METRIC_COSINE) return assign_cosine_device(x, n, d, h->coarse.ptr, h->kc, h->coarse_norms.ptr, assign);
    return ivf_assign_metric_device(x, n, d, h->coarse.ptr, h->kc, h->p.metric, nullptr, assign);
}

// IVF-Flat candidate scan (IVFIndex.swift:1023-1039): exact distance per candidate of the probed
// lists in the reference's order (Direct16 / Ip4), API distance (sqrt / negate), (distance, id) order.
__global__ void __launch_bounds__(256)
ivfflat_scan_kernel(const float* __restrict__ queries, int64_t nq, int d, const int32_t* __restrict__ probes,
                    int nprobe, const int64_t* __restrict__ list_off, const int32_t* __restrict__ list_len, int kc,
                    const float* __restrict__ slot_vecs, const int64_t* __restrict__ slot_ids, int metric, int k,
                    int P, const uint64_t* __restrict__ filter, int64_t filter_cap, int filter_deny,
                    float* __restrict__ out_dist, int64_t* __restrict__ out_ids) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    u64* keys = reinterpret_cast<u64*>(smem_raw);
    float* s_q = reinterpret_cast<float*>(keys + P);
    __shared__ int s_cnt;
    __shared__ u64 s_thr;
    for (int64_t qi = blockIdx.x; qi < nq; qi += gridDim.x) {
        __syncthreads();
        for (int e = threadIdx.x; e < d; e += blockDim.x) s_q[e] = queries[qi * (int64_t)d + e];
        BlockQueue q{keys, &s_cnt, &s_thr, k, P};
        q.init();
        const float qmag2 = (metric == VIX_METRIC_COSINE) ? seq_sumsq(s_q, d) : 0.0f;
        for (int p = 0; p < nprobe; ++p) {
            const int l = probes[qi * (int64_t)nprobe + p];
            if ((unsigned)l >= (unsigned)kc) continue;           // -1 padding, or an id no list has
            const int64_t b = list_off[l];
            const int len = list_len[l];
            for (int base = 0; base < len; base += blockDim.x) {
                q.flush_if_needed(blockDim.x);
                const int i = base + threadIdx.x;
                if (i < len && (!filter || id_filter_pass(filter, filter_cap, filter_deny, slot_ids[b + i]))) {
                    const float* v = slot_vecs + (b + i) * (int64_t)d;
                    float dist;
                    if (metric == VIX_METRIC_L2) dist = __fsqrt_rn(exact_pair<SpecDirect16L2>(s_q, v, d));
                    else if (metric == VIX_METRIC_IP) dist = -exact_pair<SpecIp4>(s_q, v, d);
                    else dist = cosine_distance(exact_pair<SpecIp4>(s_q, v, d), qmag2, seq_sumsq(v, d));
                    q.push(make_key(dist, (uint32_t)slot_ids[b + i], 0));
                }
            }
        }
        q.flush();
        for (int i = threadIdx.x; i < k; i += blockDim.x) {
            const u64 key = keys[i];
            const size_t o = (size_t)qi * k + i;
            if (key == kEmptyKey) { out_dist[o] = __int_as_float(0x7fc00000); out_ids[o] = -1; }
            else { out_dist[o] = key_score(key, 0); out_ids[o] = (int64_t)key_id(key); }
        }
    }
}

// Range variant of the candidate scan: the same candidates and arithmetic, every candidate whose API distance is within the
// radius appended to the range output (vix_range.cuh) with a per-query count.
__global__ void __launch_bounds__(256)
ivfflat_range_kernel(const float* __restrict__ queries, int64_t nq, int d, const int32_t* __restrict__ probes,
                     int nprobe, const int64_t* __restrict__ list_off, const int32_t* __restrict__ list_len, int kc,
                     const float* __restrict__ slot_vecs, const int64_t* __restrict__ slot_ids, int metric,
                     const uint64_t* __restrict__ filter, int64_t filter_cap, int filter_deny, RangeOut out) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float* s_q = reinterpret_cast<float*>(smem_raw);
    __shared__ int s_cnt;
    for (int64_t qi = blockIdx.x; qi < nq; qi += gridDim.x) {
        __syncthreads();
        for (int e = threadIdx.x; e < d; e += blockDim.x) s_q[e] = queries[qi * (int64_t)d + e];
        if (threadIdx.x == 0) s_cnt = 0;
        __syncthreads();
        const float qmag2 = (metric == VIX_METRIC_COSINE) ? seq_sumsq(s_q, d) : 0.0f;
        const uint32_t qbound = out.bound ? out.bound[qi] : 0xFFFFFFFFu;
        for (int p = 0; p < nprobe; ++p) {
            const int l = probes[qi * (int64_t)nprobe + p];
            if ((unsigned)l >= (unsigned)kc) continue;           // -1 padding, or an id no list has
            const int64_t b = list_off[l];
            const int len = list_len[l];
            for (int base = 0; base < len; base += blockDim.x) {
                const int i = base + threadIdx.x;
                bool pass = false;
                u64 key = 0;
                if (i < len && (!filter || id_filter_pass(filter, filter_cap, filter_deny, slot_ids[b + i]))) {
                    const float* v = slot_vecs + (b + i) * (int64_t)d;
                    float dist;
                    if (metric == VIX_METRIC_L2) dist = __fsqrt_rn(exact_pair<SpecDirect16L2>(s_q, v, d));
                    else if (metric == VIX_METRIC_IP) dist = -exact_pair<SpecIp4>(s_q, v, d);
                    else dist = cosine_distance(exact_pair<SpecIp4>(s_q, v, d), qmag2, seq_sumsq(v, d));
                    key = make_key(dist, (uint32_t)slot_ids[b + i], 0);
                    pass = out.bound ? (uint32_t)(key >> 32) <= qbound : dist <= out.radius;
                }
                const unsigned ball = __ballot_sync(0xFFFFFFFFu, pass);
                if (ball) {
                    range_append(out, ball, pass, key, (uint32_t)qi);
                    if ((threadIdx.x & 31) == 0) atomicAdd(&s_cnt, __popc(ball));
                }
            }
        }
        __syncthreads();
        if (threadIdx.x == 0) out.counts[qi] = (unsigned long long)s_cnt;
    }
}

// ------------------------------------------------------------------------------------------------
// host-side index logic
// ------------------------------------------------------------------------------------------------
// flat / linear-scan pre-filter: bit r of the mask set <=> row r fails the id filter (64 rows per thread)
__global__ void filter_row_mask_kernel(const int64_t* __restrict__ ids, int64_t n, const uint64_t* __restrict__ filter,
                                       int64_t filter_cap, int filter_deny, uint64_t* __restrict__ mask) {
    const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (w * 64 >= n) return;
    uint64_t bits = 0;
    for (int b = 0; b < 64; ++b) {
        const int64_t r = w * 64 + b;
        if (r < n && !id_filter_pass(filter, filter_cap, filter_deny, ids[r])) bits |= 1ull << b;
    }
    mask[w] = bits;
}

__global__ void gather_ids_kernel(const int64_t* __restrict__ rows, const int64_t* __restrict__ ids,
                                  int64_t* __restrict__ out, int64_t n) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = rows[i] >= 0 ? ids[rows[i]] : -1;
}

// codebooks [m][ks][dsub] -> code-major copy [ks][m][dsub] (coalesced LUT build of the scan)
__global__ void transpose_codebooks_kernel(const float* __restrict__ cb, int m, int ks, int dsub, float* __restrict__ out) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (int64_t)m * ks * dsub) return;
    const int t = (int)(e % dsub);
    const int64_t r = e / dsub;
    const int j = (int)(r % m), c = (int)(r / m);
    out[e] = cb[((size_t)j * ks + c) * dsub + t];
}

static int update_codebooks_t(vix_index* h) {
    const int m = h->p.m, ks = h->p.ks, dsub = h->p.d / m;
    const int64_t total = (int64_t)m * ks * dsub;
    VIX_TRY(h->codebooks_t.resize((size_t)total, false));
    transpose_codebooks_kernel<<<(unsigned)((total + 255) / 256), 256, 0, ctx().stream>>>(h->codebooks.ptr, m, ks, dsub,
                                                                                          h->codebooks_t.ptr);
    VIX_LAUNCH_CHECK();
    if (tc_decode_table_shape(m, ks, dsub)) {
        VIX_TRY(h->tc_table.resize(kTcTableWords, false));
        VIX_TRY(h->tc_meta.resize(4, false));
        VIX_TRY(tc_decode_table(h->codebooks.ptr, m, h->tc_table.ptr, h->tc_meta.ptr));
    } else {
        h->tc_table.free_all();
        h->tc_meta.free_all();
    }
    return VIX_OK;
}

// device-resident ids (the multi-GPU build hands over what the exchange delivered): same contract, checked by a kernel
static int check_ids_device(const int64_t* ids, int64_t n) {
    if (n <= 0) return VIX_OK;
    Scratch<unsigned long long> flag;
    VIX_TRY(flag.alloc(1));
    cudaStream_t s = ctx().stream;
    VIX_CUDA(cudaMemsetAsync(flag.ptr, 0, 8, s));
    count_invalid_ids_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(ids, n, flag.ptr);
    VIX_LAUNCH_CHECK();
    unsigned long long bad = 0;
    VIX_CUDA(cudaMemcpyAsync(&bad, flag.ptr, 8, cudaMemcpyDeviceToHost, s));
    VIX_CUDA(cudaStreamSynchronize(s));
    VIX_REQUIRE(bad == 0, VIX_ERR_INVALID_PARAM,
                "ids must lie in [0, 2^32 - 1) (the reference's TopK id type is Int32, TopK.swift:59); %llu of %lld device-resident "
                "ids do not", bad, (long long)n);
    return VIX_OK;
}

static int check_ids_host(const int64_t* ids, int64_t n) {
    for (int64_t i = 0; i < n; ++i)
        VIX_REQUIRE(ids[i] >= 0 && ids[i] < 0xFFFFFFFFLL, VIX_ERR_INVALID_PARAM,
                    "ids must lie in [0, 2^32 - 1) (the reference's TopK id type is Int32, TopK.swift:59); got %lld",
                    (long long)ids[i]);
    return VIX_OK;
}

// An IVF-Flat index may hold vectors before it has a coarse quantiser (the reference's insert -> optimize() -> search,
// IVFIndex.swift:279-451; until then searches are linear scans, :820-832): once centroids exist, every stored row gets
// its list.
static int assign_stored_rows(vix_index* h) {
    if (h->p.kind != VIX_INDEX_IVF_FLAT || h->n == 0) return VIX_OK;
    VIX_TRY(h->assign.resize((size_t)h->n));
    const int64_t chunk = 1 << 20;
    for (int64_t b = 0; b < h->n; b += chunk) {
        const int64_t cn = (h->n - b < chunk) ? (h->n - b) : chunk;
        VIX_TRY(assign_lists_device(h, h->vecs.ptr + (size_t)b * h->p.d, cn, h->assign.ptr + b));
    }
    h->dirty = true;
    return VIX_OK;
}

// residual PQ codes of rows whose lists are known: ks = 256 => pq_encode_residual_u8_f32 with default opts => the C
// ..._with_csq entry (PQEncode.swift:247-286); ks = 16 => cpq_encode_residual_u4_f32 (direct L2, packed nibbles,
// pq_encode.c:692-739)
int encode_rows_device(vix_index* h, const float* x, int64_t n, const int32_t* assign, uint8_t* codes) {
    if (h->p.ks == 16)
        return pq_encode_device(x, n, h->p.d, h->p.m, 16, h->codebooks.ptr, nullptr, h->coarse.ptr, assign, codes, 0, PQ_LAYOUT_AOS,
                                64, 8, 1);
    return pq_encode_device(x, n, h->p.d, h->p.m, h->p.ks, h->codebooks.ptr, h->cb_norms.ptr, h->coarse.ptr, assign, codes, 1,
                            PQ_LAYOUT_AOS, 64, 8, 0);
}

static int index_add_locked(vix_index* h, const float* x, const int64_t* ids, int64_t n) {
    const int d = h->p.d;
    cudaStream_t s = ctx().stream;
    if (n == 0) return VIX_OK;
    VIX_REQUIRE(h->n + n < 0x7FFFFFFFLL, VIX_ERR_INVALID_PARAM, "index shard limited to 2^31 - 1 rows");
    if (h->p.kind == VIX_INDEX_IVF_PQ) {
        VIX_REQUIRE(h->has_coarse, VIX_ERR_NOT_TRAINED, "index_add: coarse quantiser not trained / set");
        VIX_REQUIRE(h->has_pq, VIX_ERR_NOT_TRAINED, "index_add: PQ codebooks not trained / set");
    }
    if (ids) VIX_TRY(is_device_ptr(ids) ? check_ids_device(ids, n) : check_ids_host(ids, n));
    if (!ids) VIX_REQUIRE(h->next_auto_id + n < 0xFFFFFFFFLL, VIX_ERR_INVALID_PARAM, "automatic ids exceed 2^32 - 1");

    const int64_t n0 = h->n;
    VIX_TRY(h->ids.resize((size_t)(n0 + n)));
    if (ids) VIX_CUDA(cudaMemcpyAsync(h->ids.ptr + n0, ids, (size_t)n * 8, cudaMemcpyDefault, s));
    else {
        // (after a removal the count no longer names an unused id: automatic ids continue from the last one handed out)
        VIX_TRY(iota<int64_t>(h->ids.ptr + n0, n, h->next_auto_id));
    }

    if (h->p.kind == VIX_INDEX_FLAT || h->p.kind == VIX_INDEX_IVF_FLAT) {
        VIX_TRY(h->vecs.resize((size_t)(n0 + n) * d));
        VIX_CUDA(cudaMemcpyAsync(h->vecs.ptr + (size_t)n0 * d, x, (size_t)n * d * 4, cudaMemcpyDefault, s));
    }
    if (h->p.kind != VIX_INDEX_FLAT && h->has_coarse) {          // (IVF-Flat without centroids: rows wait for optimize())
        VIX_TRY(h->assign.resize((size_t)(n0 + n)));
        if (h->p.kind == VIX_INDEX_IVF_PQ) VIX_TRY(h->codes.resize((size_t)(n0 + n) * h->code_bytes()));
        // chunked so that host inputs of any size stage through a bounded device buffer
        const int64_t chunk = 1 << 20;
        Scratch<float> stage;
        const bool host_x = !is_device_ptr(x);
        if (host_x && h->p.kind == VIX_INDEX_IVF_PQ) VIX_TRY(stage.alloc((size_t)(n < chunk ? n : chunk) * d));
        for (int64_t b = 0; b < n; b += chunk) {
            const int64_t cn = (n - b < chunk) ? (n - b) : chunk;
            const float* xc;
            if (h->p.kind == VIX_INDEX_IVF_FLAT) xc = h->vecs.ptr + (size_t)(n0 + b) * d;
            else if (host_x) {
                VIX_CUDA(cudaMemcpyAsync(stage.ptr, x + (size_t)b * d, (size_t)cn * d * 4, cudaMemcpyHostToDevice, s));
                xc = stage.ptr;
            } else xc = x + (size_t)b * d;
            int32_t* ac = h->assign.ptr + n0 + b;
            // list assignment: euclidean => _vi_km12_assignAOS (IVFIndex.swift:362-375);
            // dot product => first-min of the CentroidBatchScore row (IVFIndex.swift:376-435)
            VIX_TRY(assign_lists_device(h, xc, cn, ac));
            if (h->p.kind == VIX_INDEX_IVF_PQ) {
                // a row whose scores are all NaN has no list (-1): the residual encoder must not read coarse[-1]
                unsigned long long invalid = 0;
                VIX_TRY(count_invalid_assign(ac, cn, h->kc, &invalid));
                if (invalid) { h->ids.size = (size_t)n0; h->assign.size = (size_t)n0; h->codes.size = (size_t)n0 * h->code_bytes(); }
                VIX_REQUIRE(invalid == 0, VIX_ERR_INVALID_PARAM,
                            "index_add: %llu rows have no nearest list (NaN components?); nothing was added", invalid);
                // pq_encode_residual_u8_f32 with default opts => C ..._with_csq (PQEncode.swift:247-286)
                VIX_TRY(encode_rows_device(h, xc, cn, ac, h->codes.ptr + (size_t)(n0 + b) * h->code_bytes()));
            }
        }
    }
    h->n = n0 + n;
    h->next_auto_id += n;
    h->dirty = true;
    return finish(true);
}

// ------------------------------------------------------------------------------------------------
// removal: compaction of the add-order rows.  The lists and the decode layout are derived from these rows, so they are
// only marked dirty here and build_lists() rebuilds them, as after an add.
// ------------------------------------------------------------------------------------------------
// ids in [0, 2^32 - 1) (checked): the low 32 bits are the whole id, so the sort key is 4 bytes whatever the ids are
__global__ void ids_to_keys_kernel(const int64_t* __restrict__ ids, int64_t n, uint32_t* __restrict__ keys) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) keys[i] = (uint32_t)ids[i];
}

// keep[i] = 0 when the id of row i is in the sorted set (binary search), 1 otherwise; keep[n] = 0 closes the scan
__global__ void mark_removed_kernel(const int64_t* __restrict__ row_ids, int64_t n, const uint32_t* __restrict__ sorted,
                                    int64_t ns, int32_t* __restrict__ keep) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n) return;
    if (i == n) { keep[n] = 0; return; }
    const uint32_t id = (uint32_t)row_ids[i];
    int64_t lo = 0, hi = ns;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (__ldg(sorted + mid) < id) lo = mid + 1; else hi = mid;
    }
    keep[i] = (lo < ns && __ldg(sorted + lo) == id) ? 0 : 1;
}

// dst row pos[r] = src row r for every kept row; rows of w units U, one thread per unit (reads coalesced, writes in runs)
template <typename U>
__global__ void __launch_bounds__(256)
compact_rows_kernel(const U* __restrict__ src, int64_t n, int w, const int32_t* __restrict__ keep,
                    const int32_t* __restrict__ pos, U* __restrict__ dst) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t units = n * w;
    if (i >= units) return;
    const int64_t row = units <= 0xFFFFFFFFLL ? (int64_t)((uint32_t)i / (uint32_t)w) : i / w;
    if (__ldg(keep + row)) dst[(int64_t)__ldg(pos + row) * w + (i - row * w)] = src[i];
}

template <typename U>
static int launch_compact(const void* src, int64_t n, int64_t row_bytes, const int32_t* keep, const int32_t* pos, void* dst) {
    const int w = (int)(row_bytes / (int64_t)sizeof(U));
    const int64_t blocks = (n * w + 255) / 256;
    compact_rows_kernel<U><<<(unsigned)blocks, 256, 0, ctx().stream>>>(static_cast<const U*>(src), n, w, keep, pos,
                                                                        static_cast<U*>(dst));
    VIX_LAUNCH_CHECK();
    return VIX_OK;
}

// the kept rows of one add-order array (row_bytes per row) into an exactly sized new array, swapped in
template <typename T>
static int compact_array(DevBuf<T>& buf, int64_t n, int64_t row_elems, int64_t kept, const int32_t* keep, const int32_t* pos) {
    if (kept == 0) { buf.size = 0; return VIX_OK; }
    const int64_t row_bytes = row_elems * (int64_t)sizeof(T);
    T* out = nullptr;
    VIX_CUDA(cudaMalloc(reinterpret_cast<void**>(&out), (size_t)(kept * row_bytes)));
    int rc;
    if (row_bytes % 16 == 0) rc = launch_compact<uint4>(buf.ptr, n, row_bytes, keep, pos, out);         // (cudaMalloc: 256 B aligned)
    else if (row_bytes % 8 == 0) rc = launch_compact<uint2>(buf.ptr, n, row_bytes, keep, pos, out);
    else if (row_bytes % 4 == 0) rc = launch_compact<uint32_t>(buf.ptr, n, row_bytes, keep, pos, out);
    else if (row_bytes % 2 == 0) rc = launch_compact<uint16_t>(buf.ptr, n, row_bytes, keep, pos, out);
    else rc = launch_compact<uint8_t>(buf.ptr, n, row_bytes, keep, pos, out);
    cudaError_t e = rc == VIX_OK ? cudaStreamSynchronize(ctx().stream) : cudaSuccess;
    if (rc != VIX_OK || e != cudaSuccess) { cudaFree(out); if (rc != VIX_OK) return rc; VIX_CUDA(e); }
    buf.adopt(out, (size_t)(kept * row_elems));
    return VIX_OK;
}

static int index_remove_locked(vix_index* h, const int64_t* ids, int64_t n, int64_t* removed) {
    *removed = 0;
    if (n == 0) return VIX_OK;
    // the id contract of add, checked before anything changes
    const bool dev_ids = is_device_ptr(ids);
    VIX_TRY(dev_ids ? check_ids_device(ids, n) : check_ids_host(ids, n));
    const int64_t rows = h->n;
    if (rows == 0) return VIX_OK;
    cudaStream_t s = ctx().stream;
    In<int64_t> did;
    VIX_TRY(did.stage(ids, (size_t)n));
    // 1. the requested ids, sorted (4-byte keys: scratch independent of the id range)
    Scratch<uint32_t> keys_in, keys;
    VIX_TRY(keys_in.alloc((size_t)n));
    VIX_TRY(keys.alloc((size_t)n));
    ids_to_keys_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(did.dev, n, keys_in.ptr);
    VIX_LAUNCH_CHECK();
    VIX_TRY(sort_keys(keys_in.ptr, keys.ptr, n));
    // 2. per stored row: keep flag; 3. new positions of the kept rows, and their number
    Scratch<int32_t> keep, pos;
    VIX_TRY(keep.alloc((size_t)rows + 1));
    VIX_TRY(pos.alloc((size_t)rows + 1));
    mark_removed_kernel<<<(unsigned)((rows + 1 + 255) / 256), 256, 0, s>>>(h->ids.ptr, rows, keys.ptr, n, keep.ptr);
    VIX_LAUNCH_CHECK();
    VIX_TRY(exclusive_sum(keep.ptr, pos.ptr, rows + 1));
    int32_t kept32 = 0;
    VIX_CUDA(cudaMemcpyAsync(&kept32, pos.ptr + rows, 4, cudaMemcpyDeviceToHost, s));
    VIX_CUDA(cudaStreamSynchronize(s));
    const int64_t kept = kept32;
    if (kept == rows) return VIX_OK;                              // nothing matched: the handle is untouched (lists stay built)
    // 4. gather the kept rows of every add-order array, largest first: once its copy is made, the memory it frees holds
    //    every later copy, so a call that gets past the first allocation completes
    struct Part { int which; int64_t bytes; };
    Part parts[4];
    int np = 0;
    parts[np++] = {0, rows * 8};
    if (h->assign.size == (size_t)rows) parts[np++] = {1, rows * 4};
    if (h->p.kind == VIX_INDEX_IVF_PQ) parts[np++] = {2, rows * (int64_t)h->code_bytes()};
    else parts[np++] = {3, rows * (int64_t)h->p.d * 4};
    for (int a = 1; a < np; ++a)
        for (int b = a; b > 0 && parts[b].bytes > parts[b - 1].bytes; --b) { Part t = parts[b]; parts[b] = parts[b - 1]; parts[b - 1] = t; }
    for (int a = 0; a < np; ++a) {
        switch (parts[a].which) {
            case 0: VIX_TRY(compact_array(h->ids, rows, 1, kept, keep.ptr, pos.ptr)); break;
            case 1: VIX_TRY(compact_array(h->assign, rows, 1, kept, keep.ptr, pos.ptr)); break;
            case 2: VIX_TRY(compact_array(h->codes, rows, h->code_bytes(), kept, keep.ptr, pos.ptr)); break;
            default: VIX_TRY(compact_array(h->vecs, rows, h->p.d, kept, keep.ptr, pos.ptr)); break;
        }
    }
    // 5. the lists, the scan layouts and the decode layout follow at the next call that reads them
    h->n = kept;
    h->dirty = true;
    *removed = rows - kept;
    return VIX_OK;
}

int ivf_range_scan(vix_index* h, const float* dq, int64_t nq, int nprobe, const int32_t* probes, const FilterArgs* filter,
                   IvfRangeScan& out) {
    const int d = h->p.d;
    cudaStream_t s = ctx().stream;
    if (h->p.kind == VIX_INDEX_IVF_PQ) {
        ScanArgs a{};
        a.queries = dq; a.nq = nq; a.d = d; a.m = h->p.m; a.ks = h->p.ks; a.dsub = d / h->p.m;
        a.nprobe = nprobe; a.coarse = h->coarse.ptr; a.kc = h->kc; a.codebooks = h->codebooks.ptr;
        a.list_off = h->list_off.ptr; a.list_len = h->list_len.ptr;
        a.slot_codes = h->slot_codes.ptr; a.slot_tx = h->slot_tx.ptr; a.slot_ids = h->slot_ids.ptr;
        a.metric = h->p.metric; a.codebooks_t = h->codebooks_t.ptr;
        if (filter) { a.filter = filter->words; a.filter_cap = filter->cap; a.filter_deny = filter->deny; }
        VIX_TRY(out.work_counter.alloc(2));
        a.work_counter = out.work_counter.ptr;
        const bool fast = scan_layout(a.m).fast && a.ks == 256;
        if (fast && nq > 2 * num_sms()) {
            VIX_TRY(query_order(probes, nq, nprobe, h->list_len.ptr, h->kc, out.order));
            a.order = out.order.ptr;
        }
        if (fast) snprintf(out.kernel, sizeof out.kernel, "fast G %d", a.m / 16);
        else snprintf(out.kernel, sizeof out.kernel, "generic");
        out.run = [a](const int32_t* pr, const RangeOut& o) {
            ScanArgs b = a;
            b.probes = pr;
            b.range = o;
            return launch_ivfpq_scan_classic(b);
        };
        return VIX_OK;
    }
    snprintf(out.kernel, sizeof out.kernel, "ivfflat");
    const size_t smem = (size_t)d * 4;
    VIX_CUDA(cudaFuncSetAttribute(ivfflat_range_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int64_t grid = std::min<int64_t>((int64_t)num_sms() * 4, nq);
    const FilterArgs f = filter ? *filter : FilterArgs{};
    out.run = [=](const int32_t* pr, const RangeOut& o) -> int {
        ivfflat_range_kernel<<<(unsigned)grid, 256, smem, s>>>(dq, nq, d, pr, nprobe, h->list_off.ptr, h->list_len.ptr, h->kc,
                                                             h->slot_vecs.ptr, h->slot_ids.ptr, h->p.metric, f.words, f.cap,
                                                             f.deny, o);
        VIX_LAUNCH_CHECK();
        return VIX_OK;
    };
    return VIX_OK;
}

// k-NN search for VIX_MAX_K < k <= VIX_MAX_K_LARGE (vix_knn_large.cu): the candidates of index_search_locked (every row,
// or the probed lists of the same probe selection / the caller's given_probes), a seed pass and a collect pass through the
// kind's range kernel, the sorted rows cut at k.  Synchronises the stream (the collect's size depends on the data); not
// traced.  The handle keeps only the collect's capacity hint, written once the call has succeeded.
static int index_knn_large_locked(vix_index* h, const float* queries, int64_t nq, int k, int nprobe, float* out_dist,
                                  int64_t* out_ids, int32_t* out_probes, vix_search_stats* stats,
                                  const int32_t* given_probes, const FilterArgs* filter) {
    const int d = h->p.d;
    cudaStream_t s = ctx().stream;
    const bool linear = h->p.kind == VIX_INDEX_FLAT || !h->has_coarse;
    VIX_REQUIRE(!linear || h->p.kind != VIX_INDEX_IVF_PQ, VIX_ERR_NOT_TRAINED, "index_search: IVF-PQ index is not trained");
    VIX_REQUIRE(nq < 0x7FFFFFFFLL, VIX_ERR_INVALID_PARAM, "index_search: k > %d needs nq < 2^31 - 1", VIX_MAX_K);
    if (!linear) {
        if (nprobe <= 0) nprobe = h->p.nprobe;
        VIX_REQUIRE(nprobe > 0 && nprobe <= VIX_MAX_K, VIX_ERR_INVALID_K, "index_search: nprobe = %d (1 .. %d)", nprobe,
                    VIX_MAX_K);
    }
    In<float> dq;
    Out<float> dd;
    Out<int64_t> di;
    Out<int32_t> dp;
    VIX_TRY(dq.stage(queries, (size_t)nq * d));
    VIX_TRY(dd.stage(out_dist, (size_t)nq * k));
    VIX_TRY(di.stage(out_ids, (size_t)nq * k));
    cudaEvent_t* ev = h->ev;
    if (stats && !ev[0]) for (int e = 0; e < 5; ++e) VIX_CUDA(cudaEventCreate(&ev[e]));
    if (stats) VIX_CUDA(cudaEventRecord(ev[0], s));
    size_t cap = h->knn_cap;
    KnnInfo info;
    char kernel[32] = "flat";
    if (linear) {
        // a flat index, or an IVF-Flat index before optimize(): the flat engine over the stored rows, row indices as ids
        Scratch<uint64_t> mask;
        if (filter && h->n > 0) {
            const int64_t words = (h->n + 63) / 64;
            VIX_TRY(mask.alloc((size_t)words));
            filter_row_mask_kernel<<<(unsigned)((words + 255) / 256), 256, 0, s>>>(h->ids.ptr, h->n, filter->words, filter->cap,
                                                                                filter->deny, mask.ptr);
            VIX_LAUNCH_CHECK();
        }
        if (stats) VIX_CUDA(cudaEventRecord(ev[1], s));
        Scratch<int64_t> rows;
        VIX_TRY(rows.alloc((size_t)nq * k));
        VIX_TRY(flat_knn_large_device(dq.dev, nq, h->vecs.ptr, h->n, d, h->p.metric, k, mask.ptr, cap, dd.dev, rows.ptr, &info));
        gather_ids_kernel<<<(unsigned)((nq * k + 255) / 256), 256, 0, s>>>(rows.ptr, h->ids.ptr, di.dev, nq * (int64_t)k);
        VIX_LAUNCH_CHECK();
    } else {
        if (h->dirty) VIX_TRY(build_lists(h));
        VIX_TRY(dp.stage(out_probes, out_probes ? (size_t)nq * nprobe : 0));
        Scratch<int32_t> probe_buf;
        In<int32_t> gp;
        const int32_t* probes = nullptr;
        if (given_probes) {
            VIX_TRY(gp.stage(given_probes, (size_t)nq * nprobe));
            if (dp.dev) VIX_CUDA(cudaMemcpyAsync(dp.dev, gp.dev, (size_t)nq * nprobe * 4, cudaMemcpyDeviceToDevice, s));
            probes = gp.dev;
        } else {
            int32_t* pp = dp.dev;
            if (!pp) { VIX_TRY(probe_buf.alloc((size_t)nq * nprobe)); pp = probe_buf.ptr; }
            if (h->p.metric == VIX_METRIC_COSINE)
                VIX_TRY(probe_select_cosine_device(dq.dev, nq, h->coarse.ptr, h->kc, d, h->coarse_norms.ptr, nprobe, pp));
            else
                VIX_TRY(probe_select_fast_device(dq.dev, nq, h->coarse.ptr, h->kc, d, h->p.metric, nprobe, h->coarse_norms.ptr, pp,
                                                 nullptr, h->coarse_norm_max.ptr));
            probes = pp;
        }
        if (stats) VIX_CUDA(cudaEventRecord(ev[1], s));
        Scratch<int32_t> prefix;
        VIX_TRY(prefix.alloc((size_t)nq * nprobe));
        size_t seed_cap = 0, max_entries = 0;
        VIX_TRY(knn_probe_prefix(probes, nq, nprobe, h->list_len.ptr, h->kc, k, prefix.ptr, &seed_cap, &max_entries));
        IvfRangeScan scan;
        VIX_TRY(ivf_range_scan(h, dq.dev, nq, nprobe, probes, filter, scan));
        snprintf(kernel, sizeof kernel, "%s", scan.kernel);
        const std::function<int(const RangeOut&)> seed = [&](const RangeOut& o) { return scan.run(prefix.ptr, o); };
        const std::function<int(const RangeOut&)> collect = [&](const RangeOut& o) { return scan.run(probes, o); };
        // (IVF-PQ reports a zero inner-product distance as -0, IVF-Flat keys the distance itself: +0)
        KnnDecode dec;
        dec.neg_zero = h->p.kind == VIX_INDEX_IVF_PQ && h->p.metric == VIX_METRIC_IP;
        VIX_TRY(knn_large_run(nq, k, dec, seed_cap, &seed, collect, max_entries, cap, dd.dev, di.dev, &info));
        VIX_TRY(dp.commit());
    }
    if (stats) VIX_CUDA(cudaEventRecord(ev[2], s));
    VIX_TRY(dd.commit());
    VIX_TRY(di.commit());
    const int rc = finish(true);
    if (rc != VIX_OK) return rc;
    h->knn_cap = cap;
    if (stats) {
        VIX_CUDA(cudaEventSynchronize(ev[2]));
        cudaEventElapsedTime(&stats->ms_coarse, ev[0], ev[1]);
        cudaEventElapsedTime(&stats->ms_scan, ev[1], ev[2]);
        cudaEventElapsedTime(&stats->ms_total, ev[0], ev[2]);
        stats->scan_path = 2;
        stats->merge_candidates = info.collect.total;
    }
    if (getenv("VIX_SCAN_DEBUG"))
        fprintf(stderr, "[vix knn] kind %s, kernel %s, filter %d, k %d, seed %lld, total %lld, passes %d, max_row %lld\n",
                h->p.kind == VIX_INDEX_FLAT ? "flat" : h->p.kind == VIX_INDEX_IVF_FLAT ? "ivfflat" : "ivfpq", kernel,
                filter != nullptr, k, (long long)info.seed, (long long)info.collect.total, info.collect.passes,
                (long long)info.collect.max_row);
    return VIX_OK;
}

int index_search_locked(vix_index* h, const float* queries, int64_t nq, int k, int nprobe, float* out_dist,
                        int64_t* out_ids, int32_t* out_probes, vix_search_stats* stats,
                        const int32_t* given_probes, const FilterArgs* filter) {
    const int d = h->p.d;
    cudaStream_t s = ctx().stream;
    if (stats) memset(stats, 0, sizeof(*stats));
    if (k <= 0 || nq <= 0) return VIX_OK;                      // IVFIndex.swift:866
    VIX_REQUIRE(queries && out_dist && out_ids, VIX_ERR_NULL_PTR, "index_search: null pointer");
    VIX_REQUIRE(k <= VIX_MAX_K_LARGE, VIX_ERR_INVALID_K, "index_search: k > %d", VIX_MAX_K_LARGE);
    if (k > VIX_MAX_K)
        return index_knn_large_locked(h, queries, nq, k, nprobe, out_dist, out_ids, out_probes, stats, given_probes, filter);
    In<float> dq;
    Out<float> dd;
    Out<int64_t> di;
    Out<int32_t> dp;
    VIX_TRY(dq.stage(queries, (size_t)nq * d));
    VIX_TRY(dd.stage(out_dist, (size_t)nq * k));
    VIX_TRY(di.stage(out_ids, (size_t)nq * k));

    cudaEvent_t* ev = h->ev;
    if (stats && !ev[0]) for (int e = 0; e < 5; ++e) VIX_CUDA(cudaEventCreate(&ev[e]));
    const bool traced = !stats && h->trace_n < h->trace_cap;
    cudaEvent_t* tev = traced ? &h->trace_ev[5 * (size_t)h->trace_n] : nullptr;
    if (stats) VIX_CUDA(cudaEventRecord(ev[0], s));
    if (traced) VIX_CUDA(cudaEventRecord(tev[0], s));

    if (h->p.kind == VIX_INDEX_FLAT || !h->has_coarse) {
        // un-optimised IVF => linear scan (IVFIndex.swift:820-832)
        VIX_REQUIRE(h->p.kind != VIX_INDEX_IVF_PQ, VIX_ERR_NOT_TRAINED, "index_search: IVF-PQ index is not trained");
        Scratch<int64_t> rows;
        VIX_TRY(rows.alloc((size_t)nq * k));
        if (filter && h->n > 0) {
            Scratch<uint64_t> mask;
            const int64_t words = (h->n + 63) / 64;
            VIX_TRY(mask.alloc((size_t)words));
            filter_row_mask_kernel<<<(unsigned)((words + 255) / 256), 256, 0, s>>>(h->ids.ptr, h->n, filter->words, filter->cap,
                                                                                filter->deny, mask.ptr);
            VIX_LAUNCH_CHECK();
            VIX_TRY(flat_search_masked_device(dq.dev, nq, h->vecs.ptr, h->n, d, h->p.metric, k, mask.ptr, dd.dev, rows.ptr));
        } else
        VIX_TRY(flat_search_auto_device(dq.dev, nq, h->vecs.ptr, h->n, d, h->p.metric, k, nullptr, dd.dev, rows.ptr, false));
        // row index -> user id
        gather_ids_kernel<<<(unsigned)((nq * k + 255) / 256), 256, 0, s>>>(rows.ptr, h->ids.ptr, di.dev, nq * (int64_t)k);
        VIX_LAUNCH_CHECK();
        if (stats) for (int e = 1; e < 5; ++e) VIX_CUDA(cudaEventRecord(ev[e], s));
        if (traced) for (int e = 1; e < 5; ++e) VIX_CUDA(cudaEventRecord(tev[e], s));
    } else {
        if (nprobe <= 0) nprobe = h->p.nprobe;
        VIX_REQUIRE(nprobe > 0 && nprobe <= VIX_MAX_K, VIX_ERR_INVALID_K, "index_search: nprobe = %d (1 .. %d)", nprobe,
                    VIX_MAX_K);
        if (h->dirty) VIX_TRY(build_lists(h));
        VIX_TRY(dp.stage(out_probes, out_probes ? (size_t)nq * nprobe : 0));
        Scratch<int32_t> probes;
        int32_t* pp = dp.dev;
        if (!pp) { VIX_TRY(probes.alloc((size_t)nq * nprobe)); pp = probes.ptr; }
        In<int32_t> gp;
        if (given_probes) {
            // probe lists chosen by the caller (sharded search: the globally merged top-nprobe)
            VIX_TRY(gp.stage(given_probes, (size_t)nq * nprobe));
            if (dp.dev) VIX_CUDA(cudaMemcpyAsync(dp.dev, gp.dev, (size_t)nq * nprobe * 4, cudaMemcpyDeviceToDevice, s));
            pp = const_cast<int32_t*>(gp.dev);
        } else if (h->p.metric == VIX_METRIC_COSINE) {
            VIX_TRY(probe_select_cosine_device(dq.dev, nq, h->coarse.ptr, h->kc, d, h->coarse_norms.ptr, nprobe, pp));
        } else {
            VIX_TRY(probe_select_fast_device(dq.dev, nq, h->coarse.ptr, h->kc, d, h->p.metric, nprobe,
                                             h->coarse_norms.ptr, pp, nullptr, h->coarse_norm_max.ptr));
        }
        // ([3], [4]: around the dominant kernel of the scan stage -- the IVF-PQ launchers record them again)
        if (stats) { VIX_CUDA(cudaEventRecord(ev[1], s)); VIX_CUDA(cudaEventRecord(ev[3], s)); VIX_CUDA(cudaEventRecord(ev[4], s)); }
        if (traced) { VIX_CUDA(cudaEventRecord(tev[1], s)); VIX_CUDA(cudaEventRecord(tev[3], s)); VIX_CUDA(cudaEventRecord(tev[4], s)); }
        int scan_path = 0;
        DevBuf<unsigned long long>& scanned = h->scanned;
        if (stats) { VIX_TRY(scanned.resize(16, false)); VIX_CUDA(cudaMemsetAsync(scanned.ptr, 0, 128, s)); }
        if (h->p.kind == VIX_INDEX_IVF_PQ) {
            ScanArgs a{};
            a.queries = dq.dev; a.nq = nq; a.d = d; a.m = h->p.m; a.ks = h->p.ks; a.dsub = d / h->p.m;
            a.probes = pp; a.nprobe = nprobe; a.coarse = h->coarse.ptr; a.kc = h->kc; a.codebooks = h->codebooks.ptr;
            a.list_off = h->list_off.ptr; a.list_len = h->list_len.ptr;
            a.slot_codes = h->slot_codes.ptr; a.slot_tx = h->slot_tx.ptr; a.slot_ids = h->slot_ids.ptr;
            a.tc_codes = h->tc_codes.ptr;
            a.metric = h->p.metric; a.k = k; a.out_dist = dd.dev; a.out_ids = di.dev;
            a.scanned = stats ? scanned.ptr : (traced ? h->trace_scanned.ptr + h->trace_n : nullptr);
            a.phase_cycles = stats ? scanned.ptr + 1 : nullptr;
            a.codebooks_t = h->codebooks_t.ptr;
            a.tc_table = h->tc_table.ptr; a.tc_meta = h->tc_meta.ptr;
            if (filter) { a.filter = filter->words; a.filter_cap = filter->cap; a.filter_deny = filter->deny; }
            // the work queue head belongs to THIS call (stream-ordered scratch): two threads searching the same handle on
            // different streams in asynchronous mode do not share it
            Scratch<int> work_counter;
            VIX_TRY(work_counter.alloc(2));
            a.work_counter = work_counter.ptr;
            Scratch<int32_t> order;
            // (the list-major path does not go query by query: no order to compute)
            if (scan_layout(a.m).fast && a.ks == 256 && nq > 2 * num_sms() && !tc_scan_supported(a)) {
                VIX_TRY(query_order(pp, nq, nprobe, h->list_len.ptr, h->kc, order));
                a.order = order.ptr;
            }
            if (stats) { a.ev_kernel[0] = ev[3]; a.ev_kernel[1] = ev[4]; }
            if (traced) { a.ev_kernel[0] = tev[3]; a.ev_kernel[1] = tev[4]; }
            VIX_TRY(launch_ivfpq_scan(a));
            scan_path = a.path;
            if (traced) h->trace_path[(size_t)h->trace_n] = a.path;
        } else {
            const int P = next_pow2(k + 256);
            const size_t smem = (size_t)P * 8 + (size_t)d * 4;
            VIX_CUDA(cudaFuncSetAttribute(ivfflat_scan_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            int64_t grid = (int64_t)num_sms() * 4;
            if (grid > nq) grid = nq;
            ivfflat_scan_kernel<<<(unsigned)grid, 256, smem, s>>>(dq.dev, nq, d, pp, nprobe, h->list_off.ptr,
                                                                 h->list_len.ptr, h->kc, h->slot_vecs.ptr, h->slot_ids.ptr,
                                                                 h->p.metric, k, P, filter ? filter->words : nullptr,
                                                                 filter ? filter->cap : 0, filter ? filter->deny : 0, dd.dev, di.dev);
            VIX_LAUNCH_CHECK();
        }
        if (traced) VIX_CUDA(cudaEventRecord(tev[2], s));
        if (stats) {
            VIX_CUDA(cudaEventRecord(ev[2], s));
            unsigned long long sc4[16] = {0};
            VIX_CUDA(cudaMemcpyAsync(sc4, scanned.ptr, 128, cudaMemcpyDeviceToHost, s));
            VIX_CUDA(cudaStreamSynchronize(s));
#ifdef VIX_SCAN_DIAG
            fprintf(stderr, "[vix diag] chunks %llu, queue flushes %llu, chunks with a passing entry %llu, barrier wait summed over warps %llu cycles\n",
                    sc4[9], sc4[10], sc4[11], sc4[12]);
#endif
            const unsigned long long sc = sc4[0];
            stats->codes_scanned = (int64_t)sc;
            stats->cycles_prologue = (int64_t)sc4[1]; stats->cycles_scan = (int64_t)sc4[2]; stats->cycles_tail = (int64_t)sc4[3];
            stats->cycles_select = (int64_t)sc4[4]; stats->cycles_probe_table = (int64_t)sc4[5]; stats->cycles_lut = (int64_t)sc4[6];
            stats->merge_candidates = (int64_t)sc4[7];
            stats->scan_path = scan_path;
            stats->code_bytes_scanned = (int64_t)sc * (h->p.kind == VIX_INDEX_IVF_PQ ? h->code_bytes() : d * 4);
        }
        VIX_TRY(dp.commit());
    }
    VIX_TRY(dd.commit());
    VIX_TRY(di.commit());
    if (traced) h->trace_n += 1;
    int rc = finish(dd.is_host() || di.is_host() || dp.is_host() || stats != nullptr);
    if (stats) {
        VIX_CUDA(cudaEventSynchronize(ev[2]));
        cudaEventElapsedTime(&stats->ms_coarse, ev[0], ev[1]);
        cudaEventElapsedTime(&stats->ms_scan, ev[1], ev[2]);
        cudaEventElapsedTime(&stats->ms_total, ev[0], ev[2]);
        if (h->p.kind != VIX_INDEX_FLAT && h->has_coarse) cudaEventElapsedTime(&stats->ms_scan_kernel, ev[3], ev[4]);
    }
    return rc;
}

// One range search of an index whose mutex the caller holds: the candidates of index_search_locked (every row, or the probed
// lists of the same probe selection, or the caller's given_probes), each kind through its range kernel, the output path of
// vix_range.cu.  keys_out: stop before decoding and hand back the sorted keys and lims (out is not touched).
int index_range_locked(vix_index* h, const float* queries, int64_t nq, float radius, int nprobe, const FilterArgs* filter,
                       vix_range_result** out, const int32_t* given_probes, RangeKeys* keys_out) {
    const int d = h->p.d;
    cudaStream_t s = ctx().stream;
    const bool linear = h->p.kind == VIX_INDEX_FLAT || !h->has_coarse;
    if (!linear) {
        if (nprobe <= 0) nprobe = h->p.nprobe;
        VIX_REQUIRE(nprobe > 0 && nprobe <= VIX_MAX_K, VIX_ERR_INVALID_K, "vix_index_range_search: nprobe = %d (1 .. %d)", nprobe,
                    VIX_MAX_K);
    }
    if (nq == 0) return range_empty(0, out);
    In<float> dq;
    VIX_TRY(dq.stage(queries, (size_t)nq * d));
    size_t cap = h->range_cap;
    RangeInfo info;
    char kernel[32] = "flat";
    int rc;
    auto collect = [&](bool neg_zero, const std::function<int(const RangeOut&)>& scan) {
        if (keys_out) return range_collect_keys(nq, radius, cap, scan, *keys_out, &info);
        return range_collect(nq, radius, cap, neg_zero, scan, out, &info);
    };
    if (linear) {
        // a flat index, or an IVF-Flat index before optimize(): the flat engine over the stored rows (IVFIndex.swift:820-832)
        Scratch<uint64_t> mask;
        if (filter && h->n > 0) {
            const int64_t words = (h->n + 63) / 64;
            VIX_TRY(mask.alloc((size_t)words));
            filter_row_mask_kernel<<<(unsigned)((words + 255) / 256), 256, 0, s>>>(h->ids.ptr, h->n, filter->words, filter->cap,
                                                                                filter->deny, mask.ptr);
            VIX_LAUNCH_CHECK();
        }
        rc = collect(h->p.metric == VIX_METRIC_IP, [&](const RangeOut& o) {
            return flat_range_device(dq.dev, nq, h->vecs.ptr, h->n, d, h->p.metric, h->ids.ptr, mask.ptr, o);
        });
    } else {
        if (h->dirty) VIX_TRY(build_lists(h));
        Scratch<int32_t> probe_buf;
        In<int32_t> gp;
        const int32_t* probes = nullptr;
        if (given_probes) {
            // probe lists chosen by the caller (sharded range search: the lists of the whole batch, exchanged)
            VIX_TRY(gp.stage(given_probes, (size_t)nq * nprobe));
            probes = gp.dev;
        } else {
            VIX_TRY(probe_buf.alloc((size_t)nq * nprobe));
            if (h->p.metric == VIX_METRIC_COSINE)
                VIX_TRY(probe_select_cosine_device(dq.dev, nq, h->coarse.ptr, h->kc, d, h->coarse_norms.ptr, nprobe, probe_buf.ptr));
            else
                VIX_TRY(probe_select_fast_device(dq.dev, nq, h->coarse.ptr, h->kc, d, h->p.metric, nprobe, h->coarse_norms.ptr,
                                                 probe_buf.ptr, nullptr, h->coarse_norm_max.ptr));
            probes = probe_buf.ptr;
        }
        if (h->p.kind == VIX_INDEX_IVF_PQ) {
            ScanArgs a{};
            a.queries = dq.dev; a.nq = nq; a.d = d; a.m = h->p.m; a.ks = h->p.ks; a.dsub = d / h->p.m;
            a.probes = probes; a.nprobe = nprobe; a.coarse = h->coarse.ptr; a.kc = h->kc; a.codebooks = h->codebooks.ptr;
            a.list_off = h->list_off.ptr; a.list_len = h->list_len.ptr;
            a.slot_codes = h->slot_codes.ptr; a.slot_tx = h->slot_tx.ptr; a.slot_ids = h->slot_ids.ptr;
            a.metric = h->p.metric; a.codebooks_t = h->codebooks_t.ptr;
            if (filter) { a.filter = filter->words; a.filter_cap = filter->cap; a.filter_deny = filter->deny; }
            Scratch<int> work_counter;
            VIX_TRY(work_counter.alloc(2));
            a.work_counter = work_counter.ptr;
            const bool fast = scan_layout(a.m).fast && a.ks == 256;
            Scratch<int32_t> order;
            if (fast && nq > 2 * num_sms()) {
                VIX_TRY(query_order(probes, nq, nprobe, h->list_len.ptr, h->kc, order));
                a.order = order.ptr;
            }
            if (fast) snprintf(kernel, sizeof kernel, "fast G %d", a.m / 16);
            else snprintf(kernel, sizeof kernel, "generic");
            // never the list-major tensor-core scan: the query-major one with its range instantiations
            rc = collect(h->p.metric == VIX_METRIC_IP, [&](const RangeOut& o) {
                ScanArgs b = a;
                b.range = o;
                return launch_ivfpq_scan_classic(b);
            });
        } else {
            snprintf(kernel, sizeof kernel, "ivfflat");
            const size_t smem = (size_t)d * 4;
            VIX_CUDA(cudaFuncSetAttribute(ivfflat_range_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            int64_t grid = (int64_t)num_sms() * 4;
            if (grid > nq) grid = nq;
            // (the IVF-Flat scan keys the distance itself, so its zeros are +0 as in k-NN search)
            rc = collect(false, [&](const RangeOut& o) -> int {
                ivfflat_range_kernel<<<(unsigned)grid, 256, smem, s>>>(dq.dev, nq, d, probes, nprobe, h->list_off.ptr,
                                                                     h->list_len.ptr, h->kc, h->slot_vecs.ptr, h->slot_ids.ptr,
                                                                     h->p.metric, filter ? filter->words : nullptr,
                                                                     filter ? filter->cap : 0, filter ? filter->deny : 0, o);
                VIX_LAUNCH_CHECK();
                return VIX_OK;
            });
        }
    }
    VIX_TRY(rc);
    h->range_cap = cap;
    if (getenv("VIX_SCAN_DEBUG"))
        fprintf(stderr, "[vix range] kind %s, kernel %s, filter %d, passes %d, total %lld, max_row %lld, sorted_long %lld\n",
                h->p.kind == VIX_INDEX_FLAT ? "flat" : h->p.kind == VIX_INDEX_IVF_FLAT ? "ivfflat" : "ivfpq", kernel,
                filter != nullptr, info.passes, (long long)info.total, (long long)info.max_row, (long long)info.sorted_long);
    return VIX_OK;
}

// gather rows of the sorted list layout back to add order / CSR export
__global__ void export_lists_kernel(const int32_t* __restrict__ slot_row, const int64_t* __restrict__ off,
                                    const int32_t* __restrict__ len, int kc, const uint8_t* __restrict__ codes,
                                    const int64_t* __restrict__ ids, int m, int64_t* __restrict__ off_out,
                                    uint8_t* __restrict__ codes_out, int64_t* __restrict__ ids_out,
                                    const int64_t* __restrict__ off_raw) {
    const int l = blockIdx.x;
    if (l >= kc) return;
    const int64_t b = off[l], o = off_raw[l];
    for (int i = threadIdx.x; i < len[l]; i += blockDim.x) {
        const int row = slot_row[b + i];
        if (ids_out) ids_out[o + i] = ids[row];
        if (codes_out) for (int j = 0; j < m; ++j) codes_out[(o + i) * (int64_t)m + j] = codes[(int64_t)row * m + j];
    }
    if (threadIdx.x == 0 && off_out) { off_out[l] = o; if (l == kc - 1) off_out[kc] = off_raw[kc]; }
}

__global__ void expand_assign_kernel(const int64_t* __restrict__ off, int kc, int32_t* __restrict__ assign) {
    const int l = blockIdx.x;
    if (l >= kc) return;
    for (int64_t i = off[l] + threadIdx.x; i < off[l + 1]; i += blockDim.x) assign[i] = l;
}

}  // namespace vix

extern "C" {

void vix_index_params_default(vix_index_params* p) {
    if (!p) return;
    memset(p, 0, sizeof(*p));
    p->kind = VIX_INDEX_IVF_PQ; p->d = 0; p->metric = VIX_METRIC_L2;
    p->nlist = 256; p->nprobe = 8;           // IVFIndex.Configuration (IVFIndex.swift:15-22)
    p->m = 16; p->ks = 256; p->shard_rank = 0; p->shard_world = 1;
}

int vix_index_create(const vix_index_params* p, vix_index_t** out) {
    VIX_TRY(ensure_device());
    VIX_REQUIRE(p && out, VIX_ERR_NULL_PTR, "vix_index_create: null pointer");
    VIX_REQUIRE(p->d > 0, VIX_ERR_INVALID_DIM, "vix_index_create: d must be > 0");
    VIX_REQUIRE(p->kind >= VIX_INDEX_FLAT && p->kind <= VIX_INDEX_IVF_PQ, VIX_ERR_INVALID_PARAM, "vix_index_create: kind");
    VIX_REQUIRE(p->metric == VIX_METRIC_L2 || p->metric == VIX_METRIC_IP ||
                    (p->metric == VIX_METRIC_COSINE && p->kind != VIX_INDEX_IVF_PQ),
                VIX_ERR_INVALID_PARAM, "vix_index_create: metric must be L2 or IP (cosine: FLAT and IVF_FLAT indexes only)");
    if (p->kind != VIX_INDEX_FLAT) VIX_REQUIRE(p->nlist > 0, VIX_ERR_INVALID_K, "vix_index_create: nlist must be > 0");
    if (p->kind == VIX_INDEX_IVF_PQ) {
        VIX_REQUIRE(p->m > 0 && p->d % p->m == 0, VIX_ERR_INVALID_DIM, "vix_index_create: d %% m != 0");
        VIX_REQUIRE(p->ks == 256 || (p->ks == 16 && p->m % 2 == 0), VIX_ERR_INVALID_K,
                    "vix_index_create: ks must be 256 (u8 codes) or 16 with an even m (u4 codes, two per byte)");
    }
    vix_index* h = new (std::nothrow) vix_index();
    VIX_REQUIRE(h, VIX_ERR_OOM, "vix_index_create: out of host memory");
    h->p = *p;
    if (h->p.nprobe <= 0) h->p.nprobe = 8;
    *out = h;
    return VIX_OK;
}

void vix_index_destroy(vix_index_t* h) {
    if (!h) return;
    cudaDeviceSynchronize();
    for (auto& e : h->ev) if (e) cudaEventDestroy(e);
    for (auto& e : h->trace_ev) if (e) cudaEventDestroy(e);
    delete h;
}

int vix_index_set_coarse(vix_index_t* h, const float* centroids, int kc) {
    VIX_REQUIRE(h && centroids, VIX_ERR_NULL_PTR, "vix_index_set_coarse: null pointer");
    VIX_REQUIRE(kc > 0, VIX_ERR_INVALID_K, "vix_index_set_coarse: kc must be > 0");
    std::lock_guard<std::mutex> lk(h->mu);
    VIX_REQUIRE(h->n == 0 || h->p.kind == VIX_INDEX_IVF_FLAT, VIX_ERR_CONTRACT, "vix_index_set_coarse: index already holds vectors");
    h->kc = kc;
    VIX_TRY(h->coarse.assign_from(centroids, (size_t)kc * h->p.d));
    VIX_TRY(h->coarse_norms.resize((size_t)kc, false));
    VIX_TRY(row_norms_device(h->coarse.ptr, kc, h->p.d, h->coarse_norms.ptr));   // IVFIndex.swift:470-485
    VIX_TRY(h->coarse_norm_max.resize(1, false));
    VIX_TRY(max_sqrt_device(h->coarse_norms.ptr, kc, h->coarse_norm_max.ptr));
    h->has_coarse = true;
    h->dirty = true;
    VIX_TRY(assign_stored_rows(h));
    return finish(true);
}

int vix_index_set_codebooks(vix_index_t* h, const float* codebooks, const float* centroid_norms) {
    VIX_REQUIRE(h && codebooks, VIX_ERR_NULL_PTR, "vix_index_set_codebooks: null pointer");
    std::lock_guard<std::mutex> lk(h->mu);
    VIX_REQUIRE(h->p.kind == VIX_INDEX_IVF_PQ, VIX_ERR_INVALID_PARAM, "vix_index_set_codebooks: not an IVF-PQ index");
    VIX_REQUIRE(h->n == 0, VIX_ERR_CONTRACT, "vix_index_set_codebooks: index already holds vectors");
    const int m = h->p.m, ks = h->p.ks, dsub = h->p.d / m;
    VIX_TRY(h->codebooks.assign_from(codebooks, (size_t)m * ks * dsub));
    if (centroid_norms) VIX_TRY(h->cb_norms.assign_from(centroid_norms, (size_t)m * ks));
    else {
        // PQTrain.swift:299-307: sequential sum of squares per centroid
        VIX_TRY(h->cb_norms.resize((size_t)m * ks, false));
        VIX_TRY(seq_norms(h->codebooks.ptr, (int64_t)m * ks, dsub, h->cb_norms.ptr));
    }
    VIX_TRY(update_codebooks_t(h));
    h->has_pq = true;
    return finish(true);
}

int vix_index_get_coarse(vix_index_t* h, float* centroids_out, int* kc_out) {
    VIX_REQUIRE(h, VIX_ERR_NULL_PTR, "vix_index_get_coarse: null handle");
    std::lock_guard<std::mutex> lk(h->mu);
    VIX_REQUIRE(h->has_coarse, VIX_ERR_NOT_TRAINED, "vix_index_get_coarse: not trained");
    if (kc_out) *kc_out = h->kc;
    if (centroids_out) {
        VIX_CUDA(cudaMemcpyAsync(centroids_out, h->coarse.ptr, (size_t)h->kc * h->p.d * 4, cudaMemcpyDefault, ctx().stream));
        return finish(true);
    }
    return VIX_OK;
}

int vix_index_get_codebooks(vix_index_t* h, float* codebooks_out, float* centroid_norms_out) {
    VIX_REQUIRE(h, VIX_ERR_NULL_PTR, "vix_index_get_codebooks: null handle");
    std::lock_guard<std::mutex> lk(h->mu);
    VIX_REQUIRE(h->has_pq, VIX_ERR_NOT_TRAINED, "vix_index_get_codebooks: not trained");
    const size_t cnt = (size_t)h->p.ks * h->p.d;
    if (codebooks_out) VIX_CUDA(cudaMemcpyAsync(codebooks_out, h->codebooks.ptr, cnt * 4, cudaMemcpyDefault, ctx().stream));
    if (centroid_norms_out)
        VIX_CUDA(cudaMemcpyAsync(centroid_norms_out, h->cb_norms.ptr, (size_t)h->p.m * h->p.ks * 4, cudaMemcpyDefault,
                                 ctx().stream));
    return finish(true);
}

int vix_index_train(vix_index_t* h, const float* x, int64_t n, const vix_kmeans_cfg* kcfg, const vix_pq_train_cfg* pcfg) {
    VIX_TRY(ensure_device());
    VIX_REQUIRE(h, VIX_ERR_NULL_PTR, "vix_index_train: null pointer");
    std::lock_guard<std::mutex> lk(h->mu);
    if (h->p.kind == VIX_INDEX_FLAT) return VIX_OK;
    // x == NULL on an IVF-Flat index that holds vectors: optimize() over the stored vectors (IVFIndex.swift:279-341)
    if (!x && h->p.kind == VIX_INDEX_IVF_FLAT && h->n > 0) { x = h->vecs.ptr; n = h->n; }
    VIX_REQUIRE(x, VIX_ERR_NULL_PTR, "vix_index_train: null pointer");
    VIX_REQUIRE(n > 0, VIX_ERR_EMPTY_INPUT, "vix_index_train: empty training set");
    VIX_REQUIRE(h->n == 0 || h->p.kind == VIX_INDEX_IVF_FLAT, VIX_ERR_CONTRACT, "vix_index_train: index already holds vectors");
    const int d = h->p.d;
    In<float> dx;
    VIX_TRY(dx.stage(x, (size_t)n * d));
    const int kc = (int)(h->p.nlist < n ? h->p.nlist : n);          // nlist clamped to n (IVFIndex.swift:320)
    VIX_TRY(h->coarse.resize((size_t)kc * d, false));
    // mode 0: the reference's trainer (k-means++ + mini-batch, IVFIndex.swift:337-341, 668-681); mode 1: GPU Lloyd
    if (kcfg && kcfg->mode == 0) VIX_TRY(kmeans_parity_device(dx.dev, n, d, kc, nullptr, kcfg, h->coarse.ptr, nullptr));
    else VIX_TRY(train_coarse_device(dx.dev, n, d, kc, h->p.metric, kcfg, h->coarse.ptr));
    h->kc = kc;
    VIX_TRY(h->coarse_norms.resize((size_t)kc, false));
    VIX_TRY(row_norms_device(h->coarse.ptr, kc, d, h->coarse_norms.ptr));
    VIX_TRY(h->coarse_norm_max.resize(1, false));
    VIX_TRY(max_sqrt_device(h->coarse_norms.ptr, kc, h->coarse_norm_max.ptr));
    h->has_coarse = true;
    if (h->p.kind == VIX_INDEX_IVF_PQ) {
        Scratch<int32_t> asg;
        VIX_TRY(asg.alloc((size_t)n));
        if (h->p.metric == VIX_METRIC_L2) VIX_TRY(ivf_assign_auto_device(dx.dev, n, d, h->coarse.ptr, kc, asg.ptr, nullptr));
        else VIX_TRY(ivf_assign_metric_device(dx.dev, n, d, h->coarse.ptr, kc, h->p.metric, nullptr, asg.ptr));
        const int m = h->p.m, ks = h->p.ks;
        VIX_TRY(h->codebooks.resize((size_t)ks * d, false));
        VIX_TRY(h->cb_norms.resize((size_t)m * ks, false));
        if (pcfg && pcfg->mode == 0) VIX_TRY(pq_train_parity_device(dx.dev, n, d, m, ks, h->coarse.ptr, asg.ptr, pcfg, h->codebooks.ptr, h->cb_norms.ptr));
        else VIX_TRY(train_pq_device(dx.dev, n, d, m, ks, h->coarse.ptr, asg.ptr, pcfg, h->codebooks.ptr, h->cb_norms.ptr));
        VIX_TRY(update_codebooks_t(h));
        h->has_pq = true;
    }
    h->dirty = true;
    VIX_TRY(assign_stored_rows(h));
    return finish(true);
}

int vix_index_add(vix_index_t* h, const float* x, const int64_t* ids, int64_t n) {
    VIX_TRY(ensure_device());
    VIX_REQUIRE(h && (x || n == 0), VIX_ERR_NULL_PTR, "vix_index_add: null pointer");
    VIX_REQUIRE(n >= 0, VIX_ERR_INVALID_PARAM, "vix_index_add: n < 0");
    std::lock_guard<std::mutex> lk(h->mu);
    return index_add_locked(h, x, ids, n);
}

int vix_index_import_lists(vix_index_t* h, const int64_t* list_offsets, const uint8_t* codes, const int64_t* ids) {
    VIX_TRY(ensure_device());
    VIX_REQUIRE(h && list_offsets && codes && ids, VIX_ERR_NULL_PTR, "vix_index_import_lists: null pointer");
    std::lock_guard<std::mutex> lk(h->mu);
    VIX_REQUIRE(h->p.kind == VIX_INDEX_IVF_PQ, VIX_ERR_INVALID_PARAM, "vix_index_import_lists: not an IVF-PQ index");
    VIX_REQUIRE(h->has_coarse && h->has_pq, VIX_ERR_NOT_TRAINED, "vix_index_import_lists: set coarse + codebooks first");
    VIX_REQUIRE(!is_device_ptr(list_offsets), VIX_ERR_INVALID_PARAM, "vix_index_import_lists: list_offsets must be a host pointer");
    const int kc = h->kc;
    const int64_t n = list_offsets[kc];
    VIX_REQUIRE(list_offsets[0] == 0 && n >= 0 && n < 0x7FFFFFFFLL, VIX_ERR_INVALID_PARAM, "vix_index_import_lists: bad offsets");
    for (int l = 0; l < kc; ++l)
        VIX_REQUIRE(list_offsets[l + 1] >= list_offsets[l], VIX_ERR_INVALID_PARAM, "vix_index_import_lists: offsets not monotone");
    VIX_TRY(is_device_ptr(ids) ? check_ids_device(ids, n) : check_ids_host(ids, n));
    VIX_TRY(h->codes.assign_from(codes, (size_t)n * h->code_bytes()));
    VIX_TRY(h->ids.assign_from(ids, (size_t)n));
    VIX_TRY(h->assign.resize((size_t)n, false));
    Scratch<int64_t> doff;
    VIX_TRY(doff.alloc((size_t)kc + 1));
    VIX_CUDA(cudaMemcpyAsync(doff.ptr, list_offsets, (size_t)(kc + 1) * 8, cudaMemcpyHostToDevice, ctx().stream));
    expand_assign_kernel<<<kc, 128, 0, ctx().stream>>>(doff.ptr, kc, h->assign.ptr);
    VIX_LAUNCH_CHECK();
    h->n = n;
    h->next_auto_id = n;
    h->dirty = true;
    return finish(true);
}

int64_t vix_index_count(vix_index_t* h) {
    if (!h) return 0;
    std::lock_guard<std::mutex> lk(h->mu);
    return h->n;
}

int vix_index_list_sizes(vix_index_t* h, int64_t* sizes_out) {
    VIX_REQUIRE(h && sizes_out, VIX_ERR_NULL_PTR, "vix_index_list_sizes: null pointer");
    std::lock_guard<std::mutex> lk(h->mu);
    VIX_REQUIRE(h->has_coarse, VIX_ERR_NOT_TRAINED, "vix_index_list_sizes: not trained");
    if (h->dirty) VIX_TRY(build_lists(h));
    std::vector<int32_t> len((size_t)h->kc);
    VIX_CUDA(cudaMemcpyAsync(len.data(), h->list_len.ptr, (size_t)h->kc * 4, cudaMemcpyDeviceToHost, ctx().stream));
    VIX_CUDA(cudaStreamSynchronize(ctx().stream));
    for (int l = 0; l < h->kc; ++l) sizes_out[l] = len[l];
    return VIX_OK;
}

int vix_index_export_lists(vix_index_t* h, int64_t* list_offsets, uint8_t* codes, int64_t* ids,
                           int32_t* assignments_in_add_order) {
    VIX_REQUIRE(h, VIX_ERR_NULL_PTR, "vix_index_export_lists: null handle");
    std::lock_guard<std::mutex> lk(h->mu);
    VIX_REQUIRE(h->has_coarse, VIX_ERR_NOT_TRAINED, "vix_index_export_lists: not trained");
    if (h->dirty) VIX_TRY(build_lists(h));
    const int kc = h->kc, m = h->code_bytes();                        // bytes per stored code
    const int64_t n = h->n;
    Scratch<int64_t> off_raw;
    VIX_TRY(off_raw.alloc((size_t)kc + 1));
    VIX_TRY(offsets_from_counts(h->list_len.ptr, kc, 1, off_raw.ptr, nullptr));
    Out<int64_t> doff, dids;
    Out<uint8_t> dcodes;
    VIX_TRY(doff.stage(list_offsets, list_offsets ? (size_t)kc + 1 : 0));
    const bool want_codes = codes && h->p.kind == VIX_INDEX_IVF_PQ;
    VIX_TRY(dcodes.stage(want_codes ? codes : nullptr, want_codes ? (size_t)n * m : 0));
    VIX_TRY(dids.stage(ids, ids ? (size_t)n : 0));
    export_lists_kernel<<<kc, 128, 0, ctx().stream>>>(h->slot_row.ptr, h->list_off.ptr, h->list_len.ptr, kc,
                                                     h->codes.ptr, h->ids.ptr, m, doff.dev, dcodes.dev, dids.dev,
                                                     off_raw.ptr);
    VIX_LAUNCH_CHECK();
    VIX_TRY(doff.commit());
    VIX_TRY(dcodes.commit());
    VIX_TRY(dids.commit());
    if (assignments_in_add_order && n > 0)
        VIX_CUDA(cudaMemcpyAsync(assignments_in_add_order, h->assign.ptr, (size_t)n * 4, cudaMemcpyDefault, ctx().stream));
    return finish(true);
}

int vix_debug_tc_codes(vix_index_t* h, uint8_t* out, int64_t cap, int64_t* bytes_out) {
    VIX_REQUIRE(h && bytes_out, VIX_ERR_NULL_PTR, "vix_debug_tc_codes: null pointer");
    std::lock_guard<std::mutex> lk(h->mu);
    VIX_REQUIRE(h->p.kind == VIX_INDEX_IVF_PQ && h->has_coarse, VIX_ERR_NOT_TRAINED, "vix_debug_tc_codes: not a trained IVF-PQ index");
    if (h->dirty) VIX_TRY(build_lists(h));
    const int64_t bytes = h->tc_codes.ptr ? h->nslots * h->p.m : 0;
    *bytes_out = bytes;
    if (out && bytes) {
        VIX_REQUIRE(cap >= bytes, VIX_ERR_INVALID_PARAM, "vix_debug_tc_codes: %lld bytes do not fit %lld", (long long)bytes, (long long)cap);
        VIX_CUDA(cudaMemcpyAsync(out, h->tc_codes.ptr, (size_t)bytes, cudaMemcpyDefault, ctx().stream));
    }
    return finish(true);
}

int vix_debug_tc_seed(vix_index_t* h, const float* queries, int64_t nq, int k, const int32_t* probes, int nprobe, float* thr) {
    VIX_TRY(ensure_device());
    VIX_REQUIRE(h && queries && probes && thr, VIX_ERR_NULL_PTR, "vix_debug_tc_seed: null pointer");
    VIX_REQUIRE(nq > 0 && nq < 0x7FFFFFFFLL && nprobe > 0 && nprobe <= VIX_MAX_K, VIX_ERR_INVALID_PARAM,
                "vix_debug_tc_seed: nq must lie in [1, 2^31 - 1), nprobe in [1, %d]", VIX_MAX_K);
    VIX_REQUIRE(k >= 1 && k <= 64, VIX_ERR_INVALID_K, "vix_debug_tc_seed: k must lie in [1, 64]");
    std::lock_guard<std::mutex> lk(h->mu);
    VIX_REQUIRE(h->p.kind == VIX_INDEX_IVF_PQ && h->has_coarse && h->has_pq, VIX_ERR_NOT_TRAINED,
                "vix_debug_tc_seed: not a trained IVF-PQ index");
    VIX_REQUIRE(tc_codes_shape(h->p.metric, h->p.m, h->p.ks, h->p.d / h->p.m), VIX_ERR_INVALID_PARAM,
                "vix_debug_tc_seed: the list-major scan does not take this shape");
    if (h->dirty) VIX_TRY(build_lists(h));
    In<float> dq;
    In<int32_t> dp;
    Out<float> dt;
    VIX_TRY(dq.stage(queries, (size_t)nq * h->p.d));
    VIX_TRY(dp.stage(probes, (size_t)nq * nprobe));
    VIX_TRY(dt.stage(thr, (size_t)nq));
    ScanArgs a{};
    a.queries = dq.dev; a.nq = nq; a.d = h->p.d; a.m = h->p.m; a.ks = h->p.ks; a.dsub = h->p.d / h->p.m;
    a.probes = const_cast<int32_t*>(dp.dev); a.nprobe = nprobe; a.coarse = h->coarse.ptr; a.kc = h->kc; a.k = k;
    a.list_off = h->list_off.ptr; a.list_len = h->list_len.ptr; a.slot_codes = h->slot_codes.ptr; a.slot_tx = h->slot_tx.ptr;
    a.codebooks_t = h->codebooks_t.ptr; a.metric = h->p.metric;
    VIX_TRY(tc_seed_thresholds(a, dt.dev));
    VIX_TRY(dt.commit());
    return finish(dt.is_host());
}

int vix_index_clear(vix_index_t* h) {
    VIX_REQUIRE(h, VIX_ERR_NULL_PTR, "vix_index_clear: null handle");
    std::lock_guard<std::mutex> lk(h->mu);
    h->n = 0;
    h->next_auto_id = 0;
    h->vecs.size = h->ids.size = h->assign.size = h->codes.size = 0;
    h->dirty = true;
    return VIX_OK;
}

int vix_index_remove(vix_index_t* h, const int64_t* ids, int64_t n, int64_t* removed_out) {
    if (removed_out) *removed_out = 0;
    VIX_TRY(ensure_device());
    VIX_REQUIRE(h && (ids || n == 0), VIX_ERR_NULL_PTR, "vix_index_remove: null pointer");
    VIX_REQUIRE(n >= 0 && n < 0x7FFFFFFFLL, VIX_ERR_INVALID_PARAM, "vix_index_remove: n must lie in [0, 2^31 - 1)");
    std::lock_guard<std::mutex> lk(h->mu);
    int64_t removed = 0;
    VIX_TRY(index_remove_locked(h, ids, n, &removed));
    if (removed_out) *removed_out = removed;
    return VIX_OK;
}

__global__ void offset_ids_kernel(int32_t* ids, int64_t n, int offset) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && ids[i] >= 0) ids[i] += offset;
}

int vix_index_search_with_probes(vix_index_t* h, const float* queries, int64_t nq, int k, const int32_t* probes, int nprobe,
                                 float* out_dist, int64_t* out_ids) {
    VIX_TRY(ensure_device());
    VIX_REQUIRE(h && probes, VIX_ERR_NULL_PTR, "vix_index_search_with_probes: null pointer");
    VIX_REQUIRE(nprobe > 0, VIX_ERR_INVALID_K, "vix_index_search_with_probes: nprobe must be > 0");
    std::lock_guard<std::mutex> lk(h->mu);
    VIX_REQUIRE(h->p.kind != VIX_INDEX_FLAT && h->has_coarse, VIX_ERR_NOT_TRAINED, "vix_index_search_with_probes: IVF index not trained");
    return index_search_locked(h, queries, nq, k, nprobe, out_dist, out_ids, nullptr, nullptr, probes);
}

int vix_index_search_filtered(vix_index_t* h, const float* queries, int64_t nq, int k, int nprobe,
                              const uint64_t* filter_words, int64_t filter_capacity, int filter_mode,
                              float* out_dist, int64_t* out_ids) {
    VIX_TRY(ensure_device());
    VIX_REQUIRE(h != nullptr, VIX_ERR_NULL_PTR, "vix_index_search_filtered: null handle");
    VIX_REQUIRE(filter_mode == VIX_FILTER_ALLOW || filter_mode == VIX_FILTER_DENY, VIX_ERR_INVALID_PARAM,
                "vix_index_search_filtered: filter_mode must be VIX_FILTER_ALLOW or VIX_FILTER_DENY");
    VIX_REQUIRE(filter_capacity >= 0, VIX_ERR_INVALID_PARAM, "vix_index_search_filtered: negative capacity");
    std::lock_guard<std::mutex> lk(h->mu);
    if (!filter_words) return index_search_locked(h, queries, nq, k, nprobe, out_dist, out_ids, nullptr, nullptr);
    In<uint64_t> fw;
    VIX_TRY(fw.stage(filter_words, (size_t)((filter_capacity + 63) / 64)));
    FilterArgs f;
    f.words = fw.dev; f.cap = filter_capacity; f.deny = filter_mode == VIX_FILTER_DENY;
    return index_search_locked(h, queries, nq, k, nprobe, out_dist, out_ids, nullptr, nullptr, nullptr, &f);
}

int vix_index_range_search(vix_index_t* h, const float* queries, int64_t nq, float radius, int nprobe,
                           const uint64_t* filter_words, int64_t filter_capacity, int filter_mode, vix_range_result_t** out) {
    VIX_TRY(ensure_device());
    VIX_REQUIRE(h && out, VIX_ERR_NULL_PTR, "vix_index_range_search: null pointer");
    *out = nullptr;
    VIX_REQUIRE(queries || nq == 0, VIX_ERR_NULL_PTR, "vix_index_range_search: null queries");
    VIX_REQUIRE(nq >= 0 && nq < 0x7FFFFFFFLL, VIX_ERR_INVALID_PARAM, "vix_index_range_search: nq must lie in [0, 2^31 - 1)");
    VIX_REQUIRE(radius == radius, VIX_ERR_INVALID_PARAM, "vix_index_range_search: radius is NaN");
    VIX_REQUIRE(filter_mode == VIX_FILTER_ALLOW || filter_mode == VIX_FILTER_DENY, VIX_ERR_INVALID_PARAM,
                "vix_index_range_search: filter_mode must be VIX_FILTER_ALLOW or VIX_FILTER_DENY");
    VIX_REQUIRE(filter_capacity >= 0, VIX_ERR_INVALID_PARAM, "vix_index_range_search: negative capacity");
    std::lock_guard<std::mutex> lk(h->mu);
    VIX_REQUIRE(h->p.kind != VIX_INDEX_IVF_PQ || (h->has_coarse && h->has_pq), VIX_ERR_NOT_TRAINED,
                "vix_index_range_search: IVF-PQ index is not trained");
    if (!filter_words) return index_range_locked(h, queries, nq, radius, nprobe, nullptr, out);
    In<uint64_t> fw;
    VIX_TRY(fw.stage(filter_words, (size_t)((filter_capacity + 63) / 64)));
    FilterArgs f;
    f.words = fw.dev; f.cap = filter_capacity; f.deny = filter_mode == VIX_FILTER_DENY;
    return index_range_locked(h, queries, nq, radius, nprobe, &f, out);
}

int vix_index_search_with_probes_ex(vix_index_t* h, const float* queries, int64_t nq, int k, const int32_t* probes,
                                    int nprobe, float* out_dist, int64_t* out_ids, vix_search_stats* stats) {
    VIX_TRY(ensure_device());
    VIX_REQUIRE(h && probes, VIX_ERR_NULL_PTR, "vix_index_search_with_probes_ex: null pointer");
    VIX_REQUIRE(nprobe > 0, VIX_ERR_INVALID_K, "vix_index_search_with_probes_ex: nprobe must be > 0");
    std::lock_guard<std::mutex> lk(h->mu);
    VIX_REQUIRE(h->p.kind != VIX_INDEX_FLAT && h->has_coarse, VIX_ERR_NOT_TRAINED, "vix_index_search_with_probes_ex: IVF index not trained");
    return index_search_locked(h, queries, nq, k, nprobe, out_dist, out_ids, nullptr, stats, probes);
}

int vix_index_probe_range(vix_index_t* h, const float* queries, int64_t nq, int nprobe, int list_begin, int list_count,
                          int32_t* list_ids_out, float* list_scores_out) {
    VIX_TRY(ensure_device());
    VIX_REQUIRE(h && queries && list_ids_out, VIX_ERR_NULL_PTR, "vix_index_probe_range: null pointer");
    std::lock_guard<std::mutex> lk(h->mu);
    VIX_REQUIRE(h->has_coarse, VIX_ERR_NOT_TRAINED, "vix_index_probe_range: not trained");
    VIX_REQUIRE(h->p.metric != VIX_METRIC_COSINE, VIX_ERR_UNSUPPORTED, "vix_index_probe_range: cosine indexes are not sharded");
    VIX_REQUIRE(nprobe > 0 && nprobe <= VIX_MAX_K, VIX_ERR_INVALID_K, "vix_index_probe_range: nprobe");
    VIX_REQUIRE(list_begin >= 0 && list_count > 0 && list_begin + list_count <= h->kc, VIX_ERR_INVALID_PARAM,
                "vix_index_probe_range: list range [%d, %d) outside [0, %d)", list_begin, list_begin + list_count, h->kc);
    if (nq <= 0) return VIX_OK;
    const int d = h->p.d;
    In<float> dq;
    Out<int32_t> di;
    Out<float> ds;
    VIX_TRY(dq.stage(queries, (size_t)nq * d));
    VIX_TRY(di.stage(list_ids_out, (size_t)nq * nprobe));
    VIX_TRY(ds.stage(list_scores_out, list_scores_out ? (size_t)nq * nprobe : 0));
    VIX_TRY(probe_select_fast_device(dq.dev, nq, h->coarse.ptr + (size_t)list_begin * d, list_count, d, h->p.metric, nprobe,
                                     h->coarse_norms.ptr + list_begin, di.dev, ds.dev, h->coarse_norm_max.ptr));
    if (list_begin > 0) {
        const int64_t total = nq * (int64_t)nprobe;
        offset_ids_kernel<<<(unsigned)((total + 255) / 256), 256, 0, ctx().stream>>>(di.dev, total, list_begin);
        VIX_LAUNCH_CHECK();
    }
    VIX_TRY(di.commit());
    VIX_TRY(ds.commit());
    return finish(di.is_host() || ds.is_host());
}

int vix_index_encode(vix_index_t* h, const float* x, int64_t n, int32_t* assign_out, uint8_t* codes_out) {
    VIX_TRY(ensure_device());
    VIX_REQUIRE(h && x && assign_out, VIX_ERR_NULL_PTR, "vix_index_encode: null pointer");
    std::lock_guard<std::mutex> lk(h->mu);
    VIX_REQUIRE(h->p.kind != VIX_INDEX_FLAT && h->has_coarse, VIX_ERR_NOT_TRAINED, "vix_index_encode: coarse quantiser not trained / set");
    const bool pq = h->p.kind == VIX_INDEX_IVF_PQ;
    if (pq) VIX_REQUIRE(h->has_pq && codes_out, VIX_ERR_NOT_TRAINED, "vix_index_encode: PQ codebooks not trained / codes_out missing");
    if (n <= 0) return VIX_OK;
    const int d = h->p.d;
    In<float> dx;
    Out<int32_t> da;
    Out<uint8_t> dc;
    VIX_TRY(dx.stage(x, (size_t)n * d));
    VIX_TRY(da.stage(assign_out, (size_t)n));
    VIX_TRY(dc.stage(pq ? codes_out : nullptr, pq ? (size_t)n * h->code_bytes() : 0));
    VIX_TRY(assign_lists_device(h, dx.dev, n, da.dev));
    if (pq) {
        unsigned long long invalid = 0;                 // rows without a list: the residual encoder would read coarse[-1]
        VIX_TRY(count_invalid_assign(da.dev, n, h->kc, &invalid));
        VIX_REQUIRE(invalid == 0, VIX_ERR_INVALID_PARAM, "vix_index_encode: %llu rows have no nearest list (NaN components?)", invalid);
    }
    if (pq) VIX_TRY(encode_rows_device(h, dx.dev, n, da.dev, dc.dev));
    VIX_TRY(da.commit());
    VIX_TRY(dc.commit());
    return finish(da.is_host() || dc.is_host());
}

}  // extern "C"
namespace vix {
int index_add_encoded_locked(vix_index* h, const int32_t* assign, const uint8_t* codes, const int64_t* ids, int64_t n) {
    VIX_REQUIRE(h->p.kind == VIX_INDEX_IVF_PQ && h->has_coarse && h->has_pq, VIX_ERR_NOT_TRAINED,
                "vix_index_add_encoded: needs a trained IVF-PQ index");
    if (n <= 0) return VIX_OK;
    VIX_REQUIRE(h->n + n < 0x7FFFFFFFLL, VIX_ERR_INVALID_PARAM, "index shard limited to 2^31 - 1 rows");
    VIX_TRY(is_device_ptr(ids) ? check_ids_device(ids, n) : check_ids_host(ids, n));
    cudaStream_t s = ctx().stream;
    {   // every row must name one of this index's lists: the scan layout is built from these ids
        In<int32_t> da;
        VIX_TRY(da.stage(assign, (size_t)n));
        unsigned long long invalid = 0;
        VIX_TRY(count_invalid_assign(da.dev, n, h->kc, &invalid));
        VIX_REQUIRE(invalid == 0, VIX_ERR_INVALID_PARAM, "vix_index_add_encoded: %llu of %lld list assignments lie outside [0, %d)",
                    invalid, (long long)n, h->kc);
    }
    const int64_t n0 = h->n;
    VIX_TRY(h->ids.resize((size_t)(n0 + n)));
    VIX_TRY(h->assign.resize((size_t)(n0 + n)));
    VIX_TRY(h->codes.resize((size_t)(n0 + n) * h->code_bytes()));
    VIX_CUDA(cudaMemcpyAsync(h->ids.ptr + n0, ids, (size_t)n * 8, cudaMemcpyDefault, s));
    VIX_CUDA(cudaMemcpyAsync(h->assign.ptr + n0, assign, (size_t)n * 4, cudaMemcpyDefault, s));
    VIX_CUDA(cudaMemcpyAsync(h->codes.ptr + (size_t)n0 * h->code_bytes(), codes, (size_t)n * h->code_bytes(), cudaMemcpyDefault, s));
    h->n = n0 + n;
    h->next_auto_id += n;
    h->dirty = true;
    return finish(true);
}

// The IVF-Flat sibling: rows whose lists are known, filed as index_add_locked files them (vectors, ids and assignments
// appended in order; the lists are rebuilt at the next search).  The assignment is taken as given, not recomputed.
int index_add_assigned_locked(vix_index* h, const int32_t* assign, const float* x, const int64_t* ids, int64_t n) {
    VIX_REQUIRE(h->p.kind == VIX_INDEX_IVF_FLAT && h->has_coarse, VIX_ERR_NOT_TRAINED,
                "index_add_assigned: needs an IVF-Flat index with coarse centroids");
    if (n <= 0) return VIX_OK;
    VIX_REQUIRE(h->n + n < 0x7FFFFFFFLL, VIX_ERR_INVALID_PARAM, "index shard limited to 2^31 - 1 rows");
    VIX_TRY(is_device_ptr(ids) ? check_ids_device(ids, n) : check_ids_host(ids, n));
    cudaStream_t s = ctx().stream;
    {
        In<int32_t> da;
        VIX_TRY(da.stage(assign, (size_t)n));
        unsigned long long invalid = 0;
        VIX_TRY(count_invalid_assign(da.dev, n, h->kc, &invalid));
        VIX_REQUIRE(invalid == 0, VIX_ERR_INVALID_PARAM, "index_add_assigned: %llu of %lld list assignments lie outside [0, %d)",
                    invalid, (long long)n, h->kc);
    }
    const int64_t n0 = h->n, d = h->p.d;
    VIX_TRY(h->ids.resize((size_t)(n0 + n)));
    VIX_TRY(h->assign.resize((size_t)(n0 + n)));
    VIX_TRY(h->vecs.resize((size_t)(n0 + n) * d));
    VIX_CUDA(cudaMemcpyAsync(h->ids.ptr + n0, ids, (size_t)n * 8, cudaMemcpyDefault, s));
    VIX_CUDA(cudaMemcpyAsync(h->assign.ptr + n0, assign, (size_t)n * 4, cudaMemcpyDefault, s));
    VIX_CUDA(cudaMemcpyAsync(h->vecs.ptr + (size_t)n0 * d, x, (size_t)n * d * 4, cudaMemcpyDefault, s));
    h->n = n0 + n;
    h->next_auto_id += n;
    h->dirty = true;
    return finish(true);
}

int index_add_rows_locked(vix_index* h, const float* x, const int64_t* ids, int64_t n) {
    return index_add_locked(h, x, ids, n);
}

int count_invalid_ids_device(const int64_t* ids, int64_t n, unsigned long long* count_dev) {
    if (n <= 0) return VIX_OK;
    count_invalid_ids_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx().stream>>>(ids, n, count_dev);
    VIX_LAUNCH_CHECK();
    return VIX_OK;
}

int select_probes_device(vix_index* h, const float* q, int64_t nq, int nprobe, int32_t* out) {
    if (h->p.metric == VIX_METRIC_COSINE)
        return probe_select_cosine_device(q, nq, h->coarse.ptr, h->kc, h->p.d, h->coarse_norms.ptr, nprobe, out);
    return probe_select_fast_device(q, nq, h->coarse.ptr, h->kc, h->p.d, h->p.metric, nprobe, h->coarse_norms.ptr, out, nullptr,
                                    h->coarse_norm_max.ptr);
}

int filter_row_mask(vix_index* h, const FilterArgs* filter, Scratch<uint64_t>& mask) {
    if (!filter || h->n == 0) return VIX_OK;
    const int64_t words = (h->n + 63) / 64;
    VIX_TRY(mask.alloc((size_t)words));
    filter_row_mask_kernel<<<(unsigned)((words + 255) / 256), 256, 0, ctx().stream>>>(h->ids.ptr, h->n, filter->words, filter->cap,
                                                                                    filter->deny, mask.ptr);
    VIX_LAUNCH_CHECK();
    return VIX_OK;
}
}  // namespace vix
extern "C" {

int vix_index_add_encoded(vix_index_t* h, const int32_t* assign, const uint8_t* codes, const int64_t* ids, int64_t n) {
    VIX_TRY(ensure_device());
    VIX_REQUIRE(h && (n == 0 || (assign && codes && ids)), VIX_ERR_NULL_PTR, "vix_index_add_encoded: null pointer");
    std::lock_guard<std::mutex> lk(h->mu);
    return index_add_encoded_locked(h, assign, codes, ids, n);
}

int vix_index_trace(vix_index_t* h, int capacity) {
    VIX_TRY(ensure_device());
    VIX_REQUIRE(h, VIX_ERR_NULL_PTR, "vix_index_trace: null handle");
    VIX_REQUIRE(capacity >= 0 && capacity <= 65536, VIX_ERR_INVALID_PARAM, "vix_index_trace: capacity");
    std::lock_guard<std::mutex> lk(h->mu);
    while ((int)h->trace_ev.size() < 5 * capacity) {
        cudaEvent_t e = nullptr;
        VIX_CUDA(cudaEventCreate(&e));
        h->trace_ev.push_back(e);
    }
    if (capacity > 0) {
        VIX_TRY(h->trace_scanned.resize((size_t)capacity, false));
        VIX_CUDA(cudaMemsetAsync(h->trace_scanned.ptr, 0, (size_t)capacity * 8, ctx().stream));
    }
    h->trace_path.assign((size_t)capacity, 0);
    h->trace_cap = capacity;
    h->trace_n = 0;
    return VIX_OK;
}

int vix_index_trace_get(vix_index_t* h, int i, vix_search_stats* out) {
    VIX_REQUIRE(h && out, VIX_ERR_NULL_PTR, "vix_index_trace_get: null pointer");
    std::lock_guard<std::mutex> lk(h->mu);
    VIX_REQUIRE(i >= 0 && i < h->trace_n, VIX_ERR_INVALID_PARAM, "vix_index_trace_get: %d of %d traced calls", i, h->trace_n);
    memset(out, 0, sizeof(*out));
    cudaEvent_t* ev = &h->trace_ev[5 * (size_t)i];
    VIX_CUDA(cudaEventSynchronize(ev[2]));
    unsigned long long sc = 0;
    VIX_CUDA(cudaMemcpy(&sc, h->trace_scanned.ptr + i, 8, cudaMemcpyDeviceToHost));
    out->codes_scanned = (int64_t)sc;
    out->code_bytes_scanned = (int64_t)sc * (h->p.kind == VIX_INDEX_IVF_PQ ? h->code_bytes() : h->p.d * 4);
    cudaEventElapsedTime(&out->ms_coarse, ev[0], ev[1]);
    cudaEventElapsedTime(&out->ms_scan, ev[1], ev[2]);
    cudaEventElapsedTime(&out->ms_total, ev[0], ev[2]);
    cudaEventElapsedTime(&out->ms_scan_kernel, ev[3], ev[4]);
    out->scan_path = h->trace_path[(size_t)i];
    return VIX_OK;
}

// Step 7 of the IVF-PQ query (docs/kernel-specs/DONE_22_adc_scan.md:873-878; IVFIndex.swift:1380-1439 does the same for
// its Kernel#30 lists): the ADC search keeps the R best candidates of a query, Kernel #40 re-scores them exactly against the
// original vectors and returns the k best by (exact score, smaller id).
int vix_index_search_rerank(vix_index_t* h, const float* queries, int64_t nq, int k, int nprobe, int rerank_r,
                            const float* xb, int64_t N, const float* xb_sq_norms, float* out_scores, int64_t* out_ids) {
    VIX_TRY(ensure_device());
    VIX_REQUIRE(h, VIX_ERR_NULL_PTR, "vix_index_search_rerank: null handle");
    if (k <= 0 || nq <= 0) return VIX_OK;
    VIX_REQUIRE(queries && xb && out_scores && out_ids, VIX_ERR_NULL_PTR, "vix_index_search_rerank: null pointer");
    VIX_REQUIRE(rerank_r >= k, VIX_ERR_INVALID_K, "vix_index_search_rerank: rerank_r (%d) must be >= k (%d) (ExactRerank.swift:730)", rerank_r, k);
    VIX_REQUIRE(rerank_r <= VIX_MAX_K_LARGE, VIX_ERR_INVALID_K, "vix_index_search_rerank: rerank_r > %d", VIX_MAX_K_LARGE);
    VIX_REQUIRE(h->p.metric != VIX_METRIC_COSINE, VIX_ERR_UNSUPPORTED, "vix_index_search_rerank: L2 / IP (Kernel #40's metrics on this path)");
    In<float> dq;
    VIX_TRY(dq.stage(queries, (size_t)nq * h->p.d));
    Scratch<float> cdist;
    Scratch<int64_t> cids;
    VIX_TRY(cdist.alloc((size_t)nq * rerank_r));
    VIX_TRY(cids.alloc((size_t)nq * rerank_r));
    {
        std::lock_guard<std::mutex> lk(h->mu);
        // candidates: approximate top-R (ids -1 pad short rows; the re-rank skips them as missing)
        const bool was_async = ctx().async;
        ctx().async = true;                                   // device outputs: no need to wait between the two stages
        const int rc = index_search_locked(h, dq.dev, nq, rerank_r, nprobe, cdist.ptr, cids.ptr, nullptr, nullptr);
        ctx().async = was_async;
        VIX_TRY(rc);
    }
    return vix_rerank_exact_topk_f32(dq.dev, nq, h->p.d, h->p.metric, cids.ptr, rerank_r, k, xb, N, xb_sq_norms, out_scores, out_ids);
}

int vix_index_search(vix_index_t* h, const float* queries, int64_t nq, int k, int nprobe, float* out_dist,
                     int64_t* out_ids) {
    return vix_index_search_ex(h, queries, nq, k, nprobe, out_dist, out_ids, nullptr, nullptr);
}

int vix_index_search_ex(vix_index_t* h, const float* queries, int64_t nq, int k, int nprobe, float* out_dist,
                        int64_t* out_ids, int32_t* out_probes, vix_search_stats* stats) {
    VIX_TRY(ensure_device());
    VIX_REQUIRE(h, VIX_ERR_NULL_PTR, "vix_index_search: null handle");
    std::lock_guard<std::mutex> lk(h->mu);
    return index_search_locked(h, queries, nq, k, nprobe, out_dist, out_ids, out_probes, stats);
}

}  // extern "C"
