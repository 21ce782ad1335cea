// vix_ivfpq_scan.cu -- the fused IVF-PQ list scan (query-only LUT -> ADC over the probed lists -> top-k).
//
// Reference composition: pq_lut_residual_l2_f32 -> adc_scan_u8 -> selectTopK -> mergeTopK
// (/root/reference/docs/kernel-specs/DONE_22_adc_scan.md:831-881; PQLUT.swift:266-386;
// ADCScan.swift:190-283; TopK.swift:54-176).  One persistent CTA per SM serves one query at a time:
//
//   ||q - x^||^2 = ||q - c_l||^2 + (||r^||^2 + 2<c_l, r^>) - 2<q, r^>,   x^ = c_l + r^
//                  bias (per probe)  t_x (per stored vector)     sum_j T[j][code_j],  T = -2<q_j, cb_j[.]>
//
// so ONE table per query serves every probed list (the reference builds one residual LUT per
// (query, list)); the result agrees with the reference's sum to fp32 rounding (1e-5, tested).
//
// The scan is bound by shared-memory look-ups (one per code byte; an SM retires 32 per clock, which at
// 1.9 GHz x 148 SMs is just above the HBM rate of the code stream), so the kernel spends exactly one
// conflict-free LDS, one PRMT and one FADD per code byte and nothing else in the inner loop:
//
//   * one stored vector per lane (no cross-lane reduction); a warp streams 32-slot chunks of the probed
//     lists with fully coalesced 128-bit loads (chunk-blocked code layout), the next chunk prefetched into registers;
//   * the table is code-major, T[code][64 slots] (256 B per code, 64 KB per table, one table per 32
//     sub-quantisers).  A 32-slot half row holds ONE group of 16 sub-quantisers twice (replica 0 | 1);
//     codes are stored "rotated" -- byte b of slot g holds sub-quantiser (b & ~15) | ((b ^ g) & 15) -- so
//     at byte position b the 16 lanes of a half-warp ask for 16 different sub-quantisers and the two
//     half-warps use the two replicas: every warp-wide look-up touches 32 different banks whatever the
//     codes are;
//   * the tables start at a 64 KB-aligned SHARED address, so the complete LDS address
//     (table | code << 8 | 4 * slot) is ONE byte-permute of the packed code word with a per-lane
//     constant; the group / table select is the LDS immediate.
//
// Top-k: per-warp shared-memory queues keyed (score, id) under a CTA-wide acceptance threshold that every warp re-reads
// each chunk; the k-th smallest of a warp's first chunk seeds it, and the k-th smallest of every 32 accepted entries
// lowers it (one shuffle network) -- a queue is sorted only when it overflows.  At the end of a query every warp
// publishes the entries that can still make the top k.  No distance array ever reaches HBM.
//
// Pipeline across queries (one CTA per SM, 16 warps): while the CTA scans query i, warp 1 first stages what query i + 1
// needs besides its table -- the query (to shared memory), the probe table of the lists that are not empty on this GPU
// and their bias terms -- and warp 0 first selects the k best of what query i - 1 published; chunks are handed out
// dynamically (runs of 4, 2, 1), so nobody waits for either.  The per-query serial part is the table build (all warps)
// between two CTA barriers.  Queries are handed out by an atomic counter in an order sorted by the first probed list that
// holds vectors here, so CTAs running concurrently scan neighbouring lists and share them through L2.
// Large d / large codebooks: the bias terms and the tables are built batch-wide instead (probe_bias_kernel,
// lut_image_kernel) and the scan copies a query's table image with cp.async.
#include <stdlib.h>

#include "vix_common.cuh"
#include "vix_topk.cuh"
#include "vix_scan.cuh"
#include "vix_scan_select.cuh"

namespace vix {

#ifndef VIX_SCAN_THREADS
#define VIX_SCAN_THREADS 512
#endif
#ifndef VIX_SCAN_FN
#define VIX_SCAN_FN __noinline__
#endif
#ifndef VIX_SCAN_GUIDED
#define VIX_SCAN_GUIDED 1    // runs shrink towards the end of a query
#endif
constexpr int kFastThreads = VIX_SCAN_THREADS;   // one CTA per SM
constexpr int kScanWarps = 8;              // generic kernel
constexpr int kScanThreads = kScanWarps * 32;

template <int IMM>
__device__ __forceinline__ float lds_imm(uint32_t addr) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1+%2];" : "=f"(v) : "r"(addr), "n"(IMM));
    return v;
}

// two look-ups whose results land in a 64-bit register pair, added to a pair of running sums with ONE packed
// add (add.rn.f32x2, sm_100): (lo, hi) += (T[a0], T[a1])
template <int IMM>
__device__ __forceinline__ void lookup2(uint32_t a0, uint32_t a1, unsigned long long& acc) {
    asm volatile(
        "{\n\t.reg .f32 lo, hi;\n\t.reg .b64 pr;\n\t"
        "ld.shared.f32 lo, [%1+%3];\n\t"
        "ld.shared.f32 hi, [%2+%3];\n\t"
        "mov.b64 pr, {lo, hi};\n\t"
        "add.rn.f32x2 %0, %0, pr;\n\t}"
        : "+l"(acc)
        : "r"(a0), "r"(a1), "n"(IMM));
}

// one group of 16 sub-quantisers: 16 look-ups of one lane, 4 running sums kept as two f32x2 pairs (s0, s1), (s2, s3).
// Group T: table T / 2, half row T % 2.
template <int T>
__device__ __forceinline__ void lookup16(const uint4& w, const uint32_t (&pre)[8], unsigned long long& s01,
                                         unsigned long long& s23) {
    constexpr int IMM = (T & 1) * 128 + (T >> 1) * 65536;
    const uint32_t x[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        // result bytes: [0] = 4 * slot (lane constant; two per register), [1] = code, [2..3] = table address >> 16
        lookup2<IMM>(__byte_perm(x[i], pre[2 * i + 0], 0x7604), __byte_perm(x[i], pre[2 * i + 0], 0x7615), s01);
        lookup2<IMM>(__byte_perm(x[i], pre[2 * i + 1], 0x7624), __byte_perm(x[i], pre[2 * i + 1], 0x7635), s23);
    }
}

// codes of slot g: chunk-blocked layout -- inside a 32-slot chunk the 16-byte piece c of every slot is stored
// contiguously ([c][slot][16]), so each of the G 128-bit loads of a warp reads 512 consecutive bytes (16 full sectors)
template <int G>
__device__ __forceinline__ void load_codes(uint4 (&w)[G], const uint8_t* __restrict__ codes, uint32_t g) {
    // every slot of a chunk exists in memory (lists are padded to whole chunks; padding holds code 0), so the
    // loads need no predicate
    const uint4* src = reinterpret_cast<const uint4*>(codes + (size_t)(g >> 5) * (512u * G)) + (g & 31u);
#pragma unroll
    for (int c = 0; c < G; ++c) w[c] = __ldg(src + 32 * c);
}

__device__ __forceinline__ u64 shfl_xor_u64(u64 v, int o) {
    return __shfl_xor_sync(0xFFFFFFFFu, v, o);
}

// per-probe term of the decomposition, ||q - c_l||^2 (L2) or <q, c_l> (IP), batch-wide: one warp per (query, probe) whose
// list holds vectors here.  Used when d is large: inside the scan kernel ONE warp per CTA computes these terms for the
// next query while the others scan, which stops being free once d x nprobe outgrows a query's scan time.
__global__ void __launch_bounds__(256)
probe_bias_kernel(const float* __restrict__ queries, const int32_t* __restrict__ probes, const float* __restrict__ coarse,
                  const int32_t* __restrict__ list_len, int kc, int64_t npairs, int nprobe, int d, int order_max,
                  float* __restrict__ bias) {
    const int lane = threadIdx.x & 31;
    const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (w >= npairs) return;
    const int l = probes[w];
    float part = 0.0f;
    if ((unsigned)l < (unsigned)kc && __ldg(list_len + l) > 0) {
        const float* q = queries + (w / nprobe) * (int64_t)d;
        const float* c = coarse + (int64_t)l * d;
        if (order_max) for (int e = lane; e < d; e += 32) part = fmaf(__ldg(q + e), __ldg(c + e), part);
        else for (int e = lane; e < d; e += 32) { const float df = __ldg(q + e) - __ldg(c + e); part = fmaf(df, df, part); }
    }
    for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xFFFFFFFFu, part, o);
    if (lane == 0) bias[w] = part;
}

// one warp, while the other warps scan the previous query: everything a query needs besides its look-up table.
//   * the query itself, copied to shared memory (the table build reads it from there);
//   * the probe table -- first slot / 32, length and exclusive prefix of the chunk counts of the probed lists that are
//     NOT EMPTY here (a shard holds only its block of lists; the other probes are dropped, so the scan never walks
//     over them);
//   * the per-probe term of the decomposition, ||q - c_l||^2 (L2) or <q, c_l> (IP), for those lists.
__device__ VIX_SCAN_FN void build_probe_table(const float* __restrict__ q, int d, const float* __restrict__ coarse,
                                               int order_max, const int32_t* __restrict__ qprobes,
                                               const float* __restrict__ qbias, int nprobe,
                                               const int64_t* __restrict__ list_off, const int32_t* __restrict__ list_len, int kc,
                                               int* s_start, int* s_len, int* s_pref, float* s_bias, int* s_np,
                                               float* s_q) {
    const int lane = threadIdx.x & 31;
    int lv[8], lenv[8];
    int64_t offv[8];
    float bv[8];
#pragma unroll
    for (int it = 0; it < 8; ++it) {
        const int p = 32 * it + lane;
        lv[it] = (p < nprobe) ? __ldg(qprobes + p) : -1;
        bv[it] = (qbias && p < nprobe) ? __ldg(qbias + p) : 0.0f;
    }
    for (int e = lane; e < d; e += 32) s_q[e] = __ldg(q + e);
#pragma unroll
    for (int it = 0; it < 8; ++it) {
        offv[it] = 0; lenv[it] = 0;
        if ((unsigned)lv[it] < (unsigned)kc) { offv[it] = __ldg(list_off + lv[it]); lenv[it] = __ldg(list_len + lv[it]); }
    }
    int carry = 0, np = 0;
    int* s_list = reinterpret_cast<int*>(s_bias);          // list ids first, overwritten by the bias below
#pragma unroll
    for (int it = 0; it < 8; ++it) {
        if (32 * it < nprobe) {
            const int nch = (lenv[it] + 31) >> 5;
            int inc = nch;
            for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xFFFFFFFFu, inc, o); if (lane >= o) inc += t; }
            const unsigned ball = __ballot_sync(0xFFFFFFFFu, nch > 0);
            if (nch > 0) {
                const int p = np + __popc(ball & ((1u << lane) - 1u));
                s_start[p] = (int)(offv[it] >> 5); s_len[p] = lenv[it]; s_pref[p] = carry + inc - nch;
                if (qbias) s_bias[p] = bv[it]; else s_list[p] = lv[it];
            }
            np += __popc(ball);
            carry += __shfl_sync(0xFFFFFFFFu, inc, 31);
        }
    }
    // probes 256 .. VIX_MAX_K - 1 (rare): the same rounds, one at a time
    for (int p0 = 256; p0 < nprobe; p0 += 32) {
        const int pp = p0 + lane;
        const int l = (pp < nprobe) ? __ldg(qprobes + pp) : -1;
        const bool ok = (unsigned)l < (unsigned)kc;
        const int len = ok ? __ldg(list_len + l) : 0;
        const int nch = (len + 31) >> 5;
        int inc = nch;
        for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xFFFFFFFFu, inc, o); if (lane >= o) inc += t; }
        const unsigned ball = __ballot_sync(0xFFFFFFFFu, nch > 0);
        if (nch > 0) {
            const int p = np + __popc(ball & ((1u << lane) - 1u));
            s_start[p] = (int)(__ldg(list_off + l) >> 5); s_len[p] = len; s_pref[p] = carry + inc - nch;
            if (qbias) s_bias[p] = __ldg(qbias + pp); else s_list[p] = l;
        }
        np += __popc(ball);
        carry += __shfl_sync(0xFFFFFFFFu, inc, 31);
    }
    if (lane == 0) { s_pref[np] = carry; *s_np = np; }
    __syncwarp();
    if (qbias) return;                                     // precomputed batch-wide (probe_bias_kernel)
    // bias: lane-strided partial sums, xor-tree across the warp; four lists in flight
    for (int p0 = 0; p0 < np; p0 += 4) {
        float part[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            part[u] = 0.0f;
            if (p0 + u < np) {
                const float* c = coarse + (int64_t)s_list[p0 + u] * d;
                if (order_max) for (int e = lane; e < d; e += 32) part[u] = fmaf(s_q[e], __ldg(c + e), part[u]);
                else for (int e = lane; e < d; e += 32) { const float df = s_q[e] - __ldg(c + e); part[u] = fmaf(df, df, part[u]); }
            }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u)
            for (int o = 16; o > 0; o >>= 1) part[u] += __shfl_xor_sync(0xFFFFFFFFu, part[u], o);
        if (lane < 4 && p0 + lane < np) s_bias[p0 + lane] = lane == 0 ? part[0] : lane == 1 ? part[1] : lane == 2 ? part[2] : part[3];
    }
}

// every warp: T[c][slot(j)] = scale * <q_j, cb_j[c]>.  Thread t of the `nthr` builders owns ONE sub-quantiser
// j = t % M (its query slice stays in registers) and walks the codes c = t / M, t / M + nthr / M, ...;
// codebooks_t is [256][M][dsub], so the M threads of a code read consecutive memory.  The build is bound by the
// latency of those (L2-resident) reads, so as many codes as the registers hold are in flight per thread: all of
// a thread's codes at dsub = 2 (one round trip), eight otherwise.  The two replicas of an entry are written in
// opposite order by the two half-warps, so a warp-wide store touches 32 different banks.  Group t16 goes to table t16 / 2,
// half row t16 % 2.
template <int M>
__device__ VIX_SCAN_FN void build_lut(float* __restrict__ s_lut, const float* __restrict__ q,
                                      const float* __restrict__ codebooks_t, int dsub, float lut_scale, int t, int nthr) {
    const int ngroups = nthr / M;
    if (t >= ngroups * M) return;
    const int j = t % M, c0 = t / M;
    const int rep_first = (threadIdx.x & 31) >> 4;
    const int t16 = j >> 4;
    float* col = s_lut + (t16 >> 1) * 16384 + (t16 & 1) * 32 + (j & 15);
    float* colA = col + 16 * rep_first;
    float* colB = col + 16 * (rep_first ^ 1);
    constexpr int U = 8;
    if (dsub == 2) {
        // codes per thread with a full CTA of builders: ceil(256 / (512 / M))
        constexpr int U2 = (256 + (kFastThreads / M) - 1) / (kFastThreads / M);
        const float q0 = q[j * 2] * lut_scale, q1 = q[j * 2 + 1] * lut_scale;
        for (int c = c0; c < 256; c += U2 * ngroups) {
            float2 v[U2];
#pragma unroll
            for (int u = 0; u < U2; ++u) {
                const int cu = min(c + u * ngroups, 255);
                v[u] = __ldg(reinterpret_cast<const float2*>(codebooks_t + ((size_t)cu * M + j) * 2));
            }
#pragma unroll
            for (int u = 0; u < U2; ++u) {
                const int cu = c + u * ngroups;
                const float dot = lut_entry2(q0, q1, v[u]);
                if (cu < 256) { colA[cu * 64] = dot; colB[cu * 64] = dot; }
            }
        }
    } else if (dsub <= 16) {
        float qv[16];
#pragma unroll
        for (int e = 0; e < 16; ++e) qv[e] = (e < dsub) ? q[j * dsub + e] * lut_scale : 0.0f;
        for (int c = c0; c < 256; c += U * ngroups) {
            float dot[U];
            if ((dsub & 3) == 0) {
#pragma unroll
                for (int u = 0; u < U; ++u) dot[u] = 0.0f;
#pragma unroll
                for (int e = 0; e < 16; e += 4) {
                    if (e < dsub) {
                        float4 v[U];
#pragma unroll
                        for (int u = 0; u < U; ++u) {
                            const int cu = min(c + u * ngroups, 255);
                            v[u] = __ldg(reinterpret_cast<const float4*>(codebooks_t + ((size_t)cu * M + j) * dsub + e));
                        }
#pragma unroll
                        for (int u = 0; u < U; ++u)
                            dot[u] = fmaf(qv[e + 3], v[u].w, fmaf(qv[e + 2], v[u].z, fmaf(qv[e + 1], v[u].y, fmaf(qv[e], v[u].x, dot[u]))));
                    }
                }
            } else {
#pragma unroll
                for (int u = 0; u < U; ++u) dot[u] = 0.0f;
#pragma unroll
                for (int e = 0; e < 16; ++e) {
                    if (e < dsub) {
#pragma unroll
                        for (int u = 0; u < U; ++u) {
                            const int cu = min(c + u * ngroups, 255);
                            dot[u] = fmaf(qv[e], __ldg(codebooks_t + ((size_t)cu * M + j) * dsub + e), dot[u]);
                        }
                    }
                }
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int cu = c + u * ngroups;
                if (cu < 256) { colA[cu * 64] = dot[u]; colB[cu * 64] = dot[u]; }
            }
        }
    } else {
        for (int c = c0; c < 256; c += ngroups) {
            const float* cw = codebooks_t + ((size_t)c * M + j) * dsub;
            float dot = 0.0f;
            for (int e = 0; e < dsub; ++e) dot = fmaf(q[j * dsub + e], __ldg(cw + e), dot);
            dot *= lut_scale;
            colA[c * 64] = dot; colB[c * 64] = dot;
        }
    }
}

// the table was built batch-wide (lut_image_kernel): copy its image with asynchronous 16-byte copies -- every piece of
// a thread is in flight at once and none of them holds a register.  The image is COMPACT ([table][code][32 slots]: one
// copy of every entry, half the bytes to write and to read back); the two replicas of a shared-memory row are made here,
// each 16-byte source piece going to both.
__device__ VIX_SCAN_FN void copy_lut_image(float* __restrict__ s_lut, const float* __restrict__ image, int npieces, int t, int nthr) {
    const float4* src = reinterpret_cast<const float4*>(image);
    const uint32_t dst = (uint32_t)__cvta_generic_to_shared(s_lut);
    for (int i = t; i < npieces; i += nthr) {
        // piece i: table i / 2048, code (i / 8) % 256, group parity (i / 4) % 2, four entries 4 (i % 4) .. of the group
        const uint32_t row = (uint32_t)(i >> 3), w = (uint32_t)i & 7u;
        const uint32_t d0 = dst + row * 256u + (w >> 2) * 128u + (w & 3u) * 16u;
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d0), "l"(src + i));
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d0 + 64u), "l"(src + i));
    }
    asm volatile("cp.async.commit_group;");
    asm volatile("cp.async.wait_group 0;" ::: "memory");
}

// The same tables for a whole batch, written to global memory as images of the scan's shared-memory layout
// ([query][table][code][64 slots], both replicas).  Building a table inside the scan kernel re-reads the codebooks
// (m x 256 x dsub floats) from L2 once per query and CTA: at dsub = 12, m = 64 that is 786 KB per query against 64 KB of
// table, and the scan kernel sits at the L2 bandwidth for a third of its time.  Here a CTA takes one table (32
// sub-quantisers) and kImgQT queries; a WARP takes one code at a time and lane = sub-quantiser, so the 32 codebook vectors
// of a code are one contiguous read (codebooks_t is [code][m][dsub]) shared by the kImgQT queries, and the warp writes the
// code's whole 256-byte row (2 groups x 2 replicas x 16) of every query.  Same operation order as build_lut (query
// pre-scaled, ascending fused multiply-adds), so both paths give the same bits.
constexpr int kImgQT = 8;       // queries per CTA
template <int M>
__global__ void __launch_bounds__(256)
lut_image_kernel(const float* __restrict__ queries, int64_t nq, int d, const float* __restrict__ codebooks_t, int dsub,
                 float lut_scale, float* __restrict__ image) {
    constexpr int NTAB = (M / 16 + 1) / 2;
    __shared__ float s_q[kImgQT][32 * 17];                 // [query][sub-quantiser][dsub <= 16], pitch 17: conflict-free
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int tab = blockIdx.y;                            // table = 32 sub-quantisers
    const int64_t q0 = (int64_t)blockIdx.x * kImgQT;
    const int j = tab * 32 + lane;                         // this lane's sub-quantiser
    const bool live = j < M;
    for (int i = threadIdx.x; i < kImgQT * 32 * dsub; i += blockDim.x) {
        const int qi = i / (32 * dsub), r = i - qi * 32 * dsub, jj = r / dsub, e = r - jj * dsub;
        const bool ok = q0 + qi < nq && tab * 32 + jj < M;
        s_q[qi][jj * 17 + e] = ok ? __ldg(queries + (q0 + qi) * d + (tab * 32 + jj) * dsub + e) * lut_scale : 0.0f;
    }
    __syncthreads();
    // compact image: [table][code][32 slots], slot = 16 * ((j / 16) & 1) + j % 16 = the lane (copy_lut_image makes the replicas)
    float* rowbase = image + (size_t)q0 * (NTAB * 8192) + (size_t)tab * 8192 + lane;
    for (int c = warp; c < 256; c += 8) {
        float cv[16];
        if (live) {
            const float* src = codebooks_t + ((size_t)c * M + j) * dsub;
            if ((dsub & 3) == 0) {
#pragma unroll
                for (int e = 0; e < 16; e += 4)
                    if (e < dsub) {
                        const float4 v = __ldg(reinterpret_cast<const float4*>(src + e));
                        cv[e] = v.x; cv[e + 1] = v.y; cv[e + 2] = v.z; cv[e + 3] = v.w;
                    }
            } else {
#pragma unroll
                for (int e = 0; e < 16; ++e) if (e < dsub) cv[e] = __ldg(src + e);
            }
        }
#pragma unroll
        for (int qi = 0; qi < kImgQT; ++qi) {
            float dot = 0.0f;
#pragma unroll
            for (int e = 0; e < 16; ++e) if (e < dsub) dot = fmaf(s_q[qi][lane * 17 + e], cv[e], dot);
            if (live && q0 + qi < nq) {
                rowbase[(size_t)qi * (NTAB * 8192) + c * 32] = dot;      // one coalesced 128-byte row per warp
            }
        }
    }
}

// one warp: sort the queue (k best first), refresh the thresholds
__device__ __noinline__ uint32_t flush_queue(u64* wq, int Pw, int k, int cnt, bool sorted_valid, uint32_t thr_u, int* s_thr) {
    const int lane = threadIdx.x & 31;
    if (!sorted_valid) for (int t = lane; t < k; t += 32) wq[t] = kEmptyKey;
    for (int t = k + cnt + lane; t < Pw; t += 32) wq[t] = kEmptyKey;
    __syncwarp();
    bitonic_sort_keys<true>(wq, Pw, lane, 32);
    const u64 t = wq[k - 1];
    if (t != kEmptyKey) {
        const uint32_t tu = (uint32_t)(t >> 32);
        if (tu < thr_u) thr_u = tu;
        if (lane == 0) atomicMin(reinterpret_cast<unsigned int*>(s_thr), tu);
    }
    return thr_u;
}

// m = 16 G; FILTER: an id filter is active; STATS: the phase counters of vix_search_stats are kept (separate
// instantiations, so the production kernel pays neither in instructions nor in registers).
template <int G, bool FILTER, bool STATS>
__global__ void __launch_bounds__(kFastThreads, 1)
ivfpq_scan_kernel(ScanArgs a) {
    constexpr int m = 16 * G;
    constexpr int NTAB = (G + 1) / 2;
    constexpr int kGrab = 4;                             // largest run of chunks handed to a warp at once
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int tid = (int)threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nwarps = (int)(blockDim.x >> 5);

    // ---- shared-memory map: bookkeeping first, then the tables ----
    // probe tables, double buffered (the next query's is built while this one is scanned):
    // [bias nprobe][first slot / 32 nprobe][length nprobe][chunk prefix nprobe + 1]
    const int pt_words = 4 * a.nprobe + 1;
    int* s_pt = reinterpret_cast<int*>(smem_raw);                         // [2][pt_words]
    float* s_qv = reinterpret_cast<float*>(s_pt + 2 * pt_words);          // [2][d] the queries themselves
    int* s_np = reinterpret_cast<int*>(s_qv + 2 * a.d);                   // [2] non-empty probes of the query
    int* s_item = s_np + 2;                                               // [2] work items (double buffered)
    int* s_thr = s_item + 2;                                              // [1] CTA acceptance threshold
    int* s_ncand = s_thr + 1;                                             // [2] candidates published for the merge
    int* s_next = s_ncand + 2;                                            // [1] next chunk to hand out
    u64* s_wq = reinterpret_cast<u64*>((reinterpret_cast<uintptr_t>(s_next + 1) + 15) & ~(uintptr_t)15);
    u64* s_cand = s_wq + (size_t)nwarps * a.Pw;                           // [2][nwarps * Pw] published candidates
    unsigned char* misc_end = reinterpret_cast<unsigned char*>(s_cand + 2 * (size_t)nwarps * a.Pw);
    const uint32_t dyn_abs = (uint32_t)__cvta_generic_to_shared(smem_raw);
    // tables at the first 64 KB boundary behind the bookkeeping (the address travels in the lane constants)
    const uint32_t tab_abs = (dyn_abs + (uint32_t)(misc_end - smem_raw) + 65535u) & ~65535u;
    float* s_lut = reinterpret_cast<float*>(smem_raw + (tab_abs - dyn_abs)); // NTAB x [256][64]
    if (tab_abs - dyn_abs + NTAB * 65536u > (uint32_t)a.smem_bytes) {
        if (threadIdx.x == 0 && blockIdx.x == 0 && a.status) *a.status = 1;
        return;
    }

    const int order_max = (a.metric == VIX_METRIC_IP);
    const float lut_scale = order_max ? 1.0f : -2.0f;
    u64* wq = s_wq + (size_t)warp * a.Pw;
    unsigned long long scanned_local = 0;
#ifdef VIX_SCAN_DIAG
    unsigned long long diag = 0;     // chunks [0, 24) | queue flushes [24, 44) | chunks with a passing entry [44, 64)
#endif
    volatile uint32_t* cta_thr = reinterpret_cast<volatile uint32_t*>(s_thr);
    volatile int* v_next = reinterpret_cast<volatile int*>(s_next);

    // per-lane look-up constants
    // (byte b of a group: slot byte offset 4 * (16 * replica + ((b ^ lane) & 15)); packed two per register under
    // the table address, whose low 16 bits are zero)
    uint32_t pre[8];
#pragma unroll
    for (int b = 0; b < 16; b += 2) {
        const uint32_t c0 = 4u * (16u * (lane >> 4) + ((b ^ lane) & 15));
        const uint32_t c1 = 4u * (16u * (lane >> 4) + (((b + 1) ^ lane) & 15));
        pre[b >> 1] = tab_abs | c0 | (c1 << 8);
        asm volatile("" : "+r"(pre[b >> 1]));  // opaque: keep the constants in registers, never recompute them
    }

    // probe table of work item `item` into buffer b (one warp)
    // work items: every query, or (tensor-core path: the queries it hands back) the first *nq_dev entries of `order`
    const int nq_items = a.nq_dev ? *a.nq_dev : (int)a.nq;
    auto probe_table = [&](int item, int b) {
        if (item >= nq_items) return;
        const int64_t qn = a.order ? a.order[item] : item;
        int* pt = s_pt + b * pt_words;
        build_probe_table(a.queries + qn * (int64_t)a.d, a.d, a.coarse, order_max, a.probes + qn * (int64_t)a.nprobe,
                          a.bias ? a.bias + qn * (int64_t)a.nprobe : nullptr, a.nprobe, a.list_off, a.list_len, a.kc,
                          pt + a.nprobe, pt + 2 * a.nprobe, pt + 3 * a.nprobe, reinterpret_cast<float*>(pt), s_np + b,
                          s_qv + b * a.d);
    };

    if (tid == 32) { s_item[0] = atomicAdd(a.work_counter, 1); s_ncand[0] = 0; s_ncand[1] = 0; }
    __syncthreads();
    if (warp == 1) {
        probe_table(s_item[0], 0);
        if (lane == 0) s_item[1] = atomicAdd(a.work_counter, 1);
    }
    __syncthreads();
    int buf = 0;
    bool have_prev = false;
    int64_t prev_qi = 0;
    long long t_mark = STATS ? clock64() : 0;
    unsigned long long cyc_pro = 0, cyc_scan = 0, cyc_tail = 0;
    for (;;) {
        const int item = s_item[buf];
        const bool more = item < nq_items;
        const int64_t qi = more ? (a.order ? a.order[item] : item) : 0;
        const float* q = s_qv + buf * a.d;
        const int* pt = s_pt + buf * pt_words;
        const float* p_bias = reinterpret_cast<const float*>(pt);
        const int* p_start = pt + a.nprobe;
        const int* p_len = pt + 2 * a.nprobe;
        const int* p_pref = pt + 3 * a.nprobe;
        const int nchunks = more ? p_pref[s_np[buf]] : 0;

        if (more) {
            // ---- prologue: the table; the first run of chunks of every warp is fixed (warp w: chunks [4 w, 4 w + 4)) ----
            if (tid == 32) { *cta_thr = 0xFFFFFFFFu; *s_next = nwarps * kGrab; }
            const long long t0 = STATS ? clock64() : 0;
            if (nchunks > 0) {
                if (a.lut_image) copy_lut_image(s_lut, a.lut_image + (size_t)qi * (NTAB * 8192), NTAB * 2048, tid, (int)blockDim.x);
                else build_lut<m>(s_lut, q, a.codebooks_t, a.dsub, lut_scale, tid, (int)blockDim.x);
            }
            if (STATS && a.phase_cycles && tid == 64) atomicAdd(a.phase_cycles + 5, (unsigned long long)(clock64() - t0));
        }
        __syncthreads();                               // (1) table ready; s_item[buf] has been read by everybody
        // ---- warp 0 first selects the k best of the candidates published for the PREVIOUS query and warp 1 builds
        //      the NEXT query's probe table; the other warps are already scanning, and chunks are handed out
        //      dynamically, so nobody waits for either
        if (warp == 0 && have_prev) {
            const long long t0 = STATS ? clock64() : 0;
            if (STATS && a.phase_cycles && lane == 0) atomicAdd(a.phase_cycles + 6, (unsigned long long)s_ncand[buf ^ 1]);
            select_and_write(s_cand + (size_t)(buf ^ 1) * nwarps * a.Pw, s_ncand[buf ^ 1], a.k, order_max, prev_qi, a.out_dist,
                             a.out_ids);
            __syncwarp();
            if (lane == 0) s_ncand[buf ^ 1] = 0;
            if (STATS && a.phase_cycles && lane == 0) atomicAdd(a.phase_cycles + 3, (unsigned long long)(clock64() - t0));
        }
        if (!more) break;
        if (warp == 1) {
            const long long t0 = STATS ? clock64() : 0;
            probe_table(s_item[buf ^ 1], buf ^ 1);
            if (lane == 0) s_item[buf] = atomicAdd(a.work_counter, 1);   // the item after the next
            if (STATS && a.phase_cycles && lane == 0) atomicAdd(a.phase_cycles + 4, (unsigned long long)(clock64() - t0));
        }
        if (STATS) { const long long t = clock64(); cyc_pro += (unsigned long long)(t - t_mark); t_mark = t; }

        // ---- scan: 32-slot chunks of the probed lists, handed out dynamically ----
        int cnt = 0;                                       // unsorted candidates behind the k sorted ones
        bool sorted_valid = false;                         // wq[0, k) holds a sorted best list
        uint32_t thr_u = 0xFFFFFFFFu;
        int p = 0;
        uint4 wA[G], wB[G];
        // Chunks are handed out CTA-wide in runs of 4, 2 and, near the end, 1 (so the warps finish together); a warp
        // takes its next run when the current one [ch, grab_end) is used up.  (Measured and dropped: taking a run ahead
        // and prefetch.global.L2-ing it -- 7 % slower; L2 prefetch of just the next chunk -- no gain; stepping through a
        // run with pointer increments instead of re-locating every chunk -- fewer instructions, yet 7 % slower.)
        int grab_end = warp * kGrab + kGrab;
        auto grab = [&](int prev) {
            if (prev + 1 < grab_end) return prev + 1;
            int c = 0, g = 0;
            if (lane == 0) {
#if VIX_SCAN_GUIDED
                const int rem = nchunks - *v_next;
                g = rem >= 8 * nwarps ? kGrab : (rem >= 3 * nwarps ? 2 : 1);
#else
                g = kGrab;
#endif
                c = atomicAdd(s_next, g);
            }
            c = __shfl_sync(0xFFFFFFFFu, c, 0);
            grab_end = c + __shfl_sync(0xFFFFFFFFu, g, 0);
            return c;
        };
        int ch = warp * kGrab;
        // the probe the warp is in is cached in registers: chunk range [pb, pe), first slot / 32, length, bias
        int pb = 0, pe = 0, pstart = 0, plen = 0;
        float pbias = 0.0f;
        uint32_t cg = 0;                                   // slot of this lane in the current chunk (< 2^31 slots)
        bool cvalid = false;
        float ctx_ = 0.0f, cbias = 0.0f;                   // t_x and bias of the current chunk (prefetched)
        auto locate = [&]() {                              // position of chunk `ch` (chunk indices only grow)
            if (ch >= pe) {
                while (ch >= p_pref[p + 1]) ++p;
                pb = p_pref[p]; pe = p_pref[p + 1]; pstart = p_start[p]; plen = p_len[p]; pbias = p_bias[p];
            }
            const int within = (ch - pb) * 32 + lane;
            cvalid = within < plen;
            cg = ((uint32_t)pstart << 5) + (uint32_t)within;
            cbias = pbias;
        };
        if (ch < nchunks) {
            locate();
            load_codes<G>(wA, a.slot_codes, cg);
            ctx_ = __ldg(a.slot_tx + cg);                  // padding slots hold t_x = 0
        }
        // one chunk: prefetch this warp's next chunk into wn, look the current one (wc) up, select
        auto do_chunk = [&](uint4 (&wc)[G], uint4 (&wn)[G]) {
            const float tx = ctx_;
            const uint32_t g = cg;
            const bool valid = cvalid;
            const float bias = cbias;
            const uint32_t cta_t = *cta_thr;               // the CTA-wide acceptance threshold, refreshed every chunk
#ifdef VIX_SCAN_DIAG
            diag += 1ull;
#endif
#define VIX_ADVANCE()                                                         \
            ch = grab(ch);                                                        \
            if (ch < nchunks) {                                                   \
                locate();                                                         \
                load_codes<G>(wn, a.slot_codes, cg);                              \
                ctx_ = __ldg(a.slot_tx + cg);                                     \
            }
#ifndef VIX_SCAN_NOPREFETCH
            VIX_ADVANCE()
#endif
            unsigned long long s01 = 0ull, s23 = 0ull;     // (s0, s1), (s2, s3) as f32x2 pairs
            lookup16<0>(wc[0], pre, s01, s23);
            if (G > 1) lookup16<1>(wc[G > 1 ? 1 : 0], pre, s01, s23);
            if (G > 2) lookup16<2>(wc[G > 2 ? 2 : 0], pre, s01, s23);
            if (G > 3) lookup16<3>(wc[G > 3 ? 3 : 0], pre, s01, s23);
            const float s0 = __uint_as_float((uint32_t)s01), s1 = __uint_as_float((uint32_t)(s01 >> 32));
            const float s2 = __uint_as_float((uint32_t)s23), s3 = __uint_as_float((uint32_t)(s23 >> 32));
#ifdef VIX_SCAN_NOPREFETCH
            VIX_ADVANCE()
#endif
#undef VIX_ADVANCE
            const float sum = (bias + tx) + ((s0 + s1) + (s2 + s3));
            if (valid) ++scanned_local;
            const u64 key = make_key(sum, 0u, order_max);
            uint32_t ku = valid ? (uint32_t)(key >> 32) : 0xFFFFFFFFu;
            thr_u = min(thr_u, cta_t);
            uint32_t fid = 0;
            bool fchecked = false, fdrop = false;
            if (FILTER && thr_u == 0xFFFFFFFFu) {
                // no threshold yet: every entry of the chunk meets the filter now (the bound below must only count
                // entries that can be returned); afterwards only entries that beat the threshold are looked up
                if (valid) {
                    fid = (uint32_t)a.slot_ids[g];
                    fdrop = !id_filter_pass(a.filter, a.filter_cap, a.filter_deny, (int64_t)fid);
                    if (fdrop) ku = 0xFFFFFFFFu;
                }
                fchecked = true;
            }
            if (thr_u == 0xFFFFFFFFu && a.k <= 32) {
                // no threshold yet: the k-th smallest of this chunk bounds the final k-th best
                const uint32_t kth = warp_kth_smallest(ku, a.k - 1, lane);
                if (kth != 0xFFFFFFFFu) {
                    thr_u = kth;
                    if (lane == 0) atomicMin(reinterpret_cast<unsigned int*>(s_thr), kth);
                }
            }
            bool pass = valid && !fdrop && (ku <= thr_u);
            if (FILTER && !fchecked && pass) {
                fid = (uint32_t)a.slot_ids[g];
                pass = id_filter_pass(a.filter, a.filter_cap, a.filter_deny, (int64_t)fid);
            }
            const unsigned ball = __ballot_sync(0xFFFFFFFFu, pass);
            if (ball) {
                if (cnt + 32 > a.Pw - a.k) {
                    thr_u = flush_queue(wq, a.Pw, a.k, cnt, sorted_valid, thr_u, s_thr);   // make room: keep the k best
                    cnt = 0; sorted_valid = true;
#ifdef VIX_SCAN_DIAG
                    diag += 1ull << 24;
#endif
                }
#ifdef VIX_SCAN_DIAG
                diag += 1ull << 44;
#endif
                if (pass) {
                    const uint32_t id = FILTER ? fid : (uint32_t)a.slot_ids[g];
                    wq[a.k + cnt + __popc(ball & ((1u << lane) - 1u))] = key | (u64)id;
                }
                const int ncnt = cnt + __popc(ball);
                __syncwarp();
                if (a.k <= 32 && (ncnt >> 5) != (cnt >> 5)) {
                    // 32 more entries have been accepted since the last look: each beat the threshold of its time, so
                    // their k-th smallest is a tighter bound on the final k-th best -- far cheaper than sorting the queue
                    const u64 e = wq[a.k + (ncnt & ~31) - 32 + lane];
                    const uint32_t kth = warp_kth_smallest((uint32_t)(e >> 32), a.k - 1, lane);
                    if (kth < thr_u) {
                        thr_u = kth;
                        if (lane == 0) atomicMin(reinterpret_cast<unsigned int*>(s_thr), kth);
                    }
                }
                cnt = ncnt;
            }
        };
#ifdef VIX_SCAN_NOPREFETCH
        (void)wB;
        while (ch < nchunks) do_chunk(wA, wA);
#else
        while (ch < nchunks) {
            do_chunk(wA, wB);
            if (ch >= nchunks) break;
            do_chunk(wB, wA);
        }
#endif
        // ---- publish the entries that can still make the top k into the CTA candidate buffer ----
        {
            const uint32_t t = *cta_thr;
            if (t < thr_u) thr_u = t;
            const int lo = sorted_valid ? 0 : a.k;
            const int hi = a.k + cnt;
            for (int base = lo; base < hi; base += 32) {
                const int i = base + lane;
                const u64 key = (i < hi) ? wq[i] : kEmptyKey;
                const bool keep = key != kEmptyKey && (uint32_t)(key >> 32) <= thr_u;
                const unsigned ball = __ballot_sync(0xFFFFFFFFu, keep);
                if (ball) {
                    int pos = 0;
                    if (lane == 0) pos = atomicAdd(s_ncand + buf, __popc(ball));
                    pos = __shfl_sync(0xFFFFFFFFu, pos, 0);
                    if (keep) s_cand[(size_t)buf * nwarps * a.Pw + pos + __popc(ball & ((1u << lane) - 1u))] = key;
                }
            }
        }
        if (STATS) { const long long t = clock64(); cyc_scan += (unsigned long long)(t - t_mark); t_mark = t; }
        __syncthreads();                               // (2) scan finished everywhere, candidates published
        if (STATS) { const long long t = clock64(); cyc_tail += (unsigned long long)(t - t_mark); t_mark = t; }
        have_prev = true;
        prev_qi = qi;
        buf ^= 1;
    }
    if (a.scanned) {
        for (int o = 16; o > 0; o >>= 1) scanned_local += __shfl_xor_sync(0xFFFFFFFFu, scanned_local, o);
        if (lane == 0 && scanned_local) atomicAdd(a.scanned, scanned_local);
    }
#ifdef VIX_SCAN_DIAG
    if (a.phase_cycles && lane == 0) {
        atomicAdd(a.phase_cycles + 8, diag & 0xFFFFFFull);
        atomicAdd(a.phase_cycles + 9, (diag >> 24) & 0xFFFFFull);
        atomicAdd(a.phase_cycles + 10, diag >> 44);
    }
#endif
#ifdef VIX_SCAN_DIAG
    if (a.phase_cycles && lane == 0) atomicAdd(a.phase_cycles + 11, cyc_tail);    // barrier wait summed over ALL warps
#endif
    if (STATS && a.phase_cycles && tid == 64) {            // one scanning warp per CTA reports its phase split
        atomicAdd(a.phase_cycles + 0, cyc_pro);
        atomicAdd(a.phase_cycles + 1, cyc_scan);
        atomicAdd(a.phase_cycles + 2, cyc_tail);
    }
}

// ------------------------------------------------------------------------------------------------
// generic m (not 32 F + {0, 8, 16}): plain AoS codes, [m][256] table, one stored vector per thread
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kScanThreads)
ivfpq_scan_generic_kernel(ScanArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int m = a.m;
    const int ks = a.ks;                                        // 256, or 16 (packed nibbles, low nibble = even sub-quantiser)
    const int cbytes = ks == 16 ? m / 2 : m;
    float* s_lut = reinterpret_cast<float*>(smem_raw);          // [m][ks]
    float* s_q = s_lut + (size_t)m * ks;
    float* s_bias = s_q + a.d;
    int* s_start = reinterpret_cast<int*>(s_bias + a.nprobe);
    int* s_len = s_start + a.nprobe;
    int* s_pref = s_len + a.nprobe;
    u64* s_wq = reinterpret_cast<u64*>((reinterpret_cast<uintptr_t>(s_pref + a.nprobe + 1) + 15) & ~(uintptr_t)15);
    u64* s_merge = s_wq + (size_t)kScanWarps * a.Pw;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int order_max = (a.metric == VIX_METRIC_IP);
    const float lut_scale = order_max ? 1.0f : -2.0f;
    u64* wq = s_wq + (size_t)warp * a.Pw;
    unsigned long long scanned_local = 0;

    for (int64_t qi = blockIdx.x; qi < a.nq; qi += gridDim.x) {
        __syncthreads();
        for (int e = tid; e < a.d; e += kScanThreads) s_q[e] = a.queries[qi * (int64_t)a.d + e];
        for (int p = tid; p < a.nprobe; p += kScanThreads) {
            const int l = a.probes[qi * (int64_t)a.nprobe + p];
            const bool ok = (unsigned)l < (unsigned)a.kc;
            s_start[p] = ok ? (int)(a.list_off[l] >> 5) : 0;
            s_len[p] = ok ? a.list_len[l] : 0;
        }
        __syncthreads();
        if (tid == 0) {
            int acc = 0;
            for (int p = 0; p < a.nprobe; ++p) { s_pref[p] = acc; acc += (s_len[p] + 31) >> 5; }
            s_pref[a.nprobe] = acc;
        }
        for (int p = warp; p < a.nprobe; p += kScanWarps) {
            const int l = a.probes[qi * (int64_t)a.nprobe + p];
            float part = 0.0f;
            if ((unsigned)l < (unsigned)a.kc) {
                const float* c = a.coarse + (int64_t)l * a.d;
                if (order_max) for (int e = lane; e < a.d; e += 32) part = fmaf(s_q[e], c[e], part);
                else for (int e = lane; e < a.d; e += 32) { float df = s_q[e] - c[e]; part = fmaf(df, df, part); }
            }
            for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xFFFFFFFFu, part, o);
            if (lane == 0) s_bias[p] = part;
        }
        for (int e = tid; e < m * ks; e += kScanThreads) {
            const int j = e / ks;
            const float* cw = a.codebooks + (size_t)e * a.dsub;
            const float* qj = s_q + j * a.dsub;
            float dot = 0.0f;
            for (int t = 0; t < a.dsub; ++t) dot = fmaf(qj[t], __ldg(cw + t), dot);
            s_lut[e] = lut_scale * dot;
        }
        for (int i = lane; i < a.Pw; i += 32) wq[i] = kEmptyKey;
        __syncthreads();

        const int nchunks = s_pref[a.nprobe];
        int cnt = 0;
        float thr_s = order_max ? -INFINITY : INFINITY;
        int p = 0;
        for (int ch = warp; ch < nchunks; ch += kScanWarps) {
            while (ch >= s_pref[p + 1]) ++p;
            const int within = (ch - s_pref[p]) * 32 + lane;
            const bool valid = within < s_len[p];
            const int64_t g = ((int64_t)s_start[p] << 5) + within;
            const uint8_t* src = a.slot_codes + g * (int64_t)cbytes;
            float s0 = 0.f;
            if (valid) {
                if (ks == 16) {
                    for (int j = 0; j < m; j += 2) {
                        const int byte = src[j >> 1];
                        s0 += s_lut[(size_t)j * 16 + (byte & 15)];
                        s0 += s_lut[(size_t)(j + 1) * 16 + (byte >> 4)];
                    }
                } else for (int j = 0; j < m; ++j) s0 += s_lut[(size_t)j * ks + src[j]];
            }
            const float tx = valid ? a.slot_tx[g] : 0.0f;
            const float sum = (s_bias[p] + tx) + s0;
            if (valid) ++scanned_local;
            bool pass = valid && (order_max ? !(sum < thr_s) : !(sum > thr_s));
            uint32_t id = 0;
            if (pass) {
                id = (uint32_t)a.slot_ids[g];
                if (a.filter) pass = id_filter_pass(a.filter, a.filter_cap, a.filter_deny, (int64_t)id);
            }
            const unsigned ball = __ballot_sync(0xFFFFFFFFu, pass);
            if (ball) {
                if (pass) wq[a.k + cnt + __popc(ball & ((1u << lane) - 1u))] = make_key(sum, id, order_max);
                cnt += __popc(ball);
                __syncwarp();
                if (cnt + 32 > a.Pw - a.k) {
                    for (int i = a.k + cnt + lane; i < a.Pw; i += 32) wq[i] = kEmptyKey;
                    __syncwarp();
                    bitonic_sort_keys<true>(wq, a.Pw, lane, 32);
                    cnt = 0;
                    const u64 t = wq[a.k - 1];
                    if (t != kEmptyKey) thr_s = key_score(t, order_max);
                }
            }
        }
        if (cnt > 0) {
            for (int i = a.k + cnt + lane; i < a.Pw; i += 32) wq[i] = kEmptyKey;
            __syncwarp();
            bitonic_sort_keys<true>(wq, a.Pw, lane, 32);
        }
        __syncwarp();
        for (int i = lane; i < a.k; i += 32) s_merge[warp * a.k + i] = wq[i];
        for (int i = kScanWarps * a.k + tid; i < a.P2; i += kScanThreads) s_merge[i] = kEmptyKey;
        __syncthreads();
        bitonic_sort_keys<false>(s_merge, a.P2, tid, kScanThreads);
        for (int i = tid; i < a.k; i += kScanThreads) {
            const u64 key = s_merge[i];
            const size_t o = (size_t)qi * a.k + i;
            if (key == kEmptyKey) { a.out_dist[o] = __int_as_float(0x7fc00000); a.out_ids[o] = -1; }
            else {
                const float sc = key_score(key, order_max);
                a.out_dist[o] = order_max ? -sc : sc;
                a.out_ids[o] = (int64_t)key_id(key);
            }
        }
    }
    if (a.scanned) {
        for (int o = 16; o > 0; o >>= 1) scanned_local += __shfl_xor_sync(0xFFFFFFFFu, scanned_local, o);
        if (lane == 0 && scanned_local) atomicAdd(a.scanned, scanned_local);
    }
}

// ------------------------------------------------------------------------------------------------
// layout + launch
// ------------------------------------------------------------------------------------------------
ScanLayout scan_layout(int m) {
    ScanLayout L;
    L.fast = m > 0 && m % 16 == 0 && m <= 64;
    L.align = 32;
    return L;
}

static size_t generic_smem_bytes(const ScanArgs& a) {
    size_t s = (size_t)a.m * a.ks * 4;
    s += (size_t)a.d * 4 + (size_t)a.nprobe * 12 + (size_t)(a.nprobe + 1) * 4 + 16;
    s += (size_t)kScanWarps * a.Pw * 8 + (size_t)a.P2 * 8;
    return s;
}

// Warps and shared memory of the fast kernel for (m, d, k, nprobe), with a.Pw set.  The tables start at a 64 KB boundary of
// the shared window; the bookkeeping (probe tables, queries, selection queues) sits in front of them, behind the <= 1 KB
// the system keeps at the start of the window.  Two tables must start at 64 KB (they end at 192 of 227 KB); one table
// may also start at 128 KB.  Large d / nprobe / k are paid for with fewer warps (smaller queues): 16 unless k is large,
// at least 3 while that fits, and 2 (warps 0 and 1 carry every role of the pipeline) when only that fits -- two
// tables with k > 448 (Pw = 1024).  nwarps = 0: not even that fits (two tables, k > 448 and 4 nprobe + d > 1912).
struct FastPlan { int nwarps; size_t misc, misc_limit, smem; };
static FastPlan fast_plan(const ScanArgs& a) {
    const int NTAB = (a.m / 16 + 1) / 2;
    FastPlan f;
    f.misc_limit = (NTAB == 2) ? 65536 - 1024 : 100 * 1024;
    auto misc_bytes = [&](int w) {
        return 2 * ((size_t)a.nprobe * 16 + 4) + 2 * (size_t)a.d * 4 + 40 + 16 + 3 * (size_t)w * a.Pw * 8;
    };
    f.nwarps = kFastThreads / 32;
    while (f.nwarps > 3 && (3 * (size_t)f.nwarps * a.Pw * 8 > 56 * 1024 || misc_bytes(f.nwarps) > f.misc_limit)) --f.nwarps;
    if (misc_bytes(f.nwarps) > f.misc_limit) f.nwarps = 2;
    f.misc = misc_bytes(f.nwarps);
    if (f.misc > f.misc_limit) f.nwarps = 0;
    f.smem = f.misc + 65535 + (size_t)NTAB * 65536;
    if (f.smem > 227 * 1024) f.smem = 227 * 1024;
    return f;
}

template <int G, bool FILTER>
static int launch_fast(ScanArgs& a, const FastPlan& f) {
    const bool stats = a.phase_cycles != nullptr;
    const size_t smem = f.smem;
    a.smem_bytes = (int)smem;
    auto kern = stats ? ivfpq_scan_kernel<G, FILTER, true> : ivfpq_scan_kernel<G, FILTER, false>;
    VIX_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int64_t grid = num_sms();
    if (grid > a.nq) grid = a.nq;
    if (a.ev_kernel[0]) VIX_CUDA(cudaEventRecord(a.ev_kernel[0], ctx().stream));
    kern<<<(unsigned)grid, 32 * f.nwarps, smem, ctx().stream>>>(a);
    VIX_LAUNCH_CHECK();
    if (a.ev_kernel[1]) VIX_CUDA(cudaEventRecord(a.ev_kernel[1], ctx().stream));
    return VIX_OK;
}

// the same terms, one warp per QUERY (its row stays in shared memory, four probed lists in flight): the batch-wide form
// the list-major path uses for every (query, probe) pair.  Lane-strided partial sums and xor tree as above: identical bits.
__global__ void __launch_bounds__(256)
probe_bias_rows_kernel(const float* __restrict__ queries, const int32_t* __restrict__ probes, const float* __restrict__ coarse,
                       const int32_t* __restrict__ list_len, int kc, int64_t nq, int nprobe, int d, int order_max,
                       const int* __restrict__ only_flagged, float* __restrict__ bias) {
    extern __shared__ float s_rows[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t q = (int64_t)blockIdx.x * 8 + warp;
    if (q >= nq || (only_flagged && !only_flagged[q])) return;
    float* sq = s_rows + (size_t)warp * d;
    for (int e = lane; e < d; e += 32) sq[e] = __ldg(queries + q * d + e);
    __syncwarp();
    for (int p0 = 0; p0 < nprobe; p0 += 4) {
        float part[4];
        const float* c[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            part[u] = 0.0f;
            c[u] = nullptr;
            if (p0 + u < nprobe) {
                const int l = __ldg(probes + q * nprobe + p0 + u);
                if ((unsigned)l < (unsigned)kc && __ldg(list_len + l) > 0) c[u] = coarse + (int64_t)l * d;
            }
        }
        if (order_max) {
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (c[u]) for (int e = lane; e < d; e += 32) part[u] = fmaf(sq[e], __ldg(c[u] + e), part[u]);
        } else {
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (c[u]) for (int e = lane; e < d; e += 32) { const float df = sq[e] - __ldg(c[u] + e); part[u] = fmaf(df, df, part[u]); }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u)
            for (int o = 16; o > 0; o >>= 1) part[u] += __shfl_xor_sync(0xFFFFFFFFu, part[u], o);
        if (lane < 4 && p0 + lane < nprobe)
            bias[q * nprobe + p0 + lane] = lane == 0 ? part[0] : lane == 1 ? part[1] : lane == 2 ? part[2] : part[3];
    }
}

int launch_probe_bias(const ScanArgs& a, float* bias, const int* only_flagged) {
    if ((size_t)a.d * 4 * 8 <= 48 * 1024) {
        probe_bias_rows_kernel<<<(unsigned)((a.nq + 7) / 8), 256, (size_t)a.d * 4 * 8, ctx().stream>>>(
            a.queries, a.probes, a.coarse, a.list_len, a.kc, a.nq, a.nprobe, a.d, a.metric == VIX_METRIC_IP, only_flagged, bias);
        VIX_LAUNCH_CHECK();
        return VIX_OK;
    }
    const int64_t npairs = a.nq * (int64_t)a.nprobe;
    probe_bias_kernel<<<(unsigned)((npairs * 32 + 255) / 256), 256, 0, ctx().stream>>>(
        a.queries, a.probes, a.coarse, a.list_len, a.kc, npairs, a.nprobe, a.d, a.metric == VIX_METRIC_IP, bias);
    VIX_LAUNCH_CHECK();
    return VIX_OK;
}

bool tc_scan_supported(const ScanArgs& a);
int launch_ivfpq_scan_tc(ScanArgs& a);

int launch_ivfpq_scan(ScanArgs& a) {
    const ScanLayout L = scan_layout(a.m);
    a.path = 0;
    if (L.fast && tc_scan_supported(a)) { a.path = 1; return launch_ivfpq_scan_tc(a); }   // list-major, tensor cores (vix_ivfpq_tc.cu)
    return launch_ivfpq_scan_classic(a);
}

// query-major: one look-up table per query
int launch_ivfpq_scan_classic(ScanArgs& a) {
    const ScanLayout L = scan_layout(a.m);
    const bool debug = getenv("VIX_SCAN_DEBUG") != nullptr;
    VIX_REQUIRE(a.nprobe > 0 && a.nprobe <= VIX_MAX_K, VIX_ERR_INVALID_K, "ivfpq scan: nprobe = %d (1 .. %d)", a.nprobe, VIX_MAX_K);
    if (!L.fast || a.ks != 256) {
        a.Pw = next_pow2(a.k + 32);
        a.P2 = next_pow2(kScanWarps * a.k);
        const size_t smem = generic_smem_bytes(a);
        VIX_REQUIRE(smem <= 227 * 1024, VIX_ERR_UNSUPPORTED,
                    "ivfpq scan: m = %d, k = %d, nprobe = %d need %zu bytes of shared memory", a.m, a.k, a.nprobe, smem);
        if (debug)
            fprintf(stderr, "[vix scan] kernel generic, filter %d, stats %d, warps %d, Pw %d, P2 %d, table kernel, bias kernel, "
                    "order no, items %lld\n", a.filter != nullptr, a.phase_cycles != nullptr, kScanWarps, a.Pw, a.P2,
                    (long long)a.nq);
        VIX_CUDA(cudaFuncSetAttribute(ivfpq_scan_generic_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int occ = 1;
        VIX_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, ivfpq_scan_generic_kernel, kScanThreads, smem));
        int64_t grid = (int64_t)num_sms() * (occ < 1 ? 1 : occ);
        if (grid > a.nq) grid = a.nq;
        if (a.ev_kernel[0]) VIX_CUDA(cudaEventRecord(a.ev_kernel[0], ctx().stream));
        ivfpq_scan_generic_kernel<<<(unsigned)grid, kScanThreads, smem, ctx().stream>>>(a);
        VIX_LAUNCH_CHECK();
        if (a.ev_kernel[1]) VIX_CUDA(cudaEventRecord(a.ev_kernel[1], ctx().stream));
        return VIX_OK;
    }
    a.Pw = next_pow2(a.k + 64);
    a.P2 = 0;
    const FastPlan plan = fast_plan(a);
    VIX_REQUIRE(plan.nwarps > 0, VIX_ERR_UNSUPPORTED,
                "ivfpq scan: d = %d, k = %d, nprobe = %d need %zu bytes of bookkeeping shared memory (limit %zu)", a.d, a.k,
                a.nprobe, plan.misc, plan.misc_limit);
    VIX_REQUIRE(a.work_counter != nullptr, VIX_ERR_NULL_PTR, "ivfpq scan: work counter missing");
    VIX_CUDA(cudaMemsetAsync(a.work_counter, 0, 2 * sizeof(int), ctx().stream));
    // a kernel that finds its shared-memory layout does not fit refuses loudly: it raises the mapped host flag that the
    // next synchronising call reports (vix_runtime.cu), not a device word nobody reads
    int* const loud = pipeline_error_flag();
    a.status = loud ? loud : a.work_counter + 1;
    Scratch<float> bias;
    const char* bias_src = a.bias ? "given" : "kernel";
    if (!a.bias && (int64_t)a.d * a.nprobe > 8192) {
        bias_src = (size_t)a.d * 4 * 8 <= 48 * 1024 ? "rows" : "pairs";      // launch_probe_bias's choice
        // one staging warp per CTA cannot hide this much bias arithmetic behind a query's scan: do it batch-wide
        VIX_TRY(bias.alloc((size_t)(a.nq * (int64_t)a.nprobe)));
        VIX_TRY(launch_probe_bias(a, bias.ptr));
        a.bias = bias.ptr;
    }
    Scratch<float> image;
    const size_t cb_bytes = (size_t)a.m * 256 * a.dsub * 4;
    const size_t img_floats = (size_t)((a.m / 16 + 1) / 2) * 8192;      // compact: [table][256 codes][32 slots]
    if (cb_bytes >= 512 * 1024 && a.dsub <= 16 && (size_t)a.nq * img_floats * 4 <= (4ull << 30) && !getenv("VIX_DISABLE_LUT_IMAGE")) {
        // large codebooks: build every query's table once, batch-wide, instead of once per query inside the scan
        // (C4: the table's share of a query 31 k -> 2.9 k cycles for a 0.46 ms batch kernel; scan stage 3.36 -> 2.86 ms)
        VIX_TRY(image.alloc((size_t)a.nq * img_floats));
        const dim3 grid((unsigned)((a.nq + kImgQT - 1) / kImgQT), (unsigned)((a.m + 31) / 32));
        const float scale = a.metric == VIX_METRIC_IP ? 1.0f : -2.0f;
#define VIX_IMG(MM) lut_image_kernel<MM><<<grid, 256, 0, ctx().stream>>>(a.queries, a.nq, a.d, a.codebooks_t, a.dsub, scale, image.ptr)
        switch (a.m) {
            case 16: VIX_IMG(16); break;
            case 32: VIX_IMG(32); break;
            case 48: VIX_IMG(48); break;
            case 64: VIX_IMG(64); break;
        }
#undef VIX_IMG
        VIX_LAUNCH_CHECK();
        a.lut_image = image.ptr;
    }
    if (debug) {
        // work items: the batch, or (queries handed back by the list-major scan) a count only the device knows
        char items[32] = "device";
        if (!a.nq_dev) snprintf(items, sizeof items, "%lld", (long long)a.nq);
        fprintf(stderr, "[vix scan] kernel fast G %d, filter %d, stats %d, warps %d, Pw %d, P2 %d, table %s, bias %s, "
                "order %s, items %s\n", a.m / 16, a.filter != nullptr, a.phase_cycles != nullptr, plan.nwarps, a.Pw, a.P2,
                a.lut_image ? "image" : "kernel", bias_src, a.order && !a.nq_dev ? "yes" : "no", items);
    }
    switch (a.m) {
        case 16: return a.filter ? launch_fast<1, true>(a, plan) : launch_fast<1, false>(a, plan);
        case 32: return a.filter ? launch_fast<2, true>(a, plan) : launch_fast<2, false>(a, plan);
        case 48: return a.filter ? launch_fast<3, true>(a, plan) : launch_fast<3, false>(a, plan);
        case 64: return a.filter ? launch_fast<4, true>(a, plan) : launch_fast<4, false>(a, plan);
    }
    set_error("ivfpq scan: unsupported m = %d", a.m);
    return VIX_ERR_UNSUPPORTED;
}

}  // namespace vix
