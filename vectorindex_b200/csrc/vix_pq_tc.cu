// vix_pq_tc.cu -- PQ encoding with a tensor-core shortlist (SURVEY.md 7: "tensor shortlist + exact rescoring").
//
// The reference's encoder (pq_encode.c:332-410) is a per (vector, sub-space) argmin over 256 codewords of
// x2 + csq[k] - 2 <x_j, c_k>; on CUDA cores that is 2 * dsub + 3 unfused fp32 operations per pair in the reference's
// order (vix_pq_encode.cu: fp32-issue bound).  Here the dot products come from the tensor cores and only the FINALISTS
// are evaluated in the reference's arithmetic:
//
//   MMA       one row tile (128 vectors) x one K-block (32 dimensions = 32 / dsub sub-spaces): the A tile is read once by
//             TMA; B is the same 32 columns of the code-major codebooks [256 x d] (row c = codeword c of every
//             sub-space side by side), so sub-space s of the block is ONE tcgen05.mma kind::tf32 M128 N256 K8 (dsub / 8
//             of them) on the 32 s-byte slices of both tiles: D_s[128 x 256] = <x_j, c_k> for all 256 codewords, in
//             TMEM.  No block-diagonal zeros, no wasted flops.
//   shortlist two threads share one (vector, sub-space), 128 codewords each: S~_k = csq[k] - 2 D[k]; pass 1 finds min S~ (the
//             two halves' minima meet in shared memory), pass 2 re-reads TMEM and keeps every k with S~_k <= min + 2 eps,
//             eps = rel ||x_j|| max||c|| (TF32 operand truncation + accumulation, the bound of vix_gemm.cu) + the rounding of
//             the fp32 evaluation itself.  The exact argmin is among them.  (Measured and dropped: ONE pass that collects
//             everything within 2 eps of the running minimum -- half the TMEM reads, but four times the exact evaluations.)
//   exact     the finalists (1-2 as a rule; a half's 128 codewords if more than four qualify) are evaluated by the very device function
//             of the CUDA-core encoder (encode_chunk: the reference's operation order, unfused) in ascending k with its
//             strict '<', i.e. tie -> smaller k (pq_encode.c:74-80): the codes are bit-identical.
//
// Warp roles as in vix_gemm.cu: warp 0 TMA producer (3-stage ring of A 16 KB | B 32 KB), warp 1 MMA issuer, warps 2-17 two
// epilogue teams of eight warps, one team per TMEM accumulator buffer (2 x 256 columns), two threads per (vector,
// sub-space) with 128 codewords each; codes are staged per row tile in shared memory and leave as one contiguous
// [128 x m] byte slab.  Residual variants: r = x - g is materialised once (the shortlist's A operand); the exact stage reads x
// and g and follows the reference's residual arithmetic.  PTX wrappers, bounded mbarrier waits (mbar_wait): vix_tcgen05.cuh.
#include "vix_common.cuh"
#include "vix_pq_encode.cuh"
#include "vix_tcgen05.cuh"

#include <stdlib.h>

namespace vix {

namespace pqtc {

constexpr int kM = 128, kN = 256, kKB = 32;
constexpr int kStages = 3;
constexpr int kStageBytes = (kM + kN) * kKB * 4;       // 48 KB
constexpr int kThreads = 64 + 512;                     // producer, MMA issuer, 2 teams x 2 column halves x 4 epilogue warps
constexpr int kCap = 4;                                // finalists kept per (vector, sub-space)
constexpr uint32_t kIdesc = idesc_tf32(kM, kN);

struct Args {
    const float* x;                 // [n x d] the rows (exact arithmetic)
    const float* coarse;            // residual modes: [kc x d]
    const int32_t* assign;          // residual modes: [n]
    int64_t n;
    int d, m, mtiles, ngroups;
    const float* codebooks;         // [m][256][dsub]
    const float* csq;               // [m][256] the caller's centroid norms (CSQ modes) / sequential norms (DOT modes)
    const float* cmax;              // [m] sqrt(max_k ||c_jk||^2)
    uint8_t* codes;                 // [n x m] AoS
    float rel;
    int* error;
    int* error_host;
};

__device__ __forceinline__ float4 lds_f4(uint32_t addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}

template <int MODE, int DSUB>
__global__ void __launch_bounds__(kThreads, 1)
pq_tc_encode_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, Args a) {
    constexpr bool kRes = (MODE == ENC_CSQ_RES || MODE == ENC_DOT_RES);
    constexpr int kSteps = DSUB / 8;                                  // tcgen05 K-steps per sub-space
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char* base = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    unsigned char* ring = base;                                                      // kStages x (A 16 KB | B 32 KB)
    uint64_t* full = reinterpret_cast<uint64_t*>(ring + (size_t)kStages * kStageBytes);
    uint64_t* empty = full + kStages;
    uint64_t* tfull = empty + kStages;                                               // [2]
    uint64_t* tempty = tfull + 2;                                                    // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
    float* s_csq = reinterpret_cast<float*>(tmem_slot + 4);                          // [m][256]
    float* s_ex = s_csq + (size_t)a.m * 256;                                          // [2 parities][2 teams][128 rows][4] pair exchange words
    uint8_t* s_codes = reinterpret_cast<uint8_t*>(s_ex + 2 * 2 * kM * 4);            // [2][128 x m]

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == 0 && lane == 0) {
        for (int s = 0; s < kStages; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(tfull + b, 1); mbar_init(tempty + b, 8); }
        mbar_init_fence();
    }
    for (int e = threadIdx.x; e < a.m * 256; e += kThreads) s_csq[e] = a.csq[e];
    if (warp == 1) tmem_alloc(tmem_slot, 512);
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;
    const int per_group = kKB / DSUB;                                  // sub-spaces per K-block

    if (warp == 0) {
        // ================= TMA producer =================
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            bool ok = true;
            for (int mt = blockIdx.x; mt < a.mtiles && ok; mt += gridDim.x) {
                for (int g = 0; g < a.ngroups; ++g) {
                    if (!mbar_wait(empty + stage, phase ^ 1, a.error, a.error_host)) { ok = false; break; }
                    unsigned char* sA = ring + (size_t)stage * kStageBytes;
                    mbar_expect_tx(full + stage, kStageBytes);
                    tma_load_2d(sA, &mapA, full + stage, g * kKB, mt * kM);
                    tma_load_2d(sA + kM * kKB * 4, &mapB, full + stage, g * kKB, 0);
                    if (++stage == kStages) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer =================
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            int acc = 0; uint32_t aphase = 0;
            bool ok = true;
            for (int mt = blockIdx.x; mt < a.mtiles && ok; mt += gridDim.x) {
                for (int g = 0; g < a.ngroups && ok; ++g) {
                    if (!mbar_wait(full + stage, phase, a.error, a.error_host)) { ok = false; break; }
                    fence_after_sync();
                    const uint32_t sA = smem_u32(ring + (size_t)stage * kStageBytes);
                    const uint64_t da = make_desc_sw128(sA), db = make_desc_sw128(sA + kM * kKB * 4);
                    const int nsub = min(per_group, a.m - g * per_group);
                    for (int s = 0; s < nsub; ++s) {
                        if (!mbar_wait(tempty + acc, aphase ^ 1, a.error, a.error_host)) { ok = false; break; }
                        fence_after_sync();
                        const uint32_t tmem_d = tmem_base + (uint32_t)acc * kN;
#pragma unroll
                        for (int k = 0; k < kSteps; ++k)               // 8 tf32 = 32 B per step: +2 in 16-byte units
                            mma_tf32(tmem_d, da + 2 * (s * kSteps + k), db + 2 * (s * kSteps + k), kIdesc, k ? 1u : 0u);
                        mma_commit(tfull + acc);
                        if (++acc == 2) { acc = 0; aphase ^= 1; }
                    }
                    if (!ok) break;
                    mma_commit(empty + stage);                         // the ring slot is free when these MMAs retire
                    if (++stage == kStages) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else {
        // ================= epilogue: team = accumulator buffer; a (vector, sub-space) is shared by TWO threads =================
        // 16 warps: team (2) x column half (2) x TMEM lane quarter (4).  The two threads of a pair each take 128 of the 256
        // codewords: pass 1 -> their minima meet in shared memory (one 64-thread named barrier) -> pass 2 -> each evaluates
        // ITS finalists in the reference's arithmetic -> the partial results meet again and the lower half decides
        // (ascending k, strict '<': a tie goes to the smaller k).
        const int e16 = warp - 2;
        const int team = e16 >> 3;
        const int half = (e16 >> 2) & 1;
        const int quarter = warp & 3;                                  // TMEM lane quarter this warp may read
        const int etid = (int)threadIdx.x - 64;                        // 0 .. 511 among the epilogue threads
        const int pair_bar = 2 + team * 4 + quarter;                   // named barrier of the two warps of a pair
        uint32_t aphase = 0;
        int seq = 0;                                                   // (row tile, sub-space) pairs seen so far, both teams
        int cbuf = 0;
        int units = 0;                                                 // units this pair has finished
        bool ok = true;
        for (int mt = blockIdx.x; mt < a.mtiles; mt += gridDim.x) {
            const int rloc = quarter * 32 + lane;
            const int64_t row = (int64_t)mt * kM + rloc;
            const bool live = row < a.n;
            const float* xi = a.x + (live ? row : 0) * (int64_t)a.d;
            const float* gi = nullptr;
            if (kRes) gi = a.coarse + (int64_t)(live ? a.assign[row] : 0) * a.d;
            uint8_t* my_codes = s_codes + (size_t)cbuf * kM * a.m + (size_t)rloc * a.m;
            float* ex0 = s_ex + ((size_t)team * kM + rloc) * 4;        // the pair's exchange words: min h0 | min h1 | bd h1 | bk h1 (x 2 unit parities)
            // this thread's sub-vector of the unit it handles next (loaded one unit ahead: the L2 round trip hides behind
            // the current unit's passes)
            float xn[DSUB], gn[DSUB];
            auto load_sub = [&](int j) {
#pragma unroll
                for (int e = 0; e < DSUB; e += 4) {
                    const bool in = live && j < a.m;
                    const float4 v = in ? __ldg(reinterpret_cast<const float4*>(xi + (size_t)j * DSUB + e)) : make_float4(0.f, 0.f, 0.f, 0.f);
                    xn[e] = v.x; xn[e + 1] = v.y; xn[e + 2] = v.z; xn[e + 3] = v.w;
                    if (kRes) {
                        const float4 w = in ? __ldg(reinterpret_cast<const float4*>(gi + (size_t)j * DSUB + e)) : make_float4(0.f, 0.f, 0.f, 0.f);
                        gn[e] = w.x; gn[e + 1] = w.y; gn[e + 2] = w.z; gn[e + 3] = w.w;
                    } else { gn[e] = gn[e + 1] = gn[e + 2] = gn[e + 3] = 0.0f; }
                }
            };
            load_sub(((seq & 1) == team) ? 0 : 1);
            for (int j = 0; j < a.m; ++j, ++seq) {
                if ((seq & 1) != team) continue;
                float xr[DSUB], gr[DSUB];
#pragma unroll
                for (int e = 0; e < DSUB; ++e) { xr[e] = xn[e]; gr[e] = gn[e]; }
                load_sub(j + 2);
                float base2 = 0.0f;                                    // x2 / r2, sequential (pq_encode.c:340, 380)
#pragma unroll
                for (int e = 0; e < DSUB; ++e) {
                    const float ri = kRes ? fsub(xr[e], gr[e]) : xr[e];
                    base2 = fadd(base2, fmul(ri, ri));
                }
                const float cm = a.cmax[j];
                const float eps = a.rel * sqrtf(base2) * cm + 4e-7f * (base2 + cm * cm);
                const uint32_t cs = smem_u32(s_csq + (size_t)j * 256 + half * 128);
                // double buffered by unit parity: a thread may be a whole unit ahead of its partner's reads
                float* ex = ex0 + (size_t)(units & 1) * (2 * kM * 4);
                ++units;
                uint32_t cands = 0;                                    // up to four finalists of this half, one byte each, ascending k
                int ncand = 0;
                if (ok && !mbar_wait(tfull + team, aphase, a.error, a.error_host)) ok = false;
                const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)team * kN + (uint32_t)half * 128;
                // pass 1: min_k S~_k over this half, S~_k = csq[k] - 2 D[k]
                float mn = INFINITY;
                if (ok) {
                    fence_after_sync();
#pragma unroll 1
                    for (int ck = 0; ck < 4; ++ck) {
                        uint32_t v[32];
                        tmem_ld32_issue(taddr + ck * 32, v);
                        tmem_ld32_wait(v);
#pragma unroll
                        for (int i4 = 0; i4 < 8; ++i4) {
                            const float4 n4 = lds_f4(cs + 128u * ck + 16u * i4);
                            mn = fminf(mn, fminf(fminf(fmaf(-2.0f, __uint_as_float(v[4 * i4]), n4.x), fmaf(-2.0f, __uint_as_float(v[4 * i4 + 1]), n4.y)),
                                                 fminf(fmaf(-2.0f, __uint_as_float(v[4 * i4 + 2]), n4.z), fmaf(-2.0f, __uint_as_float(v[4 * i4 + 3]), n4.w))));
                        }
                    }
                }
                ex[half] = mn;
                asm volatile("bar.sync %0, 64;" ::"r"(pair_bar) : "memory");
                mn = fminf(ex[0], ex[1]);
                // pass 2 (the accumulators are read again: 128 scores do not fit a thread's registers): every k of this half
                // with S~_k <= min + 2 eps
                if (ok) {
                    const float thr = mn + 2.0f * eps;
#pragma unroll 1
                    for (int ck = 0; ck < 4; ++ck) {
                        uint32_t v[32];
                        tmem_ld32_issue(taddr + ck * 32, v);
                        tmem_ld32_wait(v);
                        uint32_t hit = 0;
#pragma unroll
                        for (int i4 = 0; i4 < 8; ++i4) {
                            const float4 n4 = lds_f4(cs + 128u * ck + 16u * i4);
                            if (fmaf(-2.0f, __uint_as_float(v[4 * i4]), n4.x) <= thr) hit |= 1u << (4 * i4);
                            if (fmaf(-2.0f, __uint_as_float(v[4 * i4 + 1]), n4.y) <= thr) hit |= 2u << (4 * i4);
                            if (fmaf(-2.0f, __uint_as_float(v[4 * i4 + 2]), n4.z) <= thr) hit |= 4u << (4 * i4);
                            if (fmaf(-2.0f, __uint_as_float(v[4 * i4 + 3]), n4.w) <= thr) hit |= 8u << (4 * i4);
                        }
                        while (hit) {
                            const int i = __ffs((int)hit) - 1;
                            hit &= hit - 1;
                            if (ncand < kCap) cands |= (uint32_t)(half * 128 + ck * 32 + i) << (8 * ncand);
                            ++ncand;
                        }
                    }
                    fence_before_sync();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(tempty + team);         // eight arrivals hand the accumulator back
                }
                aphase ^= 1;
                // this half's finalists in the reference's arithmetic, ascending k, strict '<' (tie -> smaller k)
                const float* cbj = a.codebooks + (size_t)j * 256 * DSUB;
                const float* csqj = a.csq + (size_t)j * 256;
                auto xf = [&](int e) -> float { return xr[e]; };
                auto gf = [&](int e) -> float { return gr[e]; };
                float bd = 0.0f;
                int bk = -1;                                           // -1: this half has no finalist
                if (ncand > kCap || !ok) {
                    // more finalists than the list holds: this half's 128 codewords, all of them
                    int kk = 0;
                    encode_chunk<MODE, DSUB>(xf, gf, cbj + (size_t)half * 128 * DSUB, csqj + half * 128, 0, 128, DSUB, base2, bd, kk);
                    bk = half * 128 + kk;
                } else {
                    for (int t = 0; t < ncand; ++t) {
                        const int k = (int)((cands >> (8 * t)) & 0xFFu);
                        float dk = 0.0f;
                        int kk = 0;
                        // one codeword: encode_chunk over [0, 1) of a table that starts at k evaluates exactly the reference's `dist`
                        encode_chunk<MODE, DSUB>(xf, gf, cbj + (size_t)k * DSUB, csqj + k, 0, 1, DSUB, base2, dk, kk);
                        if (bk < 0 || dk < bd) { bd = dk; bk = k; }
                    }
                }
                if (half == 1) { ex[2] = bd; ex[3] = __int_as_float(bk); }
                asm volatile("bar.sync %0, 64;" ::"r"(pair_bar) : "memory");
                if (half == 0) {
                    const float bd1 = ex[2];
                    const int bk1 = __float_as_int(ex[3]);
                    if (bk < 0 && bk1 < 0) {
                        // no finalist at all (NaN scores): the reference's full scan decides
                        encode_chunk<MODE, DSUB>(xf, gf, cbj, csqj, 0, 256, DSUB, base2, bd, bk);
                    } else if (bk < 0 || (bk1 >= 0 && bd1 < bd)) {
                        bk = bk1;
                    }
                    my_codes[j] = (uint8_t)bk;
                }
            }
            // the row tile is complete when both teams are: one barrier of the 512 epilogue threads, then the slab leaves
            asm volatile("bar.sync 1, 512;" ::: "memory");
            {
                const int64_t r0 = (int64_t)mt * kM;
                const int64_t rows = a.n - r0 < kM ? a.n - r0 : (int64_t)kM;
                const int64_t total = rows * a.m;
                const uint8_t* src = s_codes + (size_t)cbuf * kM * a.m;
                uint8_t* dst = a.codes + r0 * (int64_t)a.m;
                if (((reinterpret_cast<uintptr_t>(dst) | (uintptr_t)(kM * a.m)) & 15) == 0) {
                    const int64_t nv = total >> 4;
                    for (int64_t e = etid; e < nv; e += 512) reinterpret_cast<uint4*>(dst)[e] = reinterpret_cast<const uint4*>(src)[e];
                    for (int64_t e = (nv << 4) + etid; e < total; e += 512) dst[e] = src[e];
                } else {
                    for (int64_t e = etid; e < total; e += 512) dst[e] = src[e];
                }
            }
            cbuf ^= 1;
        }
    }
    fence_before_sync();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, 512);
}

// r = x - coarse[assign] (the shortlist's A operand of the residual variants)
__global__ void residual_rows_kernel(const float* __restrict__ x, const float* __restrict__ coarse, const int32_t* __restrict__ assign,
                                     int64_t n, int d, float* __restrict__ r) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n * (int64_t)(d / 4)) return;
    const int64_t row = i / (d / 4);
    const int e = (int)(i - row * (d / 4)) * 4;
    const float4 a = __ldg(reinterpret_cast<const float4*>(x + row * d + e));
    const float4 g = __ldg(reinterpret_cast<const float4*>(coarse + (int64_t)assign[row] * d + e));
    *reinterpret_cast<float4*>(r + row * d + e) = make_float4(fsub(a.x, g.x), fsub(a.y, g.y), fsub(a.z, g.z), fsub(a.w, g.w));
}

// codebooks [m][256][dsub] -> [256][m * dsub] (row c = codeword c of every sub-space), sequential norms, per-sub-space max
__global__ void prep_codebooks_kernel(const float* __restrict__ cb, int m, int dsub, float* __restrict__ cbt, float* __restrict__ seqn) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;               // (j, c)
    if (i >= m * 256) return;
    const int j = i >> 8, c = i & 255;
    float s = 0.0f;
    for (int e = 0; e < dsub; ++e) {
        const float v = cb[(size_t)i * dsub + e];
        cbt[(size_t)c * m * dsub + (size_t)j * dsub + e] = v;
        s = fadd(s, fmul(v, v));
    }
    seqn[i] = s;
}
__global__ void cmax_kernel(const float* __restrict__ seqn, int m, float* __restrict__ cmax) {
    const int j = blockIdx.x;
    __shared__ float s[256];
    s[threadIdx.x] = seqn[j * 256 + threadIdx.x];
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) { if ((int)threadIdx.x < o) s[threadIdx.x] = fmaxf(s[threadIdx.x], s[threadIdx.x + o]); __syncthreads(); }
    if (threadIdx.x == 0) cmax[j] = sqrtf(s[0]);
}

static size_t smem_bytes(int m) {
    return (size_t)kStages * kStageBytes + 1024 + 256 + (size_t)m * 256 * 4 + 2 * 2 * kM * 4 * 4 + 2 * (size_t)kM * m + 64;
}

template <int MODE, int DSUB>
static int launch(const CUtensorMap& mapA, const CUtensorMap& mapB, const Args& a) {
    auto kern = pq_tc_encode_kernel<MODE, DSUB>;
    const size_t smem = smem_bytes(a.m);
    VIX_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int grid = num_sms();
    if (grid > a.mtiles) grid = a.mtiles;
    kern<<<grid, kThreads, smem, ctx().stream>>>(mapA, mapB, a);
    VIX_LAUNCH_CHECK();
    return VIX_OK;
}

}  // namespace pqtc

// Whether the tensor-core encoder takes this call (else the CUDA-core kernel of vix_pq_encode.cu runs).
bool pq_encode_tc_supported(const float* x, int64_t n, int d, int m, int ks, int mode, int layout, int u4) {
    const int dsub = m > 0 ? d / m : 0;
    if (getenv("VIX_DISABLE_TC") || getenv("VIX_DISABLE_PQ_TC")) return false;
    if (ks != 256 || u4 || layout != PQ_LAYOUT_AOS || n < 4096 || n >= (1LL << 31)) return false;
    if (dsub != 8 && dsub != 16) return false;
    if (mode != ENC_CSQ && mode != ENC_CSQ_RES && mode != ENC_DOT && mode != ENC_DOT_RES) return false;
    if (m > 64 || pqtc::smem_bytes(m) > 227 * 1024) return false;
    return tc::supported(n, 256, d, x, x);
}

// Device pointers.  Same results as pq_encode_kernel<mode>: bit-identical codes.
int pq_encode_tc_device(const float* x, int64_t n, int d, int m, const float* cb, const float* csq, const float* coarse,
                        const int32_t* assign, uint8_t* codes, int mode) {
    const int dsub = d / m;
    cudaStream_t s = ctx().stream;
    VIX_TRY(check_pipeline_error());
    int* pipe_flag = pipeline_error_flag();
    VIX_REQUIRE(pipe_flag != nullptr, VIX_ERR_OOM, "cannot allocate the mapped pipeline-error flag");
    Scratch<float> cbt, seqn, cmax, resid;
    Scratch<int> err;
    VIX_TRY(cbt.alloc((size_t)256 * d));
    VIX_TRY(seqn.alloc((size_t)m * 256));
    VIX_TRY(cmax.alloc((size_t)m));
    VIX_TRY(err.alloc(1));
    VIX_CUDA(cudaMemsetAsync(err.ptr, 0, 4, s));
    pqtc::prep_codebooks_kernel<<<(m * 256 + 255) / 256, 256, 0, s>>>(cb, m, dsub, cbt.ptr, seqn.ptr);
    VIX_LAUNCH_CHECK();
    pqtc::cmax_kernel<<<m, 256, 0, s>>>(seqn.ptr, m, cmax.ptr);
    VIX_LAUNCH_CHECK();
    const bool res = (mode == ENC_CSQ_RES || mode == ENC_DOT_RES);
    const bool has_csq = (mode == ENC_CSQ || mode == ENC_CSQ_RES);
    pqtc::Args a{};
    a.x = x; a.coarse = coarse; a.assign = assign; a.d = d; a.m = m;
    a.ngroups = (d + pqtc::kKB - 1) / pqtc::kKB;
    a.codebooks = cb; a.csq = has_csq ? csq : seqn.ptr; a.cmax = cmax.ptr;
    // |S~ - S| <= 2 |dot~ - dot|: TF32 operand truncation (2 * 2^-10) + fp32 accumulation, with margin (vix_gemm.cu)
    a.rel = 2.0f * 1.25f * (2.0f / 1024.0f + (float)dsub / 2097152.0f);
    a.error = err.ptr; a.error_host = pipe_flag;
    CUtensorMap mapA, mapB;
    VIX_TRY(tc::make_map_rows(&mapB, cbt.ptr, 256, d, pqtc::kN));
    // rows are processed in slabs so that the materialised residual of the residual variants stays bounded
    const int64_t slab = res ? (int64_t)1 << 20 : n;
    if (res) VIX_TRY(resid.alloc((size_t)(n < slab ? n : slab) * d));
    for (int64_t b = 0; b < n; b += slab) {
        const int64_t cn = n - b < slab ? n - b : slab;
        const float* A = x + (size_t)b * d;
        if (res) {
            const int64_t total = cn * (d / 4);
            pqtc::residual_rows_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(A, coarse, assign + b, cn, d, resid.ptr);
            VIX_LAUNCH_CHECK();
            A = resid.ptr;
        }
        VIX_TRY(tc::make_map_rows(&mapA, A, cn, d, pqtc::kM));
        a.x = x + (size_t)b * d; a.assign = assign ? assign + b : nullptr; a.n = cn;
        a.mtiles = (int)((cn + pqtc::kM - 1) / pqtc::kM);
        a.codes = codes + (size_t)b * m;
        int rc;
        if (dsub == 8) {
            rc = mode == ENC_CSQ ? pqtc::launch<ENC_CSQ, 8>(mapA, mapB, a) : mode == ENC_CSQ_RES ? pqtc::launch<ENC_CSQ_RES, 8>(mapA, mapB, a)
               : mode == ENC_DOT ? pqtc::launch<ENC_DOT, 8>(mapA, mapB, a) : pqtc::launch<ENC_DOT_RES, 8>(mapA, mapB, a);
        } else {
            rc = mode == ENC_CSQ ? pqtc::launch<ENC_CSQ, 16>(mapA, mapB, a) : mode == ENC_CSQ_RES ? pqtc::launch<ENC_CSQ_RES, 16>(mapA, mapB, a)
               : mode == ENC_DOT ? pqtc::launch<ENC_DOT, 16>(mapA, mapB, a) : pqtc::launch<ENC_DOT_RES, 16>(mapA, mapB, a);
        }
        VIX_TRY(rc);
    }
    return VIX_OK;
}

}  // namespace vix
