// vix_gemm.cu -- tensor-core shortlist for the GEMM-shaped stages: coarse probe selection (a6-a8), IVF list
// assignment (a9) and the flat scan (a1-a4).
//
// The reference computes these stages as a dense query x centroid (or query x base) contraction followed
// by a per-row selection (Kernels/CentroidBatchScore.swift:39-88 + IVFIndex.swift:905-927;
// KMeansMiniBatchKernel.swift:341-359; FlatIndexOptimized.swift:390-477).  Parity is exact (bit-identical
// ids, tie -> lower index), so the tensor cores cannot produce the final answer -- TF32 drops 13 mantissa
// bits -- but they can produce a PROVABLY sufficient shortlist:
//
//   pass 1  S~ = ||c||^2 - 2 <q, c>  (IP: -<q, c>) on tcgen05 (kind::tf32, operands fed by TMA straight
//           from the fp32 arrays, accumulators in TMEM).  The epilogue reduces every group of `gcols`
//           columns of a row to its minimum; nothing else leaves the SM.
//   select  T_q = (k-th smallest group minimum of row q) + 2 eps_q.  k different groups hold a score
//           <= that minimum, so the exact k-th best score is <= T_q - eps_q, and every member of the exact
//           top k has S~ <= T_q.  eps_q bounds |S~ - S| for every column of the row, S being the score in
//           the reference's own fp32 evaluation (up to a constant per row: the flat scan's ||q||^2):
//             eps_q = rel ||q|| max||c|| + rel2 (||q||^2 + max||c||^2)          (shortlist_margin)
//           rel   the dot product: TF32 operand truncation 2 * 2^-10 + fp32 accumulation d * 2^-21 (x 2 for L2);
//           rel2  L2 only: the fp32 rounding that scales with the squared norms, not with ||q|| ||c|| -- the
//                 epilogue's fmaf, ||c||^2 summed in another order than the reference's (row_norms against
//                 Km12, the direct (q - x)^2 sum or the fused form), the reference's own sums (each within
//                 d u (||q|| + ||c||)^2 <= 2 d u (||q||^2 + ||c||^2), u = 2^-24) and the addition forming T_q:
//                 (3 d + 8) u, taken as 4 (d + 3) u.  Without it a row with ||q|| << max||c|| (a zero row:
//                 eps = 0) keeps only the columns whose ROUNDED norm is the smallest and can miss the column
//                 whose reference distance is smallest.  Both carry a factor 1.25 of slack.
//           IP scores have no squared-norm term; their fp32 rounding is within rel's accumulation share.
//   pass 2  the same contraction again (cheaper than keeping 10^9 scores); the epilogue emits the columns
//           with S~ <= T_q into a per-row candidate list (expected ~1.2 k entries).
//   exact   the candidates are rescored in the reference's operation order by the exact CUDA-core
//           kernels and selected by (score, index); rows whose list overflowed, or is empty (a NaN in the
//           row makes T_q NaN), fall back to the exact kernel entirely.
//
// Kernel structure (one CTA per SM, persistent over (row tile, column split) work items):
//   warp 0      TMA producer: A (128 rows x 32 tf32) and B (128 columns x 32 tf32) K-blocks, 128B swizzle,
//               into a 5-stage shared-memory ring guarded by full/empty mbarriers
//   warp 1      MMA issuer: one elected lane issues tcgen05.mma M128 N128 K8 (4 per K-block); tcgen05.commit
//               releases ring slots and publishes finished accumulators; two accumulator buffers in TMEM
//   warps 2-5   epilogue: tcgen05.ld (32 lanes x 32 columns), fused ||c||^2 term, group minima / emission
// PTX wrappers: vix_tcgen05.cuh.  Every mbarrier wait is bounded (mbar_wait there: a stuck pipeline raises an error flag).
#include "vix_common.cuh"
#include "vix_exact.cuh"
#include "vix_tcgen05.cuh"
#include "vix_group.cuh"
#include "vix_topk.cuh"

#include <stdlib.h>

#include <algorithm>
#include <atomic>
#include <mutex>

namespace vix {

int probe_select_device(const float* q, int64_t nq, const float* c, int kc, int d, int metric, int nprobe,
                        const float* cnorm, const uint64_t* disabled, int32_t* out_idx, float* out_scores);
int row_norms_device(const float* x, int64_t n, int d, float* out);

namespace tc {

constexpr int kM = 128, kN = 256, kKB = 32;            // tile rows, tile columns, tf32 elements per K-block
// (N = 256: one tcgen05.mma M128 N256 K8 is 128 clocks of tensor work.  With N = 128 the single MMA-issuing lane -- four
//  MMAs, a commit and two mbarrier round trips per K-block, ~60 instructions -- could not keep the pipe busy: 38 % active)
constexpr int kStages = 4;                            // ring stages when A and B share a stage (16 + 32 KB each)
constexpr int kStagesMax = 8;                         // ... when only B streams (32 KB each): as many as fit, up to this
constexpr int kStageBytes = (kM + kN) * kKB * 4;       // 48 KB
constexpr int kEpiWarps = 8;                          // two per TMEM lane quarter: each takes 128 of the 256 columns, 64 at a time
constexpr int kThreads = 64 + 32 * kEpiWarps;
constexpr int kTmemCols = 512;                         // two fp32 accumulators of 256 columns
constexpr uint32_t kIdesc = idesc_tf32(kM, kN);

enum Mode { MODE_WRITE = 0, MODE_MIN = 1, MODE_EMIT = 2 };

struct Args {
    int64_t nA;            // rows (queries / vectors)
    int nB;                // columns (centroids / base rows)
    int kblocks;           // ceil(d / 32)
    int ntiles;            // ceil(nB / 128)
    int tiles_per_split, nsplit, mtiles;
    int nstages;           // ring stages of this launch (set by launch())
    int mode, metric;
    const float* bnorm;    // [nB] ||c||^2 (L2) or nullptr
    int gcols, ngroups;    // MODE_MIN: columns per group (32, 64 or 128 * 2^t), groups per row
    int gshift;            // log2(gcols) when gcols < 128, else log2(gcols / 128); set by launch()
    float* gmin;           // MODE_MIN: [nA x ngroups]
    const float* thr;      // MODE_EMIT: [nA]
    int* cand_cnt;         // MODE_EMIT: [nA]
    int32_t* cand_idx;     // MODE_EMIT: [nA x cap]
    int cap;
    float* out;            // MODE_WRITE: [nA x nB]
    int* error;            // device flag, set to 1 when a barrier wait times out (the other waits then give up too)
    int* error_host;       // optional mapped host copy of the flag (raised once, never polled by the device)
};

// ---------------------------------------------------------------------------------------------- the kernel
// ARES: the row tile of A (kblocks x 16 KB, d <= 128) stays RESIDENT in shared memory for all the column tiles of a work
// item (two buffers: the next item's rows load while this item finishes) and only B streams through the ring.  Without
// it every column tile re-reads its A tile, and at d = 96 the kernel runs at the L2 -> SM bandwidth (96 KB per 128 x 128
// tile, 77 % of the chip's L2 read rate, tensor pipe 38 % busy); resident rows halve that traffic.
template <int MODE, int METRIC, bool ARES>
__global__ void __launch_bounds__(kThreads, 1)
tc_score_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, Args a) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    // 1024 B alignment for the swizzle atoms
    unsigned char* base = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    constexpr int kTileBytes = kM * kKB * 4;                                         // one K-block of the A tile: 16 KB
    constexpr int kBTileBytes = kN * kKB * 4;                                        // ... of the B tile: 32 KB
    constexpr int kRingStage = ARES ? kBTileBytes : kStageBytes;                     // B only | A + B
    const size_t a_bytes = ARES ? (size_t)a.kblocks * kTileBytes : 0;                // one resident A buffer
    unsigned char* a_res = base;                                                     // ARES: 2 x [kblocks] x 16 KB
    unsigned char* ring = base + 2 * a_bytes;                                        // kStages x (A 16 KB | B 16 KB), or x B
    uint64_t* full = reinterpret_cast<uint64_t*>(ring + (size_t)a.nstages * kRingStage);  // [kStagesMax]
    uint64_t* empty = full + kStagesMax;                                             // [kStagesMax]
    uint64_t* tfull = empty + kStagesMax;                                            // [2]
    uint64_t* tempty = tfull + 2;                                                    // [2]
    uint64_t* afull = tempty + 2;                                                    // [2] resident A buffer loaded
    uint64_t* aempty = afull + 2;                                                    // [2] ... no longer read by any MMA
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(aempty + 2);
    float* s_bn = reinterpret_cast<float*>(tmem_slot + 4);                           // [kEpiWarps][2][128] column norms

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == 0 && lane == 0) {
        for (int s = 0; s < kStagesMax; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(tfull + b, 1); mbar_init(tempty + b, kEpiWarps); }
        for (int b = 0; b < 2; ++b) { mbar_init(afull + b, 1); mbar_init(aempty + b, 1); }
        mbar_init_fence();
    }
    if (warp == 1) tmem_alloc(tmem_slot, kTmemCols);
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;
    const int nitems = a.mtiles * a.nsplit;

    if (warp == 0) {
        // ================= TMA producer =================
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            bool ok = true;
            int nitem = 0;                                             // items of this CTA so far: A buffer nitem & 1
            for (int item = blockIdx.x; item < nitems && ok; item += gridDim.x, ++nitem) {
                const int mt = item / a.nsplit, sp = item - mt * a.nsplit;
                const int nt0 = sp * a.tiles_per_split, nt1 = min(a.ntiles, nt0 + a.tiles_per_split);
                if (ARES) {
                    // the item's rows, once: all K-blocks on one barrier
                    const int ab = nitem & 1;
                    if (!mbar_wait(aempty + ab, ((uint32_t)(nitem >> 1) & 1u) ^ 1u, a.error, a.error_host)) { ok = false; break; }
                    mbar_expect_tx(afull + ab, (uint32_t)a_bytes);
                    for (int kb = 0; kb < a.kblocks; ++kb)
                        tma_load_2d(a_res + (size_t)ab * a_bytes + (size_t)kb * kTileBytes, &mapA, afull + ab, kb * kKB, mt * kM);
                }
                for (int nt = nt0; nt < nt1 && ok; ++nt) {
                    for (int kb = 0; kb < a.kblocks; ++kb) {
                        if (!mbar_wait(empty + stage, phase ^ 1, a.error, a.error_host)) { ok = false; break; }
                        unsigned char* sS = ring + (size_t)stage * kRingStage;
                        mbar_expect_tx(full + stage, kRingStage);
                        if (ARES) {
                            tma_load_2d(sS, &mapB, full + stage, kb * kKB, nt * kN);
                        } else {
                            tma_load_2d(sS, &mapA, full + stage, kb * kKB, mt * kM);
                            tma_load_2d(sS + kTileBytes, &mapB, full + stage, kb * kKB, nt * kN);      // 256 rows: 32 KB
                        }
                        if (++stage == a.nstages) { stage = 0; phase ^= 1; }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer =================
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            int acc = 0; uint32_t aphase = 0;
            bool ok = true;
            int nitem = 0;
            for (int item = blockIdx.x; item < nitems && ok; item += gridDim.x, ++nitem) {
                const int mt = item / a.nsplit, sp = item - mt * a.nsplit;
                const int nt0 = sp * a.tiles_per_split, nt1 = min(a.ntiles, nt0 + a.tiles_per_split);
                (void)mt;
                const int ab = nitem & 1;
                if (ARES) {
                    if (!mbar_wait(afull + ab, (uint32_t)(nitem >> 1) & 1u, a.error, a.error_host)) { ok = false; break; }
                    fence_after_sync();
                }
                for (int nt = nt0; nt < nt1 && ok; ++nt) {
                    if (!mbar_wait(tempty + acc, aphase ^ 1, a.error, a.error_host)) { ok = false; break; }
                    fence_after_sync();
                    const uint32_t tmem_d = tmem_base + (uint32_t)acc * kN;
                    for (int kb = 0; kb < a.kblocks; ++kb) {
                        if (!mbar_wait(full + stage, phase, a.error, a.error_host)) { ok = false; break; }
                        fence_after_sync();
                        const uint32_t sS = smem_u32(ring + (size_t)stage * kRingStage);
                        const uint32_t sA = ARES ? smem_u32(a_res + (size_t)ab * a_bytes + (size_t)kb * kTileBytes) : sS;
                        const uint64_t da = make_desc_sw128(sA), db = make_desc_sw128(ARES ? sS : sS + kTileBytes);
#pragma unroll
                        for (int k = 0; k < kKB / 8; ++k)      // K = 8 tf32 (32 B) per instruction: +2 in 16 B units
                            mma_tf32(tmem_d, da + 2 * k, db + 2 * k, kIdesc, (kb | k) ? 1u : 0u);
                        mma_commit(empty + stage);             // frees the ring slot when these MMAs retire
                        if (++stage == a.nstages) { stage = 0; phase ^= 1; }
                    }
                    if (!ok) break;
                    mma_commit(tfull + acc);                   // accumulator complete
                    if (++acc == 2) { acc = 0; aphase ^= 1; }
                }
                if (ARES && ok) mma_commit(aempty + ab);       // the resident rows are free when this item's MMAs retire
            }
        }
    } else {
        // ================= epilogue (warps 2..9; TMEM lane quarter = warp % 4, column half = (warp - 2) / 4) =================
        // a thread owns one row and 128 of the tile's 256 columns, taken in two rounds of 64 (two 32-column TMEM loads in
        // flight per round)
        const int quarter = warp & 3;
        const int half = (warp - 2) >> 2;
        int acc = 0; uint32_t aphase = 0;
        bool ok = true;
        for (int item = blockIdx.x; item < nitems && ok; item += gridDim.x) {
            const int mt = item / a.nsplit, sp = item - mt * a.nsplit;
            const int nt0 = sp * a.tiles_per_split, nt1 = min(a.ntiles, nt0 + a.tiles_per_split);
            const int64_t row = (int64_t)mt * kM + quarter * 32 + lane;
            const bool row_ok = row < a.nA;
            const float thr = (MODE == MODE_EMIT && row_ok) ? a.thr[row] : -INFINITY;
            float gmin = INFINITY;
            // this warp's 128 column norms of a tile travel one tile ahead in registers (their L2 round trip used to sit in
            // front of every tile's accumulator wait)
            float nb_next[4];
            auto load_norms = [&](int nt) {
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    const int col = nt * kN + half * 128 + t * 32 + lane;
                    nb_next[t] = (a.bnorm && nt < nt1 && col < a.nB) ? __ldg(a.bnorm + col) : 0.0f;
                }
            };
            load_norms(nt0);
            for (int nt = nt0; nt < nt1 && ok; ++nt) {
                // stage the norms (private copy per warp: no CTA-level barrier needed), start the next tile's loads
                float* bn = s_bn + ((warp - 2) * 2 + acc) * 128;
#pragma unroll
                for (int t = 0; t < 4; ++t) bn[t * 32 + lane] = nb_next[t];
                load_norms(nt + 1);
                __syncwarp();
                if (!mbar_wait(tfull + acc, aphase, a.error, a.error_host)) { ok = false; break; }
                fence_after_sync();
                const bool full_tile = nt * kN + kN <= a.nB;
                unsigned long long hits[2] = {0ull, 0ull};     // MODE_EMIT: this thread's columns with S~ <= T, per round
#pragma unroll 1
                for (int rd = 0; rd < 2; ++rd) {
                    const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)acc * kN + (uint32_t)half * 128 +
                                           (uint32_t)rd * 64;
                    const int colbase = nt * kN + half * 128 + rd * 64;
                    uint32_t vraw[2][32];
                    tmem_ld32_issue(taddr, vraw[0]);
                    tmem_ld32_issue(taddr + 32, vraw[1]);
                    tmem_ld32_wait(vraw[0], vraw[1]);
#pragma unroll
                    for (int ck = 0; ck < 2; ++ck) {
                        float v[32];
#pragma unroll
                        for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(vraw[ck][i]);
                        const float4* bn4 = reinterpret_cast<const float4*>(bn + rd * 64 + ck * 32);
                        float sc[32];
#pragma unroll
                        for (int i4 = 0; i4 < 8; ++i4) {
                            const float4 nb = (METRIC == VIX_METRIC_L2) ? bn4[i4] : make_float4(0.f, 0.f, 0.f, 0.f);
                            const float nbv[4] = {nb.x, nb.y, nb.z, nb.w};
#pragma unroll
                            for (int u = 0; u < 4; ++u) {
                                const int i = 4 * i4 + u;
                                sc[i] = (METRIC == VIX_METRIC_L2) ? fmaf(-2.0f, v[i], nbv[u]) : -v[i];
                            }
                        }
                        if (!full_tile) {                          // last column tile only: mask the columns beyond nB
#pragma unroll
                            for (int i = 0; i < 32; ++i)
                                if (colbase + ck * 32 + i >= a.nB) sc[i] = INFINITY;
                        }
                        if (MODE == MODE_WRITE) {
#pragma unroll
                            for (int i = 0; i < 32; ++i) {
                                const int col = colbase + ck * 32 + i;
                                if (row_ok && col < a.nB) a.out[row * a.nB + col] = sc[i];
                            }
                        } else if (MODE == MODE_MIN) {
                            // tree minimum of the 32 columns
#pragma unroll
                            for (int w2 = 16; w2 > 0; w2 >>= 1)
#pragma unroll
                                for (int i = 0; i < w2; ++i) sc[i] = fminf(sc[i], sc[i + w2]);
                            gmin = fminf(gmin, sc[0]);
                            // group boundary.  gcols 32 / 64 / 128: groups are whole chunks / rounds / the 128-column strip of
                            // this thread; gcols = 256 t: a group is this thread's strip of t consecutive tiles (the two
                            // column halves of a tile belong to different groups: any disjoint partition is valid)
                            bool flush;
                            int g;
                            if (a.gcols < kN) {                   // gcols and tiles-per-group are powers of two
                                const int colend = colbase + ck * 32 + 32;
                                flush = (colend & (a.gcols - 1)) == 0;
                                g = (colend - 1) >> a.gshift;
                            } else {
                                flush = rd == 1 && ck == 1 && (((nt + 1) & ((1 << a.gshift) - 1)) == 0 || nt == a.ntiles - 1);
                                g = (nt >> a.gshift) * 2 + half;
                            }
                            if (flush) {
                                if (row_ok && g < a.ngroups) a.gmin[row * a.ngroups + g] = gmin;
                                gmin = INFINITY;
                            }
                        } else {
                            uint32_t hit = 0;                      // columns of this chunk with S~ <= T
#pragma unroll
                            for (int i = 0; i < 32; ++i) hit |= (sc[i] <= thr) ? (1u << i) : 0u;
                            hits[rd] |= (unsigned long long)hit << (32 * ck);
                        }
                    }
                }
                fence_before_sync();
                __syncwarp();
                if (lane == 0) mbar_arrive(tempty + acc);      // 8 arrivals free the accumulator
                if (++acc == 2) { acc = 0; aphase ^= 1; }
                if (MODE == MODE_EMIT && (hits[0] | hits[1])) {
                    // emission AFTER the accumulator has been handed back, one counter update per thread and tile: the
                    // round trip of the global atomic (rare hits: a few hundred per row in the whole matrix) used to sit
                    // between the TMEM read and the release, once per hit
                    int pos = atomicAdd(a.cand_cnt + row, __popcll(hits[0]) + __popcll(hits[1]));
#pragma unroll
                    for (int rd = 0; rd < 2; ++rd) {
                        unsigned long long h = hits[rd];
                        const int colbase = nt * kN + half * 128 + rd * 64;
                        while (h) {
                            const int i = __ffsll((long long)h) - 1;
                            h &= h - 1;
                            if (pos < a.cap) a.cand_idx[row * a.cap + pos] = colbase + i;
                            ++pos;
                        }
                    }
                }
            }
        }
    }
    fence_before_sync();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, kTmemCols);
}

// ---------------------------------------------------------------------------------------------- host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
        else
            cudaGetLastError();
    });
    return fn;
}

int make_map_rows(CUtensorMap* map, const float* ptr, int64_t rows, int d, int box_rows) {
    EncodeTiledFn fn = encode_fn();
    VIX_REQUIRE(fn != nullptr, VIX_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
    cuuint64_t gdim[2] = {(cuuint64_t)d, (cuuint64_t)rows};
    cuuint64_t gstride[1] = {(cuuint64_t)d * 4};
    cuuint32_t box[2] = {(cuuint32_t)kKB, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(ptr), gdim, gstride, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    VIX_REQUIRE(r == CUDA_SUCCESS, VIX_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) for a %lld x %d operand", (int)r,
                (long long)rows, d);
    return VIX_OK;
}

static int make_map(CUtensorMap* map, const float* ptr, int64_t rows, int d) { return make_map_rows(map, ptr, rows, d, kM); }

bool supported(int64_t nA, int64_t nB, int d, const float* A, const float* B) {
    if (nA <= 0 || nB <= 0 || d < 4 || (d & 3) != 0) return false;            // TMA: 16-byte row pitch
    if ((reinterpret_cast<uintptr_t>(A) & 15) || (reinterpret_cast<uintptr_t>(B) & 15)) return false;
    if (nB >= (1LL << 31) - kN) return false;
    return encode_fn() != nullptr;
}

// rows resident (ARES) when both A buffers and the B ring fit: d <= 128
// (d <= 96: both A buffers + three 32 KB B stages; at d = 128 only two B stages would be left, so A streams there)
static bool a_resident(int kblocks) { return kblocks <= 3; }
static int ring_stages(int kblocks) {
    if (!a_resident(kblocks)) return kStages;
    const size_t left = 227 * 1024 - 12 * 1024 - (size_t)2 * kblocks * kM * kKB * 4;
    const int n = (int)(left / ((size_t)kN * kKB * 4));
    return n > kStagesMax ? kStagesMax : n;
}
static size_t smem_bytes(int kblocks) {
    const size_t ring = a_resident(kblocks) ? (size_t)2 * kblocks * kM * kKB * 4 + (size_t)ring_stages(kblocks) * kN * kKB * 4
                                            : (size_t)kStages * kStageBytes;
    return ring + 1024 + 512 + (size_t)kEpiWarps * 2 * 128 * 4;
}

static int launch(const float* A, int64_t nA, const float* B, int nB, int d, Args& a) {
    CUtensorMap mapA, mapB;
    VIX_TRY(make_map(&mapA, A, nA, d));
    VIX_TRY(make_map_rows(&mapB, B, nB, d, kN));
    a.nA = nA; a.nB = nB;
    a.kblocks = (d + kKB - 1) / kKB;
    a.ntiles = (nB + kN - 1) / kN;
    a.mtiles = (int)((nA + kM - 1) / kM);
    // column splits: enough work items for eight waves of the SMs (with three, the last wave of C5's probe stage ran a
    // fifth of the SMs); in MODE_MIN a split is a whole number of groups
    int nsplit = (8 * num_sms() + a.mtiles - 1) / a.mtiles;
    if (nsplit < 1) nsplit = 1;
    if (nsplit > a.ntiles) nsplit = a.ntiles;
    int tps = (a.ntiles + nsplit - 1) / nsplit;
    if (a.mode == MODE_MIN && a.gcols > kN) {
        const int tpg = a.gcols / kN;
        tps = (tps + tpg - 1) / tpg * tpg;
    }
    a.tiles_per_split = tps;
    a.nsplit = (a.ntiles + tps - 1) / tps;
    {
        int v = a.gcols < kN ? a.gcols : a.gcols / kN, sh = 0;
        while ((1 << sh) < v) ++sh;
        VIX_REQUIRE((1 << sh) == v, VIX_ERR_INVALID_PARAM, "tensor-core shortlist: group width %d is not a power of two", a.gcols);
        a.gshift = sh;
    }
    const size_t smem = smem_bytes(a.kblocks);
    const bool ares = a_resident(a.kblocks);
    a.nstages = ring_stages(a.kblocks);
    int64_t grid = (int64_t)a.mtiles * a.nsplit;
    if (grid > num_sms()) grid = num_sms();
#define VIX_TC_LAUNCH(MODE_, METRIC_)                                                                                   \
    do {                                                                                                               \
        auto kern = ares ? tc_score_kernel<MODE_, METRIC_, true> : tc_score_kernel<MODE_, METRIC_, false>;             \
        VIX_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));                  \
        kern<<<(unsigned)grid, kThreads, smem, ctx().stream>>>(mapA, mapB, a);                                         \
    } while (0)
    const bool l2 = a.metric == VIX_METRIC_L2;
    if (a.mode == MODE_MIN) { if (l2) VIX_TC_LAUNCH(MODE_MIN, VIX_METRIC_L2); else VIX_TC_LAUNCH(MODE_MIN, VIX_METRIC_IP); }
    else if (a.mode == MODE_EMIT) { if (l2) VIX_TC_LAUNCH(MODE_EMIT, VIX_METRIC_L2); else VIX_TC_LAUNCH(MODE_EMIT, VIX_METRIC_IP); }
    else { if (l2) VIX_TC_LAUNCH(MODE_WRITE, VIX_METRIC_L2); else VIX_TC_LAUNCH(MODE_WRITE, VIX_METRIC_IP); }
#undef VIX_TC_LAUNCH
    VIX_LAUNCH_CHECK();
    return VIX_OK;
}

// ---------------------------------------------------------------------------------------------- thresholds
// eps_q = rel ||q|| max||c|| + rel2 (||q||^2 + max||c||^2): the bound on |S~ - S| of the header, for all three consumers
struct Margin { float rel, rel2; };
static Margin shortlist_margin(int d, int metric) {
    const bool l2 = metric == VIX_METRIC_L2;
    return {(l2 ? 2.0f : 1.0f) * 1.25f * (2.0f / 1024.0f + (float)d / 2097152.0f),
            l2 ? 1.25f * (float)(d + 3) / 4194304.0f : 0.0f};
}
__device__ __forceinline__ float shortlist_eps(Margin m, float anorm, float bnorm_max) {
    return m.rel * sqrtf(anorm) * bnorm_max + m.rel2 * (anorm + bnorm_max * bnorm_max);
}

// T_q = (k-th smallest group minimum of the row) + margin_q.  One WARP per row: the <= 32 VPL minima of the row stay in
// registers as order-preserving 32-bit keys and the k-th smallest is found by a radix select, one bit per step
// (how many keys share the prefix found so far and have a 0 in this bit?) with warp ballots -- no shared memory, no
// CTA-wide barrier, a third of the instructions of sorting the row.
template <int VPL>
__global__ void __launch_bounds__(256)
threshold_kernel(const float* __restrict__ gmin, int64_t nrows, int ngroups, int k, const float* __restrict__ anorm,
                 const float* __restrict__ bnorm_max, Margin margin, float* __restrict__ thr) {
    const int lane = threadIdx.x & 31;
    const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (row >= nrows) return;
    uint32_t v[VPL];
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
        const int g = lane + 32 * i;
        v[i] = g < ngroups ? f32_orderable(__ldg(gmin + row * ngroups + g)) : 0xFFFFFFFFu;
    }
    float kth = INFINITY;
    if (k - 1 < ngroups) {
        uint32_t prefix = 0;
        int want = k;                                       // rank (1-based) among the keys that match the prefix
        for (int bit = 31; bit >= 0; --bit) {
            const uint32_t hi = bit == 31 ? 0u : ~((2u << bit) - 1u);      // the bits above `bit`
            int zeros = 0;
#pragma unroll
            for (int i = 0; i < VPL; ++i)
                zeros += __popc(__ballot_sync(0xFFFFFFFFu, ((v[i] ^ prefix) & hi) == 0u && !((v[i] >> bit) & 1u)));
            if (want > zeros) { want -= zeros; prefix |= 1u << bit; }
        }
        kth = f32_from_orderable(prefix);
    }
    if (lane == 0) thr[row] = kth + 2.0f * shortlist_eps(margin, anorm[row], bnorm_max[0]);
}

static int launch_threshold(const float* gmin, int64_t nrows, int ngroups, int k, const float* anorm, const float* bnorm_max,
                            Margin margin, float* thr) {
    const unsigned grid = (unsigned)((nrows * 32 + 255) / 256);
    cudaStream_t s = ctx().stream;
    if (ngroups <= 256) threshold_kernel<8><<<grid, 256, 0, s>>>(gmin, nrows, ngroups, k, anorm, bnorm_max, margin, thr);
    else if (ngroups <= 512) threshold_kernel<16><<<grid, 256, 0, s>>>(gmin, nrows, ngroups, k, anorm, bnorm_max, margin, thr);
    else if (ngroups <= 1024) threshold_kernel<32><<<grid, 256, 0, s>>>(gmin, nrows, ngroups, k, anorm, bnorm_max, margin, thr);
    else if (ngroups <= 2048) threshold_kernel<64><<<grid, 256, 0, s>>>(gmin, nrows, ngroups, k, anorm, bnorm_max, margin, thr);
    else if (ngroups <= 4096) threshold_kernel<128><<<grid, 256, 0, s>>>(gmin, nrows, ngroups, k, anorm, bnorm_max, margin, thr);
    else { set_error("threshold: %d groups per row (> 4096)", ngroups); return VIX_ERR_UNSUPPORTED; }
    VIX_LAUNCH_CHECK();
    return VIX_OK;
}

__global__ void max_sqrt_kernel(const float* __restrict__ x, int64_t n, float* __restrict__ out) {
    // single CTA: out[0] = sqrt(max x)
    __shared__ float s[256];
    float m = 0.0f;
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) m = fmaxf(m, x[i]);
    s[threadIdx.x] = m;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) { if ((int)threadIdx.x < o) s[threadIdx.x] = fmaxf(s[threadIdx.x], s[threadIdx.x + o]); __syncthreads(); }
    if (threadIdx.x == 0) out[0] = sqrtf(s[0]);
}

// ---------------------------------------------------------------------------------------------- exact rescoring
// One WARP per row: exact CentroidBatchScore value of every candidate in the reference's operation order
// (sequential dot, then -2 s + ||c||^2 / -s; Kernels/CentroidBatchScore.swift:54-64), keys (score, index),
// bitonic sort of the next power of two >= n, best `k` out.  The warp takes 32 candidates at a time: their rows
// are read 32 floats at a time with coalesced 128-byte loads (all 32 in flight) into a padded shared tile, and
// lane i then walks row i of the tile -- one sequential chain per candidate, the same operations in the same order
// as a thread reading its row straight from global memory, at a thirtieth of the L1 traffic.  Nothing in the
// kernel synchronises more than a warp.  Rows whose candidate list overflowed or is empty are flagged for the exact kernel
// below.
constexpr int kRescoreWarps = 8;
__global__ void __launch_bounds__(32 * kRescoreWarps)
rescore_probe_kernel(const float* __restrict__ A, int64_t nA, const float* __restrict__ B, int d, int metric,
                     const float* __restrict__ bnorm, const int* __restrict__ cand_cnt,
                     const int32_t* __restrict__ cand_idx, int cap, int Pmax, int k, int32_t* __restrict__ out_idx,
                     float* __restrict__ out_scores, int* __restrict__ overflow_rows, int* __restrict__ n_overflow) {
    extern __shared__ __align__(16) unsigned char smem_rs[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int dpad = (d + 31) & ~31;
    u64* keys = reinterpret_cast<u64*>(smem_rs) + (size_t)warp * Pmax;                       // [warps][Pmax]
    float* sq = reinterpret_cast<float*>(reinterpret_cast<u64*>(smem_rs) + (size_t)kRescoreWarps * Pmax) + (size_t)warp * dpad;
    float* tile = reinterpret_cast<float*>(reinterpret_cast<u64*>(smem_rs) + (size_t)kRescoreWarps * Pmax) +
                  (size_t)kRescoreWarps * dpad + (size_t)warp * (32 * 33);                   // [warps][32][33]
    const int64_t row = (int64_t)blockIdx.x * kRescoreWarps + warp;
    if (row >= nA) return;
    const int n = cand_cnt[row];
    if (n > cap || n == 0) {                                           // overflowed, or empty (T_q NaN)
        if (lane == 0) overflow_rows[atomicAdd(n_overflow, 1)] = (int)row;
        return;
    }
    const int P = next_pow2(n < 2 ? 2 : n);                            // <= Pmax
    for (int e = lane; e < dpad; e += 32) sq[e] = e < d ? A[row * d + e] : 0.0f;
    for (int i = n + lane; i < P; i += 32) keys[i] = kEmptyKey;
    __syncwarp();
    for (int base = 0; base < n; base += 32) {
        const int i = base + lane;
        const int c = cand_idx[row * cap + (i < n ? i : base)];
        float acc = 0.0f;
        for (int e0 = 0; e0 < d; e0 += 32) {
            const int w = min(32, d - e0);
            float v[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) {                             // candidate j of the batch: 128 coalesced bytes
                const int cj = __shfl_sync(0xFFFFFFFFu, c, j);
                v[j] = lane < w ? __ldg(B + (int64_t)cj * d + e0 + lane) : 0.0f;
            }
#pragma unroll
            for (int j = 0; j < 32; ++j) tile[j * 33 + lane] = v[j];
            __syncwarp();
            for (int t = 0; t < w; ++t) acc = fadd(acc, fmul(sq[e0 + t], tile[lane * 33 + t]));
            __syncwarp();
        }
        if (i < n) {
            const float s = (metric == VIX_METRIC_L2) ? fadd(fmul(-2.0f, acc), bnorm[c]) : fmul(-1.0f, acc);
            keys[i] = make_key(s, (uint32_t)c, 0);
        }
    }
    __syncwarp();
    bitonic_sort_keys<true>(keys, P, lane, 32);
    for (int i = lane; i < k; i += 32) {
        const u64 key = i < P ? keys[i] : kEmptyKey;
        const size_t o = (size_t)row * k + i;
        if (key == kEmptyKey) { out_idx[o] = -1; if (out_scores) out_scores[o] = __int_as_float(0x7fc00000); }
        else { out_idx[o] = (int32_t)key_id(key); if (out_scores) out_scores[o] = cbs_signed_zero(key_score(key, 0), key_id(key), metric, bnorm); }
    }
}

// The rows whose shortlist overflowed or is empty (normally none), without a host round trip: a fixed grid walks the list the
// kernel above left on the device; one CTA per row scores EVERY column in the same operation order and selects by
// (score, index) with a CTA-wide queue.
__global__ void __launch_bounds__(256)
probe_overflow_rows_kernel(const float* __restrict__ A, const float* __restrict__ B, int nB, int d, int metric,
                           const float* __restrict__ bnorm, const int* __restrict__ overflow_rows,
                           const int* __restrict__ n_overflow, int P, int k, int32_t* __restrict__ out_idx,
                           float* __restrict__ out_scores) {
    extern __shared__ __align__(16) unsigned char smem_po[];
    u64* keys = reinterpret_cast<u64*>(smem_po);
    float* sq = reinterpret_cast<float*>(keys + P);
    __shared__ int s_cnt;
    __shared__ u64 s_thr;
    const int nrows = *n_overflow;
    for (int r = blockIdx.x; r < nrows; r += gridDim.x) {
        const int64_t row = overflow_rows[r];
        __syncthreads();
        for (int e = threadIdx.x; e < d; e += blockDim.x) sq[e] = A[row * d + e];
        BlockQueue q{keys, &s_cnt, &s_thr, k, P};
        q.init();
        for (int base = 0; base < nB; base += blockDim.x) {
            q.flush_if_needed(blockDim.x);
            const int c = base + threadIdx.x;
            if (c < nB) {
                const float dot = exact_pair<SpecSeqDot>(sq, B + (int64_t)c * d, d);
                const float s = (metric == VIX_METRIC_L2) ? fadd(fmul(-2.0f, dot), bnorm[c]) : fmul(-1.0f, dot);
                q.push(make_key(s, (uint32_t)c, 0));
            }
        }
        q.flush();
        for (int i = threadIdx.x; i < k; i += blockDim.x) {
            const u64 key = keys[i];
            const size_t o = (size_t)row * k + i;
            if (key == kEmptyKey) { out_idx[o] = -1; if (out_scores) out_scores[o] = __int_as_float(0x7fc00000); }
            else { out_idx[o] = (int32_t)key_id(key); if (out_scores) out_scores[o] = cbs_signed_zero(key_score(key, 0), key_id(key), metric, bnorm); }
        }
    }
}

// k = 1 (assignment): T = (smallest group minimum) + margin, one thread per row
__global__ void threshold_min_kernel(const float* __restrict__ gmin, int64_t n, int ngroups, const float* __restrict__ anorm,
                                     const float* __restrict__ bnorm_max, Margin margin, float* __restrict__ thr) {
    const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= n) return;
    float m = INFINITY;
    for (int g = 0; g < ngroups; ++g) m = fminf(m, gmin[row * ngroups + g]);
    thr[row] = m + 2.0f * shortlist_eps(margin, anorm[row], bnorm_max[0]);
}

// IVF list assignment from the shortlist: one thread per vector evaluates the reference's exact distance
// (_vi_km12_l2sq_aos order, KMeansMiniBatchKernel.swift:198-225) for its few candidates and keeps
// (distance, then lower index) (:341-359).  Rows without a usable shortlist go to the exact kernel.
__global__ void __launch_bounds__(128)
rescore_assign_kernel(const float* __restrict__ X, int64_t n, const float* __restrict__ C, int d,
                      const int* __restrict__ cand_cnt, const int32_t* __restrict__ cand_idx, int cap,
                      int32_t* __restrict__ assign, float* __restrict__ dist, int* __restrict__ overflow_rows,
                      int* __restrict__ n_overflow) {
    const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= n) return;
    const int cnt = cand_cnt[row];
    if (cnt > cap || cnt == 0) {
        overflow_rows[atomicAdd(n_overflow, 1)] = (int)row;
        return;
    }
    const float* x = X + row * d;
    float bd = INFINITY;
    int bi = 0x7FFFFFFF;
    for (int i = 0; i < cnt; ++i) {
        const int c = cand_idx[row * cap + i];
        const float dd = exact_pair<SpecKm12L2>(x, C + (int64_t)c * d, d);
        if (dd < bd || (dd == bd && c < bi)) { bd = dd; bi = c; }
    }
    if (bi == 0x7FFFFFFF) { overflow_rows[atomicAdd(n_overflow, 1)] = (int)row; return; }
    assign[row] = bi;
    if (dist) dist[row] = bd;
}

__global__ void scatter_assign_rows_kernel(const int32_t* __restrict__ sub_assign, const float* __restrict__ sub_dist,
                                           const int* __restrict__ rows, int n, int32_t* __restrict__ assign,
                                           float* __restrict__ dist) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    assign[rows[i]] = sub_assign[i];
    if (dist) dist[rows[i]] = sub_dist[i];
}

// Flat scan from the shortlist: one CTA per query evaluates the reference kernel for every candidate --
// _l2sqr_single_direct (d < 256, L2SqrKernel.swift:192-238), the fused dot form with clamp (d >= 256, :411-448) or
// InnerProduct (InnerProduct.swift:115-184) -- then selects by (score, id) and maps to the API distance
// (FlatIndexOptimized.swift:457-474: sqrt for L2, -dot for IP).
__global__ void __launch_bounds__(256)
rescore_flat_kernel(const float* __restrict__ A, const float* __restrict__ B, int d, int metric, int dotfused,
                    const float* __restrict__ anorm, const float* __restrict__ bnorm, const int* __restrict__ cand_cnt,
                    const int32_t* __restrict__ cand_idx, int cap, int P, int k, int raw, float* __restrict__ out_dist,
                    int64_t* __restrict__ out_ids, int* __restrict__ overflow_rows, int* __restrict__ n_overflow) {
    extern __shared__ __align__(16) unsigned char smem_rf[];
    u64* keys = reinterpret_cast<u64*>(smem_rf);
    float* sq = reinterpret_cast<float*>(keys + P);
    const int64_t row = blockIdx.x;
    const int n = cand_cnt[row];
    if (n > cap || n == 0) {                                           // overflowed, or empty (T_q NaN)
        if (threadIdx.x == 0) overflow_rows[atomicAdd(n_overflow, 1)] = (int)row;
        return;
    }
    const int order_max = (metric == VIX_METRIC_IP);
    for (int e = threadIdx.x; e < d; e += blockDim.x) sq[e] = A[row * d + e];
    for (int i = threadIdx.x; i < P; i += blockDim.x) keys[i] = kEmptyKey;
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const int c = cand_idx[row * cap + i];
        const float* xr = B + (int64_t)c * d;
        float s;
        if (order_max) s = exact_pair<SpecIp4>(sq, xr, d);
        else if (dotfused) {
            const float dot = exact_pair<SpecDot16>(sq, xr, d);
            const float dist = fsub(fadd(anorm[row], bnorm[c]), fmul(2.0f, dot));
            s = dist < 0.0f ? 0.0f : dist;
        } else s = exact_pair<SpecDirect16L2>(sq, xr, d);
        keys[i] = make_key(s, (uint32_t)c, order_max);
    }
    __syncthreads();
    bitonic_sort_keys<false>(keys, P, threadIdx.x, blockDim.x);
    for (int i = threadIdx.x; i < k; i += blockDim.x) {
        const u64 key = keys[i];
        const size_t o = (size_t)row * k + i;
        if (key == kEmptyKey) { out_dist[o] = __int_as_float(0x7fc00000); out_ids[o] = -1; }
        else {
            float sc = key_score(key, order_max);
            if (!raw) sc = order_max ? -sc : __fsqrt_rn(sc);
            out_dist[o] = sc;
            out_ids[o] = (int64_t)key_id(key);
        }
    }
}

__global__ void scatter_flat_rows_kernel(const float* __restrict__ sub_d, const int64_t* __restrict__ sub_i, int k,
                                         const int* __restrict__ rows, int n, float* __restrict__ out_d,
                                         int64_t* __restrict__ out_i) {
    const int i = blockIdx.x;
    if (i >= n) return;
    for (int e = threadIdx.x; e < k; e += blockDim.x) {
        out_d[(int64_t)rows[i] * k + e] = sub_d[(int64_t)i * k + e];
        out_i[(int64_t)rows[i] * k + e] = sub_i[(int64_t)i * k + e];
    }
}

__global__ void scatter_probe_rows_kernel(const int32_t* __restrict__ idx, const float* __restrict__ sc, int k,
                                          const int* __restrict__ rows, int n, int32_t* __restrict__ out_idx,
                                          float* __restrict__ out_sc) {
    const int i = blockIdx.x;
    if (i >= n) return;
    for (int e = threadIdx.x; e < k; e += blockDim.x) {
        out_idx[(int64_t)rows[i] * k + e] = idx[(int64_t)i * k + e];
        if (out_sc) out_sc[(int64_t)rows[i] * k + e] = sc[(int64_t)i * k + e];
    }
}

// route evidence per shortlist kind (vix_tc_shortlist_calls / vix_tc_shortlist_exact_rows)
static std::atomic<long long> g_calls[3], g_exact_rows[3];

// number of group minima per row for a given group width (see the MODE_MIN epilogue)
static int num_groups(int64_t nB, int gcols) {
    if (gcols < kN) return (int)((nB + gcols - 1) / gcols);
    const int64_t ntiles = (nB + kN - 1) / kN, tpg = gcols / kN;
    return (int)(2 * ((ntiles + tpg - 1) / tpg));
}

// columns per group so that a row has between ~4 k and 2048 group minima
static int choose_gcols(int nB, int k) {
    if (k <= 1) return nB > 4096 ? 4096 : 128;       // assignment: only the row minimum matters
    int g = 32;
    while ((nB + g - 1) / g > 1024 && (nB + 2 * g - 1) / (2 * g) >= 8 * k) g *= 2;
    while ((nB + g - 1) / g > 2048) g *= 2;
    while (g < 128 && (nB + g - 1) / g > 64 * k && (nB + 2 * g - 1) / (2 * g) >= 8 * k) g *= 2;
    return g;
}

}  // namespace tc

// Debug / test entry: the raw tensor-core scores S~ (MODE_WRITE)
int tc_scores_device(const float* q, int64_t nq, const float* c, int kc, int d, int metric, const float* cnorm,
                     float* out) {
    VIX_REQUIRE(tc::supported(nq, kc, d, q, c), VIX_ERR_UNSUPPORTED, "tensor-core path needs d %% 4 == 0 and 16-byte aligned operands");
    Scratch<int> err;
    VIX_TRY(err.alloc(1));
    VIX_CUDA(cudaMemsetAsync(err.ptr, 0, 4, ctx().stream));
    tc::Args a{};
    a.mode = tc::MODE_WRITE; a.metric = metric; a.bnorm = cnorm; a.out = out; a.error = err.ptr;
    a.gcols = 32; a.ngroups = 0;
    VIX_TRY(tc::launch(q, nq, c, kc, d, a));
    int herr = 0;
    VIX_CUDA(cudaMemcpyAsync(&herr, err.ptr, 4, cudaMemcpyDeviceToHost, ctx().stream));
    VIX_CUDA(cudaStreamSynchronize(ctx().stream));
    VIX_REQUIRE(herr == 0, VIX_ERR_CUDA, "tensor-core pipeline timed out");
    return VIX_OK;
}

// out[0] = sqrt(max x[i]) on the device (the index caches it for its coarse-centroid norms)
int max_sqrt_device(const float* x, int64_t n, float* out) {
    tc::max_sqrt_kernel<<<1, 256, 0, ctx().stream>>>(x, n, out);
    VIX_LAUNCH_CHECK();
    return VIX_OK;
}

// Probe selection through the tensor-core shortlist; results identical to probe_select_device.
int probe_select_fast_device(const float* q, int64_t nq, const float* c, int kc, int d, int metric, int nprobe,
                             const float* cnorm, int32_t* out_idx, float* out_scores, const float* cnorm_max_sqrt) {
    const int keff = nprobe < kc ? nprobe : kc;
    const int gcols = tc::choose_gcols(kc, keff);
    const int ngroups = tc::num_groups(kc, gcols);
    const bool use_tc = getenv("VIX_DISABLE_TC") == nullptr && tc::supported(nq, kc, d, q, c) && kc >= 1024 && nq >= 16 &&
                        ngroups >= 2 * keff && keff <= 256 && d <= 4096 && (metric == VIX_METRIC_IP || cnorm != nullptr);
    const int cap = keff * 4 + 128;
    const size_t rescore_smem = (size_t)tc::kRescoreWarps * ((size_t)next_pow2(cap) * 8 + (size_t)((d + 31) & ~31) * 4 + 32 * 33 * 4);
    if (!use_tc || rescore_smem > 227 * 1024)
        return probe_select_device(q, nq, c, kc, d, metric, nprobe, cnorm, nullptr, out_idx, out_scores);
    cudaStream_t s = ctx().stream;
    VIX_TRY(check_pipeline_error());                   // a pipeline that gave up in an earlier asynchronous call
    tc::g_calls[VIX_SHORTLIST_PROBE].fetch_add(1);     // (its exact rows stay on the device: no host round trip here)
    int* pipe_flag = pipeline_error_flag();
    VIX_REQUIRE(pipe_flag != nullptr, VIX_ERR_OOM, "cannot allocate the mapped pipeline-error flag");
    Scratch<float> gmin, thr, qn, cn_tmp, cmax;
    Scratch<int> cand_cnt, flags, ovf_rows;
    Scratch<int32_t> cand_idx;
    VIX_TRY(gmin.alloc((size_t)nq * ngroups));
    VIX_TRY(thr.alloc((size_t)nq));
    VIX_TRY(qn.alloc((size_t)nq));
    VIX_TRY(cmax.alloc(1));
    VIX_TRY(cand_cnt.alloc((size_t)nq));
    VIX_TRY(cand_idx.alloc((size_t)nq * cap));
    VIX_TRY(flags.alloc(2));                           // [0] pipeline gave up, [1] number of overflow rows
    VIX_TRY(ovf_rows.alloc((size_t)nq));
    VIX_CUDA(cudaMemsetAsync(flags.ptr, 0, 8, s));
    VIX_CUDA(cudaMemsetAsync(cand_cnt.ptr, 0, (size_t)nq * 4, s));
    VIX_TRY(row_norms_device(q, nq, d, qn.ptr));
    const float* cn = cnorm;
    if (!cn) { VIX_TRY(cn_tmp.alloc((size_t)kc)); VIX_TRY(row_norms_device(c, kc, d, cn_tmp.ptr)); cn = cn_tmp.ptr; }
    const float* cmaxp = cnorm_max_sqrt;               // sqrt(max ||c||^2): cached by the index, else computed here
    if (!cmaxp) {
        tc::max_sqrt_kernel<<<1, 256, 0, s>>>(cn, kc, cmax.ptr);
        VIX_LAUNCH_CHECK();
        cmaxp = cmax.ptr;
    }

    tc::Args a{};
    a.metric = metric; a.bnorm = (metric == VIX_METRIC_L2) ? cn : nullptr; a.error = flags.ptr; a.error_host = pipe_flag;
    a.mode = tc::MODE_MIN; a.gcols = gcols; a.ngroups = ngroups; a.gmin = gmin.ptr;
    VIX_TRY(tc::launch(q, nq, c, kc, d, a));
    VIX_TRY(tc::launch_threshold(gmin.ptr, nq, ngroups, keff, qn.ptr, cmaxp, tc::shortlist_margin(d, metric), thr.ptr));
    a.mode = tc::MODE_EMIT; a.thr = thr.ptr; a.cand_cnt = cand_cnt.ptr; a.cand_idx = cand_idx.ptr; a.cap = cap;
    VIX_TRY(tc::launch(q, nq, c, kc, d, a));
    {
        const int P = next_pow2(cap);
        const size_t smem = rescore_smem;
        VIX_CUDA(cudaFuncSetAttribute(tc::rescore_probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        tc::rescore_probe_kernel<<<(unsigned)((nq + tc::kRescoreWarps - 1) / tc::kRescoreWarps), 32 * tc::kRescoreWarps, smem, s>>>(
            q, nq, c, d, metric, cn, cand_cnt.ptr, cand_idx.ptr, cap, P, nprobe, out_idx, out_scores, ovf_rows.ptr, flags.ptr + 1);
        VIX_LAUNCH_CHECK();
    }
    {
        // rows whose shortlist overflowed, if any (no host round trip: the call stays asynchronous)
        const int P = next_pow2(nprobe + 256);
        const size_t smem = (size_t)P * 8 + (size_t)d * 4;
        VIX_CUDA(cudaFuncSetAttribute(tc::probe_overflow_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        tc::probe_overflow_rows_kernel<<<(unsigned)(2 * num_sms()), 256, smem, s>>>(q, c, kc, d, metric, cn, ovf_rows.ptr,
                                                                                  flags.ptr + 1, P, nprobe, out_idx, out_scores);
        VIX_LAUNCH_CHECK();
    }
    return VIX_OK;
}

int flat_search_device(const float* q, int64_t nq, const float* xb, int64_t n, int d, int metric, int k,
                       const float* xb_norm, float* out_dist, int64_t* out_ids, bool raw_scores);

// Exact flat search (a1-a4) through the tensor-core shortlist; results identical to flat_search_device.
int flat_search_auto_device(const float* q, int64_t nq, const float* xb, int64_t n, int d, int metric, int k,
                            const float* xb_norm, float* out_dist, int64_t* out_ids, bool raw_scores) {
    if (nq == 0 || k <= 0) return VIX_OK;
    const int keff = (int)(k < n ? k : n);
    const int gcols = n > 0 ? tc::choose_gcols((int)std::min<int64_t>(n, 0x7FFFFF00), keff) : 32;
    const int64_t ngroups64 = n > 0 ? tc::num_groups(n, gcols) : 0;
    // (cosine: exact CUDA-core scan only -- the shortlist's error bound is for the unnormalised scores)
    const bool use_tc = getenv("VIX_DISABLE_TC") == nullptr && xb_norm == nullptr && n >= 4096 && n < (1LL << 31) - 256 &&
                        nq >= 16 && tc::supported(nq, n, d, q, xb) && ngroups64 >= 2 * keff && keff <= 256 && d <= 4096 &&
                        (metric == VIX_METRIC_L2 || metric == VIX_METRIC_IP);
    if (!use_tc) return flat_search_device(q, nq, xb, n, d, metric, k, xb_norm, out_dist, out_ids, raw_scores);
    tc::g_calls[VIX_SHORTLIST_FLAT].fetch_add(1);
    cudaStream_t s = ctx().stream;
    const int ngroups = (int)ngroups64;
    const int nb = (int)n;
    const int cap = keff * 4 + 128;
    Scratch<float> gmin, thr, qn, xn, xmax;
    Scratch<int> cand_cnt, flags, ovf_rows;
    Scratch<int32_t> cand_idx;
    VIX_TRY(gmin.alloc((size_t)nq * ngroups));
    VIX_TRY(thr.alloc((size_t)nq));
    VIX_TRY(qn.alloc((size_t)nq));
    VIX_TRY(xn.alloc((size_t)n));
    VIX_TRY(xmax.alloc(1));
    VIX_TRY(cand_cnt.alloc((size_t)nq));
    VIX_TRY(cand_idx.alloc((size_t)nq * cap));
    VIX_TRY(flags.alloc(2));
    VIX_TRY(ovf_rows.alloc((size_t)nq));
    VIX_CUDA(cudaMemsetAsync(flags.ptr, 0, 8, s));
    VIX_CUDA(cudaMemsetAsync(cand_cnt.ptr, 0, (size_t)nq * 4, s));
    VIX_TRY(row_norms_device(q, nq, d, qn.ptr));
    VIX_TRY(row_norms_device(xb, n, d, xn.ptr));          // Norms.l2NormSquared: also the exact ||x||^2 of the d >= 256 path
    tc::max_sqrt_kernel<<<1, 256, 0, s>>>(xn.ptr, n, xmax.ptr);
    VIX_LAUNCH_CHECK();
    tc::Args a{};
    a.metric = metric; a.bnorm = (metric == VIX_METRIC_L2) ? xn.ptr : nullptr; a.error = flags.ptr;
    a.mode = tc::MODE_MIN; a.gcols = gcols; a.ngroups = ngroups; a.gmin = gmin.ptr;
    VIX_TRY(tc::launch(q, nq, xb, nb, d, a));
    VIX_TRY(tc::launch_threshold(gmin.ptr, nq, ngroups, keff, qn.ptr, xmax.ptr, tc::shortlist_margin(d, metric), thr.ptr));
    a.mode = tc::MODE_EMIT; a.thr = thr.ptr; a.cand_cnt = cand_cnt.ptr; a.cand_idx = cand_idx.ptr; a.cap = cap;
    VIX_TRY(tc::launch(q, nq, xb, nb, d, a));
    {
        const int P = next_pow2(cap);
        const size_t smem = (size_t)P * 8 + (size_t)d * 4;
        VIX_CUDA(cudaFuncSetAttribute(tc::rescore_flat_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        tc::rescore_flat_kernel<<<(unsigned)nq, 256, smem, s>>>(q, xb, d, metric, d >= 256 ? 1 : 0, qn.ptr, xn.ptr, cand_cnt.ptr,
                                                              cand_idx.ptr, cap, P, k, raw_scores ? 1 : 0, out_dist, out_ids,
                                                              ovf_rows.ptr, flags.ptr + 1);
        VIX_LAUNCH_CHECK();
    }
    int hflags[2] = {0, 0};
    VIX_CUDA(cudaMemcpyAsync(hflags, flags.ptr, 8, cudaMemcpyDeviceToHost, s));
    VIX_CUDA(cudaStreamSynchronize(s));
    VIX_REQUIRE(hflags[0] == 0, VIX_ERR_CUDA, "tensor-core pipeline timed out");
    tc::g_exact_rows[VIX_SHORTLIST_FLAT].fetch_add(hflags[1]);
    if (hflags[1] > 0) {
        const int m = hflags[1];
        Scratch<float> sub, sub_d;
        Scratch<int64_t> sub_i;
        VIX_TRY(sub.alloc((size_t)m * d));
        VIX_TRY(sub_d.alloc((size_t)m * k));
        VIX_TRY(sub_i.alloc((size_t)m * k));
        VIX_TRY(gather_rows(q, d, ovf_rows.ptr, m, sub.ptr));
        VIX_TRY(flat_search_device(sub.ptr, m, xb, n, d, metric, k, nullptr, sub_d.ptr, sub_i.ptr, raw_scores));
        tc::scatter_flat_rows_kernel<<<m, 128, 0, s>>>(sub_d.ptr, sub_i.ptr, k, ovf_rows.ptr, m, out_dist, out_ids);
        VIX_LAUNCH_CHECK();
    }
    return VIX_OK;
}

int ivf_assign_device(const float* x, int64_t n, int d, const float* c, int kc, int32_t* assign, float* dist);

// IVF list assignment (a9) through the tensor-core shortlist; results identical to ivf_assign_device.
int ivf_assign_auto_device(const float* x, int64_t n, int d, const float* c, int kc, int32_t* assign, float* dist) {
    if (n == 0) return VIX_OK;
    const bool use_tc = getenv("VIX_DISABLE_TC") == nullptr && tc::supported(n, kc, d, x, c) && kc >= 1024 && n >= 1024 &&
                        d <= 4096 && n < (1LL << 31);
    if (!use_tc) return ivf_assign_device(x, n, d, c, kc, assign, dist);
    tc::g_calls[VIX_SHORTLIST_ASSIGN].fetch_add(1);
    cudaStream_t s = ctx().stream;
    const int gcols = tc::choose_gcols(kc, 1);
    const int ngroups = tc::num_groups(kc, gcols);
    const int cap = 32;
    Scratch<float> gmin, thr, xn, cn, cmax;
    Scratch<int> cand_cnt, flags, ovf_rows;
    Scratch<int32_t> cand_idx;
    VIX_TRY(gmin.alloc((size_t)n * ngroups));
    VIX_TRY(thr.alloc((size_t)n));
    VIX_TRY(xn.alloc((size_t)n));
    VIX_TRY(cn.alloc((size_t)kc));
    VIX_TRY(cmax.alloc(1));
    VIX_TRY(cand_cnt.alloc((size_t)n));
    VIX_TRY(cand_idx.alloc((size_t)n * cap));
    VIX_TRY(flags.alloc(2));
    VIX_TRY(ovf_rows.alloc((size_t)n));
    VIX_CUDA(cudaMemsetAsync(flags.ptr, 0, 8, s));
    VIX_CUDA(cudaMemsetAsync(cand_cnt.ptr, 0, (size_t)n * 4, s));
    VIX_TRY(row_norms_device(x, n, d, xn.ptr));
    VIX_TRY(row_norms_device(c, kc, d, cn.ptr));
    tc::max_sqrt_kernel<<<1, 256, 0, s>>>(cn.ptr, kc, cmax.ptr);
    VIX_LAUNCH_CHECK();
    tc::Args a{};
    a.metric = VIX_METRIC_L2; a.bnorm = cn.ptr; a.error = flags.ptr;
    a.mode = tc::MODE_MIN; a.gcols = gcols; a.ngroups = ngroups; a.gmin = gmin.ptr;
    VIX_TRY(tc::launch(x, n, c, kc, d, a));
    tc::threshold_min_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(gmin.ptr, n, ngroups, xn.ptr, cmax.ptr,
                                                                       tc::shortlist_margin(d, VIX_METRIC_L2), thr.ptr);
    VIX_LAUNCH_CHECK();
    a.mode = tc::MODE_EMIT; a.thr = thr.ptr; a.cand_cnt = cand_cnt.ptr; a.cand_idx = cand_idx.ptr; a.cap = cap;
    VIX_TRY(tc::launch(x, n, c, kc, d, a));
    tc::rescore_assign_kernel<<<(unsigned)((n + 127) / 128), 128, 0, s>>>(x, n, c, d, cand_cnt.ptr, cand_idx.ptr, cap, assign, dist,
                                                                       ovf_rows.ptr, flags.ptr + 1);
    VIX_LAUNCH_CHECK();
    int hflags[2] = {0, 0};
    VIX_CUDA(cudaMemcpyAsync(hflags, flags.ptr, 8, cudaMemcpyDeviceToHost, s));
    VIX_CUDA(cudaStreamSynchronize(s));
    VIX_REQUIRE(hflags[0] == 0, VIX_ERR_CUDA, "tensor-core pipeline timed out");
    tc::g_exact_rows[VIX_SHORTLIST_ASSIGN].fetch_add(hflags[1]);
    if (hflags[1] > 0) {
        const int m = hflags[1];
        Scratch<float> sub, sub_dist;
        Scratch<int32_t> sub_assign;
        VIX_TRY(sub.alloc((size_t)m * d));
        VIX_TRY(sub_assign.alloc((size_t)m));
        VIX_TRY(sub_dist.alloc((size_t)m));
        VIX_TRY(gather_rows(x, d, ovf_rows.ptr, m, sub.ptr));
        VIX_TRY(ivf_assign_device(sub.ptr, m, d, c, kc, sub_assign.ptr, sub_dist.ptr));
        tc::scatter_assign_rows_kernel<<<(unsigned)((m + 255) / 256), 256, 0, s>>>(sub_assign.ptr, sub_dist.ptr, ovf_rows.ptr, m,
                                                                                assign, dist);
        VIX_LAUNCH_CHECK();
    }
    return VIX_OK;
}

}  // namespace vix

using namespace vix;

extern "C" {

/* test hook: raw tensor-core scores of the shortlist pass (not part of the reference surface) */
int vix_debug_tc_scores_f32(const float* queries, int64_t nq, const float* centroids, int kc, int d, int metric,
                            const float* centroid_norms, float* out) {
    VIX_TRY(ensure_device());
    VIX_REQUIRE(queries && centroids && out, VIX_ERR_NULL_PTR, "vix_debug_tc_scores_f32: null pointer");
    VIX_REQUIRE(is_device_ptr(queries) && is_device_ptr(centroids) && is_device_ptr(out) &&
                    (centroid_norms == nullptr || is_device_ptr(centroid_norms)),
                VIX_ERR_INVALID_PARAM, "vix_debug_tc_scores_f32: device pointers only");
    return tc_scores_device(queries, nq, centroids, kc, d, metric, centroid_norms, out);
}

int64_t vix_tc_shortlist_calls(int kind) {
    return kind >= 0 && kind < 3 ? (int64_t)tc::g_calls[kind].load() : -1;
}

int64_t vix_tc_shortlist_exact_rows(int kind) {
    return kind >= 0 && kind < 3 ? (int64_t)tc::g_exact_rows[kind].load() : -1;
}

}  // extern "C"
