// vix_ivfpq_tc.cu -- list-major IVF-PQ scan: decode once per list, score every query that probes it on the tensor cores,
// re-evaluate the finalists in the arithmetic of the look-up-table scan (vix_ivfpq_scan.cu).
//
// Reference composition: pq_lut_residual_l2_f32 -> adc_scan_u8 -> selectTopK -> mergeTopK
// (/root/reference/docs/kernel-specs/DONE_22_adc_scan.md:831-881; PQLUT.swift:266-386; ADCScan.swift:190-283).
//
// Why: the query-major scan spends one shared-memory look-up per (query, code byte) and sits on the look-up pipe
// (DESIGN 4.1: 61 wavefronts per 32 vectors and query).  A batch probes every list several times (C5: 10 k queries x 64
// probes over 65 536 lists = 9.8 queries per list), and with the decomposition the scan already uses,
//
//   ||q - x^||^2 = ||q - c_l||^2 + t_x - 2 <q, r^>          (bias per (query, list), t_x per stored vector)
//
// the only (query, vector) term is a dot product with the DECODED residual r^ = (cb_j[code_j])_j.  So per list:
//
//   decode   32 vectors per warp, one vector per lane = one TMEM lane: 16 G look-ups into ONE query-independent table (the
//            codebooks as fp16 pairs, two replicas, T[code][64 slots] x 2 sub-tables = 128 KB of shared memory) in the
//            order of the index's decode layout of the codes (vix_scan.cuh), so the 32 look-ups of a warp instruction hit 32
//            banks; a two-stage exchange network puts each value into its column and two tcgen05.st .16x128b per group
//            write them as 16 TMEM columns: the A operand never touches shared memory.  Paid once per LIST VISIT, not per
//            (query, list).
//   MMA      tcgen05.mma kind::f16 M128 N16..64 K16, A from TMEM, B = the fp16 rows of the queries probing the list
//            (gathered into a 128B-swizzled shared-memory tile): D[vector][query] = <r^, q>, fp32 accumulators in TMEM.
//   filter   one thread per vector row: D >= tau_q + h_v  <=>  bias + t_x - 2 <q, r^> <= thr_q + eps_q, where thr_q is an
//            EXACT upper bound of the query's k-th best distance (the seed: the k-th smallest exact key of 256 vectors of the
//            query's first probed list, in the look-up-table scan's arithmetic; on a shard the minimum over the ranks) and
//            eps_q bounds |fp16 tensor-core score - the look-up-table scan's fp32 sum|.  Survivors (C5: ~100 per query) are
//            appended to the filter warp's private log.
//   exact    every logged (pair, slot) is re-evaluated with the very arithmetic of the look-up-table scan (same table
//            entries, same summation order) and the k best of a query's keys are selected by (score, id): the output is
//            bit-identical to vix_ivfpq_scan.cu's.  Queries whose seed holds fewer than k vectors (and every query, should a
//            log overflow) are handed to that kernel entirely.
//
// Kernel structure (one persistent CTA per SM, 23 warps):
//   warps 0-11   decoders, three groups of four warps (a warp writes the TMEM lane quarter warp % 4)
//   warps 12-19  filter, two sets of four warps: tcgen05.ld of the accumulators, comparison, log
//   warps 20-21  MMA issuers (one lane each, alternating tiles)
//   warp 22      work: takes the next list from a global counter -- the lists with pairs in work-descending order, so that no
//                long list ends up as the kernel's tail --, publishes the item, gathers the B tile + tau
// PTX wrappers: vix_tcgen05.cuh.  Every mbarrier wait is bounded (mbar_wait_sleep there: a stuck pipeline raises the error flag).
#include <cuda_fp16.h>
#include <stdlib.h>

#include <atomic>
#include <mutex>
#include <vector>
#include <stdio.h>

#include "vix_common.cuh"
#include "vix_scan.cuh"
#include "vix_scan_select.cuh"
#include "vix_tcgen05.cuh"

namespace vix {

int launch_ivfpq_scan_classic(ScanArgs& a);
static std::atomic<long long> g_tc_launches{0};
static thread_local scan_thr_hook_t tls_thr_hook = nullptr;
static thread_local void* tls_thr_ctx = nullptr;
void set_scan_thr_hook(scan_thr_hook_t fn, void* ctx) { tls_thr_hook = fn; tls_thr_ctx = ctx; }

namespace tcs {

constexpr int kNQ = 64;                                  // query columns per item (a list probed by more queries is visited again)
constexpr int kDecGroups = 3;                            // decoder groups of four warps: group g decodes the tiles u % 3 == g
constexpr int kStagesA = 4;                              // operand stages in TMEM: tile u lives in stage u % 4 (whichever group decodes it)
constexpr int kItemRing = 4;
constexpr int kDBufs = 4;                                // accumulator buffers in TMEM (kDBufs x kNQ columns)
constexpr int kDStride = kNQ;
constexpr int kEpiSets = 2;                              // filter warp sets: set e takes the units u % kEpiSets == e
constexpr int kEpiWarps = 4 * kEpiSets;
constexpr int kMmaWarps = 2;                             // MMA issuers: issuer e takes the tiles u % kMmaWarps == e (one lane issues a
                                                         // tcgen05.mma every ~65 clocks, a commit every ~64: at N <= 64 that, not the tensor
                                                         // pipe, paces a tile)
constexpr int kDecWarps = 4 * kDecGroups, kEpiWarp0 = kDecWarps, kMmaWarp = kEpiWarp0 + kEpiWarps, kLoadWarp = kMmaWarp + kMmaWarps;
constexpr int kThreads = 32 * (kLoadWarp + 1);           // 736
static_assert(kEpiWarp0 % 4 == 0 && kDBufs % kEpiSets == 0, "a filter warp reads the TMEM lane quarter warp % 4");
constexpr uint32_t kTabAbs = 4096;                       // ABSOLUTE shared addresses: the table's travels in the LDS immediate
constexpr uint32_t kTabBytes = 2 * 65536;                // two sub-tables (groups 0-1, groups 2-3), each [256 codes][64 slots]
constexpr uint32_t kBBase = kTabAbs + kTabBytes;
constexpr uint32_t kBAtom = kNQ * 128;
constexpr uint32_t kBBuf = 2 * kBAtom;
constexpr uint32_t kEndAbs = kBBase + 2 * kBBuf;
constexpr int kACol0 = kDBufs * kDStride;                 // TMEM: accumulators in columns [0, 256), operand stages behind them
constexpr int kAStageCols = 64;                          // one operand stage: 128 rows x up to 64 columns (= sub-quantisers, fp16 pairs)
constexpr int kTmemCols = 512;
static_assert(kACol0 + kStagesA * kAStageCols <= kTmemCols, "TMEM columns");
constexpr int kSeedChunks = 8;                           // the seed looks at the first 256 vectors of a query's first list

struct Item { int first_chunk, nchunks, len, n, pair_begin, pad0, pad1, pad2; };

struct Small {                                           // the bookkeeping in front of the table
    uint64_t item_full[kItemRing], item_empty[kItemRing];
    uint64_t a_full[kStagesA], a_empty[kStagesA];
    uint64_t b_full[2], b_empty[2];
    uint64_t d_full[kDBufs], d_empty[kDBufs];
    Item items[kItemRing];
    float tau[2][kNQ];
    uint32_t pair[2][kNQ];
    uint32_t tmem_slot;
    uint32_t mma_seq;                                    // tiles whose operands an MMA issuer has claimed, in tile order
};

struct Args {
    const uint8_t* tc_codes; const float* slot_tx;      // the decode layout of the codes (vix_scan.cuh)
    const int64_t* list_off; const int32_t* list_len; int kc;
    const int32_t* pair_off;       // [kc + 1]
    const int32_t* order;          // [*n_order] the lists with pairs, most work first (list_order_*_kernel)
    const int* n_order;
    const uint32_t* pairs;         // [npairs] query * nprobe + probe position, grouped by list
    const float* bias;             // [nq x nprobe]
    const __half* qh;              // [nq x d] scaled fp16 queries
    const float* uq;               // [nq]  -thr / 2 - eps
    const uint32_t* table;         // [2][256][64] half2: the codebooks, scaled (table_kernel)
    const float* scales;           // [0] s_q, [1] s_c
    int nprobe, d, m;
    int* list_counter;
    u64* log; int* log_cnt; int log_cap;   // survivors: one private log per filter warp [grid x 4][log_cap] (no atomics, no
                                           // round trips on the filter's critical path); log_cnt[w] may exceed log_cap
    int smem_bytes;
    int* status;                   // layout refusal (loud)
    int* error; int* error_host;
    unsigned long long* diag;      // VIX_TCS_DIAG builds: waiting cycles per role and barrier kind
};

#ifdef VIX_TCS_DIAG
#define VIX_DG(i) dg[i]
#else
#define VIX_DG(i) dg_none
#endif
template <int IMM>
__device__ __forceinline__ uint32_t lds_tab(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.b32 %0, [%1+%2];" : "=r"(v) : "r"(addr), "n"(IMM));
    return v;
}
// one group of 16 sub-quantisers of the four slots r + 8 v (v = 0..3) of thread t = 4 r + c: 16 look-ups in the order of the
// decode layout (vix_scan.cuh: byte s of word v holds sub-quantiser 4 (s ^ q) + c, q = r & 3).  For one (v, s) the 16
// threads of a half-warp (q, c all different) ask for 16 different table slots and the two half-warps (h = r >> 2) read two
// replicas: the 32 look-ups hit 32 banks.  (One replica per half-warp is why some exchange remains: without one, the lanes
// that share a TMEM column in a store would all want the same slot.)  A two-stage exchange network (register s <-> s ^ 2^b where
// bit b of q is set) puts each slot's four values into column order (register k = sub-quantiser 4 k + c), and two
// tcgen05.st .16x128b write the slots r, r + 8 and r + 16, r + 24: TMEM lane = slot of the chunk, column = sub-quantiser.
template <int IMM>
__device__ __forceinline__ void decode16(const uint4& w, uint32_t pre0, uint32_t pre1, uint32_t taddr, bool q0, bool q1) {
    const uint32_t x[4] = {w.x, w.y, w.z, w.w};
    uint32_t r[4][4];
#pragma unroll
    for (int v = 0; v < 4; ++v) {
        r[v][0] = lds_tab<IMM>(__byte_perm(x[v], pre0, 0x7604));
        r[v][1] = lds_tab<IMM>(__byte_perm(x[v], pre0, 0x7615));
        r[v][2] = lds_tab<IMM>(__byte_perm(x[v], pre1, 0x7624));
        r[v][3] = lds_tab<IMM>(__byte_perm(x[v], pre1, 0x7635));
    }
#pragma unroll
    for (int v = 0; v < 4; ++v) {
#pragma unroll
        for (int b = 0; b < 2; ++b) {
            const bool bit = b == 0 ? q0 : q1;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                if ((i >> b) & 1) continue;
                const uint32_t lo = r[v][i], hi = r[v][i | (1 << b)];
                r[v][i] = bit ? hi : lo;
                r[v][i | (1 << b)] = bit ? lo : hi;
            }
        }
    }
    const uint32_t s01[8] = {r[0][0], r[1][0], r[0][1], r[1][1], r[0][2], r[1][2], r[0][3], r[1][3]};
    const uint32_t s23[8] = {r[2][0], r[3][0], r[2][1], r[3][1], r[2][2], r[3][2], r[2][3], r[3][3]};
    tmem_st16x128_x4(taddr, s01);
    tmem_st16x128_x4(taddr + (16u << 16), s23);
}

template <int G>
__global__ void __launch_bounds__(kThreads, 1)
tc_scan_kernel(Args a) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    const uint32_t dyn_abs = smem_u32(smem_raw);
    if (dyn_abs + (uint32_t)sizeof(Small) > kTabAbs || kEndAbs > dyn_abs + (uint32_t)a.smem_bytes) {
        if (threadIdx.x == 0 && blockIdx.x == 0 && a.status) *a.status = 1;
        return;
    }
    Small& S = *reinterpret_cast<Small*>(smem_raw);
    unsigned char* const abs0 = smem_raw - dyn_abs;          // generic pointer of absolute shared address 0
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned long long dg[4] = {0, 0, 0, 0}, dg_none = 0;      // VIX_TCS_DIAG: cycles this thread waited, per barrier kind
    (void)dg; (void)dg_none;
    const long long dg_t0 = clock64();

    if (threadIdx.x == 0) {
        for (int i = 0; i < kItemRing; ++i) { mbar_init(&S.item_full[i], 1); mbar_init(&S.item_empty[i], kDecWarps + kEpiWarps + kMmaWarps); }
        for (int i = 0; i < kStagesA; ++i) { mbar_init(&S.a_full[i], 128); mbar_init(&S.a_empty[i], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&S.b_full[i], 32); mbar_init(&S.b_empty[i], kEpiWarps); }
        for (int i = 0; i < kDBufs; ++i) { mbar_init(&S.d_full[i], 1); mbar_init(&S.d_empty[i], 4); }
        mbar_init_fence();
    }
    if (warp == kMmaWarp) tmem_alloc(&S.tmem_slot, kTmemCols);
    if (threadIdx.x == 32) S.mma_seq = 0;
    {   // the decode table: 2 x 64 KB, once per CTA
        const uint4* src = reinterpret_cast<const uint4*>(a.table);
        uint4* dst = reinterpret_cast<uint4*>(abs0 + kTabAbs);
        for (int i = threadIdx.x; i < (int)(kTabBytes / 16); i += kThreads) dst[i] = __ldg(src + i);
    }
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem_base = S.tmem_slot;
    const float sc = __ldg(a.scales) * __ldg(a.scales + 1);
    constexpr int m = 16 * G;
    constexpr int kKSteps = m / 8;                           // K = 16 halves per MMA, d = 2 m

    if (warp < kDecWarps) {
        // ------------------------------------------------------------------------------------------ decoders
        const int grp = warp >> 2, wi = warp & 3;
        const uint32_t h = (uint32_t)lane >> 4;
        // this warp's rows of the operand stage: TMEM lanes [32 wi, 32 wi + 32) (the lanes a warp may touch: warp % 4 == wi),
        // lane = slot of the chunk; columns kACol0 + 64 stage + sub-quantiser
        const uint32_t a_taddr0 = tmem_base + ((32u * (uint32_t)wi) << 16) + (uint32_t)kACol0;
        // thread 4 r + c looks up byte s of each code word in table slot 16 h + 4 (s ^ q) + c, q = r & 3; pre holds the four
        // byte offsets of those slots
        const uint32_t q = ((uint32_t)lane >> 2) & 3u, c4 = 4u * ((uint32_t)lane & 3u);
        const bool q0 = q & 1u, q1 = q & 2u;
        uint32_t pre[2];
#pragma unroll
        for (uint32_t s = 0; s < 4; s += 2) {
            const uint32_t b0 = 64u * h + 16u * (s ^ q) + c4, b1 = 64u * h + 16u * ((s + 1) ^ q) + c4;
            pre[s >> 1] = b0 | (b1 << 8);
            asm volatile("" : "+r"(pre[s >> 1]));
        }
        // The warp walks its units (tile t of item it with (units before the item + t) % 3 == grp) with the NEXT unit's codes
        // already in flight while it decodes the current one (two register buffers, loop unrolled by two).  Moving on may
        // cross into the next item: the descriptor of an item is copied to registers, so its ring slot is released at once.
        int it = 0, slot = 0, fc = 0, nch = 0, nt = 0, t = 0;
        long long u0 = 0;
        bool opened = false;
        // (it, t) -> this group's next unit at or behind it.  1: found; 0: the sentinel (or a time-out); 2 (only when not
        // `blocking`): the next item is not published yet.  Looking ahead must not block: the loader publishes item i + 2 only
        // after item i is finished, which may need the very unit this warp still holds.
        auto seek = [&](bool blocking) -> int {
            for (;;) {
                if (opened) {
                    if (t < nt) return 1;
                    u0 += nt;
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&S.item_empty[slot]);
                    ++it;
                    opened = false;
                }
                slot = it % kItemRing;
                const uint32_t par = (uint32_t)(it / kItemRing) & 1u;
                if (blocking) { if (!mbar_wait_sleep(&S.item_full[slot], par, a.error, a.error_host, VIX_DG(0))) return 0; }
                else if (!__all_sync(0xFFFFFFFFu, mbar_try_wait(&S.item_full[slot], par))) return 2;
                fc = S.items[slot].first_chunk; nch = S.items[slot].nchunks;
                if (nch < 0) return 0;
                nt = (nch + 3) >> 2;
                t = (int)(((long long)grp - u0 % kDecGroups + kDecGroups) % kDecGroups);
                opened = true;
            }
        };
        auto load = [&](uint4 (&w)[G], int ch) {
            if (ch < nch) {
                const uint4* src = reinterpret_cast<const uint4*>(a.tc_codes + (size_t)(fc + ch) * (512u * G)) + lane;
#pragma unroll
                for (int s = 0; s < G; ++s) w[s] = __ldg(src + 32 * s);
            }
        };
        auto process = [&](const uint4 (&w)[G], bool live, long long unit) -> bool {
            const int st = (int)(unit % kStagesA);
            const long long use = unit / kStagesA;
            const uint32_t a_taddr = a_taddr0 + (uint32_t)(st * kAStageCols);
            if (use > 0 && !mbar_wait_sleep(&S.a_empty[st], (uint32_t)(use - 1) & 1u, a.error, a.error_host, VIX_DG(1))) return false;
            if (live) {
                // group g: sub-table g / 2, slots 32 (g % 2) + 16 h + ..: the immediates are compile-time
                decode16<(int)kTabAbs>(w[0], pre[0], pre[1], a_taddr, q0, q1);
                if (G > 1) decode16<(int)kTabAbs + 128>(w[G > 1 ? 1 : 0], pre[0], pre[1], a_taddr + 16, q0, q1);
                if (G > 2) decode16<(int)kTabAbs + 65536>(w[G > 2 ? 2 : 0], pre[0], pre[1], a_taddr + 32, q0, q1);
                if (G > 3) decode16<(int)kTabAbs + 65536 + 128>(w[G > 3 ? 3 : 0], pre[0], pre[1], a_taddr + 48, q0, q1);
                tmem_wait_st();
            }
            fence_before_sync();
            mbar_arrive(&S.a_full[st]);
            return true;
        };
        uint4 wA[G], wB[G];
        if (seek(true) == 1) {
            load(wA, 4 * t + wi);
            for (;;) {
                bool live = 4 * t + wi < nch;
                long long use = u0 + t;
                t += kDecGroups;
                int r = seek(false);
                if (r == 1) load(wB, 4 * t + wi);
                if (!process(wA, live, use) || r == 0) break;
                if (r == 2) { if (seek(true) != 1) break; load(wB, 4 * t + wi); }
                live = 4 * t + wi < nch;
                use = u0 + t;
                t += kDecGroups;
                r = seek(false);
                if (r == 1) load(wA, 4 * t + wi);
                if (!process(wB, live, use) || r == 0) break;
                if (r == 2) { if (seek(true) != 1) break; load(wA, 4 * t + wi); }
            }
        }
    } else if (warp >= kMmaWarp && warp < kMmaWarp + kMmaWarps) {
        // ------------------------------------------------------------------------------------------ MMA issuers
        // Both issuers walk every item; issuer e issues the tiles u % kMmaWarps == e.  The waits on the operand stages are taken
        // in tile order (S.mma_seq): two threads waiting on DIFFERENT phases of one mbarrier would let the later one through
        // on the earlier phase's parity.
        const int me = warp - kMmaWarp;
        if (lane == 0) {
#ifdef VIX_TCS_DIAG
            unsigned long long mma_issue = 0, mma_commit_c = 0, mma_units = 0;
#endif
            int it = 0;
            long long u = 0;
            for (;;) {
                const int slot = it % kItemRing;
                if (!mbar_wait_sleep(&S.item_full[slot], (uint32_t)(it / kItemRing) & 1u, a.error, a.error_host, VIX_DG(0))) break;
                const int nch = S.items[slot].nchunks, n = S.items[slot].n;
                if (nch < 0) break;
                const int nt = (nch + 3) >> 2;
                const uint32_t idesc = idesc_f16(128, (n + 15) & ~15);
                const int buf = it & 1;
                if (!mbar_wait_sleep(&S.b_full[buf], (uint32_t)(it >> 1) & 1u, a.error, a.error_host, VIX_DG(1))) break;
                bool ok = true;
                for (int t = 0; t < nt; ++t, ++u) {
                    if ((int)(u % kMmaWarps) != me) continue;
                    const int st = (int)(u % kStagesA), db = (int)(u % kDBufs);
                    {   // my turn: every earlier tile's issuer holds its operands
                        volatile uint32_t* seq = &S.mma_seq;
                        const long long t0 = clock64();
                        for (uint32_t spins = 1; *seq != (uint32_t)u; ++spins) {
                            __nanosleep(40);
                            if ((spins & 1023u) == 0 && (clock64() - t0 > 4000000000LL || *reinterpret_cast<volatile int*>(a.error) != 0)) { ok = false; break; }
                        }
                        if (!ok) { atomicExch(a.error, 1); break; }
                    }
                    if (!mbar_wait_sleep(&S.a_full[st], (uint32_t)(u / kStagesA) & 1u, a.error, a.error_host, VIX_DG(2))) { ok = false; break; }
                    if (u >= kDBufs && !mbar_wait_sleep(&S.d_empty[db], (uint32_t)(u / kDBufs - 1) & 1u, a.error, a.error_host, VIX_DG(3))) { ok = false; break; }
                    *reinterpret_cast<volatile uint32_t*>(&S.mma_seq) = (uint32_t)(u + 1);
                    fence_after_sync();
#ifdef VIX_TCS_DIAG
                    const long long m0 = clock64();
#endif
                    const uint32_t dcol = tmem_base + (uint32_t)(db * kDStride);
#pragma unroll
                    for (int ks = 0; ks < kKSteps; ++ks) {
                        const uint64_t bd = make_desc_sw128(kBBase + (uint32_t)buf * kBBuf + (uint32_t)(ks >> 2) * kBAtom) + (uint64_t)(2 * (ks & 3));
                        // A from TMEM: 8 columns (16 halves) of the stage per K-step
                        mma_f16_ts(dcol, tmem_base + (uint32_t)(kACol0 + st * kAStageCols + 8 * ks), bd, idesc, ks > 0 ? 1u : 0u);
                    }
#ifdef VIX_TCS_DIAG
                    const long long m1 = clock64();
#endif
                    mma_commit(&S.a_empty[st]);
                    mma_commit(&S.d_full[db]);
#ifdef VIX_TCS_DIAG
                    const long long m2 = clock64();
                    mma_issue += (unsigned long long)(m1 - m0); mma_commit_c += (unsigned long long)(m2 - m1); mma_units += 1;
#endif
                }
                if (!ok) break;
                mbar_arrive(&S.item_empty[slot]);
                ++it;
            }
#ifdef VIX_TCS_DIAG
            if (a.diag) { atomicAdd(a.diag + 20, mma_issue); atomicAdd(a.diag + 21, mma_commit_c); atomicAdd(a.diag + 22, mma_units); }
#endif
        }
    } else if (warp >= kEpiWarp0 && warp < kEpiWarp0 + kEpiWarps) {
        // ------------------------------------------------------------------------------------------ filter
        const int wq = (warp - kEpiWarp0) & 3;               // = warp % 4: the TMEM lane quarter this warp may read
        const int eset = (warp - kEpiWarp0) >> 2;            // this warp's set filters the units u % kEpiSets == eset
        const uint32_t sl = (uint32_t)lane;                  // TMEM lane = tile row = slot of the chunk
        u64* const mylog = a.log + (size_t)(blockIdx.x * kEpiWarps + (warp - kEpiWarp0)) * (size_t)a.log_cap;
        int nlog = 0;
        int it = 0;
        long long u = 0;
        for (;;) {
            const int slot = it % kItemRing;
            if (!mbar_wait_sleep(&S.item_full[slot], (uint32_t)(it / kItemRing) & 1u, a.error, a.error_host, VIX_DG(0))) break;
            const int fc = S.items[slot].first_chunk, nch = S.items[slot].nchunks, len = S.items[slot].len, n = S.items[slot].n;
            if (nch < 0) break;
            const int nt = (nch + 3) >> 2;
            const int buf = it & 1;
            // t_x of this thread's row of tile t; the NEXT tile's is in flight while this one is filtered
            auto load_tx = [&](int t) {
                const int ch = 4 * t + wq;
                return (ch < nch && ch * 32 + (int)sl < len) ? __ldg(a.slot_tx + (((uint32_t)(fc + ch) << 5) + sl)) : 0.0f;
            };
            // this set's tiles of the item: t0, t0 + kEpiSets, ... ((u + t) % kEpiSets == eset)
            const int t0 = (int)(((long long)eset - u % kEpiSets + kEpiSets) % kEpiSets);
            float tx_next = load_tx(t0);
            if (!mbar_wait_sleep(&S.b_full[buf], (uint32_t)(it >> 1) & 1u, a.error, a.error_host, VIX_DG(1))) break;
            const float* tau = S.tau[buf];
            bool ok = true;
            for (int t = t0; t < nt; t += kEpiSets) {
                const long long uu = u + t;
                const int db = (int)(uu % kDBufs);
                const int ch = 4 * t + wq;
                const int within = ch * 32 + (int)sl;
                const bool valid = ch < nch && within < len;
                const uint32_t g = ((uint32_t)(fc + ch) << 5) + sl;
                const float tx = tx_next;
                tx_next = t + kEpiSets < nt ? load_tx(t + kEpiSets) : 0.0f;
                if (!mbar_wait_sleep(&S.d_full[db], (uint32_t)(uu / kDBufs) & 1u, a.error, a.error_host, VIX_DG(2))) { ok = false; break; }
                fence_after_sync();
                const float hv = sc * (0.5f * tx - 1.5e-6f * fabsf(tx));
                for (int cb = 0; cb < n; cb += 16) {
                    float dv[16];
                    tmem_ld16(tmem_base + ((uint32_t)(32 * wq) << 16) + (uint32_t)(db * kDStride + cb), dv);
                    bool any = false;
#pragma unroll
                    for (int c = 0; c < 16; ++c) any |= dv[c] >= tau[cb + c] + hv;       // tau = NaN behind the last query
                    if (__any_sync(0xFFFFFFFFu, any && valid)) {
                        // rare: append (pair, slot) records to this warp's log -- positions from a ballot, plain stores
#pragma unroll
                        for (int c = 0; c < 16; ++c) {
                            const bool hit = valid && dv[c] >= tau[cb + c] + hv;
                            const unsigned ball = __ballot_sync(0xFFFFFFFFu, hit);
                            if (ball) {
                                const int pos = nlog + __popc(ball & ((1u << lane) - 1u));
                                if (hit && pos < a.log_cap) mylog[pos] = ((u64)S.pair[buf][cb + c] << 32) | (u64)g;
                                nlog += __popc(ball);
                            }
                        }
                    }
                }
                fence_before_sync();
                __syncwarp();
                if (lane == 0) mbar_arrive(&S.d_empty[db]);
            }
            if (!ok) break;
            u += nt;
            __syncwarp();
            if (lane == 0) { mbar_arrive(&S.b_empty[buf]); mbar_arrive(&S.item_empty[slot]); }
            ++it;
        }
        if (lane == 0) a.log_cnt[blockIdx.x * kEpiWarps + (warp - kEpiWarp0)] = nlog;
    } else if (warp == kLoadWarp) {
        // ------------------------------------------------------------------------------------------ work + B tiles
        constexpr int CH = m / 4;                             // 16-byte pieces of a query row (d = 2 m halves)
        int it = 0;
        bool ok = true;
        const int n_order = *a.n_order;
        auto publish = [&](int fc, int nch, int len, int n, int pb) {
            const int slot = it % kItemRing;
            if (it >= kItemRing && !mbar_wait_sleep(&S.item_empty[slot], (uint32_t)(it / kItemRing - 1) & 1u, a.error, a.error_host, VIX_DG(0))) return false;
            if (lane == 0) {
                Item& I = S.items[slot];
                I.first_chunk = fc; I.nchunks = nch; I.len = len; I.n = n; I.pair_begin = pb;
                __threadfence_block();
                mbar_arrive(&S.item_full[slot]);
            }
            __syncwarp();
            return true;
        };
        while (ok) {
            int l = -1;
            if (lane == 0) { const int i = atomicAdd(a.list_counter, 1); if (i < n_order) l = __ldg(a.order + i); }
            l = __shfl_sync(0xFFFFFFFFu, l, 0);
            if (l < 0) break;
            const int pb = __ldg(a.pair_off + l), pe = __ldg(a.pair_off + l + 1);
            if (pe == pb) continue;
            const int len = __ldg(a.list_len + l);
            const int fc = (int)(__ldg(a.list_off + l) >> 5), nch = (len + 31) >> 5;
            for (int g0 = pb; g0 < pe && ok; g0 += kNQ) {
                const int n = min(kNQ, pe - g0);
                if (!publish(fc, nch, len, n, g0)) { ok = false; break; }
                const int buf = it & 1;
                if (it >= 2 && !mbar_wait_sleep(&S.b_empty[buf], (uint32_t)((it >> 1) - 1) & 1u, a.error, a.error_host, VIX_DG(1))) { ok = false; break; }
                const uint32_t bbase = kBBase + (uint32_t)buf * kBBuf;
                for (int idx = lane; idx < n * CH; idx += 32) {
                    const int c = idx / CH, chn = idx - c * CH;
                    const uint32_t q = __ldg(a.pairs + g0 + c) / (uint32_t)a.nprobe;
                    const uint32_t dst = bbase + (uint32_t)(chn >> 3) * kBAtom + (uint32_t)(c >> 3) * 1024u + (uint32_t)(c & 7) * 128u +
                                         (uint32_t)(((chn & 7) ^ (c & 7)) << 4);
                    const char* src = reinterpret_cast<const char*>(a.qh) + (size_t)q * (size_t)(4 * m) + (size_t)chn * 16;
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src));
                }
                asm volatile("cp.async.commit_group;");
                for (int c = lane; c < kNQ; c += 32) {
                    float tv = __int_as_float(0x7fc00000);                  // NaN behind the last query: no column value passes
                    uint32_t pr = 0;
                    if (c < n) {
                        pr = __ldg(a.pairs + g0 + c);
                        const float b = __ldg(a.bias + pr);
                        tv = sc * ((0.5f * b - 1.5e-6f * fabsf(b)) + __ldg(a.uq + pr / (uint32_t)a.nprobe));
                    }
                    S.tau[buf][c] = tv;
                    S.pair[buf][c] = pr;
                }
                asm volatile("cp.async.wait_group 0;" ::: "memory");
                fence_async_proxy();
                mbar_arrive(&S.b_full[buf]);
                ++it;
            }
        }
        if (ok) publish(0, -1, 0, 0, 0);
    }
#ifdef VIX_TCS_DIAG
    if (a.diag && lane == 0) {
        // roles: 0 decoders (12 warps), 1 filter (4 warps), 2 MMA, 3 loader; [role][4 waits] + [role] total cycles at 16 + role
        const int role = warp < kDecWarps ? 0 : warp < kMmaWarp ? 1 : warp < kLoadWarp ? 2 : 3;
        for (int i = 0; i < 4; ++i) atomicAdd(a.diag + role * 4 + i, dg[i]);
        atomicAdd(a.diag + 16 + role, (unsigned long long)(clock64() - dg_t0));
    }
#endif
    fence_before_sync();
    __syncthreads();
    if (warp == kMmaWarp) tmem_dealloc(tmem_base, kTmemCols);
}

// ---------------------------------------------------------------------------------------------- the small kernels
// decode table + its scale + the residual norm bound: one CTA.  table[sub-table][code][slot] = half2(s_c cb_j[code]), every
// entry in two replicas (one per half-warp).  meta: [1] = s_c, [2] = R_max =
// sqrt(sum_j max_c ||cb_j[c]||^2) >= ||r^|| of every stored vector.
__global__ void __launch_bounds__(1024)
table_kernel(const float* __restrict__ codebooks, int m, uint32_t* __restrict__ table, float* __restrict__ meta) {
    __shared__ float s_max[32], s_r2[64];
    __shared__ float s_scale;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    float mx = 0.0f;
    for (int i = tid; i < m * 256 * 2; i += 1024) mx = fmaxf(mx, fabsf(codebooks[i]));
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xFFFFFFFFu, mx, o));
    if (lane == 0) s_max[warp] = mx;
    // max_c ||cb_j[c]||^2: one warp per sub-quantiser
    for (int j = warp; j < m; j += 32) {
        float r2 = 0.0f;
        for (int c = lane; c < 256; c += 32) {
            const float2 v = *reinterpret_cast<const float2*>(codebooks + ((size_t)j * 256 + c) * 2);
            r2 = fmaxf(r2, v.x * v.x + v.y * v.y);
        }
        for (int o = 16; o > 0; o >>= 1) r2 = fmaxf(r2, __shfl_xor_sync(0xFFFFFFFFu, r2, o));
        if (lane == 0) s_r2[j] = r2;
    }
    __syncthreads();
    if (tid == 0) {
        float g = 0.0f;
        for (int w = 0; w < 32; ++w) g = fmaxf(g, s_max[w]);
        int e = 0;
        float s = 1.0f;
        if (g > 0.0f && g < __int_as_float(0x7f800000)) { frexpf(g, &e); s = ldexpf(1.0f, 10 - e); }
        float r2 = 0.0f;
        for (int j = 0; j < m; ++j) r2 += s_r2[j];
        s_scale = s;
        meta[1] = s;
        meta[2] = sqrtf(r2) * 1.0001f;
    }
    __syncthreads();
    const float s = s_scale;
    // [sub-table t = group / 2][code][slot = 32 (group % 2) + 16 replica + sub-quantiser % 16]: both replicas hold the same entry
    for (int i = tid; i < 2 * 256 * 64; i += 1024) {
        const int t = i >> 14, c = (i >> 6) & 255, slot = i & 63;
        const int j = 16 * (2 * t + (slot >> 5)) + (slot & 15);
        uint32_t v = 0;
        if (j < m) {
            const float2 f = *reinterpret_cast<const float2*>(codebooks + ((size_t)j * 256 + c) * 2);
            const __half2 hh = __floats2half2_rn(f.x * s, f.y * s);
            v = *reinterpret_cast<const uint32_t*>(&hh);
        }
        table[i] = v;
    }
}

// The seed: one CTA per query, one WARP per 32-vector chunk: the first kSeedChunks x 32 vectors of the query's first probed
// list that holds vectors here get their exact keys -- the same table entries (lut_entry2 from the code-major codebooks,
// L1-resident) in the same summation order as the look-up-table scan, but without building a 128 KB table -- and the CTA
// sorts them.  The k-th of ANY k stored vectors is an upper bound of the query's k-th best distance: that is the threshold
// of the filter (thr[q]; +inf when the sample holds fewer than k vectors).  (The whole list would give a tighter threshold
// and fewer finalists, but costs more than the finalists it saves: C5 1.77 ms against 0.3 ms.  One warp walking the eight
// chunks in sequence took 84 us for the 1250 queries a rank of eight seeds -- latency, not work.)  On the way the CTA
// leaves ||q|| and the batch maximum of |q_e| (the fp16 scale) for query_prep_kernel.
// A shard (only_first): only the rank that owns the query's FIRST probed list seeds it (the bounds are reduced over the
// ranks; a seed from a farther list would be looser than the owner's and cost the same).
template <int G>
__global__ void __launch_bounds__(32 * kSeedChunks)
seed_scan_kernel(const float* __restrict__ queries, int64_t nq, const int32_t* __restrict__ probes, int nprobe, int kc,
                 int only_first, const float* __restrict__ coarse, const float* __restrict__ codebooks_t,
                 const int64_t* __restrict__ list_off, const int32_t* __restrict__ list_len, const uint8_t* __restrict__ slot_codes,
                 const float* __restrict__ slot_tx, int k, float* __restrict__ qnorm, unsigned int* __restrict__ maxabs,
                 float* __restrict__ thr) {
    constexpr int m = 16 * G, d = 2 * m;
    __shared__ u64 s_keys[32 * kSeedChunks];
    __shared__ float2 s_q[m];
    __shared__ int s_list;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t q = blockIdx.x;
    const float* qv = queries + q * d;
    if (warp == 0) {
        // ||q|| and max |q_e|
        float s = 0.0f, mx = 0.0f;
        for (int e = lane; e < d; e += 32) { const float v = __ldg(qv + e); s = fmaf(v, v, s); mx = fmaxf(mx, fabsf(v)); }
        for (int o = 16; o > 0; o >>= 1) { s += __shfl_xor_sync(0xFFFFFFFFu, s, o); mx = fmaxf(mx, __shfl_xor_sync(0xFFFFFFFFu, mx, o)); }
        if (lane == 0) {
            qnorm[q] = sqrtf(s);
            if (mx == mx && mx < __int_as_float(0x7f800000)) atomicMax(maxabs, __float_as_uint(mx));
        }
        // the first probe position whose list holds vectors here
        int l = -1, p0 = -1;
        for (int base = 0; base < nprobe; base += 32) {
            const int p = base + lane;
            const int lp = p < nprobe ? __ldg(probes + q * nprobe + p) : -1;
            const bool here = (unsigned)lp < (unsigned)kc && __ldg(list_len + lp) > 0;
            const unsigned ball = __ballot_sync(0xFFFFFFFFu, here);
            if (ball) { const int src = __ffs(ball) - 1; l = __shfl_sync(0xFFFFFFFFu, lp, src); p0 = base + src; break; }
        }
        if (only_first && p0 != 0) l = -1;
        if (lane == 0) s_list = l;
    }
    for (int j = threadIdx.x; j < m; j += blockDim.x) s_q[j] = make_float2(__ldg(qv + 2 * j) * -2.0f, __ldg(qv + 2 * j + 1) * -2.0f);
    __syncthreads();
    const int l = s_list;
    if (l < 0) {
        if (threadIdx.x == 0) thr[q] = __int_as_float(0x7f800000);
        return;
    }
    // bias ||q - c_l||^2 in the order of probe_bias_kernel / build_probe_table (lane-strided partial sums, xor tree)
    float bias = 0.0f;
    {
        const float* c = coarse + (int64_t)l * d;
        for (int e = lane; e < d; e += 32) { const float df = __ldg(qv + e) - __ldg(c + e); bias = fmaf(df, df, bias); }
        for (int o = 16; o > 0; o >>= 1) bias += __shfl_xor_sync(0xFFFFFFFFu, bias, o);
    }
    const int len = __ldg(list_len + l);
    const uint32_t first = (uint32_t)(__ldg(list_off + l) >> 5);
    const float2* cbt = reinterpret_cast<const float2*>(codebooks_t);
    const uint32_t rot = (uint32_t)lane & 15u;
    u64 key = kEmptyKey;
    const int ch = warp;                                             // a SAMPLE of the list: any k vectors bound the k-th best
    if (ch * 32 + lane < len) {
        const uint32_t g = ((first + (uint32_t)ch) << 5) + (uint32_t)lane;
        const uint4* src = reinterpret_cast<const uint4*>(slot_codes + (size_t)(first + ch) * (512u * G)) + lane;
        float s[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
        for (int grp = 0; grp < G; ++grp) {
            const uint4 w = __ldg(src + 32 * grp);
            const uint32_t x[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
            for (int i4 = 0; i4 < 4; ++i4) {
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    const uint32_t b = 4 * i4 + t;
                    const uint32_t code = (x[i4] >> (8 * t)) & 255u;
                    const uint32_t j = 16u * grp + (b ^ rot);
                    const float2 v = __ldg(cbt + code * m + j);
                    const float2 qq = s_q[j];
                    s[t] = fadd(s[t], lut_entry2(qq.x, qq.y, v));
                }
            }
        }
        const float sum = fadd(fadd(bias, __ldg(slot_tx + g)), fadd(fadd(s[0], s[1]), fadd(s[2], s[3])));
        key = make_key(sum, 0u, 0) | 0xFFFFFFFFull;                  // only the score matters: any id, the same for all
    }
    s_keys[threadIdx.x] = key;
    __syncthreads();
    bitonic_sort_keys<false>(s_keys, 32 * kSeedChunks, threadIdx.x, blockDim.x);
    if (threadIdx.x == 0) {
        const u64 kth = s_keys[k - 1];
        const float t = key_score(kth, 0);
        thr[q] = (kth != kEmptyKey && t == t) ? t : __int_as_float(0x7f800000);
    }
}

// per query (one warp), after the seed scan: the fp16 row, u_q = -thr / 2 - eps_q, and whether the query can take this path
// (a finite k-th seed distance and a finite error bound)
__global__ void __launch_bounds__(256)
query_prep_kernel(const float* __restrict__ queries, int64_t nq, int d, const float* __restrict__ qnorm,
                  const unsigned int* __restrict__ maxabs, float* __restrict__ meta, const float* __restrict__ tmeta,
                  const float* __restrict__ thr_in, __half* __restrict__ qh, float* __restrict__ uq, int* __restrict__ flag) {
    const int lane = threadIdx.x & 31;
    const int64_t q = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (q >= nq) return;
    const float g = __uint_as_float(*maxabs);
    float sq = 1.0f;
    if (g > 0.0f) { int e = 0; frexpf(g, &e); sq = ldexpf(1.0f, 10 - e); }
    const float s_c = tmeta[1], rmax = tmeta[2];                // of the decode table (per codebooks; meta is this launch's)
    // The filter scales its bounds by s_q s_c (tc_scan_kernel).  Queries and codebooks both below 2^-50 make that product
    // overflow (2^64 x 2^64 at 2^-54) although every distance is a normal fp32 number: s_q is lowered to keep it at most
    // 2^126.  A smaller s_q only leaves more of the fp16 row subnormal, which the 6e-8 sqrt(d) rmax / s_q term of eps
    // bounds; a product still not normal (s_c itself not finite, or both data above 2^73) hands the queries back below.
    // tau and h_v themselves (sc times a distance) may still overflow when a distance exceeds 2^128 / sc; the sign makes
    // that harmless: +inf rejects vectors that are that far anyway, -inf passes everything (at worst the log overflows
    // and the queries are handed back).
    if (sq * s_c > 0x1p126f) sq = 0x1p126f / s_c;
    if (q == 0 && lane == 0) { meta[0] = sq; meta[1] = s_c; }
    for (int e = lane; e < d; e += 32) qh[q * d + e] = __float2half_rn(__ldg(queries + q * d + e) * sq);
    if (lane == 0) {
        const float qn = qnorm[q];
        const float thr = thr_in[q];
        // |fp16 tensor-core <q, r^> - exact| <= eta ||q|| ||r^|| + the subnormal floor of the two conversions, and the
        // look-up-table scan's own fp32 sum is within 2e-6 of (|bias| + |t_x| + 2 ||q|| ||r^||) of the exact value
        // (the |bias| and |t_x| shares ride in tau and h_v)
        const float eta = 1.05f * 0.0009765625f + (float)d * 4.8e-7f;
        const float eps = eta * qn * rmax + 6e-8f * sqrtf((float)d) * (rmax / sq + qn / s_c) + 2e-6f * qn * rmax;
        const float u = -0.5f * thr - eps - 2e-6f * fabsf(thr);
        const float sc = sq * s_c;
        const bool fine = thr == thr && fabsf(thr) < __int_as_float(0x7f800000) && u == u && fabsf(u) < __int_as_float(0x7f800000) &&
                          qn * sq < 60000.0f && sc >= 0x1p-126f && sc <= 0x1p126f;
        uq[q] = fine ? u : 0.0f;
        flag[q] = fine ? 0 : 1;
    }
}

// (query, probe position) pairs of this path, counted per list; also the entries every valid pair visits (statistics)
__global__ void __launch_bounds__(256)
pair_count_kernel(const int32_t* __restrict__ probes, int64_t npairs, int nprobe, const int32_t* __restrict__ list_len, int kc,
                  const int* __restrict__ flag, int32_t* __restrict__ hist,
                  unsigned long long* __restrict__ scanned) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long vis = 0;
    if (i < npairs) {
        const int l = __ldg(probes + i);
        if ((unsigned)l < (unsigned)kc) {
            const int len = __ldg(list_len + l);
            vis = (unsigned long long)len;
            if (len > 0 && !flag[i / nprobe]) atomicAdd(hist + l, 1);
        }
    }
    if (scanned) {
        for (int o = 16; o > 0; o >>= 1) vis += __shfl_xor_sync(0xFFFFFFFFu, vis, o);
        if ((threadIdx.x & 31) == 0 && vis) atomicAdd(scanned, vis);
    }
}
__global__ void __launch_bounds__(256)
pair_scatter_kernel(const int32_t* __restrict__ probes, int64_t npairs, int nprobe, const int32_t* __restrict__ list_len, int kc,
                    const int* __restrict__ flag, int32_t* __restrict__ cursor,
                    uint32_t* __restrict__ pairs) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npairs) return;
    const int l = __ldg(probes + i);
    if ((unsigned)l >= (unsigned)kc || __ldg(list_len + l) <= 0) return;
    if (flag[i / nprobe]) return;
    pairs[atomicAdd(cursor + l, 1)] = (uint32_t)i;
}

// exclusive prefix sums of hist[0, n) -> off[0, n], cursor[0, n) (a copy the scatter advances); two small kernels
constexpr int kScanBlock = 1024;
__global__ void __launch_bounds__(256)
block_sum_kernel(const int32_t* __restrict__ hist, int n, int32_t* __restrict__ bsum) {
    __shared__ int s_w[8];
    const int base = blockIdx.x * kScanBlock;
    int s = 0;
    for (int i = threadIdx.x; i < kScanBlock; i += 256) s += base + i < n ? hist[base + i] : 0;
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xFFFFFFFFu, s, o);
    if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) { int t = 0; for (int w = 0; w < 8; ++w) t += s_w[w]; bsum[blockIdx.x] = t; }
}
__global__ void __launch_bounds__(256)
block_scan_kernel(const int32_t* __restrict__ hist, int n, const int32_t* __restrict__ bsum, int32_t* __restrict__ off,
                  int32_t* __restrict__ cursor) {
    __shared__ int s_w[8];
    __shared__ int s_base;
    const int base = blockIdx.x * kScanBlock;
    if (threadIdx.x < 32) {
        int s = 0;
        for (int b = threadIdx.x; b < (int)blockIdx.x; b += 32) s += bsum[b];
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xFFFFFFFFu, s, o);
        if (threadIdx.x == 0) s_base = s;
    }
    // thread t owns the 4 consecutive bins base + 4 t ..
    int v[4], s = 0;
#pragma unroll
    for (int e = 0; e < 4; ++e) { const int i = base + 4 * threadIdx.x + e; v[e] = i < n ? hist[i] : 0; s += v[e]; }
    int inc = s;
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xFFFFFFFFu, inc, o); if ((int)(threadIdx.x & 31) >= o) inc += t; }
    if ((threadIdx.x & 31) == 31) s_w[threadIdx.x >> 5] = inc;
    __syncthreads();
    int run = s_base + inc - s;
    for (int w = 0; w < (int)(threadIdx.x >> 5); ++w) run += s_w[w];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        const int i = base + 4 * threadIdx.x + e;
        if (i < n) { off[i] = run; cursor[i] = run; }
        run += v[e];
        if (i == n - 1) off[n] = run;
    }
}

// bias[pair] = ||q - c_l||^2 of the pairs THIS launch visits (the lists that hold vectors here, the queries not handed
// back): a warp takes eight consecutive pairs.  The batch-wide rows kernel walks all nprobe probes of a query one after
// the other, each a chain of dependent loads -- on a shard, where seven of eight probes belong to other ranks, that chain
// (118 us at C5 on 8 GPUs) cost more than the one-GPU kernel's arithmetic.  Lane-strided partial sums and the xor tree of
// probe_bias_rows_kernel / build_probe_table: identical bits.
template <int G>
__global__ void __launch_bounds__(256)
pair_bias_kernel(const float* __restrict__ queries, const int32_t* __restrict__ probes, const float* __restrict__ coarse,
                 const uint32_t* __restrict__ pairs, const int32_t* __restrict__ npairs_dev, int nprobe,
                 float* __restrict__ bias) {
    constexpr int d = 32 * G;                                // = 2 m: the loops below unroll, all loads of a round in flight
    constexpr int U = 8;                                     // consecutive pairs of a warp: grouped by list, so the
    const int lane = threadIdx.x & 31;                       // centroid row of most of them is the same (L1)
    const int np = *npairs_dev;
    const int nwarps = (int)((gridDim.x * blockDim.x) >> 5);
    for (int i0 = U * (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5); i0 < np; i0 += U * nwarps) {
        const uint32_t mine = (lane < U && i0 + lane < np) ? __ldg(pairs + i0 + lane) : 0xFFFFFFFFu;
        const int lst = mine != 0xFFFFFFFFu ? __ldg(probes + mine) : 0;
        float part[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint32_t pr = __shfl_sync(0xFFFFFFFFu, mine, u);
            const int l = __shfl_sync(0xFFFFFFFFu, lst, u);
            part[u] = 0.0f;
            if (pr != 0xFFFFFFFFu) {
                const float* qv = queries + (size_t)(pr / (uint32_t)nprobe) * d;
                const float* cv = coarse + (size_t)l * d;
                float qe[G], ce[G];
#pragma unroll
                for (int t = 0; t < G; ++t) { qe[t] = __ldg(qv + lane + 32 * t); ce[t] = __ldg(cv + lane + 32 * t); }
#pragma unroll
                for (int t = 0; t < G; ++t) { const float df = qe[t] - ce[t]; part[u] = fmaf(df, df, part[u]); }
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u)
            for (int o = 16; o > 0; o >>= 1) part[u] += __shfl_xor_sync(0xFFFFFFFFu, part[u], o);
        float out = 0.0f;
#pragma unroll
        for (int u = 0; u < U; ++u) out = lane == u ? part[u] : out;
        if (mine != 0xFFFFFFFFu) bias[mine] = out;
    }
}

// The order in which the CTAs take the lists: most work first (work = 128-vector tiles x visits of kNQ queries), so the
// long lists do not end up as the tail of the kernel -- at one-eighth of the lists a CTA sees ~55 lists and one list of ten
// times the mean length taken last was a fifth of the kernel.  A counting sort over 256 work classes (eight per octave,
// descending); lists nobody probes are left out.  hist = pairs per list (pair_count_kernel).
constexpr int kOrderClasses = 256;
__device__ __forceinline__ int work_class(int npairs, int len) {
    const unsigned w = (unsigned)((len + 127) >> 7) * (unsigned)((npairs + kNQ - 1) / kNQ);      // >= 1
    const int e = 31 - __clz(w);
    const int frac = e >= 3 ? (int)((w >> (e - 3)) & 7u) : (int)((w << (3 - e)) & 7u);
    return kOrderClasses - 1 - (8 * e + frac);
}
__global__ void __launch_bounds__(256)
list_order_count_kernel(const int32_t* __restrict__ hist, const int32_t* __restrict__ list_len, int kc, int* __restrict__ class_cnt) {
    __shared__ int s_h[kOrderClasses];
    s_h[threadIdx.x] = 0;
    __syncthreads();
    for (int l = blockIdx.x * kScanBlock + threadIdx.x; l < min(kc, (int)(blockIdx.x + 1) * kScanBlock); l += 256) {
        const int np = hist[l];
        if (np > 0) atomicAdd(&s_h[work_class(np, __ldg(list_len + l))], 1);
    }
    __syncthreads();
    if (s_h[threadIdx.x]) atomicAdd(class_cnt + threadIdx.x, s_h[threadIdx.x]);
}
__global__ void __launch_bounds__(256)
list_order_scatter_kernel(const int32_t* __restrict__ hist, const int32_t* __restrict__ list_len, int kc,
                          const int* __restrict__ class_cnt, int* __restrict__ class_cur, int32_t* __restrict__ order,
                          int* __restrict__ n_order) {
    __shared__ int s_h[kOrderClasses], s_at[kOrderClasses], s_w[8];
    // where class c starts: the exclusive prefix sum of the class counts (every CTA recomputes the 256 sums)
    const int cnt = class_cnt[threadIdx.x];
    int inc = cnt;
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xFFFFFFFFu, inc, o); if ((int)(threadIdx.x & 31) >= o) inc += t; }
    if ((threadIdx.x & 31) == 31) s_w[threadIdx.x >> 5] = inc;
    s_h[threadIdx.x] = 0;
    __syncthreads();
    int base = inc - cnt;
    for (int w = 0; w < (int)(threadIdx.x >> 5); ++w) base += s_w[w];
    if (blockIdx.x == 0 && threadIdx.x == kOrderClasses - 1) *n_order = base + cnt;
    const int lo = blockIdx.x * kScanBlock, hi = min(kc, lo + kScanBlock);
    int cls[kScanBlock / 256], pos[kScanBlock / 256];
#pragma unroll
    for (int e = 0; e < kScanBlock / 256; ++e) {
        const int l = lo + threadIdx.x + 256 * e;
        cls[e] = -1;
        if (l < hi) {
            const int np = hist[l];
            if (np > 0) { cls[e] = work_class(np, __ldg(list_len + l)); pos[e] = atomicAdd(&s_h[cls[e]], 1); }
        }
    }
    __syncthreads();
    // this CTA's lists of class c go to one run, reserved with one atomic per (CTA, class)
    s_at[threadIdx.x] = s_h[threadIdx.x] ? base + atomicAdd(class_cur + threadIdx.x, s_h[threadIdx.x]) : 0;
    __syncthreads();
#pragma unroll
    for (int e = 0; e < kScanBlock / 256; ++e)
        if (cls[e] >= 0) order[s_at[cls[e]] + pos[e]] = lo + threadIdx.x + 256 * e;
}

// The finalists.  kLogParts CTAs per log (the logs are far from equally long: one CTA per log left the longest as the kernel's
// tail), one thread per (pair, slot) record: the record is replaced by its exact key -- the
// look-up-table scan's arithmetic: the same table entries (lut_entry2), the same four partial sums in the same order -- and
// the query it belongs to is counted.  (Per record, not per query: a few queries have thousands of survivors.)
// A log that overflowed hands every query back (flagged through *overflow).
constexpr int kLogParts = 4;
template <int G>
__global__ void __launch_bounds__(256)
log_key_kernel(u64* __restrict__ log, const int* __restrict__ log_cnt, int log_cap, uint32_t* __restrict__ log_q,
               const float* __restrict__ queries, int nprobe, const float* __restrict__ bias, const float* __restrict__ codebooks_t,
               const uint8_t* __restrict__ slot_codes, const float* __restrict__ slot_tx, const int64_t* __restrict__ slot_ids,
               int32_t* __restrict__ cand_cnt, int* __restrict__ overflow) {
    constexpr int m = 16 * G;
    const int w = blockIdx.x / kLogParts, part = blockIdx.x % kLogParts;      // a log is shared by kLogParts CTAs
    int n = log_cnt[w];
    if (n > log_cap) { if (threadIdx.x == 0) *overflow = 1; n = log_cap; }
    u64* recs = log + (size_t)w * log_cap;
    const float2* cbt = reinterpret_cast<const float2*>(codebooks_t);
    for (int i = part * 256 + threadIdx.x; i < n; i += 256 * kLogParts) {
        const u64 c = recs[i];
        const uint32_t pr = (uint32_t)(c >> 32), g = (uint32_t)c;
        const uint32_t q = pr / (uint32_t)nprobe;
        const uint32_t sl = g & 31u;
        const uint4* src = reinterpret_cast<const uint4*>(slot_codes + (size_t)(g >> 5) * (512u * G)) + sl;
        const float2* qv = reinterpret_cast<const float2*>(queries + (size_t)q * (2 * m));
        uint4 w4[G];
#pragma unroll
        for (int grp = 0; grp < G; ++grp) w4[grp] = __ldg(src + 32 * grp);
        float s[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
        for (int grp = 0; grp < G; ++grp) {
            const uint32_t x[4] = {w4[grp].x, w4[grp].y, w4[grp].z, w4[grp].w};
#pragma unroll
            for (int i4 = 0; i4 < 4; ++i4) {
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    const uint32_t b = 4 * i4 + t;
                    const uint32_t code = (x[i4] >> (8 * t)) & 255u;
                    const uint32_t j = 16u * grp + ((b ^ sl) & 15u);
                    const float2 v = __ldg(cbt + code * m + j);
                    const float2 qq = __ldg(qv + j);
                    s[t] = fadd(s[t], lut_entry2(qq.x * -2.0f, qq.y * -2.0f, v));     // the table build's pre-scaled query
                }
            }
        }
        const float sum = fadd(fadd(__ldg(bias + pr), __ldg(slot_tx + g)), fadd(fadd(s[0], s[1]), fadd(s[2], s[3])));
        recs[i] = make_key(sum, 0u, 0) | (u64)(uint32_t)slot_ids[g];
        log_q[(size_t)w * log_cap + i] = q;
        atomicAdd(cand_cnt + q, 1);
    }
}

// keys -> one contiguous run per query (cursor = the exclusive prefix sums of the counts)
__global__ void __launch_bounds__(256)
key_scatter_kernel(const u64* __restrict__ log, const int* __restrict__ log_cnt, int log_cap, const uint32_t* __restrict__ log_q,
                   int32_t* __restrict__ cursor, u64* __restrict__ keys) {
    const int w = blockIdx.x;
    const int n = min(log_cnt[w], log_cap);
    for (int i = threadIdx.x; i < n; i += 256) {
        const size_t at = (size_t)w * log_cap + i;
        keys[atomicAdd(cursor + log_q[at], 1)] = log[at];
    }
}

// one warp per query: the k best of its keys by (score, id) -- or the query is handed back.  Up to 512 keys are selected in
// registers (select_and_write); the few queries with longer runs (thousands of survivors: a warp streaming 6.7 k keys through
// its queue was the tail of this kernel, 140 us at C5) are listed for select_long_kernel.
__global__ void __launch_bounds__(128)
select_kernel(int64_t nq, const int32_t* __restrict__ off, const u64* __restrict__ keys, int k, const int* __restrict__ flag,
              const int* __restrict__ overflow, int32_t* __restrict__ fb_list, int* __restrict__ fb_count,
              int32_t* __restrict__ long_list, int* __restrict__ long_count, float* __restrict__ out_dist,
              int64_t* __restrict__ out_ids) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t q = (int64_t)blockIdx.x * 4 + warp;
    if (q >= nq) return;
    if (flag[q] || *overflow) {
        if (lane == 0) fb_list[atomicAdd(fb_count, 1)] = (int32_t)q;
        return;
    }
    // (one GPU: the seed's k vectors passed the filter, so there are at least k keys; a shard may hold fewer)
    const int n = off[q + 1] - off[q];
    if (n <= 512) { select_and_write(keys + off[q], n, k, 0, q, out_dist, out_ids); return; }
    if (lane == 0) long_list[atomicAdd(long_count, 1)] = (int32_t)q;
}

// the listed queries, one CTA at a time: the keys stream through a CTA-wide queue under a threshold (BlockQueue: k best +
// up to P - k accepted since the last sort).  A key equal to the k-th best is a second copy of it: kept out only if k copies
// are already in, which the sort guarantees.
__global__ void __launch_bounds__(256)
select_long_kernel(const int32_t* __restrict__ long_list, const int* __restrict__ long_count, const int32_t* __restrict__ off,
                   const u64* __restrict__ keys, int k, int P, float* __restrict__ out_dist, int64_t* __restrict__ out_ids) {
    extern __shared__ __align__(16) unsigned char qsm[];
    __shared__ int s_cnt;
    __shared__ u64 s_thr;
    u64* sk = reinterpret_cast<u64*>(qsm);
    const int nlong = *long_count;
    for (int r = blockIdx.x; r < nlong; r += gridDim.x) {
        const int64_t q = long_list[r];
        const u64* src = keys + off[q];
        const int n = off[q + 1] - off[q];
        __syncthreads();
        BlockQueue bq{sk, &s_cnt, &s_thr, k, P};
        bq.init();
        for (int base = 0; base < n; base += blockDim.x) {
            bq.flush_if_needed(blockDim.x);
            const int i = base + threadIdx.x;
            if (i < n) bq.push(src[i]);
        }
        bq.flush();
        for (int i = threadIdx.x; i < k; i += blockDim.x) write_result(sk[i], 0, (size_t)q * k + i, out_dist, out_ids);
    }
}

__global__ void smem_base_kernel(uint32_t* out) {
    extern __shared__ __align__(1024) unsigned char probe_raw[];
    if (threadIdx.x == 0) *out = smem_u32(probe_raw);
}

// the absolute shared address at which this device starts a kernel's dynamic shared memory (1024 on sm_100: the system's
// reserve), asked once; -1 when the layout above does not fit behind it
static int smem_base() {
    static std::once_flag once;
    static int base = -1;
    std::call_once(once, [] {
        uint32_t* d = nullptr;
        uint32_t h = 0xFFFFFFFFu;
        if (cudaMalloc(&d, 4) != cudaSuccess) return;
        smem_base_kernel<<<1, 32, 1024>>>(d);
        if (cudaMemcpy(&h, d, 4, cudaMemcpyDeviceToHost) == cudaSuccess && h + sizeof(Small) <= kTabAbs &&
            kEndAbs - h <= 227u * 1024u)
            base = (int)h;
        cudaFree(d);
        (void)cudaGetLastError();
    });
    return base;
}

}  // namespace tcs

// L2, dsub = 2, rotated lists, no filter, no phase statistics; batches large enough that lists are shared.
// VIX_TC_SCAN=0 disables the path, =1 takes it whenever the shape allows.
// VIX_TC_SCAN_TIMES=1: CUDA events between the stages of every list-major launch (no synchronisation: the events of a launch are
// read when the NEXT launch of this thread starts, or at exit), summed and printed at process exit.  For multi-GPU runs, where
// ncu cannot look: which of the small stages a rank's step consists of.
namespace tcs {
constexpr int kTimeMarks = 10;
static const char* const kTimeNames[kTimeMarks - 1] = {"setup", "norms+seed_scan", "bounds over ranks", "prep+pairs+order",
                                                        "probe_bias", "tc_scan", "log_key", "scatter+select", "handed_back"};
struct StageTimes {
    cudaEvent_t ev[kTimeMarks] = {};
    bool have = false, pending = false;
    double sum[kTimeMarks - 1] = {};
    long long launches = 0;
    void collect() {
        if (!pending) return;
        if (cudaEventSynchronize(ev[kTimeMarks - 1]) == cudaSuccess) {
            for (int i = 0; i + 1 < kTimeMarks; ++i) { float ms = 0; if (cudaEventElapsedTime(&ms, ev[i], ev[i + 1]) == cudaSuccess) sum[i] += ms; }
            ++launches;
        }
        pending = false;
    }
    ~StageTimes() {
        collect();
        if (!launches) return;
        const char* r = getenv("RANK");
        double tot = 0;
        for (int i = 0; i + 1 < kTimeMarks; ++i) tot += sum[i];
        fprintf(stderr, "[vix tc times] rank %s, %lld launches, %.1f us per launch:", r ? r : "-", launches, 1e3 * tot / launches);
        for (int i = 0; i + 1 < kTimeMarks; ++i) fprintf(stderr, " %s %.1f", kTimeNames[i], 1e3 * sum[i] / launches);
        fprintf(stderr, "\n");
    }
};
static StageTimes* stage_times() {
    static const bool on = [] { const char* e = getenv("VIX_TC_SCAN_TIMES"); return e && e[0] == '1'; }();
    if (!on) return nullptr;
    static thread_local StageTimes st;
    if (!st.have) {
        for (int i = 0; i < kTimeMarks; ++i) if (cudaEventCreate(&st.ev[i]) != cudaSuccess) return nullptr;
        st.have = true;
    }
    return &st;
}
}  // namespace tcs

bool tc_decode_table_shape(int m, int ks, int dsub) { return dsub == 2 && ks == 256 && (m == 16 || m == 32 || m == 48 || m == 64); }
bool tc_codes_shape(int metric, int m, int ks, int dsub) { return metric == VIX_METRIC_L2 && tc_decode_table_shape(m, ks, dsub); }
int tc_decode_table(const float* codebooks, int m, uint32_t* table, float* meta) {
    tcs::table_kernel<<<1, 1024, 0, ctx().stream>>>(codebooks, m, table, meta);
    VIX_LAUNCH_CHECK();
    return VIX_OK;
}

bool tc_scan_supported(const ScanArgs& a) {
    const char* env = getenv("VIX_TC_SCAN");
    if (env && env[0] == '0') return false;
    if (!tc_codes_shape(a.metric, a.m, a.ks, a.dsub)) return false;
    if (a.filter || a.phase_cycles || a.nq_dev || a.k > 64) return false;
    if (a.nq * (int64_t)a.nprobe >= (1LL << 32) || a.nq < 1) return false;
    if (!(env && env[0] == '1') && a.nq * (int64_t)a.nprobe < 32768) return false;
    return tcs::smem_base() >= 0;
}

int launch_ivfpq_scan_tc(ScanArgs& a) {
    using namespace tcs;
    cudaStream_t s = ctx().stream;
    const int64_t nq = a.nq, npairs = a.nq * (int64_t)a.nprobe;
    const int k = a.k, m = a.m, d = a.d, G = m / 16;

    Scratch<uint32_t> table, pairs;
    Scratch<float> meta, qnorm, uq, bias;
    Scratch<unsigned int> maxabs;
    Scratch<int32_t> hist, off, cursor, bsum, fb_list, long_list;
    Scratch<int> flag, counters, wc_fb;
    Scratch<int32_t> cand_cnt, cand_off, cand_cur;
    Scratch<uint32_t> log_q;
    Scratch<__half> qh;
    Scratch<u64> cand;
    const bool own_table = !(a.tc_table && a.tc_meta);          // callers without a handle: the table of this launch
    if (own_table) VIX_TRY(table.alloc(kTcTableWords));
    Scratch<float> own_meta;
    if (own_table) VIX_TRY(own_meta.alloc(4));
    const uint32_t* const table_ptr = own_table ? table.ptr : a.tc_table;
    const float* const tmeta_ptr = own_table ? own_meta.ptr : a.tc_meta;
    VIX_TRY(meta.alloc(4));
    VIX_TRY(qnorm.alloc((size_t)nq));
    VIX_TRY(uq.alloc((size_t)nq));
    VIX_TRY(maxabs.alloc(1));
    VIX_TRY(flag.alloc((size_t)nq));
    VIX_TRY(qh.alloc((size_t)nq * d));
    VIX_TRY(hist.alloc((size_t)a.kc + 1));
    VIX_TRY(off.alloc((size_t)a.kc + 1));
    VIX_TRY(cursor.alloc((size_t)a.kc + 1));
    const int nblk = (a.kc + kScanBlock - 1) / kScanBlock;
    VIX_TRY(bsum.alloc((size_t)nblk));
    VIX_TRY(pairs.alloc((size_t)npairs));
    VIX_TRY(bias.alloc((size_t)npairs));
    Scratch<int32_t> order;
    VIX_TRY(order.alloc((size_t)a.kc));
    // [0] list counter, [1] error, [2] fall-back count, [3] status, [4] log overflow, [5] lists in `order`, [6] queries with
    // more than 512 finalists;
    // [8, 264) lists per work class, [264, 520) the scatter's cursors
    VIX_TRY(counters.alloc(8 + 2 * kOrderClasses));
    VIX_TRY(cand_cnt.alloc((size_t)nq + 1));
    VIX_TRY(cand_off.alloc((size_t)nq + 1));
    VIX_TRY(cand_cur.alloc((size_t)nq + 1));
    VIX_TRY(fb_list.alloc((size_t)nq));
    VIX_TRY(long_list.alloc((size_t)nq));
    VIX_TRY(wc_fb.alloc(2));
    VIX_CUDA(cudaMemsetAsync(maxabs.ptr, 0, 4, s));
    VIX_CUDA(cudaMemsetAsync(hist.ptr, 0, ((size_t)a.kc + 1) * 4, s));
    VIX_CUDA(cudaMemsetAsync(counters.ptr, 0, (8 + 2 * kOrderClasses) * sizeof(int), s));
    VIX_CUDA(cudaMemsetAsync(cand_cnt.ptr, 0, (size_t)nq * 4, s));
    StageTimes* const times = stage_times();
    if (times) times->collect();
    int mark_i = 0;
    auto mark = [&] { if (times && mark_i < kTimeMarks) cudaEventRecord(times->ev[mark_i++], s); };
    mark();

    if (own_table) VIX_TRY(tc_decode_table(a.codebooks, m, table.ptr, own_meta.ptr));
    const unsigned qwarps = (unsigned)((nq * 32 + 255) / 256);
    mark();
    Scratch<float> thr;
    VIX_TRY(thr.alloc((size_t)nq));
    {   // norms + seed: one CTA per query, one warp per sampled chunk
        static_assert(32 * kSeedChunks >= 64, "k <= 64 keys out of the sample");
#define VIX_SEED(GG)                                                                                                       \
        do {                                                                                                               \
            seed_scan_kernel<GG><<<(unsigned)nq, 32 * kSeedChunks, 0, s>>>(a.queries, nq, a.probes, a.nprobe, a.kc,          \
                tls_thr_hook != nullptr, a.coarse, a.codebooks_t, a.list_off, a.list_len, a.slot_codes, a.slot_tx, k,       \
                qnorm.ptr, maxabs.ptr, thr.ptr);                                                                           \
            VIX_LAUNCH_CHECK();                                                                                            \
        } while (0)
        switch (G) {
            case 1: VIX_SEED(1); break;
            case 2: VIX_SEED(2); break;
            case 3: VIX_SEED(3); break;
            case 4: VIX_SEED(4); break;
        }
#undef VIX_SEED
    }
    mark();
    if (tls_thr_hook) VIX_TRY(tls_thr_hook(tls_thr_ctx, thr.ptr, nq));         // sharded: the minimum over the ranks
    mark();
    query_prep_kernel<<<qwarps, 256, 0, s>>>(a.queries, nq, d, qnorm.ptr, maxabs.ptr, meta.ptr, tmeta_ptr, thr.ptr, qh.ptr,
                                            uq.ptr, flag.ptr);
    VIX_LAUNCH_CHECK();
    const unsigned pblocks = (unsigned)((npairs + 255) / 256);
    pair_count_kernel<<<pblocks, 256, 0, s>>>(a.probes, npairs, a.nprobe, a.list_len, a.kc, flag.ptr, hist.ptr, a.scanned);
    VIX_LAUNCH_CHECK();
    block_sum_kernel<<<nblk, 256, 0, s>>>(hist.ptr, a.kc, bsum.ptr);
    VIX_LAUNCH_CHECK();
    block_scan_kernel<<<nblk, 256, 0, s>>>(hist.ptr, a.kc, bsum.ptr, off.ptr, cursor.ptr);
    VIX_LAUNCH_CHECK();
    list_order_count_kernel<<<nblk, 256, 0, s>>>(hist.ptr, a.list_len, a.kc, counters.ptr + 8);
    VIX_LAUNCH_CHECK();
    list_order_scatter_kernel<<<nblk, 256, 0, s>>>(hist.ptr, a.list_len, a.kc, counters.ptr + 8, counters.ptr + 8 + kOrderClasses,
                                                  order.ptr, counters.ptr + 5);
    VIX_LAUNCH_CHECK();
    pair_scatter_kernel<<<pblocks, 256, 0, s>>>(a.probes, npairs, a.nprobe, a.list_len, a.kc, flag.ptr, cursor.ptr,
                                               pairs.ptr);
    VIX_LAUNCH_CHECK();
    mark();
    {   // the per-pair term of this launch's pairs, plus all probes of the (rare) queries handed back, for the look-up-table
        // scan.  (The batch-wide rows kernel walks all nprobe probes of a query as one chain of dependent loads: on a shard,
        // where seven of eight probes belong to other ranks, 118 us against 73 at C5 on 8 GPUs; on one GPU the two are equal,
        // 180 / 173 us between events.)
        int64_t want = (npairs * 32 + 8 * 256 - 1) / (8 * 256);
        const int64_t cap = (int64_t)num_sms() * 8;
        const unsigned bgrid = (unsigned)(want < cap ? (want ? want : 1) : cap);
        switch (G) {
            case 1: pair_bias_kernel<1><<<bgrid, 256, 0, s>>>(a.queries, a.probes, a.coarse, pairs.ptr, off.ptr + a.kc, a.nprobe, bias.ptr); break;
            case 2: pair_bias_kernel<2><<<bgrid, 256, 0, s>>>(a.queries, a.probes, a.coarse, pairs.ptr, off.ptr + a.kc, a.nprobe, bias.ptr); break;
            case 3: pair_bias_kernel<3><<<bgrid, 256, 0, s>>>(a.queries, a.probes, a.coarse, pairs.ptr, off.ptr + a.kc, a.nprobe, bias.ptr); break;
            case 4: pair_bias_kernel<4><<<bgrid, 256, 0, s>>>(a.queries, a.probes, a.coarse, pairs.ptr, off.ptr + a.kc, a.nprobe, bias.ptr); break;
        }
        VIX_LAUNCH_CHECK();
        VIX_TRY(launch_probe_bias(a, bias.ptr, flag.ptr));
    }
    mark();

    int grid = num_sms();
    if (grid > a.kc) grid = a.kc;
    // room for 256 survivors per query over all logs (C5: ~100 per query with the sampled seed), at least 4096 per log
    const int64_t want = (nq * 256 + grid * kEpiWarps - 1) / (grid * kEpiWarps);
    const int log_cap = (int)(want < 4096 ? 4096 : want);
    Scratch<u64> log;
    Scratch<int> log_cnt;
    VIX_TRY(log.alloc((size_t)grid * kEpiWarps * log_cap));
    VIX_TRY(log_cnt.alloc((size_t)grid * kEpiWarps));
    VIX_TRY(log_q.alloc((size_t)grid * kEpiWarps * log_cap));
    VIX_TRY(cand.alloc((size_t)grid * kEpiWarps * log_cap));
    VIX_CUDA(cudaMemsetAsync(log_cnt.ptr, 0, (size_t)grid * kEpiWarps * sizeof(int), s));
    Args t{};
    t.tc_codes = a.tc_codes; t.slot_tx = a.slot_tx; t.list_off = a.list_off; t.list_len = a.list_len; t.kc = a.kc;
    t.pair_off = off.ptr; t.order = order.ptr; t.n_order = counters.ptr + 5; t.pairs = pairs.ptr; t.bias = bias.ptr; t.qh = qh.ptr;
    t.uq = uq.ptr; t.table = table_ptr;
    t.scales = meta.ptr; t.nprobe = a.nprobe; t.d = d; t.m = m;
    t.list_counter = counters.ptr; t.log = log.ptr; t.log_cnt = log_cnt.ptr; t.log_cap = log_cap;
    t.error = counters.ptr + 1; t.error_host = pipeline_error_flag();
    t.status = t.error_host ? t.error_host : counters.ptr + 3;
#ifdef VIX_TCS_DIAG
    Scratch<unsigned long long> diag;
    VIX_TRY(diag.alloc(32));
    VIX_CUDA(cudaMemsetAsync(diag.ptr, 0, 256, s));
    t.diag = diag.ptr;
#endif
    const int smem = (int)kEndAbs - smem_base();
    t.smem_bytes = smem;
#define VIX_TCS(GG)                                                                                                        \
    do {                                                                                                                   \
        VIX_CUDA(cudaFuncSetAttribute(tc_scan_kernel<GG>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));             \
        if (a.ev_kernel[0]) VIX_CUDA(cudaEventRecord(a.ev_kernel[0], s));                                                  \
        tc_scan_kernel<GG><<<grid, kThreads, smem, s>>>(t);                                                                \
        VIX_LAUNCH_CHECK();                                                                                                \
        if (a.ev_kernel[1]) VIX_CUDA(cudaEventRecord(a.ev_kernel[1], s));                                                  \
        mark();                                                                                                            \
        log_key_kernel<GG><<<grid * kEpiWarps * kLogParts, 256, 0, s>>>(log.ptr, log_cnt.ptr, log_cap, log_q.ptr, a.queries, a.nprobe, bias.ptr,  \
            a.codebooks_t, a.slot_codes, a.slot_tx, a.slot_ids, cand_cnt.ptr, counters.ptr + 4);                           \
        VIX_LAUNCH_CHECK();                                                                                                \
    } while (0)
    switch (G) {
        case 1: VIX_TCS(1); break;
        case 2: VIX_TCS(2); break;
        case 3: VIX_TCS(3); break;
        case 4: VIX_TCS(4); break;
    }
#undef VIX_TCS
    mark();
    {   // per-query runs of keys, then the selection
        const int qblk = (int)((nq + kScanBlock - 1) / kScanBlock);
        VIX_TRY(bsum.alloc((size_t)qblk));
        block_sum_kernel<<<qblk, 256, 0, s>>>(cand_cnt.ptr, (int)nq, bsum.ptr);
        VIX_LAUNCH_CHECK();
        block_scan_kernel<<<qblk, 256, 0, s>>>(cand_cnt.ptr, (int)nq, bsum.ptr, cand_off.ptr, cand_cur.ptr);
        VIX_LAUNCH_CHECK();
        key_scatter_kernel<<<grid * kEpiWarps, 256, 0, s>>>(log.ptr, log_cnt.ptr, log_cap, log_q.ptr, cand_cur.ptr, cand.ptr);
        VIX_LAUNCH_CHECK();
        select_kernel<<<(unsigned)((nq + 3) / 4), 128, 0, s>>>(nq, cand_off.ptr, cand.ptr, k, flag.ptr, counters.ptr + 4, fb_list.ptr,
                                                              counters.ptr + 2, long_list.ptr, counters.ptr + 6, a.out_dist, a.out_ids);
        VIX_LAUNCH_CHECK();
        const int P = next_pow2(k + 256);
        select_long_kernel<<<num_sms(), 256, (size_t)P * 8, s>>>(long_list.ptr, counters.ptr + 6, cand_off.ptr, cand.ptr, k, P,
                                                                a.out_dist, a.out_ids);
        VIX_LAUNCH_CHECK();
    }
    mark();
    {   // the queries handed back: all their probes through the look-up-table scan
        ScanArgs fb = a;
        fb.order = fb_list.ptr; fb.nq_dev = counters.ptr + 2;
        fb.scanned = nullptr; fb.bias = bias.ptr; fb.lut_image = nullptr;
        fb.ev_kernel[0] = fb.ev_kernel[1] = nullptr;
        fb.work_counter = wc_fb.ptr;
        VIX_TRY(launch_ivfpq_scan_classic(fb));
    }
    mark();
    if (times) times->pending = mark_i == kTimeMarks;
    g_tc_launches.fetch_add(1);
    if (getenv("VIX_TC_SCAN_DEBUG")) {
        // diagnostics (synchronises): queries handed back, candidates per query
        int hc[4] = {0, 0, 0, 0};
        std::vector<int> cc((size_t)nq);
        VIX_CUDA(cudaMemcpyAsync(hc, counters.ptr, 16, cudaMemcpyDeviceToHost, s));
        VIX_CUDA(cudaMemcpyAsync(cc.data(), cand_cnt.ptr, (size_t)nq * 4, cudaMemcpyDeviceToHost, s));
        VIX_CUDA(cudaStreamSynchronize(s));
        long long tot = 0;
        int mx = 0;
        for (int64_t i = 0; i < nq; ++i) { tot += cc[(size_t)i]; mx = cc[(size_t)i] > mx ? cc[(size_t)i] : mx; }
#ifdef VIX_TCS_DIAG
        unsigned long long hd[32];
        VIX_CUDA(cudaMemcpy(hd, diag.ptr, 256, cudaMemcpyDeviceToHost));
        const char* names[4][4] = {{"item_full", "a_empty", "-", "-"}, {"item_full", "b_full", "d_full", "-"},
                                   {"item_full", "b_full", "a_full", "d_empty"}, {"item_empty", "b_empty", "-", "-"}};
        const char* roles[4] = {"decoder", "filter", "mma", "loader"};
        const double nw[4] = {12.0 * grid, 1.0 * kEpiWarps * grid, 1.0 * kMmaWarps * grid, 1.0 * grid};
        for (int r = 0; r < 4; ++r) {
            fprintf(stderr, "[vix tc diag] %-8s total %10.0f cycles per warp; waits:", roles[r], (double)hd[16 + r] / nw[r]);
            for (int i = 0; i < 4; ++i) if (names[r][i][0] != '-') fprintf(stderr, " %s %.0f", names[r][i], (double)hd[r * 4 + i] / nw[r]);
            fprintf(stderr, "\n");
        }
#endif
#ifdef VIX_TCS_DIAG
        fprintf(stderr, "[vix tc diag] mma thread: %.0f units per CTA, %.1f cycles per unit issuing the MMAs, %.1f in the two commits\n",
                (double)hd[22] / grid, (double)hd[20] / (double)(hd[22] ? hd[22] : 1), (double)hd[21] / (double)(hd[22] ? hd[22] : 1));
#endif
        fprintf(stderr, "[vix tc scan] nq %lld, handed back %d, candidates %lld (max %d per query; %d per log), error %d\n", (long long)nq,
                hc[2], tot, mx, log_cap, hc[1]);
    }
    return VIX_OK;
}

long long tc_scan_launches() { return g_tc_launches.load(); }

}  // namespace vix
