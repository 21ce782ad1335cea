// vix_scoring.cu -- exact-arithmetic scoring and selection kernels (CUDA cores, reference order):
//
//   a1-a3  vix_l2sqr_f32_block / vix_ip_f32_block / vix_row_norms_f32
//   a1-a4  vix_flat_search_f32          pair tiles + fused per-row top-k, no [nq x n] matrix in HBM
//   a4/a5  vix_select_topk_f32 / vix_merge_topk_f32
//   a6-a8  vix_centroid_batch_score_f32 / vix_ivf_select_nprobe_batch_f32
//   a9     vix_ivf_assign_f32 / vix_ivf_assign_metric_f32      bit-exact argmin
//   a16    vix_accel_rank_candidates_f32
//
// All of them are instances of one tiled kernel (PairTile, vix_exact.cuh) with three epilogues:
// WRITE (materialise the tile), ARGMIN (running per-row minimum, tie -> lower index) and TOPK
// (per-row shared-memory selection queues keyed by (score, id); partial results of the B-splits are
// merged by merge_keys_kernel).  Distances come out bit-identical to the oracle's restatement of the
// reference, so ids match even on ties.  The tensor-core path (vix_gemm.cu) uses these kernels to
// rescore its shortlists.
#include "vix_exact.cuh"
#include "vix_topk.cuh"

#include <math.h>

namespace vix {

enum Epilogue { EPI_WRITE = 0, EPI_ARGMIN = 1, EPI_TOPK = 2 };
enum Transform {
    TR_NONE = 0,      // raw score
    TR_CBS_L2 = 1,    // -2 * s + bnorm[b]        CentroidBatchScore L2 (CentroidBatchScore.swift:54-64)
    TR_NEG = 2,       // -s                       CentroidBatchScore IP (alpha = -1)
    TR_DOTFUSED = 3,  // max(0, (anorm[a] + bnorm[b]) - 2 * s)   L2SqrKernel.swift:436-446
    TR_COSINE = 4     // clamp((s * anorm[a]) * bnorm[b], -1, 1) with inverse norms   Cosine.swift:96-119
};

struct PairArgs {
    const float* A; int64_t nA;
    const float* B; int64_t nB;
    int d, pitch;
    int transform;
    const float* anorm; const float* bnorm;
    const uint64_t* disabled;      // TOPK: bit b set => B row b skipped
    // WRITE
    float* out; int64_t ldo;
    // ARGMIN
    int32_t* arg_out; float* min_out;
    int first_min;                 // 1: plain first minimum, -1 when the row has none (IVFIndex.swift:376-435); 0: km12
    // TOPK
    int k, P, order_max, nsplit; int64_t btiles_per_split;
    u64* keys_out;                 // [nA x nsplit x k]
};

__device__ __forceinline__ float apply_transform(int tr, float s, const PairArgs& p, int64_t a, int64_t b) {
    if (tr == TR_CBS_L2) return fadd(fmul(-2.0f, s), p.bnorm[b]);
    if (tr == TR_NEG) return fmul(-1.0f, s);
    if (tr == TR_DOTFUSED) {
        float dist = fsub(fadd(p.anorm[a], p.bnorm[b]), fmul(2.0f, s));
        return dist < 0.0f ? 0.0f : dist;
    }
    if (tr == TR_COSINE) {
        const float v = fmul(fmul(s, p.anorm[a]), p.bnorm[b]);
        return fminf(1.0f, fmaxf(-1.0f, v));               // clampUnit (Cosine.swift:177)
    }
    return s;
}

template <typename Spec, int TV, int TC, int EPI>
__global__ void __launch_bounds__(256) pair_kernel(PairArgs p) {
    using Tile = PairTile<Spec, TV, TC>;
    constexpr int TA = Tile::TA, TB = Tile::TB;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float* As = reinterpret_cast<float*>(smem_raw);
    float* Bs = As + (size_t)TA * p.pitch;
    unsigned char* extra = reinterpret_cast<unsigned char*>(Bs + (size_t)TB * p.pitch);
    extra += (16 - (reinterpret_cast<uintptr_t>(extra) & 15)) & 15;

    const int tid = threadIdx.x;
    const int tx = tid & 15, ty = tid >> 4;
    const int lane = tid & 31, warp = tid >> 5;
    const int64_t a0 = (int64_t)blockIdx.x * TA;

    Tile::load_rows(As, p.pitch, p.A, a0, p.nA, TA, p.d);

    const int64_t nbt = (p.nB + TB - 1) / TB;
    int64_t bt0 = 0, bt1 = nbt;
    if (EPI == EPI_TOPK) {
        bt0 = (int64_t)blockIdx.y * p.btiles_per_split;
        bt1 = min(nbt, bt0 + p.btiles_per_split);
    }

    // ---- epilogue state ----
    float bestd[TV];
    int64_t besti[TV];
    bool nan0[TV];
    u64* qkeys = nullptr; int* qcnt = nullptr; u64* qthr = nullptr;
    if (EPI == EPI_ARGMIN) {
#pragma unroll
        for (int v = 0; v < TV; ++v) { bestd[v] = INFINITY; besti[v] = INT64_MAX; nan0[v] = false; }
    }
    if (EPI == EPI_TOPK) {
        qkeys = reinterpret_cast<u64*>(extra);                 // [TA x P]
        qthr = qkeys + (size_t)TA * p.P;                       // [TA]
        qcnt = reinterpret_cast<int*>(qthr + TA);              // [TA]
        for (int e = tid; e < TA * p.P; e += 256) qkeys[e] = kEmptyKey;
        for (int e = tid; e < TA; e += 256) { qthr[e] = kEmptyKey; qcnt[e] = 0; }
    }

    for (int64_t bt = bt0; bt < bt1; ++bt) {
        const int64_t b0 = bt * TB;
        __syncthreads();                      // previous Bs consumed (and queues initialised)
        Tile::load_rows(Bs, p.pitch, p.B, b0, p.nB, TB, p.d);
        __syncthreads();

        if (EPI == EPI_TOPK) {
            // make room: a tile can add at most TB candidates to a row
            for (int r = warp; r < TA; r += 8) {
                if (qcnt[r] > p.P - p.k - TB) {
                    WarpQueue q{qkeys + (size_t)r * p.P, qcnt + r, qthr + r, p.k, p.P};
                    q.flush(lane);
                }
            }
            __syncthreads();
        }

        float sc[TV][TC];
        Tile::compute(As, Bs, p.pitch, p.d, tx, ty, sc);

#pragma unroll
        for (int v = 0; v < TV; ++v) {
            const int64_t a = a0 + tx + 16 * v;
            if (a >= p.nA) continue;
#pragma unroll
            for (int c = 0; c < TC; ++c) {
                const int64_t b = b0 + ty + 16 * c;
                if (b >= p.nB) continue;
                const float s = apply_transform(p.transform, sc[v][c], p, a, b);
                if (EPI == EPI_WRITE) {
                    p.out[a * p.ldo + b] = s;
                } else if (EPI == EPI_ARGMIN) {
                    if (b == 0 && s != s) nan0[v] = true;
                    if (s < bestd[v] || (s == bestd[v] && b < besti[v])) { bestd[v] = s; besti[v] = b; }
                } else {
                    if (p.disabled && ((p.disabled[b >> 6] >> (b & 63)) & 1ull)) continue;
                    const int r = tx + 16 * v;
                    const u64 key = make_key(s, (uint32_t)b, p.order_max);
                    if (key < qthr[r]) {
                        int pos = atomicAdd(qcnt + r, 1);
                        qkeys[(size_t)r * p.P + p.k + pos] = key;
                    }
                }
            }
        }
    }

    if (EPI == EPI_ARGMIN) {
        // reduce over the 16 ty-threads that share an A row
        __syncthreads();
        float* rd = reinterpret_cast<float*>(extra);                       // [TA x 16]
        int64_t* ri = reinterpret_cast<int64_t*>(rd + TA * 16);            // [TA x 16]
        int* rn = reinterpret_cast<int*>(ri + TA * 16);                    // [TA]
        for (int e = tid; e < TA; e += 256) rn[e] = 0;
        __syncthreads();
#pragma unroll
        for (int v = 0; v < TV; ++v) {
            const int r = tx + 16 * v;
            rd[r * 16 + ty] = bestd[v];
            ri[r * 16 + ty] = besti[v];
            if (nan0[v]) rn[r] = 1;
        }
        __syncthreads();
        for (int r = tid; r < TA; r += 256) {
            const int64_t a = a0 + r;
            if (a >= p.nA) continue;
            float bd = rd[r * 16];
            int64_t bi = ri[r * 16];
            for (int y = 1; y < 16; ++y) {
                float s = rd[r * 16 + y];
                int64_t i = ri[r * 16 + y];
                if (s < bd || (s == bd && i < bi)) { bd = s; bi = i; }
            }
            // reference semantics with NaN (KMeansMiniBatchKernel.swift:341-359): the running best
            // starts at centroid 0 and a NaN there is never replaced
            // the first minimum of a CentroidBatchScore row instead (IVFIndex.swift:376-435: best starts at -1,
            // strict <): a row without any comparable score -- all NaN / +inf -- has no list
            if (p.first_min) { if (bi == INT64_MAX) bi = -1; }
            else if (rn[r] || bi == INT64_MAX) { bi = 0; if (rn[r]) bd = __int_as_float(0x7fc00000); }
            if (p.arg_out) p.arg_out[a] = (int32_t)bi;
            if (p.min_out) p.min_out[a] = bd;
        }
    }

    if (EPI == EPI_TOPK) {
        __syncthreads();
        for (int r = warp; r < TA; r += 8) {
            const int64_t a = a0 + r;
            if (a >= p.nA) continue;
            WarpQueue q{qkeys + (size_t)r * p.P, qcnt + r, qthr + r, p.k, p.P};
            if (qcnt[r] > 0) q.flush(lane);
            __syncwarp();
            u64* dst = p.keys_out + ((size_t)a * p.nsplit + blockIdx.y) * p.k;
            for (int i = lane; i < p.k; i += 32) dst[i] = q.keys[i];
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Merge of per-split key lists: one CTA per row, bitonic sort of P2 keys in shared memory.
// Output mapping: dist_mode 0 raw score, 1 sqrt(score) (flat L2 API distance), 2 -score (IP API
// distance, DistanceUtils.swift:40-46), 3 1 - score (cosine, FlatIndexOptimized.swift:468-470); unused slots id -1 / NaN.
// ------------------------------------------------------------------------------------------------
__global__ void merge_keys_kernel(const u64* __restrict__ keys, int nin, int P2, int k, int order_max,
                                  int dist_mode, uint32_t id_xor, float* __restrict__ out_score,
                                  int64_t* __restrict__ out_id64, int32_t* __restrict__ out_id32,
                                  int* __restrict__ out_count) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    u64* s = reinterpret_cast<u64*>(smem_raw);
    const int64_t row = blockIdx.x;
    const u64* src = keys + (size_t)row * nin;
    for (int i = threadIdx.x; i < P2; i += blockDim.x) s[i] = (i < nin) ? src[i] : kEmptyKey;
    __syncthreads();
    bitonic_sort_keys<false>(s, P2, threadIdx.x, blockDim.x);
    int cnt = 0;
    for (int i = threadIdx.x; i < k; i += blockDim.x) {
        u64 key = (i < P2) ? s[i] : kEmptyKey;
        const size_t o = (size_t)row * k + i;
        if (key == kEmptyKey) {
            if (out_score) out_score[o] = __int_as_float(0x7fc00000);
            if (out_id64) out_id64[o] = -1;
            if (out_id32) out_id32[o] = -1;
        } else {
            float sc = key_score(key, order_max);
            if (dist_mode == 1) sc = __fsqrt_rn(sc);
            else if (dist_mode == 2) sc = -sc;
            else if (dist_mode == 3) sc = fsub(1.0f, sc);
            if (out_score) out_score[o] = sc;
            const uint32_t id = key_id(key) ^ id_xor;
            if (out_id64) out_id64[o] = id_xor ? (int64_t)(int32_t)id : (int64_t)id;
            if (out_id32) out_id32[o] = (int32_t)id;
            ++cnt;
        }
    }
    if (out_count) {
        // count of valid entries (only used with a single row)
        __shared__ int total;
        if (threadIdx.x == 0) total = 0;
        __syncthreads();
        atomicAdd(&total, cnt);
        __syncthreads();
        if (threadIdx.x == 0) out_count[row] = total;
    }
}

int probe_select_fast_device(const float* q, int64_t nq, const float* c, int kc, int d, int metric, int nprobe,
                             const float* cnorm, int32_t* out_idx, float* out_scores, const float* cnorm_max_sqrt);

int ivf_assign_auto_device(const float* x, int64_t n, int d, const float* c, int kc, int32_t* assign, float* dist);

int flat_search_auto_device(const float* q, int64_t nq, const float* xb, int64_t n, int d, int metric, int k,
                            const float* xb_norm, float* out_dist, int64_t* out_ids, bool raw_scores);

int launch_merge_keys(const u64* keys, int64_t rows, int nin, int k, int order_max, int dist_mode,
                      float* out_score, int64_t* out_id64, int32_t* out_id32, int* out_count,
                      uint32_t id_xor = 0) {
    if (rows == 0 || k <= 0) return VIX_OK;
    int P2 = next_pow2(nin < 2 ? 2 : nin);
    size_t smem = (size_t)P2 * sizeof(u64);
    VIX_REQUIRE(smem <= 200 * 1024, VIX_ERR_UNSUPPORTED, "merge: %d candidates per row exceed shared memory", nin);
    VIX_CUDA(cudaFuncSetAttribute(merge_keys_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int threads = P2 / 2 < 32 ? 32 : (P2 / 2 > 512 ? 512 : P2 / 2);
    merge_keys_kernel<<<(unsigned)rows, threads, smem, ctx().stream>>>(keys, nin, P2, k, order_max, dist_mode,
                                                                       id_xor, out_score, out_id64, out_id32,
                                                                       out_count);
    VIX_LAUNCH_CHECK();
    return VIX_OK;
}

// ------------------------------------------------------------------------------------------------
// Launch helpers
// ------------------------------------------------------------------------------------------------
struct TilePlan { int tv; size_t smem; int P; };

static size_t tile_smem(int tv, int d, int epi, int P) {
    const int TA = 16 * tv, TB = 16 * tv;
    const int pitch = d | 1;
    size_t s = (size_t)(TA + TB) * pitch * 4 + 16;
    if (epi == EPI_TOPK) s += (size_t)TA * P * 8 + (size_t)TA * 12;
    if (epi == EPI_ARGMIN) s += (size_t)TA * 16 * 12 + (size_t)TA * 4;
    return s;
}

// Rows too long for the tiled engine (two 16-row tiles of whole rows no longer fit shared memory, d > ~1700; the
// reference's tests go to d = 2048, IVFSelectTests.swift:578-609): one thread per pair straight from global memory --
// the same chain, slowly.  WRITE epilogue only; selections then run on the materialised block (row_select_device).
template <typename Spec>
__global__ void __launch_bounds__(256)
pair_direct_kernel(PairArgs p) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.nA * p.nB) return;
    const int64_t a = i / p.nB, b = i - a * p.nB;
    const float s = exact_pair<Spec>(p.A + a * p.d, p.B + b * p.d, p.d);
    p.out[a * p.ldo + b] = apply_transform(p.transform, s, p, a, b);
}

// per row of a materialised [rows x n] score block: the k best columns by (score ascending, column ascending), columns
// whose bit is set in `disabled` skipped; padded with -1 / NaN.  One CTA per row at a time.
__global__ void __launch_bounds__(256)
row_select_kernel(const float* __restrict__ scores, int64_t rows, int n, int k, int P, const uint64_t* __restrict__ disabled,
                  int32_t* __restrict__ out_idx, float* __restrict__ out_scores) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    u64* keys = reinterpret_cast<u64*>(smem_raw);
    __shared__ int s_cnt;
    __shared__ u64 s_thr;
    for (int64_t r = blockIdx.x; r < rows; r += gridDim.x) {
        __syncthreads();
        BlockQueue q{keys, &s_cnt, &s_thr, k, P};
        q.init();
        for (int base = 0; base < n; base += blockDim.x) {
            q.flush_if_needed(blockDim.x);
            const int c = base + threadIdx.x;
            if (c < n && !(disabled && ((disabled[c >> 6] >> (c & 63)) & 1ull)))
                q.push(make_key(scores[r * (int64_t)n + c], (uint32_t)c, 0));
        }
        q.flush();
        for (int i = threadIdx.x; i < k; i += blockDim.x) {
            const u64 key = keys[i];
            out_idx[r * (int64_t)k + i] = key == kEmptyKey ? -1 : (int32_t)key_id(key);
            if (out_scores) out_scores[r * (int64_t)k + i] = key == kEmptyKey ? __int_as_float(0x7fc00000) : key_score(key, 0);
        }
    }
}

int row_select_device(const float* scores, int64_t rows, int n, int k, const uint64_t* disabled, int32_t* out_idx,
                      float* out_scores) {
    if (rows == 0 || k <= 0) return VIX_OK;
    const int P = next_pow2(k + 256);
    const size_t smem = (size_t)P * 8;
    VIX_REQUIRE(smem <= 200 * 1024, VIX_ERR_UNSUPPORTED, "row selection: k = %d exceeds shared memory", k);
    VIX_CUDA(cudaFuncSetAttribute(row_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int64_t grid = (int64_t)num_sms() * 4;
    if (grid > rows) grid = rows;
    row_select_kernel<<<(unsigned)grid, 256, smem, ctx().stream>>>(scores, rows, n, k, P, disabled, out_idx, out_scores);
    VIX_LAUNCH_CHECK();
    return VIX_OK;
}

static bool plan_tile(int d, int epi, int k, TilePlan* plan) {
    const size_t budget = 220 * 1024;
    for (int tv = 4; tv >= 1; tv >>= 1) {
        int P = (epi == EPI_TOPK) ? next_pow2(k + 16 * tv) : 0;
        size_t s = tile_smem(tv, d, epi, P);
        if (s <= budget) { plan->tv = tv; plan->smem = s; plan->P = P; return true; }
    }
    return false;
}

template <typename Spec, int EPI>
static int launch_pair(PairArgs& p, int k_for_plan, int64_t* nsplit_out = nullptr) {
    TilePlan plan;
    if (!plan_tile(p.d, EPI, k_for_plan, &plan)) {
        if constexpr (EPI == EPI_WRITE) {
            const int64_t total = p.nA * p.nB;
            VIX_REQUIRE(total < (1LL << 38), VIX_ERR_UNSUPPORTED, "exact scoring: %lld pairs at d = %d", (long long)total, p.d);
            if (total == 0) return VIX_OK;
            pair_direct_kernel<Spec><<<(unsigned)((total + 255) / 256), 256, 0, ctx().stream>>>(p);
            VIX_LAUNCH_CHECK();
            return VIX_OK;
        }
        set_error("exact scoring: d = %d (k = %d) does not fit the shared-memory tile", p.d, k_for_plan);
        return VIX_ERR_UNSUPPORTED;
    }
    p.pitch = p.d | 1;
    p.P = plan.P;
    const int TA = 16 * plan.tv, TB = 16 * plan.tv;
    const int64_t atiles = (p.nA + TA - 1) / TA;
    const int64_t btiles = (p.nB + TB - 1) / TB;
    dim3 grid((unsigned)atiles, 1, 1);
    if (EPI == EPI_TOPK) {
        // enough CTAs for ~3 waves of the SMs; each split yields k keys per row
        int64_t want = (3LL * num_sms() + atiles - 1) / atiles;
        int64_t maxsplit = 4096 / (p.k > 0 ? p.k : 1);
        if (maxsplit < 1) maxsplit = 1;
        int64_t nsplit = want < 1 ? 1 : want;
        if (nsplit > btiles) nsplit = btiles;
        if (nsplit > maxsplit) nsplit = maxsplit;
        if (nsplit < 1) nsplit = 1;
        p.btiles_per_split = (btiles + nsplit - 1) / nsplit;
        nsplit = (btiles + p.btiles_per_split - 1) / p.btiles_per_split;
        if (nsplit < 1) nsplit = 1;
        p.nsplit = (int)nsplit;
        grid.y = (unsigned)nsplit;
        if (nsplit_out) { *nsplit_out = nsplit; return VIX_OK; }   // planning pass
    }
#define VIX_LAUNCH_TV(TVV)                                                                                 \
    do {                                                                                                   \
        auto kern = pair_kernel<Spec, TVV, TVV, EPI>;                                                      \
        VIX_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)plan.smem)); \
        kern<<<grid, 256, plan.smem, ctx().stream>>>(p);                                                   \
    } while (0)
    if (plan.tv == 4) VIX_LAUNCH_TV(4);
    else if (plan.tv == 2) VIX_LAUNCH_TV(2);
    else VIX_LAUNCH_TV(1);
#undef VIX_LAUNCH_TV
    VIX_LAUNCH_CHECK();
    return VIX_OK;
}

// Fused "score + top-k" over device pointers.  Returns per-row best->worst results.
template <typename Spec>
static int pair_topk(PairArgs p, int k, int order_max, int dist_mode, float* out_score, int64_t* out_id64,
                     int32_t* out_id32) {
    p.k = k;
    p.order_max = order_max;
    int64_t nsplit = 1;
    VIX_TRY((launch_pair<Spec, EPI_TOPK>(p, k, &nsplit)));   // plan
    Scratch<u64> keys;
    VIX_TRY(keys.alloc((size_t)p.nA * nsplit * k));
    p.keys_out = keys.ptr;
    VIX_TRY((launch_pair<Spec, EPI_TOPK>(p, k)));
    return launch_merge_keys(keys.ptr, p.nA, (int)(nsplit * k), k, order_max, dist_mode, out_score, out_id64,
                             out_id32, nullptr);
}

// ------------------------------------------------------------------------------------------------
// Row-wise kernels (one thread per row)
// ------------------------------------------------------------------------------------------------
__global__ void row_norms_kernel(const float* __restrict__ x, int64_t n, int d, float* __restrict__ out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = exact_norm_l2sq(x + i * (int64_t)d, d);
}

// 1 / (sqrt(||x||^2) + 1e-12) per row: computeQueryInvNorm_impl and the on-the-fly row norm of Cosine.run
// (Cosine.swift:113-114, 186-190; Norms.l2NormSquared order)
__global__ void row_inv_norms_kernel(const float* __restrict__ x, int64_t n, int d, float* __restrict__ out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = __fdiv_rn(1.0f, fadd(__fsqrt_rn(exact_norm_l2sq(x + i * (int64_t)d, d)), 1e-12f));
}

// l2sqr_f32_block / ip_f32_block for ONE query: the query sits in shared memory, each thread owns
// a base row.  mode 0: direct L2^2 (Direct16), 1: dot-trick L2^2 (Dot16 + norms), 2: inner product.
__global__ void block_score_kernel(const float* __restrict__ q, const float* __restrict__ xb, int64_t n, int d,
                                   int mode, const float* __restrict__ xb_norm, float q_norm_in, int q_norm_given,
                                   float* __restrict__ out) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float* sq = reinterpret_cast<float*>(smem_raw);
    __shared__ float s_qn;
    for (int e = threadIdx.x; e < d; e += blockDim.x) sq[e] = q[e];
    __syncthreads();
    if (mode == 1 && threadIdx.x == 0) s_qn = q_norm_given ? q_norm_in : exact_norm_l2sq(sq, d);
    __syncthreads();
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* row = xb + i * (int64_t)d;
    if (mode == 0) {
        out[i] = exact_pair<SpecDirect16L2>(sq, row, d);
    } else if (mode == 2) {
        out[i] = exact_pair<SpecIp4>(sq, row, d);
    } else {
        float dot = exact_pair<SpecDot16>(sq, row, d);
        float xn = xb_norm ? xb_norm[i] : exact_norm_l2sq(row, d);
        float dist = fsub(fadd(s_qn, xn), fmul(2.0f, dot));
        out[i] = dist < 0.0f ? 0.0f : dist;
    }
}

int row_norms_device(const float* x, int64_t n, int d, float* out) {
    if (n == 0) return VIX_OK;
    row_norms_kernel<<<(unsigned)((n + 127) / 128), 128, 0, ctx().stream>>>(x, n, d, out);
    VIX_LAUNCH_CHECK();
    return VIX_OK;
}

// ------------------------------------------------------------------------------------------------
// Device-pointer cores used by the entry points below and by vix_index.cu
// ------------------------------------------------------------------------------------------------

// FlatIndexOptimized.fastSearchWithMicrokernels (FlatIndexOptimized.swift:390-477) for nq queries.
// raw_scores: keep kernel scores (no sqrt / negate) when true.
static int flat_search_impl(const float* q, int64_t nq, const float* xb, int64_t n, int d, int metric, int k,
                            const float* xb_norm, float* out_dist, int64_t* out_ids, bool raw_scores,
                            const uint64_t* disabled_rows);

int flat_search_device(const float* q, int64_t nq, const float* xb, int64_t n, int d, int metric, int k,
                       const float* xb_norm, float* out_dist, int64_t* out_ids, bool raw_scores) {
    return flat_search_impl(q, nq, xb, n, d, metric, k, xb_norm, out_dist, out_ids, raw_scores, nullptr);
}

// same scan with a row mask (bit b set => base row b is skipped): the pre-filter of FlatIndex.search (FlatIndex.swift:61)
int flat_search_masked_device(const float* q, int64_t nq, const float* xb, int64_t n, int d, int metric, int k,
                              const uint64_t* disabled_rows, float* out_dist, int64_t* out_ids) {
    return flat_search_impl(q, nq, xb, n, d, metric, k, nullptr, out_dist, out_ids, false, disabled_rows);
}

static int flat_search_impl(const float* q, int64_t nq, const float* xb, int64_t n, int d, int metric, int k,
                            const float* xb_norm, float* out_dist, int64_t* out_ids, bool raw_scores,
                            const uint64_t* disabled_rows) {
    if (nq == 0 || k <= 0) return VIX_OK;
    PairArgs p{};
    p.A = q; p.nA = nq; p.B = xb; p.nB = n; p.d = d; p.disabled = disabled_rows;
    if (n == 0) {
        Scratch<u64> keys;
        VIX_TRY(keys.alloc((size_t)nq));
        VIX_CUDA(cudaMemsetAsync(keys.ptr, 0xFF, (size_t)nq * 8, ctx().stream));
        return launch_merge_keys(keys.ptr, nq, 1, k, 0, 0, out_dist, out_ids, nullptr, nullptr);
    }
    if (metric == VIX_METRIC_IP) {
        p.transform = TR_NONE;
        return pair_topk<SpecIp4>(p, k, 1, raw_scores ? 0 : 2, out_dist, out_ids, nullptr);
    }
    if (metric == VIX_METRIC_COSINE) {
        // ScoreBlock.run without cached norms => Cosine.run two-pass (Cosine.swift:94-119): InnerProduct.run, then
        // (dot * qInv) * inv per row, clamped; selection .max on the similarity; API distance 1 - similarity
        Scratch<float> qi, xi;
        VIX_TRY(qi.alloc((size_t)nq));
        VIX_TRY(xi.alloc((size_t)n));
        row_inv_norms_kernel<<<(unsigned)((nq + 127) / 128), 128, 0, ctx().stream>>>(q, nq, d, qi.ptr);
        VIX_LAUNCH_CHECK();
        row_inv_norms_kernel<<<(unsigned)((n + 127) / 128), 128, 0, ctx().stream>>>(xb, n, d, xi.ptr);
        VIX_LAUNCH_CHECK();
        p.transform = TR_COSINE; p.anorm = qi.ptr; p.bnorm = xi.ptr;
        return pair_topk<SpecIp4>(p, k, 1, raw_scores ? 0 : 3, out_dist, out_ids, nullptr);
    }
    if (d >= 256 || xb_norm) {
        // dot-trick path (L2SqrKernel.swift:95-106): norms by Norms.l2NormSquared
        Scratch<float> qn, xn;
        VIX_TRY(qn.alloc((size_t)nq));
        VIX_TRY(row_norms_device(q, nq, d, qn.ptr));
        const float* xnp = xb_norm;
        if (!xnp) {
            VIX_TRY(xn.alloc((size_t)n));
            VIX_TRY(row_norms_device(xb, n, d, xn.ptr));
            xnp = xn.ptr;
        }
        p.transform = TR_DOTFUSED; p.anorm = qn.ptr; p.bnorm = xnp;
        return pair_topk<SpecDot16>(p, k, 0, raw_scores ? 0 : 1, out_dist, out_ids, nullptr);
    }
    p.transform = TR_NONE;
    return pair_topk<SpecDirect16L2>(p, k, 0, raw_scores ? 0 : 1, out_dist, out_ids, nullptr);
}

// CentroidBatchScore.swift:70-84, cosine: the block holds -<q, c>; 1 - dot qInv cInv = 1 + row qInv cInv, except where the
// near-zero-norm guard of the single-query path (IVFIndex.swift:558-561) forces the largest distance, 1.
// qn / cn = ||.||^2 by Norms.l2NormSquared; the inverse norms are 1 / (sqrt(.) + 1e-12) (IVFIndex.swift:470-485).
__global__ void cbs_cosine_epilogue_kernel(float* __restrict__ out, int64_t nq, int kc, const float* __restrict__ qn,
                                           const float* __restrict__ cn) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nq * (int64_t)kc) return;
    const int64_t qi = i / kc;
    const float qn2 = qn[qi], cn2 = cn[i - qi * kc];
    const float qinv = __fdiv_rn(1.0f, fadd(__fsqrt_rn(qn2), 1e-12f));
    const float cinv = __fdiv_rn(1.0f, fadd(__fsqrt_rn(cn2), 1e-12f));
    const float denom = __fsqrt_rn(fmul(qn2, cn2));
    out[i] = denom > 1.1920929e-07f ? fadd(1.0f, fmul(fmul(out[i], qinv), cinv)) : 1.0f;
}

int centroid_batch_score_device(const float* q, int64_t nq, const float* c, int kc, int d, int metric,
                                const float* cnorm, float* out) {
    if (nq == 0 || kc == 0) return VIX_OK;
    PairArgs p{};
    p.A = q; p.nA = nq; p.B = c; p.nB = kc; p.d = d;
    p.transform = (metric == VIX_METRIC_L2) ? TR_CBS_L2 : TR_NEG;
    p.bnorm = cnorm; p.out = out; p.ldo = kc;
    return launch_pair<SpecSeqDot, EPI_WRITE>(p, 0);
}

// the cosine block: -<q, c> in the contraction's order, then the guarded epilogue (cnorm = ||c||^2, required)
int centroid_batch_score_cosine_device(const float* q, int64_t nq, const float* c, int kc, int d, const float* cnorm,
                                       float* out) {
    if (nq == 0 || kc == 0) return VIX_OK;
    VIX_REQUIRE(nq * (int64_t)kc < (1LL << 38), VIX_ERR_UNSUPPORTED, "cosine centroid scores: block too large");
    VIX_TRY(centroid_batch_score_device(q, nq, c, kc, d, VIX_METRIC_IP, nullptr, out));
    Scratch<float> qn;
    VIX_TRY(qn.alloc((size_t)nq));
    VIX_TRY(row_norms_device(q, nq, d, qn.ptr));
    const int64_t total = nq * (int64_t)kc;
    cbs_cosine_epilogue_kernel<<<(unsigned)((total + 255) / 256), 256, 0, ctx().stream>>>(out, nq, kc, qn.ptr, cnorm);
    VIX_LAUNCH_CHECK();
    return VIX_OK;
}

// batchSearch probe stage (IVFIndex.swift:905-927): CentroidBatchScore row + ordered prefix.
// Outputs [nq x nprobe] padded with -1 / NaN beyond min(nprobe, kc).
// the selections below carry their scores in keys (make_key: -0 folded into +0); put back the sign of the zero scores
__global__ void probe_zero_sign_kernel(const int32_t* __restrict__ idx, float* __restrict__ scores, int64_t n, int metric,
                                       const float* __restrict__ cnorm) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && idx[i] >= 0) scores[i] = cbs_signed_zero(scores[i], (uint32_t)idx[i], metric, cnorm);
}

static int probe_select_keys(const float* q, int64_t nq, const float* c, int kc, int d, int metric, int nprobe,
                             const float* cnorm, const uint64_t* disabled, int32_t* out_idx, float* out_scores);

int probe_select_device(const float* q, int64_t nq, const float* c, int kc, int d, int metric, int nprobe,
                        const float* cnorm, const uint64_t* disabled, int32_t* out_idx, float* out_scores) {
    if (nq == 0 || nprobe <= 0) return VIX_OK;
    VIX_TRY(probe_select_keys(q, nq, c, kc, d, metric, nprobe, cnorm, disabled, out_idx, out_scores));
    if (out_scores) {
        const int64_t n = nq * (int64_t)nprobe;
        probe_zero_sign_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx().stream>>>(out_idx, out_scores, n, metric, cnorm);
        VIX_LAUNCH_CHECK();
    }
    return VIX_OK;
}

static int probe_select_keys(const float* q, int64_t nq, const float* c, int kc, int d, int metric, int nprobe,
                             const float* cnorm, const uint64_t* disabled, int32_t* out_idx, float* out_scores) {
    TilePlan plan;
    if (!plan_tile(d, EPI_TOPK, nprobe, &plan)) {
        // rows too long for the tiled engine: the CentroidBatchScore block of a tile of queries, then the ordered prefix
        int64_t tile = (64LL << 20) / kc;
        tile = tile < 1 ? 1 : (tile > nq ? nq : tile);
        Scratch<float> scores;
        VIX_TRY(scores.alloc((size_t)tile * kc));
        for (int64_t b = 0; b < nq; b += tile) {
            const int64_t cnt = nq - b < tile ? nq - b : tile;
            VIX_TRY(centroid_batch_score_device(q + (size_t)b * d, cnt, c, kc, d, metric, cnorm, scores.ptr));
            VIX_TRY(row_select_device(scores.ptr, cnt, kc, nprobe, disabled, out_idx + (size_t)b * nprobe,
                                      out_scores ? out_scores + (size_t)b * nprobe : nullptr));
        }
        return VIX_OK;
    }
    PairArgs p{};
    p.A = q; p.nA = nq; p.B = c; p.nB = kc; p.d = d;
    p.transform = (metric == VIX_METRIC_L2) ? TR_CBS_L2 : TR_NEG;
    p.bnorm = cnorm; p.disabled = disabled;
    return pair_topk<SpecSeqDot>(p, nprobe, 0, 0, out_scores, nullptr, out_idx);
}

int ivf_assign_device(const float* x, int64_t n, int d, const float* c, int kc, int32_t* assign, float* dist) {
    if (n == 0) return VIX_OK;
    PairArgs p{};
    p.A = x; p.nA = n; p.B = c; p.nB = kc; p.d = d;
    p.transform = TR_NONE; p.arg_out = assign; p.min_out = dist;
    return launch_pair<SpecKm12L2, EPI_ARGMIN>(p, 0);
}

int ivf_assign_metric_device(const float* x, int64_t n, int d, const float* c, int kc, int metric,
                             const float* cnorm, int32_t* assign) {
    if (n == 0) return VIX_OK;
    PairArgs p{};
    p.A = x; p.nA = n; p.B = c; p.nB = kc; p.d = d;
    p.transform = (metric == VIX_METRIC_L2) ? TR_CBS_L2 : TR_NEG;
    p.bnorm = cnorm; p.arg_out = assign; p.first_min = 1;
    return launch_pair<SpecSeqDot, EPI_ARGMIN>(p, 0);
}

// ------------------------------------------------------------------------------------------------
// Kernel #40 exact re-rank (Operations/Rerank/ExactRerank.swift:698-814), DenseArray backend: one CTA per
// query scores its C candidate rows with the reference kernel (L2Sqr.run: direct for d < 256 without norms,
// fused dot form otherwise; InnerProduct.run), skips missing ids (skipMissing), selects the K best by
// (score per the metric's ordering, then smaller candidate id) and pads with the sentinel / id -1.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
rerank_kernel(const float* __restrict__ Q, int d, int metric, const int64_t* __restrict__ cand, int C, int K,
              const float* __restrict__ xb, int64_t N, const float* __restrict__ xnorm, int dotfused, int P,
              float* __restrict__ out_scores, int64_t* __restrict__ out_ids) {
    extern __shared__ __align__(16) unsigned char smem_rr[];
    u64* keys = reinterpret_cast<u64*>(smem_rr);
    float* sq = reinterpret_cast<float*>(keys + P);
    __shared__ float s_qn;
    const int64_t row = blockIdx.x;
    const int order_max = (metric == VIX_METRIC_IP);
    for (int e = threadIdx.x; e < d; e += blockDim.x) sq[e] = Q[row * d + e];
    for (int i = threadIdx.x; i < P; i += blockDim.x) keys[i] = kEmptyKey;
    __syncthreads();
    if (threadIdx.x == 0) {
        // ||q||^2: with caller-supplied base norms the re-rank passes its own sequential sum (ExactRerank.swift:243, 276);
        // otherwise L2Sqr.run computes Norms.l2NormSquared itself (L2SqrKernel.swift:95-106)
        float qn = 0.0f;
        if (!order_max && dotfused) {
            if (xnorm) for (int e = 0; e < d; ++e) qn = fadd(qn, fmul(sq[e], sq[e]));
            else qn = exact_norm_l2sq(sq, d);
        }
        s_qn = qn;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < C; i += blockDim.x) {
        const int64_t id = cand[row * C + i];
        if (id < 0 || id >= N) continue;                                  // missing row
        const float* xr = xb + id * d;
        float s;
        if (order_max) s = exact_pair<SpecIp4>(sq, xr, d);
        else if (dotfused) {
            const float dot = exact_pair<SpecDot16>(sq, xr, d);
            const float xn = xnorm ? xnorm[id] : exact_norm_l2sq(xr, d);
            const float dist = fsub(fadd(s_qn, xn), fmul(2.0f, dot));
            s = dist < 0.0f ? 0.0f : dist;
        } else s = exact_pair<SpecDirect16L2>(sq, xr, d);
        keys[i] = make_key(s, (uint32_t)id, order_max);
    }
    __syncthreads();
    bitonic_sort_keys<false>(keys, P, threadIdx.x, blockDim.x);
    for (int i = threadIdx.x; i < K; i += blockDim.x) {
        const u64 key = (i < P) ? keys[i] : kEmptyKey;
        const size_t o = (size_t)row * K + i;
        if (key == kEmptyKey) { out_scores[o] = order_max ? -INFINITY : INFINITY; out_ids[o] = -1; }
        else { out_scores[o] = key_score(key, order_max); out_ids[o] = (int64_t)key_id(key); }
    }
}

__global__ void narrow_ids_kernel(const int64_t* __restrict__ in, int32_t* __restrict__ out, int64_t n) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (int32_t)in[i];
}

// ------------------------------------------------------------------------------------------------
// selectTopK (Operations/Selection/TopK.swift:127-164) over a score array: each CTA selects the k
// best of its chunk with a shared-memory queue, merge_keys_kernel merges the chunks.  ids are int32
// (TopK.swift:59); they are biased by 0x80000000 inside the key so that "smaller id" is the signed
// order.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
select_chunk_kernel(const float* __restrict__ scores, const int32_t* __restrict__ ids, int64_t n, int64_t chunk,
                    int k, int P, int order_max, u64* __restrict__ keys_out) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int s_cnt;
    __shared__ u64 s_thr;
    BlockQueue q{reinterpret_cast<u64*>(smem_raw), &s_cnt, &s_thr, k, P};
    q.init();
    const int64_t b = (int64_t)blockIdx.x * chunk;
    const int64_t e = min(n, b + chunk);
    for (int64_t base = b; base < e; base += blockDim.x) {
        q.flush_if_needed(blockDim.x);
        const int64_t i = base + threadIdx.x;
        if (i < e) {
            const int32_t id = ids ? ids[i] : (int32_t)i;
            q.push(make_key(scores[i], (uint32_t)id ^ 0x80000000u, order_max));
        }
    }
    q.flush();
    for (int i = threadIdx.x; i < k; i += blockDim.x) keys_out[(size_t)blockIdx.x * k + i] = q.keys[i];
}

int select_topk_device(const float* scores, const int32_t* ids, int64_t n, int k, int ordering,
                       float* out_scores, int32_t* out_ids, int* out_count) {
    const int P = next_pow2(k + 256);
    int64_t nchunks = (n + 16383) / 16384;
    const int64_t maxchunks = 4096 / k > 0 ? 4096 / k : 1;
    if (nchunks > maxchunks) nchunks = maxchunks;
    if (nchunks < 1) nchunks = 1;
    const int64_t chunk = (n + nchunks - 1) / nchunks;
    nchunks = (n + chunk - 1) / chunk;
    Scratch<u64> keys;
    VIX_TRY(keys.alloc((size_t)nchunks * k));
    select_chunk_kernel<<<(unsigned)nchunks, 256, (size_t)P * 8, ctx().stream>>>(scores, ids, n, chunk, k, P,
                                                                                ordering == VIX_ORDER_MAX, keys.ptr);
    VIX_LAUNCH_CHECK();
    return launch_merge_keys(keys.ptr, 1, (int)(nchunks * k), k, ordering == VIX_ORDER_MAX, 0, out_scores, nullptr,
                             out_ids, out_count, 0x80000000u);
}

// ------------------------------------------------------------------------------------------------
// mergeTopK (Operations/Selection/TopKMerge.swift:11-61) for `batch` rows of nlists best->worst lists.
// (score, id) is a total order, so merging == selecting the k smallest keys of the union; exact
// duplicates (same score, same id) are indistinguishable in the output, which makes the reference's
// "smaller list index" rule unobservable.
// ------------------------------------------------------------------------------------------------
__global__ void lists_to_keys_kernel(const float* __restrict__ scores, const int64_t* __restrict__ ids,
                                     const int32_t* __restrict__ lens, int64_t batch, int nlists, int stride,
                                     int order_max, u64* __restrict__ keys) {
    const int64_t total = batch * nlists * stride;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t bl = e / stride;
        const int i = (int)(e - bl * stride);
        const int len = lens ? lens[bl] : stride;
        u64 key = kEmptyKey;
        if (i < len && ids[e] >= 0) key = make_key(scores[e], (uint32_t)ids[e], order_max);
        keys[e] = key;
    }
}

int merge_lists_device(const float* scores, const int64_t* ids, const int32_t* lens, int64_t batch, int nlists,
                       int stride, int k, int order_max, int dist_mode, float* out_scores, int64_t* out_ids) {
    if (batch == 0 || k <= 0) return VIX_OK;
    const int64_t total = batch * nlists * stride;
    Scratch<u64> keys;
    VIX_TRY(keys.alloc((size_t)(total > 0 ? total : 1)));
    if (total > 0) {
        int64_t blocks = (total + 255) / 256;
        if (blocks > 65535) blocks = 65535;
        lists_to_keys_kernel<<<(unsigned)blocks, 256, 0, ctx().stream>>>(scores, ids, lens, batch, nlists, stride,
                                                                        order_max, keys.ptr);
        VIX_LAUNCH_CHECK();
    }
    return launch_merge_keys(keys.ptr, batch, nlists * stride, k, order_max, dist_mode, out_scores, out_ids, nullptr,
                             nullptr);
}

}  // namespace vix

using namespace vix;

extern "C" {

int vix_l2sqr_f32_block(const float* q, const float* xb, int64_t n, int d, float* out, const float* xb_norm,
                        float q_norm) {
    VIX_TRY(ensure_device());
    // @_cdecl l2sqr_f32_block silently returns on null pointers (CABIBridge.swift:13)
    VIX_REQUIRE(q && xb && out, VIX_ERR_NULL_PTR, "vix_l2sqr_f32_block: null pointer");
    VIX_REQUIRE(d > 0 && n >= 0, VIX_ERR_INVALID_DIM, "vix_l2sqr_f32_block: bad n/d");
    if (n == 0) return VIX_OK;
    In<float> dq, dx, dn;
    Out<float> dout;
    VIX_TRY(dq.stage(q, (size_t)d));
    VIX_TRY(dx.stage(xb, (size_t)n * d));
    VIX_TRY(dn.stage(xb_norm, xb_norm ? (size_t)n : 0));
    VIX_TRY(dout.stage(out, (size_t)n));
    const bool qn_given = !(q_norm != q_norm);
    const bool use_dot = xb_norm != nullptr || qn_given || d >= 256;   // L2SqrKernel.swift:95-106
    block_score_kernel<<<(unsigned)((n + 127) / 128), 128, (size_t)d * 4, ctx().stream>>>(
        dq.dev, dx.dev, n, d, use_dot ? 1 : 0, dn.dev, q_norm, qn_given ? 1 : 0, dout.dev);
    VIX_LAUNCH_CHECK();
    VIX_TRY(dout.commit());
    return finish(dout.is_host());
}

int vix_ip_f32_block(const float* q, const float* xb, int64_t n, int d, float* out) {
    VIX_TRY(ensure_device());
    VIX_REQUIRE(q && xb && out, VIX_ERR_NULL_PTR, "vix_ip_f32_block: null pointer");
    VIX_REQUIRE(d >= 0 && n >= 0, VIX_ERR_INVALID_DIM, "vix_ip_f32_block: bad n/d");
    if (n == 0) return VIX_OK;
    In<float> dq, dx;
    Out<float> dout;
    VIX_TRY(dq.stage(q, (size_t)d));
    VIX_TRY(dx.stage(xb, (size_t)n * d));
    VIX_TRY(dout.stage(out, (size_t)n));
    block_score_kernel<<<(unsigned)((n + 127) / 128), 128, (size_t)(d > 0 ? d : 1) * 4, ctx().stream>>>(
        dq.dev, dx.dev, n, d, 2, nullptr, 0.0f, 0, dout.dev);
    VIX_LAUNCH_CHECK();
    VIX_TRY(dout.commit());
    return finish(dout.is_host());
}

int vix_row_norms_f32(const float* x, int64_t n, int d, float* out) {
    VIX_TRY(ensure_device());
    VIX_REQUIRE(x && out, VIX_ERR_NULL_PTR, "vix_row_norms_f32: null pointer");
    VIX_REQUIRE(d >= 0 && n >= 0, VIX_ERR_INVALID_DIM, "vix_row_norms_f32: bad n/d");
    In<float> dx;
    Out<float> dout;
    VIX_TRY(dx.stage(x, (size_t)n * d));
    VIX_TRY(dout.stage(out, (size_t)n));
    VIX_TRY(row_norms_device(dx.dev, n, d, dout.dev));
    VIX_TRY(dout.commit());
    return finish(dout.is_host());
}

int vix_flat_search_f32(const float* queries, int64_t nq, const float* xb, int64_t n, int d, int metric, int k,
                        float* out_dist, int64_t* out_ids) {
    VIX_TRY(ensure_device());
    if (k <= 0 || nq == 0) return VIX_OK;   // k <= 0 => [] (IVFIndex.swift:787; FlatIndex.swift:57)
    VIX_REQUIRE(queries && out_dist && out_ids && (xb || n == 0), VIX_ERR_NULL_PTR, "vix_flat_search_f32: null pointer");
    VIX_REQUIRE(d > 0 && n >= 0 && nq >= 0, VIX_ERR_INVALID_DIM, "vix_flat_search_f32: bad shape");
    VIX_REQUIRE(metric == VIX_METRIC_L2 || metric == VIX_METRIC_IP || metric == VIX_METRIC_COSINE, VIX_ERR_INVALID_PARAM,
                "vix_flat_search_f32: metric");
    VIX_REQUIRE(k <= VIX_MAX_K, VIX_ERR_INVALID_K, "vix_flat_search_f32: k > %d", VIX_MAX_K);
    VIX_REQUIRE(n < (1LL << 32) - 1, VIX_ERR_INVALID_PARAM, "vix_flat_search_f32: n must be < 2^32 - 1");
    In<float> dq, dx;
    Out<float> dd;
    Out<int64_t> di;
    VIX_TRY(dq.stage(queries, (size_t)nq * d));
    VIX_TRY(dx.stage(xb, (size_t)n * d));
    VIX_TRY(dd.stage(out_dist, (size_t)nq * k));
    VIX_TRY(di.stage(out_ids, (size_t)nq * k));
    VIX_TRY(flat_search_auto_device(dq.dev, nq, dx.dev, n, d, metric, k, nullptr, dd.dev, di.dev, false));   // tensor-core shortlist + exact rescoring
    VIX_TRY(dd.commit());
    VIX_TRY(di.commit());
    return finish(dd.is_host() || di.is_host());
}

int vix_accel_rank_candidates_f32(const float* queries, int64_t nq, const float* candidates, int64_t c, int d,
                                  int metric, int k, int32_t* out_indices, float* out_distances) {
    VIX_TRY(ensure_device());
    if (k <= 0 || nq == 0) return VIX_OK;
    VIX_REQUIRE(queries && out_indices && out_distances && (candidates || c == 0), VIX_ERR_NULL_PTR,
                "vix_accel_rank_candidates_f32: null pointer");
    VIX_REQUIRE(d > 0 && c >= 0, VIX_ERR_INVALID_DIM, "vix_accel_rank_candidates_f32: bad shape");
    VIX_REQUIRE(k <= VIX_MAX_K, VIX_ERR_INVALID_K, "vix_accel_rank_candidates_f32: k > %d", VIX_MAX_K);
    VIX_REQUIRE(c < (1LL << 31), VIX_ERR_INVALID_PARAM, "vix_accel_rank_candidates_f32: c must fit int32");
    In<float> dq, dx;
    Out<float> dd;
    Out<int32_t> di;
    Scratch<int64_t> id64;
    VIX_TRY(dq.stage(queries, (size_t)nq * d));
    VIX_TRY(dx.stage(candidates, (size_t)c * d));
    VIX_TRY(dd.stage(out_distances, (size_t)nq * k));
    VIX_TRY(di.stage(out_indices, (size_t)nq * k));
    VIX_TRY(id64.alloc((size_t)nq * k));
    VIX_TRY(flat_search_auto_device(dq.dev, nq, dx.dev, c, d, metric, k, nullptr, dd.dev, id64.ptr, false));
    // narrow ids to int32 (AcceleratedResults.indices, AccelerableIndex.swift:60-75)
    {
        int64_t total = nq * (int64_t)k;
        narrow_ids_kernel<<<(unsigned)((total + 255) / 256), 256, 0, ctx().stream>>>(id64.ptr, di.dev, total);
        VIX_LAUNCH_CHECK();
    }
    VIX_TRY(dd.commit());
    VIX_TRY(di.commit());
    return finish(true);
}

int vix_rerank_exact_topk_f32(const float* queries, int64_t nq, int d, int metric, const int64_t* cand_ids, int C, int K,
                              const float* xb, int64_t N, const float* xb_sq_norms, float* top_scores, int64_t* top_ids) {
    VIX_TRY(ensure_device());
    if (nq <= 0 || K <= 0) return VIX_OK;
    VIX_REQUIRE(queries && cand_ids && xb && top_scores && top_ids, VIX_ERR_NULL_PTR, "vix_rerank_exact_topk_f32: null pointer");
    VIX_REQUIRE(d > 0 && N >= 0, VIX_ERR_INVALID_DIM, "vix_rerank_exact_topk_f32: bad shape");
    VIX_REQUIRE(metric == VIX_METRIC_L2 || metric == VIX_METRIC_IP, VIX_ERR_INVALID_PARAM, "vix_rerank_exact_topk_f32: metric");
    VIX_REQUIRE(K <= C, VIX_ERR_INVALID_K, "vix_rerank_exact_topk_f32: K must be <= C (ExactRerank.swift:730)");
    VIX_REQUIRE(C <= 16384, VIX_ERR_UNSUPPORTED, "vix_rerank_exact_topk_f32: at most 16384 candidates per query");
    VIX_REQUIRE(N < 0xFFFFFFFFLL, VIX_ERR_INVALID_PARAM, "vix_rerank_exact_topk_f32: N must be < 2^32 - 1");
    In<float> dq, dx, dn;
    In<int64_t> dc;
    Out<float> ds;
    Out<int64_t> di;
    VIX_TRY(dq.stage(queries, (size_t)nq * d));
    VIX_TRY(dc.stage(cand_ids, (size_t)nq * C));
    VIX_TRY(dx.stage(xb, (size_t)N * d));
    VIX_TRY(dn.stage(xb_sq_norms, xb_sq_norms ? (size_t)N : 0));
    VIX_TRY(ds.stage(top_scores, (size_t)nq * K));
    VIX_TRY(di.stage(top_ids, (size_t)nq * K));
    const int P = next_pow2(C < 2 ? 2 : C);
    const size_t smem = (size_t)P * 8 + (size_t)d * 4;
    VIX_REQUIRE(smem <= 200 * 1024, VIX_ERR_UNSUPPORTED, "vix_rerank_exact_topk_f32: C = %d, d = %d exceed shared memory", C, d);
    VIX_CUDA(cudaFuncSetAttribute(rerank_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int dotfused = (xb_sq_norms != nullptr || d >= 256) ? 1 : 0;       // L2SqrKernel.swift:95-106
    rerank_kernel<<<(unsigned)nq, 256, smem, ctx().stream>>>(dq.dev, d, metric, dc.dev, C, K, dx.dev, N, dn.dev, dotfused, P, ds.dev,
                                                            di.dev);
    VIX_LAUNCH_CHECK();
    VIX_TRY(ds.commit());
    VIX_TRY(di.commit());
    return finish(ds.is_host() || di.is_host());
}

int vix_select_topk_f32(const float* scores, const int32_t* ids, int64_t n, int k, int ordering,
                        float* out_scores, int32_t* out_ids, int* out_count) {
    VIX_TRY(ensure_device());
    if (out_count && !is_device_ptr(out_count)) *out_count = 0;
    if (k <= 0 || n <= 0) return VIX_OK;
    VIX_REQUIRE(scores && out_scores && out_ids, VIX_ERR_NULL_PTR, "vix_select_topk_f32: null pointer");
    VIX_REQUIRE(k <= VIX_MAX_K, VIX_ERR_INVALID_K, "vix_select_topk_f32: k > %d", VIX_MAX_K);
    In<float> ds;
    In<int32_t> dids;
    Out<float> dos;
    Out<int32_t> doi;
    Out<int> dcnt;
    VIX_TRY(ds.stage(scores, (size_t)n));
    VIX_TRY(dids.stage(ids, ids ? (size_t)n : 0));
    const int keff = (int)(k < n ? k : n);
    VIX_TRY(dos.stage(out_scores, (size_t)keff));
    VIX_TRY(doi.stage(out_ids, (size_t)keff));
    VIX_TRY(dcnt.stage(out_count, out_count ? 1 : 0));
    VIX_TRY(select_topk_device(ds.dev, dids.dev, n, keff, ordering, dos.dev, doi.dev, dcnt.dev));
    VIX_TRY(dos.commit());
    VIX_TRY(doi.commit());
    VIX_TRY(dcnt.commit());
    return finish(true);
}

int vix_merge_topk_f32(const float* scores, const int64_t* ids, const int32_t* lens, int64_t batch, int nlists,
                       int list_stride, int k, int ordering, float* out_scores, int64_t* out_ids) {
    VIX_TRY(ensure_device());
    if (k <= 0 || batch <= 0) return VIX_OK;
    VIX_REQUIRE(out_scores && out_ids, VIX_ERR_NULL_PTR, "vix_merge_topk_f32: null output");
    VIX_REQUIRE(nlists >= 0 && list_stride >= 0, VIX_ERR_INVALID_PARAM, "vix_merge_topk_f32: bad shape");
    VIX_REQUIRE((scores && ids) || nlists * list_stride == 0, VIX_ERR_NULL_PTR, "vix_merge_topk_f32: null input");
    VIX_REQUIRE(k <= VIX_MAX_K, VIX_ERR_INVALID_K, "vix_merge_topk_f32: k > %d", VIX_MAX_K);
    const size_t total = (size_t)batch * nlists * list_stride;
    In<float> ds;
    In<int64_t> di;
    In<int32_t> dl;
    Out<float> dos;
    Out<int64_t> doi;
    VIX_TRY(ds.stage(scores, total));
    VIX_TRY(di.stage(ids, total));
    VIX_TRY(dl.stage(lens, lens ? (size_t)batch * nlists : 0));
    VIX_TRY(dos.stage(out_scores, (size_t)batch * k));
    VIX_TRY(doi.stage(out_ids, (size_t)batch * k));
    VIX_TRY(merge_lists_device(ds.dev, di.dev, dl.dev, batch, nlists, list_stride, k, ordering == VIX_ORDER_MAX, 0,
                               dos.dev, doi.dev));
    VIX_TRY(dos.commit());
    VIX_TRY(doi.commit());
    return finish(dos.is_host() || doi.is_host());
}

int vix_centroid_batch_score_f32(const float* queries, int64_t q, const float* centroids, int kc, int d, int metric,
                                 const float* centroid_norms, float* out) {
    VIX_TRY(ensure_device());
    VIX_REQUIRE(queries && centroids && out, VIX_ERR_NULL_PTR, "vix_centroid_batch_score_f32: null pointer");
    VIX_REQUIRE(d > 0 && kc > 0 && q >= 0, VIX_ERR_INVALID_DIM, "vix_centroid_batch_score_f32: bad shape");
    VIX_REQUIRE(metric == VIX_METRIC_L2 || metric == VIX_METRIC_IP || metric == VIX_METRIC_COSINE, VIX_ERR_INVALID_PARAM,
                "vix_centroid_batch_score_f32: metric");
    if (q == 0) return VIX_OK;
    In<float> dq, dc, dn;
    Out<float> dout;
    Scratch<float> cn;
    VIX_TRY(dq.stage(queries, (size_t)q * d));
    VIX_TRY(dc.stage(centroids, (size_t)kc * d));
    VIX_TRY(dout.stage(out, (size_t)q * kc));
    const float* cnp = nullptr;
    if (metric != VIX_METRIC_IP) {
        if (centroid_norms) { VIX_TRY(dn.stage(centroid_norms, (size_t)kc)); cnp = dn.dev; }
        else { VIX_TRY(cn.alloc((size_t)kc)); VIX_TRY(row_norms_device(dc.dev, kc, d, cn.ptr)); cnp = cn.ptr; }
    }
    if (metric == VIX_METRIC_COSINE) {
        VIX_TRY(centroid_batch_score_cosine_device(dq.dev, q, dc.dev, kc, d, cnp, dout.dev));
    } else {
        VIX_TRY(centroid_batch_score_device(dq.dev, q, dc.dev, kc, d, metric, cnp, dout.dev));
    }
    VIX_TRY(dout.commit());
    return finish(dout.is_host());
}

int vix_ivf_select_nprobe_batch_f32(const float* Q, int64_t b, int d, const float* centroids, int kc, int metric,
                                    int nprobe, const float* centroid_norms, const uint64_t* disabled_lists,
                                    int32_t* list_ids_out, float* list_scores_out) {
    VIX_TRY(ensure_device());
    VIX_REQUIRE(Q && centroids && list_ids_out, VIX_ERR_NULL_PTR, "vix_ivf_select_nprobe_batch_f32: null pointer");
    VIX_REQUIRE(d > 0 && kc > 0 && b >= 0, VIX_ERR_INVALID_DIM, "vix_ivf_select_nprobe_batch_f32: bad shape");
    VIX_REQUIRE(nprobe > 0 && nprobe <= VIX_MAX_K, VIX_ERR_INVALID_K, "vix_ivf_select_nprobe_batch_f32: nprobe");
    VIX_REQUIRE(metric == VIX_METRIC_L2 || metric == VIX_METRIC_IP, VIX_ERR_INVALID_PARAM, "metric");
    if (b == 0) return VIX_OK;
    In<float> dq, dc, dn;
    In<uint64_t> dmask;
    Out<int32_t> dids;
    Out<float> dsc;
    Scratch<float> cn;
    VIX_TRY(dq.stage(Q, (size_t)b * d));
    VIX_TRY(dc.stage(centroids, (size_t)kc * d));
    VIX_TRY(dmask.stage(disabled_lists, disabled_lists ? (size_t)((kc + 63) / 64) : 0));
    VIX_TRY(dids.stage(list_ids_out, (size_t)b * nprobe));
    VIX_TRY(dsc.stage(list_scores_out, list_scores_out ? (size_t)b * nprobe : 0));
    const float* cnp = nullptr;
    if (metric == VIX_METRIC_L2) {
        if (centroid_norms) { VIX_TRY(dn.stage(centroid_norms, (size_t)kc)); cnp = dn.dev; }
        else { VIX_TRY(cn.alloc((size_t)kc)); VIX_TRY(row_norms_device(dc.dev, kc, d, cn.ptr)); cnp = cn.ptr; }
    }
    // no list mask: tensor-core shortlist + exact rescoring (vix_gemm.cu; identical results); else the exact kernel
    if (dmask.dev == nullptr) VIX_TRY(probe_select_fast_device(dq.dev, b, dc.dev, kc, d, metric, nprobe, cnp, dids.dev, dsc.dev, nullptr));
    else VIX_TRY(probe_select_device(dq.dev, b, dc.dev, kc, d, metric, nprobe, cnp, dmask.dev, dids.dev, dsc.dev));
    VIX_TRY(dids.commit());
    VIX_TRY(dsc.commit());
    return finish(true);
}

int vix_ivf_assign_f32(const float* x, int64_t n, int d, const float* centroids, int kc, int32_t* assign_out,
                       float* dist_out) {
    VIX_TRY(ensure_device());
    VIX_REQUIRE(x && centroids && assign_out, VIX_ERR_NULL_PTR, "vix_ivf_assign_f32: null pointer");
    VIX_REQUIRE(d > 0 && n >= 0, VIX_ERR_INVALID_DIM, "vix_ivf_assign_f32: bad shape");
    VIX_REQUIRE(kc > 0, VIX_ERR_INVALID_K, "vix_ivf_assign_f32: kc must be > 0");
    if (n == 0) return VIX_OK;
    In<float> dx, dc;
    Out<int32_t> da;
    Out<float> dd;
    VIX_TRY(dx.stage(x, (size_t)n * d));
    VIX_TRY(dc.stage(centroids, (size_t)kc * d));
    VIX_TRY(da.stage(assign_out, (size_t)n));
    VIX_TRY(dd.stage(dist_out, dist_out ? (size_t)n : 0));
    VIX_TRY(ivf_assign_auto_device(dx.dev, n, d, dc.dev, kc, da.dev, dd.dev));   // tensor-core shortlist + exact rescoring
    VIX_TRY(da.commit());
    VIX_TRY(dd.commit());
    return finish(true);
}

int vix_ivf_assign_metric_f32(const float* x, int64_t n, int d, const float* centroids, int kc, int metric,
                              const float* centroid_norms, int32_t* assign_out) {
    VIX_TRY(ensure_device());
    VIX_REQUIRE(x && centroids && assign_out, VIX_ERR_NULL_PTR, "vix_ivf_assign_metric_f32: null pointer");
    VIX_REQUIRE(d > 0 && n >= 0, VIX_ERR_INVALID_DIM, "vix_ivf_assign_metric_f32: bad shape");
    VIX_REQUIRE(kc > 0, VIX_ERR_INVALID_K, "vix_ivf_assign_metric_f32: kc must be > 0");
    VIX_REQUIRE(metric == VIX_METRIC_L2 || metric == VIX_METRIC_IP, VIX_ERR_INVALID_PARAM, "metric");
    if (n == 0) return VIX_OK;
    In<float> dx, dc, dn;
    Out<int32_t> da;
    Scratch<float> cn;
    VIX_TRY(dx.stage(x, (size_t)n * d));
    VIX_TRY(dc.stage(centroids, (size_t)kc * d));
    VIX_TRY(da.stage(assign_out, (size_t)n));
    const float* cnp = nullptr;
    if (metric == VIX_METRIC_L2) {
        if (centroid_norms) { VIX_TRY(dn.stage(centroid_norms, (size_t)kc)); cnp = dn.dev; }
        else { VIX_TRY(cn.alloc((size_t)kc)); VIX_TRY(row_norms_device(dc.dev, kc, d, cn.ptr)); cnp = cn.ptr; }
    }
    VIX_TRY(ivf_assign_metric_device(dx.dev, n, d, dc.dev, kc, metric, cnp, da.dev));
    VIX_TRY(da.commit());
    return finish(true);
}

}  // extern "C"
