/*
 * vindex_cuda.h -- C ABI of libvindex_b200: the B200-native (sm_100a) implementation of
 * gifton/VectorIndex's batched search hot path.
 *
 * Conventions (same as the reference's C module Sources/CPQEncode/include/cpq_encode.h and its
 * @_cdecl exports Sources/VectorIndex/Operations/Scoring/CABIBridge.swift:5-30):
 *   - plain C, caller-owned row-major buffers, `int64_t n`, `int d, m, ks`, nullable option structs;
 *   - every pointer may be a HOST pointer or a CUDA DEVICE pointer (detected per call).  Host inputs
 *     are copied to HBM, host outputs are copied back and the call returns after they are valid;
 *   - new entry points return an int status: 0 = ok, negative = error.  The first five codes are the
 *     reference's KMeansMBStatus (Sources/VectorIndex/Kernels/KMeansMiniBatchKernel.swift:131-138);
 *     nothing aborts; vix_last_error() describes the failure;
 *   - there is NO CPU fallback: without a usable CUDA device every entry point returns
 *     VIX_ERR_NO_DEVICE;
 *   - thread-safe: stateless entry points are re-entrant; an index handle serialises the HOST side of its calls
 *     (a mutex per handle: one add / search enqueues at a time, the reference's actor isolation, IVFIndex.swift:13).
 *     Device work of calls issued from different threads is ordered only by their streams: every search owns its
 *     work queue and scratch (stream-ordered allocations), so concurrent asynchronous searches of one handle on
 *     different streams are independent; a call that CHANGES the handle (add, remove, train, set_*, clear, the lazy list
 *     rebuild of the first search after an add or a removal) must not overlap other calls still running on another
 *     stream -- synchronise (vix_synchronize) before it;
 *   - ids live in [0, 2^32 - 1) (the reference's top-k id type is Int32, TopK.swift:59), checked for host AND device
 *     id arrays; adding an id that is already stored APPENDS a second row (the reference's Dictionary store replaces,
 *     IVFIndex.swift:42): callers that need replacement call vix_index_remove with the id, then add the new row;
 *     duplicates are returned as separate results;
 *   - list ids (assignments handed to vix_index_add_encoded, probe lists handed to *_with_probes*) outside [0, kc) are
 *     rejected (assignments) or skipped like the -1 padding (probes); rows whose scores are all NaN get no list:
 *     IVF_FLAT keeps them unreachable as the reference does (IVFIndex.swift:376-435 "guard best >= 0"), IVF_PQ add fails.
 *
 * Environment switches (tests, A/B measurements and diagnostics; none is needed in production, none changes a result):
 *   VIX_TC_SCAN=0 | 1        never / whenever the shape allows take the list-major tensor-core IVF-PQ scan (default: L2,
 *                            d = 2 m, ks = 256, nq x nprobe >= 32768)
 *   VIX_TC_SCAN_DEBUG=1      per launch (synchronises): queries handed back, finalists per query
 *   VIX_TC_SCAN_TIMES=1      CUDA events between the stages of every list-major launch, summed, printed at exit
 *   VIX_SCAN_DEBUG=1         per query-major IVF-PQ scan launch (no synchronisation), one stderr line "[vix scan] ...": the
 *                            kernel (fast G = m / 16, or generic), filter and stats instantiation, warps, Pw, P2, the
 *                            table source (image: batch-wide lut_image_kernel; kernel: built in the scan), the bias source
 *                            (kernel: in the scan; rows: probe_bias_rows_kernel; pairs: probe_bias_kernel; given: by the
 *                            list-major scan), the locality order (yes / no) and the work items (query count, or device:
 *                            the queries the list-major scan hands back); and per vix_index_range_search call one line
 *                            "[vix range] kind K, kernel fast G n | generic | ivfflat | flat, filter 0|1, passes 1|2, total T,
 *                            max_row M, sorted_long L" (L: rows longer than the in-shared-memory sort, merged in global memory);
 *                            and per vix_sharded_range_search call and rank (world > 1) one line "[vix sharded range] world W,
 *                            peer 0|1, local T_r, total T, max_row M, grown 0|1" (T_r: this rank's entries, M: the longest
 *                            merged row, grown: the range region of the communicator was (re)allocated by the call); and
 *                            per vix_sharded_search / _filtered call with k > VIX_MAX_K and rank (world > 1) one line
 *                            "[vix sharded knn] world W, peer 0|1, k K, seed S_r, local T_r, sent X_r, total T, max_row M,
 *                            grown 0|1" (S_r: this rank's seed entries, T_r: its collected entries, X_r: those left after
 *                            each row is cut at k, T: the merged entries before the cut at k)
 *   VIX_DISABLE_TC, VIX_DISABLE_PQ_TC, VIX_DISABLE_LUT_IMAGE
 *                            exact CUDA-core kernels instead of the tensor-core shortlists / per-query tables built inside
 *                            the scan instead of batch-wide (the parity tests compare both ways)
 *   VIX_NO_P2P=1             vix_sharded_* / vix_replicated_*: NCCL all-gathers instead of peer memory; VIX_NCCL_PATH: the libnccl to dlopen
 *
 * Each declaration cites the reference interface it replaces (paths relative to
 * /root/reference/Sources/VectorIndex unless another root is given).
 */
#ifndef VINDEX_CUDA_H
#define VINDEX_CUDA_H

#include <stdbool.h>
#include <stddef.h>
#include <stdint.h>

#include "cpq_encode.h"

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------------------------------------ */
/* Status, metrics, orderings                                                                       */
/* ------------------------------------------------------------------------------------------------ */
typedef enum {
    VIX_OK                 = 0,
    VIX_ERR_INVALID_DIM    = -1,   /* KMeansMBStatus.invalidDim    */
    VIX_ERR_INVALID_K      = -2,   /* KMeansMBStatus.invalidK      */
    VIX_ERR_NULL_PTR       = -3,   /* KMeansMBStatus.nullPtr       */
    VIX_ERR_INVALID_LAYOUT = -4,   /* KMeansMBStatus.invalidLayout */
    VIX_ERR_INVALID_PARAM  = -5,   /* VectorIndexError(.invalidParameter)  */
    VIX_ERR_NOT_TRAINED    = -6,   /* index used before train / set_* */
    VIX_ERR_EMPTY_INPUT    = -7,   /* VectorIndexError(.emptyInput)        */
    VIX_ERR_CONTRACT       = -8,   /* VectorIndexError(.contractViolation) */
    VIX_ERR_UNSUPPORTED    = -9,
    VIX_ERR_CUDA           = -100,
    VIX_ERR_NO_DEVICE      = -101,
    VIX_ERR_OOM            = -102,
    VIX_NO_CONVERGENCE     = 1     /* KMeansMBStatus.noConvergence */
} vix_status;

/* SupportedDistanceMetric subset on the hot path: euclidean, dotProduct (ScoreBlock.swift:24-70) */
/* cosine: flat search / FLAT index (Cosine.run two-pass, distance = 1 - similarity), vix_centroid_batch_score_f32 and the
 * IVF_FLAT index (guarded CentroidBatchScore rows, DistanceUtils.swift:22-38 candidate distances); IVF_PQ takes L2 / IP */
typedef enum { VIX_METRIC_L2 = 0, VIX_METRIC_IP = 1, VIX_METRIC_COSINE = 2 } vix_metric;

/* HeapOrdering (Operations/Selection/TopK.swift:8-31): ties always go to the smaller id */
typedef enum { VIX_ORDER_MIN = 0, VIX_ORDER_MAX = 1 } vix_ordering;

#define VIX_MAX_K 512      /* largest k / nprobe served by the fused selection kernels */
#define VIX_MAX_K_LARGE 16384  /* largest k of index / flat k-NN search: VIX_MAX_K < k <= VIX_MAX_K_LARGE takes the exact
                                  two-pass route over the range-search scans (and the largest rerank_r) */

/* ------------------------------------------------------------------------------------------------ */
/* Library / context                                                                                */
/* ------------------------------------------------------------------------------------------------ */
int         vix_version(void);
const char* vix_last_error(void);            /* thread-local description of the last failure       */
void        vix_clear_error(void);           /* reset it (the void cpq_* calls report only through it) */
int         vix_device_count(void);
int         vix_set_device(int device);      /* cudaSetDevice for the calling thread               */
int         vix_set_stream(void* cuda_stream);  /* thread-local stream (NULL = legacy default)     */
int         vix_set_async(int enabled);      /* 1: do not synchronise when all outputs are device ptrs */
int         vix_get_async(void);             /* the calling thread's current setting (0 / 1)        */
int         vix_synchronize(void);           /* wait for the calling thread's stream               */
int64_t     vix_kernel_launches(int reset);  /* kernels launched by this thread (bench bookkeeping) */
int64_t     vix_scan_tc_launches(void);      /* IVF-PQ searches of this process that took the list-major tensor-core
                                                scan (csrc/vix_ivfpq_tc.cu) rather than the query-major one (tests, bench) */
/* the tensor-core shortlist of the GEMM-shaped stages (csrc/vix_gemm.cu), per kind: coarse probe selection, flat search,
 * IVF list assignment (vix_index_add, k-means, vix_ivf_assign_f32) */
typedef enum { VIX_SHORTLIST_PROBE = 0, VIX_SHORTLIST_FLAT = 1, VIX_SHORTLIST_ASSIGN = 2 } vix_shortlist_kind;
int64_t     vix_tc_shortlist_calls(int kind);       /* calls of this process that took the shortlist rather than the exact
                                                       CUDA-core kernel alone (-1: no such kind) */
int64_t     vix_tc_shortlist_exact_rows(int kind);  /* rows of those calls whose shortlist overflowed or was empty and that the
                                                       exact kernel computed instead; flat and assignment only (probe
                                                       selection hands them over on the device and counts 0) */

/* ------------------------------------------------------------------------------------------------ */
/* a1-a3  Flat scoring.  Replaces @_cdecl l2sqr_f32_block / ip_f32_block                            */
/* (Operations/Scoring/CABIBridge.swift:5-30; kernels L2SqrKernel.swift:78-138, InnerProduct.swift: */
/* 8-101).  out[i] = L2^2(q, xb[i]) (no sqrt) or <q, xb[i]>.  q_norm = NaN means "absent";          */
/* algorithm selection as the reference: dot-trick iff norms are given or d >= 256.                 */
/* ------------------------------------------------------------------------------------------------ */
int vix_l2sqr_f32_block(const float* q, const float* xb, int64_t n, int d, float* out,
                        const float* xb_norm, float q_norm);
int vix_ip_f32_block(const float* q, const float* xb, int64_t n, int d, float* out);

/* Norms.l2NormSquared per row (Operations/Support/Norms.swift:105-130; IVFIndex.swift:470-485) */
int vix_row_norms_f32(const float* x, int64_t n, int d, float* out);

/* a1-a4  Batched exact search = ScoreBlock.run + selectTopK + API distance mapping
 * (FlatIndexOptimized.swift:390-477) for nq queries at once, top-k fused into the scan (no [nq x n]
 * matrix is written).  ids are base row indices.  out_dist: L2 => sqrt(L2^2), IP => -dot.
 * Rows with fewer than k results are padded with id -1 / NaN.  k <= VIX_MAX_K_LARGE: above VIX_MAX_K the exact two-pass
 * route of vix_index_search (same results, ties to the smaller row), which synchronises the stream. */
int vix_flat_search_f32(const float* queries, int64_t nq, const float* xb, int64_t n, int d,
                        int metric, int k, float* out_dist, int64_t* out_ids);

/* a4  selectTopK (Operations/Selection/TopK.swift:127-151): k best of n (score, id); ids == NULL
 * => 0..n-1; outputs best -> worst (extractSorted); *out_count = min(k, n). */
int vix_select_topk_f32(const float* scores, const int32_t* ids, int64_t n, int k, int ordering,
                        float* out_scores, int32_t* out_ids, int* out_count);

/* Kernel #40 rerank_exact_topk_batch (Operations/Rerank/ExactRerank.swift:698-814; spec step 7 of
 * docs/kernel-specs/DONE_22_adc_scan.md:873-878), DenseArray backend: cand_ids [nq x C] are rows of xb [N x d];
 * ids outside [0, N) are missing and skipped; scores are the raw kernel values (L2^2 without sqrt / dot);
 * ordering .min for L2, .max for IP, ties -> smaller candidate id; padded with +-inf / id -1. */
int vix_rerank_exact_topk_f32(const float* queries, int64_t nq, int d, int metric, const int64_t* cand_ids, int C, int K,
                              const float* xb, int64_t N, const float* xb_sq_norms /* nullable */, float* top_scores,
                              int64_t* top_ids);

/* a5  mergeTopK (Operations/Selection/TopKMerge.swift:11-61): nlists best->worst lists stored as
 * rows of [nlists x list_stride] with lens[l] valid entries, for `batch` independent queries
 * (scores/ids are [batch x nlists x list_stride], lens [batch x nlists]); ties: smaller id, then
 * smaller list index.  Outputs [batch x k] padded with id -1 / NaN.  This is also the multi-GPU
 * reduction applied to the all-gathered per-rank results. */
int vix_merge_topk_f32(const float* scores, const int64_t* ids, const int32_t* lens, int64_t batch,
                       int nlists, int list_stride, int k, int ordering,
                       float* out_scores, int64_t* out_ids);

/* ------------------------------------------------------------------------------------------------ */
/* a6-a9  Coarse quantiser                                                                          */
/* ------------------------------------------------------------------------------------------------ */
/* CentroidBatchScore.run (Kernels/CentroidBatchScore.swift:39-88): out[q x kc], smaller is better:
 * L2 => ||c||^2 - 2<q,c> (||q||^2 omitted), IP => -<q,c>, cosine => 1 - <q,c> qInv cInv with the near-zero-norm
 * guard (sqrt(||q||^2 ||c||^2) <= ulpOfOne => 1; :70-84).  centroid_norms = ||c||^2 (Norms.l2NormSquared,
 * IVFIndex.swift:470-485), may be NULL (computed). */
int vix_centroid_batch_score_f32(const float* queries, int64_t q, const float* centroids, int kc,
                                 int d, int metric, const float* centroid_norms, float* out);

/* ivf_select_nprobe_batch_f32 (Kernels/IVFSelect.swift:242-315) with the batchSearch ordering
 * (IVFIndex.swift:593-595, 905-927): per query the nprobe best lists by (score asc, index asc);
 * list_ids_out[b x nprobe] int32, padded with -1 (scores NaN) beyond min(nprobe, kc);
 * list_scores_out (optional) in the CentroidBatchScore convention, "smaller is better": L2 => ||c||^2 - 2<q,c>,
 * IP => -<q,c>.  IVFSelect's own listScoresOut (||q||^2 + ||c||^2 - 2<q,c> / <q,c>, IVFSelect.swift:436-479) differ by
 * a per-query constant / the sign, which leaves the selected lists and their order unchanged; the Swift shim of
 * INTEGRATION.md restores them;
 * disabled_lists: optional bitmask, bit i set => list i skipped (IVFSelect.swift:366-395). */
int vix_ivf_select_nprobe_batch_f32(const float* Q, int64_t b, int d, const float* centroids, int kc,
                                    int metric, int nprobe, const float* centroid_norms,
                                    const uint64_t* disabled_lists,
                                    int32_t* list_ids_out, float* list_scores_out);

/* _vi_km12_assignAOS over all rows (Kernels/KMeansMiniBatchKernel.swift:341-359, 689-706):
 * assign_out[i] = argmin_c L2^2(x_i, C_c), tie -> lower c; BIT-EXACT with the reference's 8-lane
 * summation order.  dist_out optional. */
int vix_ivf_assign_f32(const float* x, int64_t n, int d, const float* centroids, int kc,
                       int32_t* assign_out, float* dist_out);

/* metric-aware list assignment of IVFIndex.optimize for dot-product indexes
 * (IVFIndex.swift:376-435): first-min argmin of the CentroidBatchScore row. */
int vix_ivf_assign_metric_f32(const float* x, int64_t n, int d, const float* centroids, int kc,
                              int metric, const float* centroid_norms, int32_t* assign_out);

/* ------------------------------------------------------------------------------------------------ */
/* a13  PQ look-up tables (Operations/Quantization/PQLUT.swift)                                     */
/* ------------------------------------------------------------------------------------------------ */
typedef struct {
    int  use_dot_trick;     /* -1 auto (centroid_norms given && ks >= 64), 0, 1   (PQLutOpts.useDotTrick) */
    bool include_q_norm;    /* default true                                      (includeQNorm)          */
    bool strict_fp;         /* scalar sequential sums instead of the 8-lane order (strictFP)             */
} vix_pq_lut_opts;

/* pq_query_subnorms_f32 (PQLUT.swift:174-187): out[q][j] = ||q_j||^2 in the LUT kernels' own reduction order (_simd_dot),
 * for nq queries at once; computed once and reused across the LUTs of a query's probed lists. */
int vix_pq_query_subnorms_f32(const float* queries, int64_t nq, int d, int m, float* out /* [nq x m] */);

/* pq_lut_batch_l2_f32 (PQLUT.swift:392-465) / pq_lut_l2_f32 (:191-261) for nq queries:
 * luts[nq x m x ks]. */
int vix_pq_lut_batch_l2_f32(const float* queries, int64_t nq, int d, int m, int ks,
                            const float* codebooks, float* luts, const float* centroid_norms,
                            const vix_pq_lut_opts* opts);

/* pq_lut_residual_l2_f32 (PQLUT.swift:266-386) for nq (query, coarse centroid) pairs:
 * coarse_ids[nq] indexes coarse_centroids[kc x d]; luts[nq x m x ks]. */
int vix_pq_lut_residual_l2_f32(const float* queries, const int32_t* coarse_ids, int64_t nq, int d,
                               const float* coarse_centroids, int m, int ks, const float* codebooks,
                               float* luts, const float* centroid_norms, const vix_pq_lut_opts* opts);

/* ------------------------------------------------------------------------------------------------ */
/* a14  ADC scan (Operations/Quantization/ADCScan.swift:99-149)                                     */
/* ------------------------------------------------------------------------------------------------ */
typedef struct {
    int   layout;            /* 0 = AoS [n][m], 1 = interleavedBlock [n/g][m][g]  (ADCLayout) */
    int   group_size;        /* g for layout 1                                                 */
    int   stride;            /* AoS row stride in bytes, 0 => m (u8) or m/2 (u4)               */
    float add_bias;          /* added after the accumulator sum                                */
    bool  strict_fp;         /* Kahan summation when m >= 64                                   */
} vix_adc_scan_opts;

/* out[i] = sum_j lut[j*ks + code(i,j)] + bias, reference accumulation order (4 accumulators for u8,
 * sequential for u4, Kahan when strict_fp && m >= 64).  ks must be 256 (u8) / 16 (u4). */
int vix_adc_scan_u8(const uint8_t* codes, int64_t n, int m, int ks, const float* lut, float* out,
                    const vix_adc_scan_opts* opts);
int vix_adc_scan_u4(const uint8_t* codes, int64_t n, int m, int ks, const float* lut, float* out,
                    const vix_adc_scan_opts* opts);

/* ------------------------------------------------------------------------------------------------ */
/* a10 / a12  Trainers                                                                              */
/* ------------------------------------------------------------------------------------------------ */
typedef struct {
    int      batch_size;          /* KMeansMBConfig.batchSize   (default 1024)                 */
    int      epochs;              /* KMeansMBConfig.epochs      (default 10)                   */
    float    tol;                 /* KMeansMBConfig.tol         (default 1e-4)                 */
    uint64_t seed;                /* KMeansMBConfig.seed                                       */
    uint64_t stream_id;           /* KMeansMBConfig.streamID                                   */
    bool     compute_assignments; /* KMeansMBConfig.computeAssignments                         */
    int      mode;                /* 0 = reference-parity (replays RNG + quirks of finding 6),
                                     1 = sane (Lloyd on a sample, standard empty-cluster split) */
} vix_kmeans_cfg;

/* kmeansPlusPlusSeed (Kernels/KMeansSeeding.swift:167-292) */
int vix_kmeanspp_seed_f32(const float* data, int64_t n, int d, int k, uint64_t seed, uint64_t stream_id,
                          float* centroids_out, int64_t* chosen_out);

/* kmeans_minibatch_f32 (Kernels/KMeansMiniBatchKernel.swift:401-724); init_centroids NULL =>
 * k-means++ with cfg.seed.  assign_out optional [n]. */
int vix_kmeans_minibatch_f32(const float* x, int64_t n, int d, int kc, const float* init_centroids,
                             const vix_kmeans_cfg* cfg, float* centroids_out, int32_t* assign_out);

typedef struct {
    int      algorithm;      /* 0 lloyd, 1 minibatch            (PQTrainConfig.algo)        */
    int      max_iters;      /* default 25                                                  */
    float    tol;            /* default 1e-4                                                */
    int      batch_size;     /* default 1024                                                */
    int64_t  sample_n;       /* default 0 (all rows)                                        */
    uint64_t seed;           /* default 42                                                  */
    int      stream_id;      /* default 0                                                   */
    int      empty_policy;   /* 0 split, 1 reseed, 2 ignore                                 */
    int      mode;           /* 0 = reference-parity, 1 = sane                              */
} vix_pq_train_cfg;

/* pq_train_f32 (Kernels/PQTrain.swift:83-388).  coarse_centroids/assignments both NULL or both
 * given (residual training).  codebooks_out[m x ks x dsub], centroid_norms_out[m x ks] optional. */
int vix_pq_train_f32(const float* x, int64_t n, int d, int m, int ks, const float* coarse_centroids,
                     const int32_t* assignments, const vix_pq_train_cfg* cfg, float* codebooks_out,
                     float* centroid_norms_out);

/* pq_train_streaming_f32 (Kernels/PQTrain.swift:391-706): the mini-batch trainer over `nchunks` row blocks that the host
 * hands over one pointer each (host or device, valid for the call; no residual form).  Reference parity only (the
 * reference's RNG streams, per-chunk permutations, Bernoulli row sampling, running-mean blend and pass-level repair are
 * replayed; distances and argmins run on the GPU): bit-identical codebooks, incl. the reference's own golden vector
 * (Tests/VectorIndexTests/PQTrainTests.swift:724-817).  Defaults as the reference: max_iters 15, batch_size 8192,
 * sample_n 2000 when more rows are given. */
int vix_pq_train_streaming_f32(const float* const* chunks, const int64_t* chunk_n, int nchunks, int d, int m, int ks,
                               const vix_pq_train_cfg* cfg, float* codebooks_out, float* centroid_norms_out /* nullable */);

/* ------------------------------------------------------------------------------------------------ */
/* a15  Index handles: build / train / add / search with device-resident state.                     */
/* Mirrors VectorIndexProtocol (IndexProtocols.swift:50-103) for FlatIndex(Optimized), IVFIndex     */
/* (IVF-Flat) and the IVF-PQ composition of docs/kernel-specs/DONE_22_adc_scan.md:831-881.          */
/* ------------------------------------------------------------------------------------------------ */
typedef struct vix_index vix_index_t;

typedef enum { VIX_INDEX_FLAT = 0, VIX_INDEX_IVF_FLAT = 1, VIX_INDEX_IVF_PQ = 2 } vix_index_kind;

typedef struct {
    int kind;          /* vix_index_kind                                                      */
    int d;             /* dimension                                                           */
    int metric;        /* vix_metric                                                          */
    int nlist;         /* IVFIndex.Configuration.nlist (default 256), clamped to n at train   */
    int nprobe;        /* IVFIndex.Configuration.nprobe (default 8)                           */
    int m;             /* PQ sub-quantisers (IVF_PQ)                                          */
    int ks;            /* PQ codebook size, 256                                               */
    int shard_rank;    /* multi-GPU: this rank ...                                            */
    int shard_world;   /* ... of shard_world ranks (lists / row ranges are partitioned); 0/1 = no sharding */
} vix_index_params;

void vix_index_params_default(vix_index_params* p);
int  vix_index_create(const vix_index_params* p, vix_index_t** out);
void vix_index_destroy(vix_index_t* h);

/* optimize(): coarse k-means (+ PQ codebooks on residuals) from a training sample.  An IVF_FLAT index may already hold
 * vectors (the reference's insert -> optimize() -> search; until it has centroids its searches are linear scans,
 * IVFIndex.swift:820-832): they are filed into their lists, and x == NULL trains on them (IVFIndex.swift:279-341).
 * An IVF_PQ index keeps codes, not vectors: train / set_* first. */
int vix_index_train(vix_index_t* h, const float* x, int64_t n, const vix_kmeans_cfg* kcfg,
                    const vix_pq_train_cfg* pcfg);
/* stage-wise parity / import: install externally trained parameters */
int vix_index_set_coarse(vix_index_t* h, const float* centroids, int kc);
int vix_index_set_codebooks(vix_index_t* h, const float* codebooks, const float* centroid_norms);
int vix_index_get_coarse(vix_index_t* h, float* centroids_out, int* kc_out);
int vix_index_get_codebooks(vix_index_t* h, float* codebooks_out, float* centroid_norms_out);

/* batchInsert: ids NULL => consecutive ids continuing after the last automatic id this handle handed out, counting every
 * row added since the handle was created, cleared or imported into.  Without removals that is the current count; after
 * one, automatic ids never repeat an id that may still be stored. */
int vix_index_add(vix_index_t* h, const float* x, const int64_t* ids, int64_t n);
/* remove(id:): remove every stored row whose id is in ids[0..n) (host or device array; duplicates and ids that are not
 * stored are allowed).  A row stored twice under one id is removed twice.  *removed_out (nullable, host) = rows removed.
 * Ids are checked as by add (VIX_ERR_INVALID_PARAM outside [0, 2^32 - 1)) before anything changes: a call rejected for
 * its input removes nothing.  The remaining rows keep their order, so the index then equals one built by adding only them: same lists,
 * same slots, same search results.  The rows are compacted on the device (one extra copy of the largest row array at
 * the peak) and the lists are rebuilt by the next call that reads them, as after an add; a call that matches no row
 * changes nothing.  Every index kind.  On a shard it removes what THIS rank holds: a sharded host passes the same ids to
 * every rank and sums the counts itself. */
int vix_index_remove(vix_index_t* h, const int64_t* ids, int64_t n, int64_t* removed_out);
/* import of prebuilt inverted lists in the reference's AoS list format (Kernels/IVFAppend.swift:
 * 220-236): CSR offsets[kc+1], codes[N x m], ids[N] */
int vix_index_import_lists(vix_index_t* h, const int64_t* list_offsets, const uint8_t* codes,
                           const int64_t* ids);
int64_t vix_index_count(vix_index_t* h);       /* vectors stored on THIS shard */
int     vix_index_list_sizes(vix_index_t* h, int64_t* sizes_out /* [nlist] */);
int     vix_index_export_lists(vix_index_t* h, int64_t* list_offsets, uint8_t* codes, int64_t* ids,
                               int32_t* assignments_in_add_order /* nullable */);
int     vix_index_clear(vix_index_t* h);

/* batchSearch: out_dist/out_ids [nq x k] ascending by API distance, padded with id -1 / NaN.
 * nprobe <= 0 => the index's configured nprobe; nprobe > VIX_MAX_K => VIX_ERR_INVALID_K.  k <= 0 => VIX_OK with nothing written
 * (IVFIndex.swift:866).  IVF-PQ probes: -1, ids outside [0, kc) and empty lists are skipped; a list probed twice in one
 * row is scanned twice, so its vectors can come back twice (both copies with the same distance bits).  Shared-memory
 * limits of the query-major scan, refused with VIX_ERR_UNSUPPORTED before any kernel runs: m in {48, 64} (ks = 256)
 * with k > 448 needs 4 nprobe + d <= 1912; the generic kernel (other m, or ks = 16) needs
 * 4 (m ks + d + 4 nprobe) + 64 next_pow2(k + 32) + 8 next_pow2(8 k) <= 227 KB.
 * Non-finite values (IVF-PQ): results rank by (distance, id), NaN after every number, equal distances by the smaller id
 * (the oracle keeps its scan order among equal or NaN distances).  A NaN query component makes every probed distance
 * NaN (the row is the k smallest probed ids); an infinite one can give NaN where the oracle gives +-inf, because the scan
 * adds the per-probe and per-code terms of its decomposition (+inf + -inf); a query whose L2 distances overflow gets +inf.
 * With sharding the result is this shard's local top-k (merge with
 * vix_merge_topk_f32 after an all-gather).
 * k <= VIX_MAX_K_LARGE (above: VIX_ERR_INVALID_K).  VIX_MAX_K < k <= VIX_MAX_K_LARGE takes an exact two-pass route over the
 * range-search scans (every kind, metric and filter; the same outputs, padding, tie and NaN rules, and search(k)[:, :k2]
 * == search(k2) bit for bit): a seed pass bounds each query's k-th distance from a subset of its candidates (IVF: the
 * probes, in order, that hold about 2 k vectors; flat: the fused top-512 of 2 k / 512 row blocks), a collect pass keeps
 * every candidate within that bound, and the rows are sorted by (distance, id) and cut at k.  IVF-PQ takes the query-major
 * scan on this route.  The route synchronises its stream, even in asynchronous mode (the size of the collect depends on
 * the data); a collect that does not fit in device memory returns VIX_ERR_OOM with the handle unchanged; it is not
 * recorded by vix_index_trace; vix_search_stats reports scan_path = 2, merge_candidates = the entries collected (the
 * row lengths before the cut), the three ms_* times, cycle counters 0.  VIX_SCAN_DEBUG=1 prints one line per call:
 * "[vix knn] kind K, kernel fast G n | generic | ivfflat | flat, filter 0|1, k K, seed S, total T, passes P, max_row M"
 * (S seed entries, T collected entries, P scans of the collect: 2 when it outgrew the capacity the handle remembers). */
int vix_index_search(vix_index_t* h, const float* queries, int64_t nq, int k, int nprobe,
                     float* out_dist, int64_t* out_ids);

/* stage outputs for parity tests and profiling */
typedef struct {
    int64_t codes_scanned;        /* sum over (query, probed owned list) of list length          */
    int64_t code_bytes_scanned;   /* codes_scanned * m  == algorithmic ADC bytes (SURVEY 8d)      */
    float   ms_coarse;            /* CUDA-event time of the probe-selection stage                 */
    float   ms_scan;              /* ... of the LUT + ADC + top-k stage                           */
    float   ms_total;
    /* fused IVF-PQ scan only: SM cycles one scanning warp per CTA spent building the per-query table and probe
     * bookkeeping / scanning / waiting for the other warps at the end of a query, summed over CTAs */
    int64_t cycles_prologue, cycles_scan, cycles_tail;
    int64_t cycles_select, cycles_probe_table, cycles_lut;   /* the three concurrent pieces of the prologue */
    int64_t merge_candidates;                                 /* entries handed to the per-query top-k merge */
    float   ms_scan_kernel;       /* CUDA-event time of the stage's dominant kernel alone (the scan proper)              */
    int32_t scan_path;            /* IVF-PQ: 0 = query-major look-up-table scan, 1 = list-major tensor-core scan;
                                     2 = the two-pass route of k > VIX_MAX_K (every kind)                                  */
} vix_search_stats;
int vix_index_search_ex(vix_index_t* h, const float* queries, int64_t nq, int k, int nprobe,
                        float* out_dist, int64_t* out_ids, int32_t* out_probes /* [nq x nprobe] nullable */,
                        vix_search_stats* stats /* nullable */);

/* Range search (Kernel #07, Operations/RangeQuery/RangeQuery.swift; rangeScanADC_u8 / _u4): for every query, EVERY stored
 * vector whose API distance is <= radius, sorted ascending by (distance, id), as CSR in a result object the library owns.
 *   - candidates: FLAT every stored row; IVF_FLAT / IVF_PQ the rows of the nprobe probed lists, chosen exactly as
 *     vix_index_search chooses them (nprobe <= 0 => the configured nprobe; nprobe > VIX_MAX_K => VIX_ERR_INVALID_K; -1, ids
 *     outside [0, kc) and empty lists skipped); an IVF_FLAT index without centroids scans every row, as its search does;
 *   - distance: what vix_index_search returns for the same (query, vector) -- FLAT / IVF_FLAT: L2 sqrt(L2^2), IP -dot,
 *     cosine 1 - similarity; IVF_PQ: L2 the ADC squared distance (no sqrt), IP -score -- bit for bit (IVF_PQ always takes
 *     the query-major scan); the test is the IEEE comparison distance <= radius on that value: NaN distances never pass,
 *     a NaN radius is VIX_ERR_INVALID_PARAM, +inf returns every candidate with a number for its distance, negative radii
 *     are valid (an IP radius of -0.8 keeps dot >= 0.8);
 *   - filter_words (nullable): the id filter of vix_index_search_filtered, applied before the radius test;
 *   - a row stored twice, or a list probed twice, comes back twice; a dirty handle rebuilds its lists first, as search
 *     does; on a shard the result is what THIS rank holds (vix_sharded_range_search merges the ranks).
 * The call synchronises its stream once, even in asynchronous mode: the size of the answer depends on the data.  It
 * normally scans once; when the answer outgrows the capacity the handle remembers from its previous call, the scan runs a
 * second time with the exact capacity.  A result that does not fit in device memory returns VIX_ERR_OOM with nothing
 * allocated and the handle unchanged.  nq == 0 gives an empty result (lims = {0}).  *out must be released with
 * vix_range_result_destroy.  VIX_SCAN_DEBUG=1 prints one "[vix range] ..." line per call (kind, kernel, filter, passes,
 * total, longest row, rows sorted in global memory). */
typedef struct vix_range_result vix_range_result_t;
int     vix_index_range_search(vix_index_t* h, const float* queries, int64_t nq, float radius, int nprobe,
                               const uint64_t* filter_words /* nullable */, int64_t filter_capacity, int filter_mode,
                               vix_range_result_t** out);
int64_t vix_range_result_nq(const vix_range_result_t* r);
int64_t vix_range_result_total(const vix_range_result_t* r);
/* CSR: lims [nq + 1] (lims[0] = 0), dist / ids [total]; each nullable; host or device pointers (host outputs are valid when
 * the call returns, device outputs as the usual asynchronous-mode rules say) */
int     vix_range_result_get(const vix_range_result_t* r, int64_t* lims, float* dist, int64_t* ids);
void    vix_range_result_destroy(vix_range_result_t* r);   /* NULL is a no-op */

/* Search with an id filter: IDFilterBitset / idFilterPass of Operations/Filtering/IDFilter.swift:13-135 -- a bitset over
 * the dense id domain [0, capacity); ids outside the domain never pass; VIX_FILTER_ALLOW keeps ids whose bit is 1,
 * VIX_FILTER_DENY keeps ids whose bit is 0.  The filter is applied BEFORE selection (the pre-filter of
 * IVFIndex.search / FlatIndex.search, IVFIndex.swift:813, 1034; FlatIndex.swift:61): the result is the k best of the
 * vectors that pass, possibly fewer than k (padding id -1 / NaN).  filter_words == NULL => unfiltered search.
 * Closure filters over metadata are host-side objects in the reference; evaluate them on the host into a bitset.
 * k as vix_index_search: up to VIX_MAX_K_LARGE, the two-pass route above VIX_MAX_K with the filter on both passes. */
enum { VIX_FILTER_ALLOW = 0, VIX_FILTER_DENY = 1 };
int vix_index_search_filtered(vix_index_t* h, const float* queries, int64_t nq, int k, int nprobe,
                              const uint64_t* filter_words /* [ceil(capacity / 64)] */, int64_t filter_capacity,
                              int filter_mode, float* out_dist, int64_t* out_ids);

/* ---- multi-GPU: inverted lists are partitioned over ranks by contiguous list-id blocks ------------------
 * Search on rank r of R:  vix_index_probe_range over r's block of centroids (local top-nprobe, GLOBAL list ids)
 *   -> all-gather + vix_merge_topk_f32 (.min; ids = list ids) = the global probe lists of IVFIndex.swift:905-927
 *   -> vix_index_search_with_probes (lists this rank does not hold are empty, so only owned lists are scanned)
 *   -> all-gather + vix_merge_topk_f32 of the per-rank [nq x k] results (TopKMerge.swift:11-61).
 * Build: any rank assigns + encodes a batch (vix_index_encode); rows are routed to the rank owning their
 * list and appended there with vix_index_add_encoded. */
int vix_index_probe_range(vix_index_t* h, const float* queries, int64_t nq, int nprobe, int list_begin, int list_count,
                          int32_t* list_ids_out /* [nq x nprobe] */, float* list_scores_out /* nullable */);
/* (k as vix_index_search: up to VIX_MAX_K_LARGE; both passes of the two-pass route use the given probes) */
int vix_index_search_with_probes(vix_index_t* h, const float* queries, int64_t nq, int k, const int32_t* probes,
                                 int nprobe, float* out_dist, int64_t* out_ids);

/* ---- the whole sharded step behind the C ABI: one process per GPU, one communicator per process ------------------
 * north_star: "the database shards by inverted list across the GPUs of one box; queries are broadcast, each GPU produces
 * a local top-k, and the per-GPU results are merged" -- here without any host-language glue: a non-Python host (the Swift
 * shim of INTEGRATION.md) calls these four entry points and nothing else.  NCCL is bound at run time (libnccl.so.2,
 * VIX_NCCL_PATH overrides); the exchanges of a search run over peer-mapped memory (cudaIpc: every rank stores its block
 * into all peers over NVLink + one barrier kernel) and fall back to ncclAllGather when the ranks cannot map each other
 * (decided once, collectively; VIX_NO_P2P=1 forces the fallback).
 *   vix_comm_unique_id   rank 0: the NCCL id (128 bytes) the host hands to every rank by its own means
 *   vix_comm_create      collective; binds the calling thread's CUDA device
 *   vix_sharded_add      collective; x / ids: the rows THIS rank contributes (any rows; n may be 0).  IVF-PQ and IVF-Flat:
 *                        rows are assigned (+ encoded) here and appended on the rank owning their list: list l belongs to
 *                        rank r iff list_bounds[r] <= l < list_bounds[r + 1] (host array [world + 1], NULL = equal-count
 *                        blocks); IVF-Flat rows travel as vectors with their assignment, which the owner keeps.  Flat: rows
 *                        stay on the rank that passes them (list_bounds must be NULL, else VIX_ERR_INVALID_PARAM).
 *                        A row with no nearest list (NaN components; IVF kinds) or an id outside [0, 2^32 - 1) on ANY rank
 *                        makes every rank return VIX_ERR_INVALID_PARAM (naming that rank) before any row is stored or
 *                        travels: no rank stores a row of the call.  An IVF-Flat index needs its centroids first
 *                        (VIX_ERR_NOT_TRAINED): the sharded layout files every row into its list
 *   vix_sharded_search   collective; every rank passes the SAME batch (host or device pointer; from a host pointer only
 *                        the rank's own 1/world block crosses PCIe) and receives the merged [nq x k] result.  Results
 *                        equal vix_index_search on one GPU holding all lists (same probe lists by construction; same
 *                        (distance, id) order: mergeTopK, TopKMerge.swift:11-61), bit for bit -- zero distances with
 *                        their sign (IP -0, L2 +0) and NaN / -1 padding included -- when that GPU holds every row in the
 *                        slot the shards do: rows inserted in the order the owners append them, i.e. rank 0's
 *                        contributions first.  A row in another slot of its list may differ in the last bit of its
 *                        distance (the slot decides the order its table entries are summed in).  Asynchronous mode: no host
 *                        synchronisation at all when the outputs are device pointers (k <= VIX_MAX_K).
 *                        k <= VIX_MAX_K_LARGE (above: VIX_ERR_INVALID_K; k > VIX_MAX_K with nq >= 2^31 - 1:
 *                        VIX_ERR_INVALID_PARAM; both on every rank before any exchange), with the same parity, and
 *                        search(k)[:, :k2] == search(k2) for every k2 <= k.  Above VIX_MAX_K (world > 1) the call takes
 *                        the two-pass route of vix_index_search with one bound per query shared by all ranks: each rank
 *                        seeds over the probes of the lists it owns that hold about 2 k vectors, the ranks take the
 *                        minimum of their k-th seed distances (peer memory or an NCCL all-reduce), each rank collects
 *                        the candidates within it from its probed lists and cuts every sorted row at k, and the cut rows
 *                        are exchanged, merged and cut at k as sharded range search exchanges its rows (at most world x k
 *                        keys per query travel).  That route synchronises the stream even in asynchronous mode.  A rank
 *                        whose local pass fails makes every rank return its code; a merged answer that does not fit
 *                        makes every rank return VIX_ERR_OOM; a merged row shorter than k within a finite bound (the two
 *                        passes disagreed on a distance) makes every rank return VIX_ERR_CONTRACT.  One rank is
 *                        vix_index_search.
 *                        Every index kind: flat, IVF-Flat (L2, IP, cosine) and IVF-PQ (L2, IP).  Flat: no probes; each rank
 *                        runs the fused flat search over its rows (k > VIX_MAX_K: the flat two-pass route with the shared
 *                        bound) and the ranks' results merge by raw score and then rank, so the answer equals one GPU
 *                        holding rank 0's rows first, then rank 1's, ..., each rank's in add order (flat search breaks ties
 *                        at one score by row, and maps scores to distances only after selecting).  IVF-Flat: as IVF-PQ
 *                        (probes exchanged, each rank scans the lists it owns); its distances are exact per pair and its
 *                        ties fall to the id, so the answer does not depend on the slots.  Zero distances keep one GPU's
 *                        sign per kind: IP -0 from flat and IVF-PQ, +0 from IVF-Flat. */
typedef struct vix_comm vix_comm_t;
int vix_comm_unique_id(void* id_out, size_t capacity /* >= 128 */);
int vix_comm_create(const void* id, size_t id_bytes, int rank, int world, vix_comm_t** out);
int vix_comm_destroy(vix_comm_t* c);
int vix_comm_rank(const vix_comm_t* c);
int vix_comm_world(const vix_comm_t* c);
int vix_comm_uses_peer_memory(const vix_comm_t* c);        /* 1 peer memory, 0 NCCL all-gathers, -1 not decided yet */
/* measurement aid: CUDA events around the three phases of the LAST vix_sharded_search, vix_sharded_search_filtered or
 * vix_sharded_range_search (or replicated search, see vix_replicated_search) on this communicator -- probe selection + exchange | fused scan (range: local scan and sort;
 * k > VIX_MAX_K: seed, bound exchange, collect and cut at k) | result exchange + merge (range: + decode; k > VIX_MAX_K:
 * + cut at k) (ms; waits for that call to finish) */
int vix_comm_trace(vix_comm_t* c, int enabled);
int vix_comm_trace_get(vix_comm_t* c, float* phase_ms /* [3] */);
/* rows [first, first + count) of a batch of nq queries are the block whose probe lists `rank` computes */
int vix_sharded_query_block(int64_t nq, int rank, int world, int64_t* first, int64_t* count);
int vix_sharded_add(vix_index_t* h, vix_comm_t* c, const int64_t* list_bounds /* nullable */, const float* x,
                    const int64_t* ids, int64_t n);
int vix_sharded_search(vix_index_t* h, vix_comm_t* c, const float* queries, int64_t nq, int k, int nprobe,
                       float* out_dist, int64_t* out_ids);

/* Sharded range search and id filters: vix_index_range_search / vix_index_search_filtered over the list-sharded layout of
 * vix_sharded_search.  Both are collective: every rank passes the same batch, radius (or k), nprobe and filter, host or
 * device pointers (from a host pointer only the rank's own block of queries crosses PCIe), and every rank receives the
 * whole merged answer.
 *   - Parity: the answer equals the one-GPU call on an index holding every row in the slot the shards hold it in (rows
 *     inserted in owner-append order, rank 0's contributions first), bit for bit: lims, ids, distance bits with the sign of
 *     zero (IP -0, L2 +0; IVF-Flat +0), the (distance, id) order, rows stored twice and lists probed twice (each comes back
 *     twice).  A flat index has no probes: each rank runs the flat range scan over its rows.
 *   - Refusals, on every rank alike and before any exchange: a NaN radius, a filter_mode other than VIX_FILTER_ALLOW /
 *     VIX_FILTER_DENY or a negative filter_capacity (VIX_ERR_INVALID_PARAM); nprobe outside 1 .. VIX_MAX_K after the default
 *     (VIX_ERR_INVALID_K; not read for a flat index); an IVF-PQ index that is not trained (VIX_ERR_NOT_TRAINED) or uses
 *     cosine (VIX_ERR_UNSUPPORTED); an IVF-Flat index without coarse centroids (VIX_ERR_NOT_TRAINED).  Flat and IVF-Flat
 *     indexes follow the parity of vix_sharded_search for their kind (flat: rows in rank order; IVF-Flat: any slots).
 *   - Range: nq == 0 gives an empty result (lims = {0}) with no exchange; one rank is vix_index_range_search.  The probes
 *     travel as in vix_sharded_search; each rank runs the query-major range scan over the probed lists it owns and sorts
 *     its rows; the ranks exchange their row starts, then their sorted keys (a second peer-mapped region of the
 *     communicator, grown collectively and geometrically, or NCCL: an all-gather of the row starts and grouped send /
 *     receive of the keys); every rank merges the world sorted runs of each row on the device and decodes them.  Host
 *     synchronisations: the local total, the global total and the collective verdict on the result's allocation.  A global
 *     answer that does not fit in device memory on some rank makes every rank return VIX_ERR_OOM with nothing allocated and
 *     the index unchanged; so does a failure of any rank's local scan (every rank returns that rank's code).  *out is
 *     released with vix_range_result_destroy.
 *   - Filtered k-NN: filter_words == NULL is vix_sharded_search; a filter sends each rank's scan down the query-major path,
 *     as on one GPU.  k as vix_sharded_search: up to VIX_MAX_K_LARGE, the filter applied on both passes on every rank. */
int vix_sharded_range_search(vix_index_t* h, vix_comm_t* c, const float* queries, int64_t nq, float radius, int nprobe,
                             const uint64_t* filter_words /* nullable */, int64_t filter_capacity, int filter_mode,
                             vix_range_result_t** out);
int vix_sharded_search_filtered(vix_index_t* h, vix_comm_t* c, const float* queries, int64_t nq, int k, int nprobe,
                                const uint64_t* filter_words /* nullable */, int64_t filter_capacity, int filter_mode,
                                float* out_dist, int64_t* out_ids);

/* ---- multi-GPU replicas: every rank holds the WHOLE index and answers its share of the batch --------------------------
 * For an index that fits one GPU this is the faster layout (no probe exchange, no merge: a query's answer never depends on
 * the other queries of its batch).  The calls take the vix_comm_t of the sharded calls and a handle whose shard_world is 0
 * or 1 (VIX_ERR_INVALID_PARAM otherwise).  All four are collective: every rank calls them in the same order with the same
 * nq, k, radius, nprobe and filter.
 *   vix_replicated_add              x / ids: the rows THIS rank contributes (any rows; n may be 0; explicit ids).  Each rank
 *                                   prepares its own rows (IVF-PQ: list assignment and codes; IVF-Flat: assignment; flat:
 *                                   nothing), the counts are all-gathered, and a row with no nearest list (IVF kinds) or an id
 *                                   outside [0, 2^32 - 1) on ANY rank makes every rank return VIX_ERR_INVALID_PARAM naming that
 *                                   rank, before any row travels: no rank stores a row of the call.  The prepared rows
 *                                   (IVF-PQ m + 12 bytes, IVF-Flat 4 d + 12, flat 4 d + 8) are all-gathered over peer memory
 *                                   (the range region, grown collectively) or NCCL grouped send / receive, and every replica
 *                                   appends all of them rank by rank, rank 0's first: every replica holds identical lists, rows
 *                                   in identical slots.  An IVF-PQ index must be trained, an IVF-Flat index needs its
 *                                   centroids (VIX_ERR_NOT_TRAINED).
 *   vix_replicated_search[_filtered] rank r answers rows vix_sharded_query_block(nq, r, world) with the one-GPU search
 *                                   (vix_index_search / _filtered: the list-major scan when the block's shape allows it, the
 *                                   two-pass route for VIX_MAX_K < k <= VIX_MAX_K_LARGE); from a host pointer only that block
 *                                   of queries crosses PCIe.  Its [cnt x k] block is stored into every peer's region at the
 *                                   block's row offset, one barrier (NCCL: an all-gather), and every rank receives the whole
 *                                   [nq x k] answer.  k <= VIX_MAX_K with device outputs in asynchronous mode: no host
 *                                   synchronisation; a rank whose local search failed then raises the pipeline error that the
 *                                   next synchronising call on every rank reports (VIX_ERR_CUDA).  Otherwise (host outputs,
 *                                   synchronous mode, or k > VIX_MAX_K, whose blocks travel through the range region, grown
 *                                   collectively) the call synchronises and every rank returns the failing rank's code.
 *   vix_replicated_range_search     each rank range-searches its block; row starts and sorted keys travel as in
 *                                   vix_sharded_range_search (statuses, global total, collective growth, allocation verdict:
 *                                   VIX_ERR_OOM on every rank when the answer does not fit on one); the rows of different ranks
 *                                   belong to different queries, so the global CSR is the ranks' rows concatenated (no merge).
 *   remove                          no collective call: every replica calls vix_index_remove with the same ids (the remaining
 *                                   rows keep their order, so the replicas stay identical).
 *   a rank that only needs ITS block (no assembly) calls vix_index_search on the rows vix_sharded_query_block gives it.
 * Contract: the collective answer equals the one-GPU call (vix_index_search, vix_index_search_filtered,
 * vix_index_range_search) on the whole batch, over an index holding the rows in the order the replicas append them, bit for
 * bit: ids, distance bits with the sign of zero, -1 / NaN padding, rows stored twice and lists probed twice, and
 * search(k)[:, :k2] == search(k2).  It rests on one fact, which tests/test_replicated.py pins for every kind, metric, route
 * and filter: a query's answer does not depend on the other queries of its batch.  One rank is the one-GPU call.
 * Refusals, on every rank alike and before any exchange, with the codes of the sharded calls: a NaN radius, a bad
 * filter_mode or negative filter_capacity (VIX_ERR_INVALID_PARAM); nprobe outside 1 .. VIX_MAX_K after the default
 * (VIX_ERR_INVALID_K; read by IVF indexes with centroids only, as on one GPU); k > VIX_MAX_K_LARGE (VIX_ERR_INVALID_K); k >
 * VIX_MAX_K with nq >= 2^31 - 1 (VIX_ERR_INVALID_PARAM); an untrained IVF-PQ index (VIX_ERR_NOT_TRAINED) or one with cosine
 * (VIX_ERR_UNSUPPORTED).  vix_comm_trace records three phases: queries in | local search | assembly (range: exchange and
 * concatenation).  VIX_SCAN_DEBUG=1 prints one "[vix replicated] world W, peer P, kind K, op knn|range|add, block B, total
 * T, grown 0|1" line per call and rank at world > 1 (B: this rank's queries or rows, T: entries of the answer or rows
 * appended). */
int vix_replicated_add(vix_index_t* h, vix_comm_t* c, const float* x, const int64_t* ids, int64_t n);
int vix_replicated_search(vix_index_t* h, vix_comm_t* c, const float* queries, int64_t nq, int k, int nprobe,
                          float* out_dist, int64_t* out_ids);
int vix_replicated_search_filtered(vix_index_t* h, vix_comm_t* c, const float* queries, int64_t nq, int k, int nprobe,
                                   const uint64_t* filter_words /* nullable */, int64_t filter_capacity, int filter_mode,
                                   float* out_dist, int64_t* out_ids);
int vix_replicated_range_search(vix_index_t* h, vix_comm_t* c, const float* queries, int64_t nq, float radius, int nprobe,
                                const uint64_t* filter_words /* nullable */, int64_t filter_capacity, int filter_mode,
                                vix_range_result_t** out);

/* Test hook: the assembly of the replicated calls on one GPU, over blocks the caller passes (host or device pointers; world
 * 1 .. 256; rank r's block is vix_sharded_query_block(nq, r, world)).  out_range == NULL: k-NN -- dist_all / ids_all [nq x
 * k] hold the ranks' [count_r x k] blocks rank by rank (raw bits; lims_all is not read); every emulated rank stores its
 * block into the other ranks' buffers as the exchange does, and out_dist / out_ids receive the last rank's buffer.
 * Otherwise range search -- lims_all: every rank's block row starts (count_r + 1 each, rank by rank: nq + world in all);
 * dist_all / ids_all: their rows (API distances, ids) rank by rank; they are keyed, laid out as the exchange holds them and
 * concatenated and decoded (kind and metric: the sign of zero distances, IP -0 but IVF-Flat +0) into a new result object. */
int vix_debug_replica_assemble(const int64_t* lims_all /* nullable for k-NN */, const float* dist_all, const int64_t* ids_all,
                               int world, int64_t nq, int k, int metric, int kind, float* out_dist, int64_t* out_ids,
                               vix_range_result_t** out_range /* nullable */);

/* f-1  The IVF-PQ query with its optional last step (docs/kernel-specs/DONE_22_adc_scan.md:873-878, "7. Optional: exact
 * rerank (kernel #40)"; IVFIndex.swift:1380-1439): ADC search for the rerank_r best candidates per query (k <= rerank_r <=
 * VIX_MAX_K_LARGE; above VIX_MAX_K through the two-pass route of vix_index_search, which synchronises; the re-rank's own
 * limits -- C <= 16384 candidates and its shared memory -- return VIX_ERR_UNSUPPORTED), then rerank_exact_topk over the ORIGINAL vectors with the DenseArray reader: id -> row of xb [N x d] (ids
 * outside [0, N) are missing and skipped).  Outputs as vix_rerank_exact_topk_f32: raw exact scores (L2^2 / dot), best
 * first by (score under the metric's ordering, smaller id), padded with +-inf / id -1.  xb may live on the device (it is
 * staged per call otherwise). */
int vix_index_search_rerank(vix_index_t* h, const float* queries, int64_t nq, int k, int nprobe, int rerank_r,
                            const float* xb, int64_t N, const float* xb_sq_norms /* nullable */, float* out_scores,
                            int64_t* out_ids);

/* same, with the stage timings / scan statistics of vix_index_search_ex (synchronises) */
int vix_index_search_with_probes_ex(vix_index_t* h, const float* queries, int64_t nq, int k, const int32_t* probes,
                                    int nprobe, float* out_dist, int64_t* out_ids, vix_search_stats* stats /* nullable */);
int vix_index_encode(vix_index_t* h, const float* x, int64_t n, int32_t* assign_out, uint8_t* codes_out /* [n x m] */);
int vix_index_add_encoded(vix_index_t* h, const int32_t* assign, const uint8_t* codes, const int64_t* ids, int64_t n);

/* Stage timing without host synchronisation (bench / profiling): after vix_index_trace(h, capacity) the
 * next `capacity` searches WITHOUT a stats struct record their stage events and scanned-code count on
 * the stream and return asynchronously; vix_index_trace_get(h, i, &st) waits for call i and reads them
 * back.  capacity 0 switches tracing off. */
int vix_index_trace(vix_index_t* h, int capacity);
int vix_index_trace_get(vix_index_t* h, int i, vix_search_stats* out);

/* Test hook (not part of the reference surface): the raw TF32 tensor-core scores S~ of the shortlist pass
 * (vix_gemm.cu), out[nq x kc]; device pointers only. */
int vix_debug_tc_scores_f32(const float* queries, int64_t nq, const float* centroids, int kc, int d, int metric,
                            const float* centroid_norms, float* out);

/* Test hook: the list-major tensor-core scan's decode layout of an IVF-PQ index's codes (vix_scan.cuh), as the next search
 * reads it (the lists are rebuilt first if rows were added).  *bytes_out = list slots x m, or 0 when the index keeps no such
 * layout (only L2 indexes with ks = 256, d = 2 m and m in {16, 32, 48, 64} do); out (host or device, nullable) receives
 * the bytes when cap holds them. */
int vix_debug_tc_codes(vix_index_t* h, uint8_t* out, int64_t cap, int64_t* bytes_out);
/* Test hook: the list-major scan's seed alone, thr[q] = the k-th smallest exact key (the query-major scan's distance) of the
 * first 256 stored vectors of the query's first probed list that holds vectors, +inf when there are fewer than k;
 * k <= 64, L2, ks = 256, dsub = 2, m in {16, 32, 48, 64} */
int vix_debug_tc_seed(vix_index_t* h, const float* queries, int64_t nq, int k, const int32_t* probes, int nprobe, float* thr);

/* Test hook: the result merge of vix_sharded_search on one GPU.  dist_all / ids_all: [world x nq x k] per-rank top-k
 * lists as the ranks' scans return them (API distances, ids; id -1 = none); they are packed into keys and merged by the
 * kernels the exchange runs, into out [nq x k] (host or device pointers). */
int vix_debug_shard_merge(const float* dist_all, const int64_t* ids_all, int world, int64_t nq, int k, int metric,
                          float* out_dist, int64_t* out_ids);

/* Test hook: the merge of vix_sharded_range_search on one GPU.  lims_all: [world x (nq + 1)] the ranks' CSR row starts;
 * dist_all / ids_all: their rows (API distances, ids), concatenated rank by rank, each row sorted by (distance, id) as
 * vix_index_range_search returns it.  They are packed into keys and merged and decoded by the kernels the exchange runs
 * (metric: the sign of zero distances), into a new result object (host or device pointers; world 1 .. 256). */
int vix_debug_shard_range_merge(const int64_t* lims_all /* [world x (nq + 1)] */, const float* dist_all,
                                const int64_t* ids_all /* concatenated rank by rank */, int world, int64_t nq, int metric,
                                vix_range_result_t** out);

/* Test hook: the merge and cut of vix_sharded_search with k > VIX_MAX_K on one GPU.  Input as vix_debug_shard_range_merge
 * (each rank's rows sorted by (distance, id), of any length); the merged rows are cut at k into out [nq x k], padded with
 * id -1 / NaN (host or device pointers; world 1 .. 256, 1 <= k <= VIX_MAX_K_LARGE). */
int vix_debug_shard_knn_merge(const int64_t* lims_all /* [world x (nq + 1)] */, const float* dist_all,
                              const int64_t* ids_all /* concatenated rank by rank */, int world, int64_t nq, int k, int metric,
                              float* out_dist, int64_t* out_ids);

/* Test hook: the merge of the flat kind's sharded k-NN search on one GPU.  lims_all: [world x (nq + 1)] the ranks' CSR row
 * starts; score_all / ids_all: their rows as the flat engine selects them -- RAW scores (L2^2, dot, cosine similarity) and
 * ids, concatenated rank by rank, each row in the flat search's order (score in the metric's order, then row).  They are
 * keyed (score word, id) and merged by the score word and then the rank, as one GPU holding the ranks' rows rank by rank
 * orders them, then mapped to API distances (sqrt, -s, 1 - s).  k > 0: the merged rows cut at k into out [nq x k], padded
 * with id -1 / NaN; k == 0: the whole merged rows into out [total] and their starts into out_lims [nq + 1] (nullable)
 * (host or device pointers; world 1 .. 256, 0 <= k <= VIX_MAX_K_LARGE). */
int vix_debug_shard_flat_merge(const int64_t* lims_all /* [world x (nq + 1)] */, const float* score_all,
                               const int64_t* ids_all /* concatenated rank by rank */, int world, int64_t nq, int k, int metric,
                               int64_t* out_lims /* nullable */, float* out_dist, int64_t* out_ids);

/* Test hook: a sharded call with every rank on one GPU.  shards: the world ranks' handles (distinct, one kind, metric and
 * dimension; each holds what that rank would hold after vix_sharded_add).  Every rank's local pass runs as in
 * vix_sharded_search / vix_sharded_search_filtered / vix_sharded_range_search (the probes of the whole batch selected once;
 * for k > VIX_MAX_K each rank's seed, the minimum of the ranks' bounds, each rank's collect cut at k) and the answer is merged
 * by the kernels the exchange runs; only the transport between the ranks is left out.  out_range == NULL: k-NN into out_dist
 * / out_ids [nq x k] (k <= 0 or nq == 0: nothing); otherwise range search with `radius` into a new result object.  Filter
 * arguments as vix_sharded_search_filtered (filter_words NULL: none). */
int vix_debug_sharded_emulate(vix_index_t* const* shards, int world, const float* queries, int64_t nq, int k, int nprobe,
                              float radius, const uint64_t* filter_words /* nullable */, int64_t filter_capacity,
                              int filter_mode, float* out_dist, int64_t* out_ids, vix_range_result_t** out_range /* nullable */);

/* a16  AccelerableIndex-shaped convenience (AccelerableIndex.swift:15-127): candidates [c x d]
 * contiguous in, (indices into candidates, distances) out, per query. */
int vix_accel_rank_candidates_f32(const float* queries, int64_t nq, const float* candidates, int64_t c,
                                  int d, int metric, int k, int32_t* out_indices, float* out_distances);

#ifdef __cplusplus
}
#endif
#endif /* VINDEX_CUDA_H */
