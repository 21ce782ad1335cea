// vix_train.cu -- coarse-quantiser and PQ-codebook training on the GPU (a10 / a12).
//
// Two modes (vix_kmeans_cfg.mode / vix_pq_train_cfg.mode):
//   mode 1 "sane"   deterministic Lloyd iterations on a strided sample with standard empty-cluster
//                   handling -- what the benchmark configurations are built with (the reference's
//                   mini-batch trainer collapses at nlist >= 1024, SURVEY.md section 0.6);
//   mode 0 "parity" the reference's control flow (RNG streams, batch composition, repairs) replayed on
//                   the host with every distance pass, argmin and f64 accumulation on the GPU in the
//                   reference's order (vix_train_parity.cu).
//
// Both modes build on the same blocks: bit-exact assignment kernels (vix_scoring.cu / vix_pq_encode.cu), the
// stable grouping of rows by assignment (vix_group.cu), and a deterministic centroid update -- each (centroid,
// component) is summed sequentially in f64 in the order of the stably sorted rows, which is exactly the
// reference's accumulation order (KMeansMiniBatchKernel.swift:582, PQTrain.swift:1111), with no atomics on the
// value path, so results are reproducible run to run and rank to rank.
#include "vix_common.cuh"
#include "vix_exact.cuh"
#include "vix_group.cuh"

#include <vector>

namespace vix {

int ivf_assign_device(const float* x, int64_t n, int d, const float* c, int kc, int32_t* assign, float* dist);
int ivf_assign_auto_device(const float* x, int64_t n, int d, const float* c, int kc, int32_t* assign, float* dist);
int pq_encode_device(const float* x, int64_t n, int d, int m, int ks, const float* cb, const float* csq,
                     const float* coarse, const int32_t* assign, uint8_t* codes, int use_dot, int layout,
                     int B, int g, int u4);

// centroid c := mean of its members, f64 sums in data order (rows sorted stably by assignment).
// One CTA per centroid, threads over components.  Empty centroids are left untouched.
__global__ void centroid_update_kernel(const float* __restrict__ x, int d, int x_ld, int x_off,
                                       const int32_t* __restrict__ sorted_rows, const int64_t* __restrict__ off,
                                       int kc, float* __restrict__ centroids, int c_ld, int c_off) {
    const int c = blockIdx.x;
    if (c >= kc) return;
    const int64_t b = off[c], e = off[c + 1];
    if (e <= b) return;
    const double inv = 1.0 / (double)(e - b);
    for (int t = threadIdx.x; t < d; t += blockDim.x) {
        double acc = 0.0;
        for (int64_t i = b; i < e; ++i) acc += (double)x[(int64_t)sorted_rows[i] * x_ld + x_off + t];
        centroids[(int64_t)c * c_ld + c_off + t] = (float)(acc * inv);
    }
}

// Deterministic repair of empty centroids: the e-th empty centroid (ascending) takes the row
// rows_by_dist_desc[e] -- the points currently farthest from their centroid (standard "split the worst
// fitted points" policy; PQTrain's .split policy uses the same farthest-first idea, PQTrain.swift:1148-1177).
__global__ void repair_empty_kernel(const float* __restrict__ x, int d, int x_ld, int x_off,
                                    const int32_t* __restrict__ cnt, int kc, const int32_t* __restrict__ far_rows,
                                    int64_t nfar, float* __restrict__ centroids, int c_ld, int c_off,
                                    int32_t* __restrict__ n_empty_out) {
    __shared__ int s_rank;
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        int e = 0;
        for (int c = 0; c < kc; ++c) if (cnt[c] == 0) {
            if (e < nfar) {
                const float* src = x + (int64_t)far_rows[e] * x_ld + x_off;
                for (int t = 0; t < d; ++t) centroids[(int64_t)c * c_ld + c_off + t] = src[t];
            }
            ++e;
        }
        *n_empty_out = e;
        s_rank = e;
    }
}

static int sort_by_assignment(const int32_t* assign, int64_t n, int kc, Scratch<int32_t>& rows_sorted,
                              Scratch<int32_t>& cnt, Scratch<int64_t>& off) {
    VIX_TRY(rows_sorted.alloc((size_t)n));
    VIX_TRY(cnt.alloc((size_t)kc));
    VIX_TRY(off.alloc((size_t)kc + 1));
    VIX_TRY(order_by_key(assign, n, kc, rows_sorted.ptr));
    return key_offsets(assign, n, kc, cnt.ptr, off.ptr);
}

// rows sorted by descending distance (ties: ascending row): keys = ~orderable(dist)
__global__ void dist_keys_kernel(const float* __restrict__ dist, int64_t n, uint32_t* __restrict__ keys) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) keys[i] = ~f32_orderable(dist[i]);
}

static int farthest_rows(const float* dist, int64_t n, Scratch<int32_t>& rows_sorted) {
    cudaStream_t s = ctx().stream;
    Scratch<uint32_t> keys, keys_out;
    Scratch<int32_t> rows_in;
    VIX_TRY(keys.alloc((size_t)n));
    VIX_TRY(keys_out.alloc((size_t)n));
    VIX_TRY(rows_in.alloc((size_t)n));
    VIX_TRY(rows_sorted.alloc((size_t)n));
    dist_keys_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(dist, n, keys.ptr);
    VIX_LAUNCH_CHECK();
    VIX_TRY(iota<int32_t>(rows_in.ptr, n, 0));
    return sort_pairs<uint32_t>(keys.ptr, keys_out.ptr, rows_in.ptr, rows_sorted.ptr, n, 32);
}

// LCG of the reference (Utilities/RNG.swift:61-65) for the deterministic sample / init choices
static inline uint64_t lcg_next(uint64_t& s) { s = 2862933555777941757ULL * s + 3037000493ULL; return s; }

// distinct pseudo-random rows: a multiplicative walk over [0, n) with a stride coprime to n
static void distinct_rows(int64_t n, int64_t count, uint64_t seed, std::vector<int64_t>& out) {
    out.resize((size_t)count);
    uint64_t s = seed ? seed : 1;
    int64_t stride = (int64_t)(lcg_next(s) % (uint64_t)n);
    if (stride == 0) stride = 1;
    auto gcd = [](int64_t a, int64_t b) { while (b) { int64_t t = a % b; a = b; b = t; } return a; };
    while (gcd(stride, n) != 1) ++stride;
    int64_t pos = (int64_t)(lcg_next(s) % (uint64_t)n);
    for (int64_t i = 0; i < count; ++i) { out[(size_t)i] = pos; pos = (pos + stride) % n; }
}

// Lloyd on device rows xs[ns x d] (sub-space [x_off, x_off + dd) of rows with leading dimension x_ld).
// assign_fn(centroids) must fill assign[ns] / dist[ns].
template <typename AssignFn>
static int lloyd_device(const float* xs, int64_t ns, int dd, int x_ld, int x_off, int kc, int iters,
                        float* centroids, int c_ld, int c_off, int32_t* assign, float* dist, AssignFn assign_fn) {
    cudaStream_t s = ctx().stream;
    Scratch<int32_t> n_empty;
    VIX_TRY(n_empty.alloc(1));
    for (int it = 0; it < iters; ++it) {
        VIX_TRY(assign_fn());
        Scratch<int32_t> rows_sorted, cnt, far;
        Scratch<int64_t> off;
        VIX_TRY(sort_by_assignment(assign, ns, kc, rows_sorted, cnt, off));
        centroid_update_kernel<<<kc, dd < 256 ? (dd < 32 ? 32 : dd) : 256, 0, s>>>(xs, dd, x_ld, x_off, rows_sorted.ptr,
                                                                                  off.ptr, kc, centroids, c_ld, c_off);
        VIX_LAUNCH_CHECK();
        VIX_TRY(farthest_rows(dist, ns, far));
        repair_empty_kernel<<<1, 32, 0, s>>>(xs, dd, x_ld, x_off, cnt.ptr, kc, far.ptr, ns, centroids, c_ld, c_off,
                                             n_empty.ptr);
        VIX_LAUNCH_CHECK();
    }
    return VIX_OK;
}

// ------------------------------------------------------------------------------------------------
// coarse quantiser, mode 1
// ------------------------------------------------------------------------------------------------
int train_coarse_device(const float* x, int64_t n, int d, int kc, int metric, const vix_kmeans_cfg* cfg,
                        float* centroids_out) {
    (void)metric;   // the reference trains with L2 k-means whatever the metric (IVFIndex.swift:337-341)
    cudaStream_t s = ctx().stream;
    const int iters = (cfg && cfg->epochs > 0) ? cfg->epochs : 10;
    const uint64_t seed = cfg ? cfg->seed : 42;
    // sample: at most 64 points per centroid
    int64_t ns = n;
    const int64_t cap = (int64_t)kc * 64;
    if (ns > cap) ns = cap;
    if (ns < kc) ns = n;
    std::vector<int64_t> rows;
    Scratch<float> xs;
    const float* xp = x;
    if (ns < n) {
        distinct_rows(n, ns, seed ^ 0x9E3779B97F4A7C15ULL, rows);
        Scratch<int64_t> drows;
        VIX_TRY(drows.alloc((size_t)ns));
        VIX_CUDA(cudaMemcpyAsync(drows.ptr, rows.data(), (size_t)ns * 8, cudaMemcpyHostToDevice, s));
        VIX_TRY(xs.alloc((size_t)ns * d));
        VIX_TRY(gather_rows(x, d, drows.ptr, ns, xs.ptr));
        VIX_CUDA(cudaStreamSynchronize(s));
        xp = xs.ptr;
    }
    // init: kc distinct sample rows
    {
        std::vector<int64_t> init;
        distinct_rows(ns, kc, seed, init);
        Scratch<int64_t> dinit;
        VIX_TRY(dinit.alloc((size_t)kc));
        VIX_CUDA(cudaMemcpyAsync(dinit.ptr, init.data(), (size_t)kc * 8, cudaMemcpyHostToDevice, s));
        VIX_TRY(gather_rows(xp, d, dinit.ptr, kc, centroids_out));
        VIX_CUDA(cudaStreamSynchronize(s));
    }
    Scratch<int32_t> assign;
    Scratch<float> dist;
    VIX_TRY(assign.alloc((size_t)ns));
    VIX_TRY(dist.alloc((size_t)ns));
    return lloyd_device(xp, ns, d, d, 0, kc, iters, centroids_out, d, 0, assign.ptr, dist.ptr, [&]() {
        return ivf_assign_auto_device(xp, ns, d, centroids_out, kc, assign.ptr, dist.ptr);
    });
}

// ------------------------------------------------------------------------------------------------
// PQ codebooks, mode 1: Lloyd per sub-space on (residual) sample rows.  The assignment of all m
// sub-spaces is ONE launch of the encode kernel (direct L2, tie -> lower k).
// ------------------------------------------------------------------------------------------------
__global__ void residual_rows_kernel(const float* __restrict__ x, int d, const int64_t* __restrict__ rows, int64_t ns,
                                     const float* __restrict__ coarse, const int32_t* __restrict__ assign,
                                     float* __restrict__ out) {
    const int64_t i = blockIdx.x;
    if (i >= ns) return;
    const int64_t r = rows ? rows[i] : i;
    const float* src = x + r * (int64_t)d;
    const float* c = coarse ? coarse + (int64_t)assign[r] * d : nullptr;
    for (int e = threadIdx.x; e < d; e += blockDim.x) out[i * (int64_t)d + e] = c ? __fsub_rn(src[e], c[e]) : src[e];
}

__global__ void codes_column_kernel(const uint8_t* __restrict__ codes, int64_t ns, int m, int j,
                                    int32_t* __restrict__ out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < ns) out[i] = codes[i * (int64_t)m + j];
}

// per-row squared distance of sub-vector j to its assigned centroid (for the empty-cluster repair)
__global__ void sub_dist_kernel(const float* __restrict__ xs, int64_t ns, int d, int j, int dsub,
                                const float* __restrict__ cb, int ks, const int32_t* __restrict__ assign,
                                float* __restrict__ dist) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ns) return;
    const float* a = xs + i * (int64_t)d + (size_t)j * dsub;
    const float* c = cb + ((size_t)j * ks + assign[i]) * dsub;
    dist[i] = exact_pair<SpecKm11L2>(a, c, dsub);
}

int train_pq_device(const float* x, int64_t n, int d, int m, int ks, const float* coarse, const int32_t* assign,
                    const vix_pq_train_cfg* cfg, float* codebooks_out, float* norms_out) {
    cudaStream_t s = ctx().stream;
    const int dsub = d / m;
    const int iters = (cfg && cfg->max_iters > 0) ? cfg->max_iters : 25;
    const uint64_t seed = cfg ? cfg->seed : 42;
    int64_t ns = n;
    int64_t cap = (cfg && cfg->sample_n > 0) ? cfg->sample_n : (int64_t)ks * 256;
    if (ns > cap) ns = cap;
    VIX_REQUIRE(ns >= 1, VIX_ERR_EMPTY_INPUT, "pq train: empty input");
    std::vector<int64_t> rows;
    Scratch<int64_t> drows;
    if (ns < n) {
        distinct_rows(n, ns, seed ^ 0xD1B54A32D192ED03ULL, rows);
        VIX_TRY(drows.alloc((size_t)ns));
        VIX_CUDA(cudaMemcpyAsync(drows.ptr, rows.data(), (size_t)ns * 8, cudaMemcpyHostToDevice, s));
    }
    Scratch<float> xs;
    VIX_TRY(xs.alloc((size_t)ns * d));
    residual_rows_kernel<<<(unsigned)ns, 128, 0, s>>>(x, d, ns < n ? drows.ptr : nullptr, ns, coarse, assign, xs.ptr);
    VIX_LAUNCH_CHECK();
    VIX_CUDA(cudaStreamSynchronize(s));
    // init: ks distinct sample rows per sub-space (same rows for every j; sub-vectors differ)
    {
        std::vector<int64_t> init;
        const int64_t take = ks <= ns ? ks : ns;
        distinct_rows(ns, take, seed, init);
        std::vector<int64_t> full((size_t)ks);
        for (int k = 0; k < ks; ++k) full[(size_t)k] = init[(size_t)(k % take)];
        Scratch<int64_t> dinit;
        Scratch<float> tmp;
        VIX_TRY(dinit.alloc((size_t)ks));
        VIX_TRY(tmp.alloc((size_t)ks * d));
        VIX_CUDA(cudaMemcpyAsync(dinit.ptr, full.data(), (size_t)ks * 8, cudaMemcpyHostToDevice, s));
        VIX_TRY(gather_rows(xs.ptr, d, dinit.ptr, ks, tmp.ptr));
        // tmp[k][j*dsub + e] -> codebooks[j][k][e]
        for (int j = 0; j < m; ++j)
            VIX_CUDA(cudaMemcpy2DAsync(codebooks_out + (size_t)j * ks * dsub, (size_t)dsub * 4, tmp.ptr + (size_t)j * dsub,
                                       (size_t)d * 4, (size_t)dsub * 4, (size_t)ks, cudaMemcpyDeviceToDevice, s));
        VIX_CUDA(cudaStreamSynchronize(s));
    }
    Scratch<uint8_t> codes;
    Scratch<int32_t> col;
    Scratch<float> dist;
    Scratch<int32_t> n_empty;
    VIX_TRY(codes.alloc((size_t)ns * m));
    VIX_TRY(col.alloc((size_t)ns));
    VIX_TRY(dist.alloc((size_t)ns));
    VIX_TRY(n_empty.alloc(1));
    for (int it = 0; it < iters; ++it) {
        // direct L2 argmin, tie -> lower k, all sub-spaces at once
        VIX_TRY(pq_encode_device(xs.ptr, ns, d, m, ks, codebooks_out, nullptr, nullptr, nullptr, codes.ptr, 0,
                                 PQ_LAYOUT_AOS, 64, 8, 0));
        for (int j = 0; j < m; ++j) {
            codes_column_kernel<<<(unsigned)((ns + 255) / 256), 256, 0, s>>>(codes.ptr, ns, m, j, col.ptr);
            VIX_LAUNCH_CHECK();
            sub_dist_kernel<<<(unsigned)((ns + 255) / 256), 256, 0, s>>>(xs.ptr, ns, d, j, dsub, codebooks_out, ks, col.ptr,
                                                                        dist.ptr);
            VIX_LAUNCH_CHECK();
            Scratch<int32_t> rows_sorted, cnt, far;
            Scratch<int64_t> off;
            VIX_TRY(sort_by_assignment(col.ptr, ns, ks, rows_sorted, cnt, off));
            float* cbj = codebooks_out + (size_t)j * ks * dsub;
            centroid_update_kernel<<<ks, 32, 0, s>>>(xs.ptr, dsub, d, j * dsub, rows_sorted.ptr, off.ptr, ks, cbj, dsub, 0);
            VIX_LAUNCH_CHECK();
            VIX_TRY(farthest_rows(dist.ptr, ns, far));
            repair_empty_kernel<<<1, 32, 0, s>>>(xs.ptr, dsub, d, j * dsub, cnt.ptr, ks, far.ptr, ns, cbj, dsub, 0,
                                                 n_empty.ptr);
            VIX_LAUNCH_CHECK();
        }
    }
    if (norms_out) VIX_TRY(seq_norms(codebooks_out, (int64_t)m * ks, dsub, norms_out));
    return VIX_OK;
}

int kmeans_parity_device(const float* x, int64_t n, int d, int kc, const float* init, const vix_kmeans_cfg* cfg,
                         float* centroids_out, int32_t* assign_out);
int kmeanspp_parity_device(const float* x, int64_t n, int d, int k, uint64_t seed, uint64_t stream, float* centroids_out,
                           int64_t* chosen_out);
int pq_train_streaming_parity_device(const float* X, const std::vector<int64_t>& chunk_n, int d, int m, int ks,
                                     const vix_pq_train_cfg* cfg, float* codebooks_out, float* norms_out);
int pq_train_parity_device(const float* x, int64_t n, int d, int m, int ks, const float* coarse, const int32_t* assign,
                           const vix_pq_train_cfg* cfg, float* codebooks_out, float* norms_out);

}  // namespace vix

using namespace vix;

extern "C" {

int vix_kmeanspp_seed_f32(const float* data, int64_t n, int d, int k, uint64_t seed, uint64_t stream_id,
                          float* centroids_out, int64_t* chosen_out) {
    VIX_TRY(ensure_device());
    VIX_REQUIRE(data && centroids_out, VIX_ERR_NULL_PTR, "vix_kmeanspp_seed_f32: null pointer");
    VIX_REQUIRE(d > 0 && n > 0, VIX_ERR_INVALID_DIM, "vix_kmeanspp_seed_f32: bad shape");
    VIX_REQUIRE(k > 0 && k <= n, VIX_ERR_INVALID_K, "vix_kmeanspp_seed_f32: need 1 <= k <= n");
    In<float> dx;
    Out<float> dc;
    VIX_TRY(dx.stage(data, (size_t)n * d));
    VIX_TRY(dc.stage(centroids_out, (size_t)k * d));
    VIX_REQUIRE(!chosen_out || !is_device_ptr(chosen_out), VIX_ERR_INVALID_PARAM, "chosen_out must be a host pointer");
    VIX_TRY(kmeanspp_parity_device(dx.dev, n, d, k, seed, stream_id, dc.dev, chosen_out));
    VIX_TRY(dc.commit());
    return finish(true);
}

int vix_kmeans_minibatch_f32(const float* x, int64_t n, int d, int kc, const float* init_centroids,
                             const vix_kmeans_cfg* cfg, float* centroids_out, int32_t* assign_out) {
    VIX_TRY(ensure_device());
    VIX_REQUIRE(x && centroids_out, VIX_ERR_NULL_PTR, "vix_kmeans_minibatch_f32: null pointer");
    VIX_REQUIRE(d > 0 && n > 0, VIX_ERR_INVALID_DIM, "vix_kmeans_minibatch_f32: bad shape");
    VIX_REQUIRE(kc > 0 && kc <= n, VIX_ERR_INVALID_K, "vix_kmeans_minibatch_f32: need 1 <= kc <= n");
    In<float> dx, dinit;
    Out<float> dc;
    Out<int32_t> da;
    VIX_TRY(dx.stage(x, (size_t)n * d));
    VIX_TRY(dinit.stage(init_centroids, init_centroids ? (size_t)kc * d : 0));
    VIX_TRY(dc.stage(centroids_out, (size_t)kc * d));
    VIX_TRY(da.stage(assign_out, assign_out ? (size_t)n : 0));
    int rc;
    if (cfg && cfg->mode == 1) {
        rc = train_coarse_device(dx.dev, n, d, kc, VIX_METRIC_L2, cfg, dc.dev);
        if (rc == VIX_OK && da.dev) rc = ivf_assign_auto_device(dx.dev, n, d, dc.dev, kc, da.dev, nullptr);
    } else {
        rc = kmeans_parity_device(dx.dev, n, d, kc, dinit.dev, cfg, dc.dev, da.dev);
    }
    if (rc < 0) return rc;
    VIX_TRY(dc.commit());
    VIX_TRY(da.commit());
    VIX_TRY(finish(true));
    return rc;
}

int vix_pq_train_f32(const float* x, int64_t n, int d, int m, int ks, const float* coarse_centroids,
                     const int32_t* assignments, const vix_pq_train_cfg* cfg, float* codebooks_out,
                     float* centroid_norms_out) {
    VIX_TRY(ensure_device());
    VIX_REQUIRE(x && codebooks_out, VIX_ERR_NULL_PTR, "vix_pq_train_f32: null pointer");
    VIX_REQUIRE(n > 0, VIX_ERR_EMPTY_INPUT, "vix_pq_train_f32: empty input");                 // PQTrain.swift:96-135
    VIX_REQUIRE(d > 0 && m > 0 && d % m == 0, VIX_ERR_INVALID_DIM, "vix_pq_train_f32: need d %% m == 0");
    VIX_REQUIRE(ks > 0 && ks <= 256, VIX_ERR_INVALID_K, "vix_pq_train_f32: ks must be in 1..256");
    VIX_REQUIRE((coarse_centroids == nullptr) == (assignments == nullptr), VIX_ERR_CONTRACT,
                "vix_pq_train_f32: coarse_centroids and assignments must be given together");
    {   // PQTrain.swift:127-135: fewer training vectors (after sampling) than centroids => .emptyInput
        const int64_t need_n = (cfg && cfg->sample_n > 0) ? cfg->sample_n : n;
        VIX_REQUIRE(need_n >= ks, VIX_ERR_EMPTY_INPUT,
                    "vix_pq_train_f32: Insufficient training data: need at least ks vectors (%lld available, ks = %d)",
                    (long long)need_n, ks);
    }
    In<float> dx, dco;
    In<int32_t> das;
    Out<float> dcb, dn;
    VIX_TRY(dx.stage(x, (size_t)n * d));
    if (coarse_centroids) {
        VIX_TRY(das.stage(assignments, (size_t)n));
        int64_t rows = 0;
        if (!is_device_ptr(coarse_centroids)) {
            VIX_REQUIRE(!is_device_ptr(assignments), VIX_ERR_INVALID_PARAM, "host coarse with device assignments");
            for (int64_t i = 0; i < n; ++i) if (assignments[i] + 1 > rows) rows = assignments[i] + 1;
        }
        VIX_TRY(dco.stage(coarse_centroids, (size_t)rows * d));
    }
    VIX_TRY(dcb.stage(codebooks_out, (size_t)ks * d));
    VIX_TRY(dn.stage(centroid_norms_out, centroid_norms_out ? (size_t)m * ks : 0));
    int rc;
    if (cfg && cfg->mode == 1) {
        VIX_REQUIRE(ks == 256, VIX_ERR_INVALID_K, "vix_pq_train_f32 (mode 1): ks must be 256");
        rc = train_pq_device(dx.dev, n, d, m, ks, coarse_centroids ? dco.dev : nullptr, coarse_centroids ? das.dev : nullptr,
                             cfg, dcb.dev, dn.dev);
    } else {
        rc = pq_train_parity_device(dx.dev, n, d, m, ks, coarse_centroids ? dco.dev : nullptr,
                                    coarse_centroids ? das.dev : nullptr, cfg, dcb.dev, dn.dev);
    }
    if (rc < 0) return rc;
    VIX_TRY(dcb.commit());
    VIX_TRY(dn.commit());
    VIX_TRY(finish(true));
    return rc;
}

int vix_pq_train_streaming_f32(const float* const* chunks, const int64_t* chunk_n, int nchunks, int d, int m, int ks,
                               const vix_pq_train_cfg* cfg, float* codebooks_out, float* centroid_norms_out) {
    VIX_TRY(ensure_device());
    VIX_REQUIRE(chunks && chunk_n && codebooks_out, VIX_ERR_NULL_PTR, "vix_pq_train_streaming_f32: null pointer");
    VIX_REQUIRE(nchunks > 0, VIX_ERR_EMPTY_INPUT, "vix_pq_train_streaming_f32: no chunks");
    VIX_REQUIRE(d > 0 && m > 0 && d % m == 0, VIX_ERR_INVALID_DIM, "vix_pq_train_streaming_f32: need d %% m == 0");
    VIX_REQUIRE(ks >= 1 && ks <= 256, VIX_ERR_INVALID_K, "vix_pq_train_streaming_f32: ks must be in 1..256");
    std::vector<int64_t> cn((size_t)nchunks);
    int64_t total = 0;
    for (int c = 0; c < nchunks; ++c) {
        VIX_REQUIRE(chunk_n[c] >= 0 && (chunk_n[c] == 0 || chunks[c]), VIX_ERR_NULL_PTR, "vix_pq_train_streaming_f32: chunk %d", c);
        cn[(size_t)c] = chunk_n[c];
        total += chunk_n[c];
    }
    VIX_REQUIRE(total >= ks, VIX_ERR_EMPTY_INPUT,
                "vix_pq_train_streaming_f32: Insufficient training data: need at least ks vectors (%lld available, ks = %d)",
                (long long)total, ks);
    // the chunks (host or device, each valid for the call) laid end to end on the device
    Scratch<float> X;
    VIX_TRY(X.alloc((size_t)total * d));
    int64_t at = 0;
    for (int c = 0; c < nchunks; ++c) {
        if (cn[(size_t)c] == 0) continue;
        VIX_CUDA(cudaMemcpyAsync(X.ptr + (size_t)at * d, chunks[c], (size_t)cn[(size_t)c] * d * 4, cudaMemcpyDefault, ctx().stream));
        at += cn[(size_t)c];
    }
    Out<float> dcb, dn;
    VIX_TRY(dcb.stage(codebooks_out, (size_t)ks * d));
    VIX_TRY(dn.stage(centroid_norms_out, centroid_norms_out ? (size_t)m * ks : 0));
    VIX_TRY(pq_train_streaming_parity_device(X.ptr, cn, d, m, ks, cfg, dcb.dev, dn.dev));
    VIX_TRY(dcb.commit());
    VIX_TRY(dn.commit());
    return finish(true);
}

}  // extern "C"
