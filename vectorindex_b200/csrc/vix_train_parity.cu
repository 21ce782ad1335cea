// vix_train_parity.cu -- reference-parity trainers (cfg.mode == 0): the reference's control flow -- RNG streams,
// batch composition, repairs, stopping rules -- replayed on the host, with every distance, argmin and f64
// centroid accumulation on the GPU in the reference's operation order.
//
//   kmeansPlusPlusSeed      Kernels/KMeansSeeding.swift:167-409         (RNGState LCG, Utilities/RNG.swift:33-104)
//   kmeans_minibatch_f32    Kernels/KMeansMiniBatchKernel.swift:401-724 (lloydMiniBatch, AoS, incl. the quirks of
//                           SURVEY.md section 0.6: batches drawn with replacement, "empties" = untouched this batch,
//                           all repaired with the batch point farthest from centroid 0)
//   pq_train_f32            Kernels/PQTrain.swift:83-388, 856-1442      (Xoroshiro128**, selection sampling, k-means++
//                           per sub-space, Lloyd with .split/.reseed/.ignore repair, mini-batch with running-mean blend)
//
// What has to be sequential in the reference stays sequential here: the f64 D^2 cumulative sums of the samplers and
// the f64 distortion sums run on the host over values computed by the GPU; the per-centroid f64 sums of Lloyd are
// taken on the GPU in row order (rows stably sorted by assignment, one sequential f64 chain per centroid component),
// which is the reference's accumulation order (PQTrain.swift:1111).
#include "vix_common.cuh"
#include "vix_exact.cuh"
#include "vix_group.cuh"

#include <algorithm>
#include <vector>

namespace vix {

int ivf_assign_device(const float* x, int64_t n, int d, const float* c, int kc, int32_t* assign, float* dist);

namespace {

// ------------------------------------------------------------------------------------------------ RNGs (host)
struct Lcg {                                                  // Utilities/RNG.swift:47-103
    uint64_t s;
    Lcg(uint64_t seed, uint64_t stream) : s((seed == 0 ? 1 : seed) ^ (stream << 32)) {}
    uint64_t next() { s = 2862933555777941757ULL * s + 3037000493ULL; return s; }
    double next_double() { return (double)(next() >> 11) / 9007199254740992.0; }
    int64_t next_int(int64_t bound) { return (int64_t)(next() % (uint64_t)bound); }
};

struct Xoro {                                                 // Kernels/PQTrain.swift:712-759
    uint64_t s0, s1;
    static uint64_t rotl(uint64_t x, unsigned k) { return (x << k) | (x >> (64 - k)); }
    static uint64_t splitmix(uint64_t& st) {
        st += 0x9E3779B97F4A7C15ULL;
        uint64_t z = st;
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
        return z ^ (z >> 31);
    }
    Xoro(uint64_t seed, uint64_t stream, uint64_t task) {
        uint64_t s = seed ^ (stream * 0xD1B54A32D192ED03ULL) ^ (task * 0x94D049BB133111EBULL);
        const uint64_t a = splitmix(s), b = splitmix(s);
        if (a != 0 || b != 0) { s0 = a; s1 = b; }
        else { s0 = 0x9E3779B97F4A7C15ULL; s1 = 0xD1B54A32D192ED03ULL; }
    }
    uint64_t u64() {
        const uint64_t r = rotl(s0 * 5, 7) * 9, t = s0 ^ s1;
        s0 = rotl(s0, 24) ^ t ^ (t << 16);
        s1 = rotl(t, 37);
        return r;
    }
    uint32_t u32() { return (uint32_t)(u64() >> 32); }
    double f64() { return (double)(u64() >> 11) * (1.0 / 9007199254740992.0); }
};

void randperm(std::vector<uint32_t>& a, Xoro& r) {            // PQTrain.swift:761-768
    for (int64_t i = (int64_t)a.size() - 1; i >= 1; --i) {
        const int64_t j = (int64_t)(((uint64_t)r.u32() * (uint64_t)(i + 1)) >> 32);
        std::swap(a[(size_t)i], a[(size_t)j]);
    }
}
int64_t sample_wo_repl(uint32_t n, uint32_t k, Xoro& r, std::vector<uint32_t>& out) {   // :770-782 selection sampling
    out.assign(k, 0);
    uint32_t t = 0, m = 0;
    while (m < k && t < n) {
        const double u = r.f64();
        if ((double)(n - t) * u >= (double)(k - m)) t += 1;
        else { out[m] = t; t += 1; m += 1; }
    }
    return m;
}

// ------------------------------------------------------------------------------------------------ device pieces
// A set of sub-vectors: row t is x[(idx ? idx[t] : t) * ld + off .. + dsub), optionally as a residual against the
// coarse centroid of its row (coarse[assign[row] * cd + off ..]).
struct SubSrc {
    const float* x; int64_t ld; int off; int dsub;
    const uint32_t* idx;
    const float* coarse; const int32_t* assign; int cd;
};
__device__ __forceinline__ void sub_ptrs(const SubSrc& s, int64_t t, const float*& xs, const float*& gs) {
    const int64_t r = s.idx ? (int64_t)s.idx[t] : t;
    xs = s.x + r * s.ld + s.off;
    gs = s.coarse ? s.coarse + (int64_t)s.assign[r] * s.cd + s.off : nullptr;
}
// PQTrain l2Sq (PQTrain.swift:797-813) and its residual form ((x - g) - c) (:833-852): two SIMD4 accumulators per
// 8-stride, lane-wise acc0 + acc1, hsum, scalar tail
__device__ __forceinline__ float pq_l2(const float* __restrict__ xs, const float* __restrict__ gs,
                                       const float* __restrict__ c, int dsub) {
    float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    const int l8 = dsub & ~7;
    for (int i = 0; i < l8; i += 8) {
#pragma unroll
        for (int l = 0; l < 8; ++l) {
            const float r = gs ? fsub(fsub(xs[i + l], gs[i + l]), c[i + l]) : fsub(xs[i + l], c[i + l]);
            acc[l] = fadd(acc[l], fmul(r, r));
        }
    }
    float s = hsum4(fadd(acc[0], acc[4]), fadd(acc[1], acc[5]), fadd(acc[2], acc[6]), fadd(acc[3], acc[7]));
    for (int i = l8; i < dsub; ++i) {
        const float r = gs ? fsub(fsub(xs[i], gs[i]), c[i]) : fsub(xs[i], c[i]);
        s = fadd(s, fmul(r, r));
    }
    return s;
}

// out[t] = dist(row t, point)            (init)    or    if (dist < out[t]) out[t] = dist     (update)
__global__ void sub_dist_point_kernel(SubSrc s, int64_t n, const float* __restrict__ point, int use_residual, int update,
                                      float* __restrict__ out) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const float *xs, *gs;
    sub_ptrs(s, t, xs, gs);
    const float dd = pq_l2(xs, use_residual ? gs : nullptr, point, s.dsub);
    if (!update || dd < out[t]) out[t] = dd;
}

// best_k[t] = argmin_k dist(row t, C[k]) (tie -> lower k), best_d[t] = that distance; C [ks x dsub] staged in smem
__global__ void __launch_bounds__(256)
sub_assign_kernel(SubSrc s, int64_t n, const float* __restrict__ C, int ks, int use_residual, int32_t* __restrict__ best_k,
                  float* __restrict__ best_d) {
    extern __shared__ __align__(16) unsigned char smem_sa[];
    float* sc = reinterpret_cast<float*>(smem_sa);
    for (int e = threadIdx.x; e < ks * s.dsub; e += blockDim.x) sc[e] = C[e];
    __syncthreads();
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const float *xs, *gs;
    sub_ptrs(s, t, xs, gs);
    if (!use_residual) gs = nullptr;
    int bk = 0;
    float bd = pq_l2(xs, gs, sc, s.dsub);
    for (int k = 1; k < ks; ++k) {
        const float dk = pq_l2(xs, gs, sc + (size_t)k * s.dsub, s.dsub);
        if (dk < bd || (dk == bd && k < bk)) { bd = dk; bk = k; }
    }
    if (best_k) best_k[t] = bk;
    if (best_d) best_d[t] = bd;
}

// dense[t][u] = x_sub[u] (- g_sub[u])
__global__ void sub_gather_kernel(SubSrc s, int64_t n, int use_residual, float* __restrict__ dense) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n * s.dsub) return;
    const int64_t t = e / s.dsub;
    const int u = (int)(e - t * s.dsub);
    const float *xs, *gs;
    sub_ptrs(s, t, xs, gs);
    dense[e] = (use_residual && gs) ? fsub(xs[u], gs[u]) : xs[u];
}

// Lloyd centroid update: rows stably sorted by assignment; centroid k := mean of its members, f64 sums in row order
// (values are the float residuals x - g when a coarse quantiser is given, PQTrain.swift:1105-1111)
__global__ void sub_centroid_update_kernel(SubSrc s, const int32_t* __restrict__ sorted_rows, const int64_t* __restrict__ off,
                                           int ks, float* __restrict__ C) {
    const int k = blockIdx.x;
    if (k >= ks) return;
    const int64_t b = off[k], e = off[k + 1];
    if (e <= b) return;
    const double inv = 1.0 / (double)(e - b);
    for (int u = threadIdx.x; u < s.dsub; u += blockDim.x) {
        double acc = 0.0;
        for (int64_t i = b; i < e; ++i) {
            const float *xs, *gs;
            sub_ptrs(s, sorted_rows[i], xs, gs);
            acc += gs ? (double)fsub(xs[u], gs[u]) : (double)xs[u];
        }
        C[(size_t)k * s.dsub + u] = (float)(acc * inv);
    }
}

// km11 D^2 update of k-means++ (KMeansSeeding.swift:302-361): d2[i] = min(d2[i], safe(L2^2(x_i, c)))
__global__ void km11_update_kernel(const float* __restrict__ x, int64_t n, int d, const float* __restrict__ c,
                                   float* __restrict__ d2) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float ds = exact_pair<SpecKm11L2>(x + i * d, c, d);
    const float safe = (isfinite(ds) && ds >= 0.0f) ? ds : 0.0f;
    if (safe < d2[i]) d2[i] = safe;
}
// dist[i] = _vi_km12_l2sq_aos(rows[i], c)
__global__ void km12_dist_to_row_kernel(const float* __restrict__ rows, int64_t n, int d, const float* __restrict__ c,
                                        float* __restrict__ dist) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dist[i] = exact_pair<SpecKm12L2>(rows + i * d, c, d);
}
// centroids[list[t]] = rows[t]
__global__ void scatter_rows_kernel(float* __restrict__ centroids, int d, const int32_t* __restrict__ list, int nlist,
                                    const float* __restrict__ rows) {
    const int t = blockIdx.x;
    if (t >= nlist) return;
    for (int e = threadIdx.x; e < d; e += blockDim.x) centroids[(int64_t)list[t] * d + e] = rows[(int64_t)t * d + e];
}
// centroids[list[t]] = v for every t
__global__ void fill_rows_kernel(float* __restrict__ centroids, int d, const int32_t* __restrict__ list, int nlist,
                                 const float* __restrict__ v) {
    const int t = blockIdx.x;
    if (t >= nlist) return;
    for (int e = threadIdx.x; e < d; e += blockDim.x) centroids[(int64_t)list[t] * d + e] = v[e];
}

inline unsigned blocks_for(int64_t n, int t = 256) { return (unsigned)((n + t - 1) / t); }

template <typename T>
int to_host(std::vector<T>& h, const T* dev, size_t n) {
    h.resize(n);
    if (n) VIX_CUDA(cudaMemcpyAsync(h.data(), dev, n * sizeof(T), cudaMemcpyDeviceToHost, ctx().stream));
    VIX_CUDA(cudaStreamSynchronize(ctx().stream));
    return VIX_OK;
}
template <typename T>
int to_device(T* dev, const std::vector<T>& h) {
    if (!h.empty()) VIX_CUDA(cudaMemcpyAsync(dev, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice, ctx().stream));
    VIX_CUDA(cudaStreamSynchronize(ctx().stream));          // h may go out of scope
    return VIX_OK;
}

}  // namespace

// ------------------------------------------------------------------------------------------------ k-means++
int kmeanspp_parity_device(const float* x, int64_t n, int d, int k, uint64_t seed, uint64_t stream, float* centroids_out,
                           int64_t* chosen_out) {
    cudaStream_t s = ctx().stream;
    Lcg rng(seed, stream);
    Scratch<float> d2;
    VIX_TRY(d2.alloc((size_t)n));
    VIX_TRY(fill<float>(d2.ptr, n, INFINITY));
    std::vector<float> w;
    int64_t sel = rng.next_int(n);                                               // KMeansSeeding.swift:223
    for (int t = 0; t < k; ++t) {
        if (t > 0) {
            // :368-409: f64 total over finite non-negative weights, threshold = nextDouble * total, first i with cum >= thr
            VIX_TRY(to_host(w, d2.ptr, (size_t)n));
            double total = 0.0;
            for (int64_t i = 0; i < n; ++i) { const double v = (double)w[(size_t)i]; if (std::isfinite(v) && v >= 0.0) total += v; }
            if (total <= 0.0) sel = rng.next_int(n);
            else {
                const double thr = rng.next_double() * total;
                double cum = 0.0;
                sel = n - 1;
                for (int64_t i = 0; i < n; ++i) {
                    const double v = (double)w[(size_t)i];
                    if (std::isfinite(v) && v >= 0.0) cum += v;
                    if (cum >= thr) { sel = i; break; }
                }
            }
        }
        if (chosen_out) chosen_out[t] = sel;
        VIX_CUDA(cudaMemcpyAsync(centroids_out + (size_t)t * d, x + sel * d, (size_t)d * 4, cudaMemcpyDeviceToDevice, s));
        km11_update_kernel<<<blocks_for(n), 256, 0, s>>>(x, n, d, centroids_out + (size_t)t * d, d2.ptr);
        VIX_LAUNCH_CHECK();
    }
    return VIX_OK;
}

// ------------------------------------------------------------------------------------------------ mini-batch k-means
int kmeans_parity_device(const float* x, int64_t n, int d, int kc, const float* init, const vix_kmeans_cfg* cfg,
                         float* centroids_out, int32_t* assign_out) {
    cudaStream_t s = ctx().stream;
    const int batch_size = (cfg && cfg->batch_size > 0) ? cfg->batch_size : 1024;
    const int epochs = cfg ? (cfg->epochs > 1 ? cfg->epochs : 1) : 10;      // max(epochs, 1) (KMeansMiniBatchKernel.swift:493)
    const float tol = cfg ? cfg->tol : 1e-4f;
    const uint64_t seed = cfg ? cfg->seed : 0, stream = cfg ? cfg->stream_id : 0;
    if (init) VIX_CUDA(cudaMemcpyAsync(centroids_out, init, (size_t)kc * d * 4, cudaMemcpyDeviceToDevice, s));
    else VIX_TRY(kmeanspp_parity_device(x, n, d, kc, seed, stream, centroids_out, nullptr));   // :430-447

    Lcg rng(seed, stream);                                                       // :474 (a fresh stream)
    Scratch<int64_t> d_bidx;
    Scratch<float> d_rows, d_dist, d_newc;
    Scratch<int32_t> d_bassign, d_list;
    const int64_t sm = n < 10000 ? n : 10000;
    const int64_t cap = std::max<int64_t>(batch_size, sm);
    VIX_TRY(d_bidx.alloc((size_t)cap));
    VIX_TRY(d_rows.alloc((size_t)cap * d));
    VIX_TRY(d_dist.alloc((size_t)cap));
    VIX_TRY(d_bassign.alloc((size_t)cap));
    VIX_TRY(d_newc.alloc((size_t)std::min<int64_t>(batch_size, kc) * d));
    VIX_TRY(d_list.alloc((size_t)kc));
    std::vector<int64_t> bidx;
    std::vector<int32_t> bassign;
    std::vector<float> rows, dist;
    std::vector<uint32_t> batch_tag((size_t)kc, 0);
    std::vector<int> sum_index((size_t)kc, -1), batch_counts((size_t)kc, 0), touched_list;
    std::vector<double> sums;
    uint32_t current_tag = 1;
    double prev_inertia = INFINITY;
    int rc = VIX_OK;
    for (int epoch = 0; epoch < epochs; ++epoch) {
        int64_t processed = 0;
        while (processed < n) {
            const int bc = (int)std::min<int64_t>(batch_size, n - processed);
            bidx.resize((size_t)bc);
            for (int bi = 0; bi < bc; ++bi) bidx[(size_t)bi] = (int64_t)(rng.next() % (uint64_t)n);   // :524-528, with replacement
            current_tag += 1;
            VIX_TRY(to_device(d_bidx.ptr, bidx));
            VIX_TRY(gather_rows(x, d, d_bidx.ptr, bc, d_rows.ptr));
            // assignments use the centroids as of batch start
            VIX_TRY(ivf_assign_device(d_rows.ptr, bc, d, centroids_out, kc, d_bassign.ptr, nullptr));
            VIX_TRY(to_host(bassign, d_bassign.ptr, (size_t)bc));
            VIX_TRY(to_host(rows, d_rows.ptr, (size_t)bc * d));
            touched_list.clear();
            sums.assign((size_t)std::min<int64_t>(bc, kc) * d, 0.0);
            for (int bi = 0; bi < bc; ++bi) {                                   // f64 sums in draw order (:582)
                const int cb = bassign[(size_t)bi];
                if (batch_tag[(size_t)cb] != current_tag) {
                    batch_tag[(size_t)cb] = current_tag;
                    sum_index[(size_t)cb] = (int)touched_list.size();
                    touched_list.push_back(cb);
                }
                double* z = sums.data() + (size_t)sum_index[(size_t)cb] * d;
                const float* v = rows.data() + (size_t)bi * d;
                for (int j = 0; j < d; ++j) z[j] += (double)v[j];
                batch_counts[(size_t)cb] += 1;
            }
            // :595-607 the centroid is REPLACED by the batch mean
            std::vector<float> newc(touched_list.size() * (size_t)d);
            std::vector<int32_t> tl(touched_list.begin(), touched_list.end());
            for (size_t t = 0; t < touched_list.size(); ++t) {
                const int c = touched_list[t];
                const double inv = 1.0 / (double)batch_counts[(size_t)c];
                for (int j = 0; j < d; ++j) newc[t * d + j] = (float)(sums[t * d + j] * inv);
                batch_counts[(size_t)c] = 0;
            }
            VIX_TRY(to_device(d_newc.ptr, newc));
            VIX_TRY(to_device(d_list.ptr, tl));
            scatter_rows_kernel<<<(unsigned)tl.size(), 128, 0, s>>>(centroids_out, d, d_list.ptr, (int)tl.size(), d_newc.ptr);
            VIX_LAUNCH_CHECK();
            // :609-627 + :290-331: empties = untouched this batch; the counts are all zero by now so the "largest"
            // cluster is centroid 0; every empty centroid := the batch point farthest from the UPDATED centroid 0
            std::vector<int32_t> empties;
            for (int c = 0; c < kc; ++c) if (batch_tag[(size_t)c] != current_tag) empties.push_back(c);
            if (!empties.empty()) {
                km12_dist_to_row_kernel<<<blocks_for(bc), 256, 0, s>>>(d_rows.ptr, bc, d, centroids_out, d_dist.ptr);
                VIX_LAUNCH_CHECK();
                VIX_TRY(to_host(dist, d_dist.ptr, (size_t)bc));
                int far = 0;
                float fard = -INFINITY;
                for (int bi = 0; bi < bc; ++bi) if (dist[(size_t)bi] > fard) { fard = dist[(size_t)bi]; far = bi; }
                VIX_TRY(to_device(d_list.ptr, empties));
                fill_rows_kernel<<<(unsigned)empties.size(), 128, 0, s>>>(centroids_out, d, d_list.ptr, (int)empties.size(),
                                                                         d_rows.ptr + (size_t)far * d);
                VIX_LAUNCH_CHECK();
            }
            processed += bc;
        }
        // :635-682 inertia on a reservoir sample of min(n, 10000) (consumes n - m draws of the same stream)
        std::vector<int64_t> res((size_t)sm);
        for (int64_t i = 0; i < sm; ++i) res[(size_t)i] = i;
        for (int64_t i = sm; i < n; ++i) {
            const int64_t j = (int64_t)(rng.next() % (uint64_t)(i + 1));
            if (j < sm) res[(size_t)j] = i;
        }
        VIX_TRY(to_device(d_bidx.ptr, res));
        VIX_TRY(gather_rows(x, d, d_bidx.ptr, sm, d_rows.ptr));
        VIX_TRY(ivf_assign_device(d_rows.ptr, sm, d, centroids_out, kc, d_bassign.ptr, d_dist.ptr));
        VIX_TRY(to_host(dist, d_dist.ptr, (size_t)sm));
        double inertia = 0.0;
        for (int64_t t = 0; t < sm; ++t) inertia += (double)dist[(size_t)t];
        if (epoch > 0) {
            const double denom = prev_inertia > 4.9406564584124654e-324 ? prev_inertia : 4.9406564584124654e-324;
            if ((prev_inertia - inertia) / denom < (double)tol) break;          // :676-681
        }
        prev_inertia = inertia;
    }
    if (assign_out) VIX_TRY(ivf_assign_device(x, n, d, centroids_out, kc, assign_out, nullptr));   // :689-706
    return rc;
}

// ------------------------------------------------------------------------------------------------ PQ training
namespace {

struct OrdT { float v; int64_t i; };
// descending by value, ties keep ascending index (Swift's sort is a stable merge sort in practice)
inline bool ord_less(const OrdT& a, const OrdT& b) { return a.v > b.v || (a.v == b.v && a.i < b.i); }

int launch_sub_assign(const SubSrc& src, int64_t n, const float* C, int ks, int use_residual, int32_t* best_k, float* best_d) {
    if (n == 0) return VIX_OK;
    const size_t smem = (size_t)ks * src.dsub * 4;
    VIX_REQUIRE(smem <= 200 * 1024, VIX_ERR_UNSUPPORTED, "pq_train: ks * dsub = %d floats exceed shared memory", ks * src.dsub);
    VIX_CUDA(cudaFuncSetAttribute(sub_assign_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    sub_assign_kernel<<<blocks_for(n), 256, smem, ctx().stream>>>(src, n, C, ks, use_residual, best_k, best_d);
    VIX_LAUNCH_CHECK();
    return VIX_OK;
}

// k-means++ over `npts` sub-vectors of `src` (PQTrain.swift:856-1019): i0 = clamp(Int(uniform * n)); then
// r = uniform * sum(dmin); first i with (r -= dmin[i]) <= 0; dmin updated with strict <
// streaming != 0: streamingKMeansppSeed (PQTrain.swift:391-706): the same draws over the chunks laid end to end, except that a
// degenerate sum falls back to row 0 WITHOUT a draw and an exhausted walk to centroid 0
int seed_subspace(const SubSrc& src, int64_t npts, int ks, int use_residual, Xoro& rng, float* C /* device [ks x dsub] */,
                  int streaming = 0) {
    cudaStream_t s = ctx().stream;
    const int dsub = src.dsub;
    Scratch<float> dmin;
    VIX_TRY(dmin.alloc((size_t)npts));
    SubSrc one = src;
    std::vector<float> h;
    auto pick_into = [&](int64_t pick, int k) -> int {
        // C[k] = sub-vector `pick` (residualised when a coarse quantiser is given)
        SubSrc p = src;
        Scratch<uint32_t> pi;
        VIX_TRY(pi.alloc(1));
        const uint32_t row = src.idx ? 0 : (uint32_t)pick;
        if (src.idx) {
            VIX_CUDA(cudaMemcpyAsync(pi.ptr, src.idx + pick, 4, cudaMemcpyDeviceToDevice, s));
        } else {
            VIX_CUDA(cudaMemcpyAsync(pi.ptr, &row, 4, cudaMemcpyHostToDevice, s));
            VIX_CUDA(cudaStreamSynchronize(s));
        }
        p.idx = pi.ptr;
        sub_gather_kernel<<<1, 256, 0, s>>>(p, 1, use_residual, C + (size_t)k * dsub);
        VIX_LAUNCH_CHECK();
        VIX_CUDA(cudaStreamSynchronize(s));
        return VIX_OK;
    };
    (void)one;
    int64_t i0 = (int64_t)(rng.f64() * (double)npts);
    if (i0 < 0) i0 = 0;
    if (i0 > npts - 1) i0 = npts - 1;
    VIX_TRY(pick_into(i0, 0));
    sub_dist_point_kernel<<<blocks_for(npts), 256, 0, s>>>(src, npts, C, use_residual, 0, dmin.ptr);
    VIX_LAUNCH_CHECK();
    for (int k = 1; k < ks; ++k) {
        VIX_TRY(to_host(h, dmin.ptr, (size_t)npts));
        double sum = 0.0;
        for (int64_t i = 0; i < npts; ++i) sum += (double)h[(size_t)i];
        int64_t pick;
        bool copy_first_centroid = false;
        if (!(sum > 0)) {
            if (streaming) pick = 0;
            else {
                pick = (int64_t)(rng.f64() * (double)npts);
                if (pick < 0) pick = 0;
                if (pick > npts - 1) pick = npts - 1;
            }
        } else {
            double r = rng.f64() * sum;
            pick = npts - 1;
            bool chosen = false;
            for (int64_t i = 0; i < npts; ++i) { r -= (double)h[(size_t)i]; if (r <= 0) { pick = i; chosen = true; break; } }
            copy_first_centroid = streaming && !chosen;
        }
        if (copy_first_centroid) VIX_CUDA(cudaMemcpyAsync(C + (size_t)k * dsub, C, (size_t)dsub * 4, cudaMemcpyDeviceToDevice, s));
        else VIX_TRY(pick_into(pick, k));
        sub_dist_point_kernel<<<blocks_for(npts), 256, 0, s>>>(src, npts, C + (size_t)k * dsub, use_residual, 1, dmin.ptr);
        VIX_LAUNCH_CHECK();
    }
    return VIX_OK;
}

// rows stably sorted by assignment + CSR offsets (device)
int sort_rows_by_code(const int32_t* best_k, int64_t n, int ks, Scratch<int32_t>& rows_sorted, Scratch<int64_t>& off,
                      std::vector<int32_t>& counts_h) {
    Scratch<int32_t> cnt;
    VIX_TRY(rows_sorted.alloc((size_t)n));
    VIX_TRY(cnt.alloc((size_t)ks));
    VIX_TRY(off.alloc((size_t)ks + 1));
    VIX_TRY(order_by_key(best_k, n, ks, rows_sorted.ptr));
    VIX_TRY(key_offsets(best_k, n, ks, cnt.ptr, off.ptr));
    return to_host(counts_h, cnt.ptr, (size_t)ks);
}

// copy raw (non-residual) sub-vectors x[rows[t]] into C[ks_list[t]]
int copy_raw_rows(const float* x, int64_t ld, int off, int dsub, const std::vector<int64_t>& rows, const std::vector<int>& ks_list,
                  float* C) {
    for (size_t t = 0; t < rows.size(); ++t)
        VIX_CUDA(cudaMemcpyAsync(C + (size_t)ks_list[t] * dsub, x + rows[t] * ld + off, (size_t)dsub * 4, cudaMemcpyDeviceToDevice,
                                 ctx().stream));
    return VIX_OK;
}

// lloydKMeansSubspace (PQTrain.swift:1023-1202)
int lloyd_subspace(const SubSrc& all, int64_t n, int j, int ks, const vix_pq_train_cfg& cfg, float* C) {
    cudaStream_t s = ctx().stream;
    const int dsub = all.dsub;
    Scratch<int32_t> best_k;
    Scratch<float> best_d;
    VIX_TRY(best_k.alloc((size_t)n));
    VIX_TRY(best_d.alloc((size_t)n));
    std::vector<float> bd_h;
    std::vector<int32_t> counts;
    double prev = INFINITY;
    const int max_iters = cfg.max_iters > 1 ? cfg.max_iters : 1;
    for (int iter = 0; iter < max_iters; ++iter) {
        VIX_TRY(launch_sub_assign(all, n, C, ks, 1, best_k.ptr, best_d.ptr));
        Scratch<int32_t> rows_sorted;
        Scratch<int64_t> off;
        VIX_TRY(sort_rows_by_code(best_k.ptr, n, ks, rows_sorted, off, counts));
        sub_centroid_update_kernel<<<ks, 32, 0, s>>>(all, rows_sorted.ptr, off.ptr, ks, C);   // non-empty centroids only
        VIX_LAUNCH_CHECK();
        VIX_TRY(to_host(bd_h, best_d.ptr, (size_t)n));
        double distortion = 0.0;                                   // f64, row order, negative distances clamped (:1131)
        for (int64_t i = 0; i < n; ++i) { float bd = bd_h[(size_t)i]; if (bd < 0) bd = 0; distortion += (double)bd; }
        std::vector<int> empties;
        for (int k = 0; k < ks; ++k) if (counts[(size_t)k] == 0) empties.push_back(k);
        if (!empties.empty()) {
            if (cfg.empty_policy == 1) {                           // .reseed (:1126-1136): raw sub-vectors, LCG picks
                uint64_t seed = cfg.seed ^ ((uint64_t)j * 0x9E3779B97F4A7C15ULL) ^ ((uint64_t)iter * 0xD1B54A32D192ED03ULL);
                std::vector<int64_t> rows;
                for (size_t t = 0; t < empties.size(); ++t) {
                    seed = 2862933555777941757ULL * seed + 3037000493ULL;
                    rows.push_back((int64_t)(seed % (uint64_t)n));
                }
                VIX_TRY(copy_raw_rows(all.x, all.ld, all.off, dsub, rows, empties, C));
            } else if (cfg.empty_policy == 0) {                    // .split (:1137-1188): farthest stride-sampled points
                const int64_t want = std::max<int64_t>(128, n / 4);
                const int64_t sample = n < want ? n : want;
                const int64_t stride = n / sample > 1 ? n / sample : 1;
                std::vector<uint32_t> pts;
                for (int64_t idx = 0; idx < n; idx += stride) pts.push_back((uint32_t)idx);
                const int64_t cnt = (int64_t)pts.size();
                Scratch<uint32_t> d_pts;
                Scratch<float> md;
                VIX_TRY(d_pts.alloc((size_t)cnt));
                VIX_TRY(md.alloc((size_t)cnt));
                VIX_TRY(to_device(d_pts.ptr, pts));
                SubSrc sub = all;
                sub.idx = d_pts.ptr;
                VIX_TRY(launch_sub_assign(sub, cnt, C, ks, 0, nullptr, md.ptr));   // NB: the repair ignores the residual (:1155)
                std::vector<float> md_h;
                VIX_TRY(to_host(md_h, md.ptr, (size_t)cnt));
                std::vector<OrdT> o((size_t)cnt);
                for (int64_t t = 0; t < cnt; ++t) o[(size_t)t] = OrdT{md_h[(size_t)t], t};
                std::stable_sort(o.begin(), o.end(), ord_less);
                std::vector<int64_t> rows;
                std::vector<int> ksl;
                for (size_t r = 0; r < empties.size() && (int64_t)r < cnt; ++r) { rows.push_back(o[r].i * stride); ksl.push_back(empties[r]); }
                VIX_TRY(copy_raw_rows(all.x, all.ld, all.off, dsub, rows, ksl, C));
            }
        }
        const double improve = (prev - distortion) / (prev == 0 ? 1 : prev);
        prev = distortion;
        if (cfg.tol > 0 && iter > 0 && improve >= 0 && improve < (double)cfg.tol) break;
    }
    VIX_CUDA(cudaStreamSynchronize(s));
    return VIX_OK;
}

// minibatchKMeansSubspace (PQTrain.swift:1206-1442), no warm start
int minibatch_subspace(const SubSrc& all, int64_t n, int ks, const vix_pq_train_cfg& cfg, int64_t sample_n_eff, int dist_eval_n,
                       Xoro& rng, float* C) {
    cudaStream_t s = ctx().stream;
    const int dsub = all.dsub;
    std::vector<uint32_t> idx((size_t)n);
    for (int64_t i = 0; i < n; ++i) idx[(size_t)i] = (uint32_t)i;
    const int B = cfg.batch_size > 1 ? cfg.batch_size : 1;
    std::vector<int64_t> gcounts((size_t)ks, 0), counts((size_t)ks);
    std::vector<double> sums((size_t)ks * dsub);
    std::vector<float> Ch((size_t)ks * dsub), sub_h;
    std::vector<int32_t> bk_h;
    Scratch<uint32_t> d_idx;
    Scratch<int32_t> d_bk;
    Scratch<float> d_sub, d_md;
    const int64_t eval_cap = std::max<int64_t>(std::max<int64_t>(B, dist_eval_n), sample_n_eff > 0 ? sample_n_eff : 0);
    VIX_TRY(d_idx.alloc((size_t)std::max<int64_t>(eval_cap, 1)));
    VIX_TRY(d_bk.alloc((size_t)std::max<int64_t>(B, 1)));
    VIX_TRY(d_sub.alloc((size_t)std::max<int64_t>(B, 1) * dsub));
    VIX_TRY(d_md.alloc((size_t)std::max<int64_t>(eval_cap, 1)));
    const int passes = cfg.max_iters > 1 ? cfg.max_iters : 1;
    for (int p = 0; p < passes; ++p) {
        randperm(idx, rng);
        const int64_t limit = sample_n_eff > 0 ? std::min<int64_t>(n, sample_n_eff) : n;
        for (int64_t sb = 0; sb < limit; sb += B) {
            const int64_t e = std::min<int64_t>(sb + B, limit), bc = e - sb;
            std::vector<uint32_t> bidx(idx.begin() + sb, idx.begin() + e);
            VIX_TRY(to_device(d_idx.ptr, bidx));
            SubSrc sub = all;
            sub.idx = d_idx.ptr;
            VIX_TRY(launch_sub_assign(sub, bc, C, ks, 1, d_bk.ptr, nullptr));
            sub_gather_kernel<<<blocks_for(bc * dsub), 256, 0, s>>>(sub, bc, 1, d_sub.ptr);
            VIX_LAUNCH_CHECK();
            VIX_TRY(to_host(bk_h, d_bk.ptr, (size_t)bc));
            VIX_TRY(to_host(sub_h, d_sub.ptr, (size_t)bc * dsub));
            VIX_TRY(to_host(Ch, C, (size_t)ks * dsub));
            std::fill(sums.begin(), sums.end(), 0.0);
            std::fill(counts.begin(), counts.end(), 0);
            for (int64_t t = 0; t < bc; ++t) {
                double* sk = sums.data() + (size_t)bk_h[(size_t)t] * dsub;
                for (int u = 0; u < dsub; ++u) sk[u] += (double)sub_h[(size_t)t * dsub + u];
                counts[(size_t)bk_h[(size_t)t]] += 1;
            }
            for (int k = 0; k < ks; ++k) {                          // running-mean blend (:1297-1316)
                const int64_t ck = counts[(size_t)k];
                if (ck <= 0) continue;
                const int64_t old_n = gcounts[(size_t)k], new_n = old_n + ck;
                gcounts[(size_t)k] = new_n;
                const double old_w = (double)old_n / (double)new_n, new_w = (double)ck / (double)new_n;
                for (int u = 0; u < dsub; ++u) {
                    const double old_val = (double)Ch[(size_t)k * dsub + u];
                    const double batch_mean = sums[(size_t)k * dsub + u] / (double)ck;
                    const float v = (float)(old_w * old_val + new_w * batch_mean);
                    Ch[(size_t)k * dsub + u] = std::isfinite(v) ? v : 0.0f;
                }
            }
            VIX_TRY(to_device(C, Ch));
        }
        // pass-level repair for clusters that never received anything (:1325-1395)
        std::vector<int> empties;
        for (int k = 0; k < ks; ++k) if (gcounts[(size_t)k] == 0) empties.push_back(k);
        if (!empties.empty()) {
            int64_t eval_lim = sample_n_eff > 0 ? sample_n_eff : dist_eval_n;
            if (eval_lim > n) eval_lim = n;
            if (eval_lim > 0) {
                std::vector<uint32_t> inds((size_t)eval_lim);
                for (int64_t t = 0; t < eval_lim; ++t) inds[(size_t)t] = idx[(size_t)(t % n)];
                VIX_TRY(to_device(d_idx.ptr, inds));
                SubSrc sub = all;
                sub.idx = d_idx.ptr;
                VIX_TRY(launch_sub_assign(sub, eval_lim, C, ks, 1, nullptr, d_md.ptr));
                std::vector<float> md_h;
                VIX_TRY(to_host(md_h, d_md.ptr, (size_t)eval_lim));
                std::vector<OrdT> o((size_t)eval_lim);
                for (int64_t t = 0; t < eval_lim; ++t) o[(size_t)t] = OrdT{md_h[(size_t)t], t};
                std::stable_sort(o.begin(), o.end(), ord_less);
                for (size_t r = 0; r < empties.size() && (int64_t)r < eval_lim; ++r) {
                    // C[k] = residualised sub-vector of the r-th farthest evaluated point
                    Scratch<uint32_t> one;
                    VIX_TRY(one.alloc(1));
                    const uint32_t row = inds[(size_t)o[r].i];
                    VIX_CUDA(cudaMemcpyAsync(one.ptr, &row, 4, cudaMemcpyHostToDevice, s));
                    VIX_CUDA(cudaStreamSynchronize(s));
                    SubSrc pk = all;
                    pk.idx = one.ptr;
                    sub_gather_kernel<<<1, 256, 0, s>>>(pk, 1, 1, C + (size_t)empties[r] * dsub);
                    VIX_LAUNCH_CHECK();
                    VIX_CUDA(cudaStreamSynchronize(s));
                    gcounts[(size_t)empties[r]] = 1;
                }
            }
        }
    }
    VIX_CUDA(cudaStreamSynchronize(s));
    return VIX_OK;
}

}  // namespace

int pq_train_parity_device(const float* x, int64_t n, int d, int m, int ks, const float* coarse, const int32_t* assign,
                           const vix_pq_train_cfg* in_cfg, float* codebooks_out, float* norms_out) {
    cudaStream_t s = ctx().stream;
    vix_pq_train_cfg cfg{};
    if (in_cfg) cfg = *in_cfg;
    else { cfg.algorithm = 0; cfg.max_iters = 25; cfg.tol = 1e-4f; cfg.batch_size = 1024; cfg.sample_n = 0; cfg.seed = 42; cfg.stream_id = 0; cfg.empty_policy = 0; }
    VIX_REQUIRE(ks >= 1 && ks <= 65536, VIX_ERR_INVALID_PARAM, "pq_train: ks must be in 1..65536");
    const int64_t need = cfg.sample_n > 0 ? cfg.sample_n : n;
    VIX_REQUIRE(need >= ks, VIX_ERR_EMPTY_INPUT, "pq_train: fewer training vectors (%lld) than centroids (%d)", (long long)need, ks);   // PQTrain.swift:96-135
    VIX_REQUIRE(n < (1LL << 31), VIX_ERR_INVALID_PARAM, "pq_train: n must be < 2^31");
    const int dsub = d / m;
    const int dist_eval_n = 2000;
    if (cfg.algorithm == 1) {                                        // :144-149
        if (cfg.sample_n <= 0 && n > dist_eval_n) cfg.sample_n = dist_eval_n;
        if (cfg.batch_size <= 0) cfg.batch_size = 512;
        cfg.empty_policy = 1;
    }
    if (cfg.max_iters <= 0) cfg.max_iters = 25;
    if (cfg.tol <= 0) cfg.tol = 1e-4f;
    for (int j = 0; j < m; ++j) {
        Xoro rng(cfg.seed, (uint64_t)cfg.stream_id, (uint64_t)j);
        SubSrc all{x, d, j * dsub, dsub, nullptr, coarse, assign, d};
        // buildSampleIndex (:784-795)
        int64_t ns = n;
        std::vector<uint32_t> idx;
        if (!(cfg.sample_n <= 0 || cfg.sample_n >= n)) { sample_wo_repl((uint32_t)n, (uint32_t)cfg.sample_n, rng, idx); ns = cfg.sample_n; }
        float* Cj = codebooks_out + (size_t)j * ks * dsub;
        VIX_CUDA(cudaMemsetAsync(Cj, 0, (size_t)ks * dsub * 4, s));
        const int64_t seeding_cap = 4LL * ks;                       // :191-193
        const bool use_subset = ns > seeding_cap;
        const int64_t ns_seed = use_subset ? seeding_cap : ns;
        if (ns == n && !use_subset) {
            VIX_TRY(seed_subspace(all, n, ks, 1, rng, Cj));          // kmeansppSeedSubspace (strided, residual aware)
        } else {
            std::vector<uint32_t> pos, rows((size_t)ns_seed);
            if (use_subset) sample_wo_repl((uint32_t)ns, (uint32_t)ns_seed, rng, pos);
            for (int64_t t = 0; t < ns_seed; ++t) {
                const int64_t pool = use_subset ? pos[(size_t)t] : t;
                rows[(size_t)t] = (ns == n) ? (uint32_t)pool : idx[(size_t)pool];
            }
            Scratch<uint32_t> d_rows;
            Scratch<float> dense;
            VIX_TRY(d_rows.alloc((size_t)ns_seed));
            VIX_TRY(dense.alloc((size_t)ns_seed * dsub));
            VIX_TRY(to_device(d_rows.ptr, rows));
            SubSrc sub = all;
            sub.idx = d_rows.ptr;
            sub_gather_kernel<<<blocks_for(ns_seed * dsub), 256, 0, s>>>(sub, ns_seed, 1, dense.ptr);   // residualised copies
            VIX_LAUNCH_CHECK();
            SubSrc dn{dense.ptr, dsub, 0, dsub, nullptr, nullptr, nullptr, 0};
            VIX_TRY(seed_subspace(dn, ns_seed, ks, 0, rng, Cj));     // kmeansppSeedSubspaceDense
        }
        if (cfg.algorithm == 1) VIX_TRY(minibatch_subspace(all, n, ks, cfg, cfg.sample_n, dist_eval_n, rng, Cj));
        else VIX_TRY(lloyd_subspace(all, n, j, ks, cfg, Cj));
    }
    if (norms_out) {                                                 // :299-307 sequential sum of squares
        std::vector<float> cb;
        VIX_TRY(to_host(cb, codebooks_out, (size_t)m * ks * dsub));
        std::vector<float> nr((size_t)m * ks);
        for (size_t r = 0; r < nr.size(); ++r) {
            float acc = 0.0f;
            for (int u = 0; u < dsub; ++u) { const float v = cb[r * dsub + u]; acc = acc + v * v; }
            nr[r] = acc;
        }
        VIX_TRY(to_device(norms_out, nr));
    }
    return VIX_OK;
}

// pq_train_streaming_f32 (Kernels/PQTrain.swift:391-706), no residual: X holds the chunks laid end to end on the device
// (row (c, i) = prefix[c] + i); the chunk structure lives on in the control flow -- one permutation per chunk and pass,
// Bernoulli sampling of the rows of a batch, the running-mean blend per batch, the pass-level repair from 512 random rows.
int pq_train_streaming_parity_device(const float* X, const std::vector<int64_t>& chunk_n, int d, int m, int ks,
                                     const vix_pq_train_cfg* in_cfg, float* codebooks_out, float* norms_out) {
    cudaStream_t s = ctx().stream;
    vix_pq_train_cfg cfg{};
    if (in_cfg) cfg = *in_cfg;
    else { cfg.seed = 42; }
    cfg.algorithm = 1;
    if (cfg.max_iters <= 0) cfg.max_iters = 15;
    if (cfg.batch_size <= 0) cfg.batch_size = 8192;
    const int nchunks = (int)chunk_n.size();
    std::vector<int64_t> prefix((size_t)nchunks + 1, 0);
    for (int c = 0; c < nchunks; ++c) prefix[(size_t)c + 1] = prefix[(size_t)c] + chunk_n[(size_t)c];
    const int64_t total = prefix[(size_t)nchunks];
    VIX_REQUIRE(total > 0 && total < (1LL << 31), VIX_ERR_EMPTY_INPUT, "pq_train_streaming: %lld rows", (long long)total);
    if (cfg.sample_n <= 0 && total > 2000) cfg.sample_n = 2000;
    const int dsub = d / m;
    const int64_t repair_eval_n = 512;
    const int B = cfg.batch_size > 1 ? cfg.batch_size : 1;
    Scratch<uint32_t> d_idx;
    Scratch<int32_t> d_bk;
    Scratch<float> d_sub, d_md;
    const int64_t cap_rows = std::max<int64_t>(std::max<int64_t>(B, repair_eval_n), 4LL * ks);
    VIX_TRY(d_idx.alloc((size_t)cap_rows));
    VIX_TRY(d_bk.alloc((size_t)cap_rows));
    VIX_TRY(d_sub.alloc((size_t)cap_rows * dsub));
    VIX_TRY(d_md.alloc((size_t)cap_rows));
    std::vector<float> Ch((size_t)ks * dsub), sub_h;
    std::vector<int32_t> bk_h;
    for (int j = 0; j < m; ++j) {
        Xoro rng(cfg.seed, (uint64_t)cfg.stream_id, (uint64_t)j);
        SubSrc all{X, d, j * dsub, dsub, nullptr, nullptr, nullptr, d};
        float* Cj = codebooks_out + (size_t)j * ks * dsub;
        VIX_CUDA(cudaMemsetAsync(Cj, 0, (size_t)ks * dsub * 4, s));
        const int64_t cap = 4LL * ks;
        if (total > cap) {                                           // seed on a sample of 4 ks rows (dense copy)
            std::vector<uint32_t> picks;
            const int64_t got = sample_wo_repl((uint32_t)total, (uint32_t)cap, rng, picks);
            (void)got;
            VIX_TRY(to_device(d_idx.ptr, picks));
            SubSrc sub = all;
            sub.idx = d_idx.ptr;
            sub_gather_kernel<<<blocks_for(cap * dsub), 256, 0, s>>>(sub, cap, 0, d_sub.ptr);
            VIX_LAUNCH_CHECK();
            SubSrc dn{d_sub.ptr, dsub, 0, dsub, nullptr, nullptr, nullptr, 0};
            VIX_TRY(seed_subspace(dn, cap, ks, 0, rng, Cj));         // kmeansppSeedSubspaceDense
        } else {
            VIX_TRY(seed_subspace(all, total, ks, 0, rng, Cj, 1));   // streamingKMeansppSeed
        }
        std::vector<int64_t> gcounts((size_t)ks, 0), counts((size_t)ks);
        std::vector<double> sums((size_t)ks * dsub);
        for (int pass = 0; pass < cfg.max_iters; ++pass) {
            const int64_t limit = cfg.sample_n > 0 ? std::min<int64_t>(total, cfg.sample_n) : total;
            double prob = (double)limit / (double)(total > 1 ? total : 1);
            if (prob < 0.0) prob = 0.0;
            if (prob > 1.0) prob = 1.0;
            for (int c = 0; c < nchunks; ++c) {
                const int64_t nc = chunk_n[(size_t)c];
                if (nc <= 0) continue;
                std::vector<uint32_t> idx((size_t)nc);               // minibatchKMeansSubspaceChunk (:1444-1575)
                for (int64_t i = 0; i < nc; ++i) idx[(size_t)i] = (uint32_t)i;
                randperm(idx, rng);
                for (int64_t sb = 0; sb < nc;) {
                    const int64_t e = std::min<int64_t>(sb + B, nc);
                    std::vector<uint32_t> rows;
                    for (int64_t t = sb; t < e; ++t) {
                        if (prob < 1.0) { const double u = rng.f64(); if (u > prob) continue; }
                        rows.push_back((uint32_t)(prefix[(size_t)c] + idx[(size_t)t]));
                    }
                    sb = e;
                    const int64_t bc = (int64_t)rows.size();
                    if (bc == 0) continue;                           // (a batch without rows blends nothing)
                    VIX_TRY(to_device(d_idx.ptr, rows));
                    SubSrc sub = all;
                    sub.idx = d_idx.ptr;
                    VIX_TRY(launch_sub_assign(sub, bc, Cj, ks, 0, d_bk.ptr, nullptr));
                    sub_gather_kernel<<<blocks_for(bc * dsub), 256, 0, s>>>(sub, bc, 0, d_sub.ptr);
                    VIX_LAUNCH_CHECK();
                    VIX_TRY(to_host(bk_h, d_bk.ptr, (size_t)bc));
                    VIX_TRY(to_host(sub_h, d_sub.ptr, (size_t)bc * dsub));
                    VIX_TRY(to_host(Ch, Cj, (size_t)ks * dsub));
                    std::fill(sums.begin(), sums.end(), 0.0);
                    std::fill(counts.begin(), counts.end(), 0);
                    for (int64_t t = 0; t < bc; ++t) {
                        double* sk = sums.data() + (size_t)bk_h[(size_t)t] * dsub;
                        for (int u = 0; u < dsub; ++u) sk[u] += (double)sub_h[(size_t)t * dsub + u];
                        counts[(size_t)bk_h[(size_t)t]] += 1;
                    }
                    for (int k = 0; k < ks; ++k) {                  // running-mean blend
                        const int64_t ck = counts[(size_t)k];
                        if (ck <= 0) continue;
                        const int64_t old_n = gcounts[(size_t)k], new_n = old_n + ck;
                        gcounts[(size_t)k] = new_n;
                        const double old_w = (double)old_n / (double)new_n, new_w = (double)ck / (double)new_n;
                        for (int u = 0; u < dsub; ++u) {
                            const double old_val = (double)Ch[(size_t)k * dsub + u];
                            const double batch_mean = sums[(size_t)k * dsub + u] / (double)ck;
                            const float v = (float)(old_w * old_val + new_w * batch_mean);
                            Ch[(size_t)k * dsub + u] = std::isfinite(v) ? v : 0.0f;
                        }
                    }
                    VIX_TRY(to_device(Cj, Ch));
                }
            }
            // pass-level repair (:543-640): clusters that never received anything take the farthest of 512 random rows
            std::vector<int> empties;
            for (int k = 0; k < ks; ++k) if (gcounts[(size_t)k] == 0) empties.push_back(k);
            if (!empties.empty()) {
                const int64_t eval_n = std::min<int64_t>(total, repair_eval_n);
                std::vector<uint32_t> rows((size_t)eval_n);
                for (int64_t t = 0; t < eval_n; ++t) {
                    int64_t g = (int64_t)(rng.f64() * (double)total);
                    // the reference walks the chunks with the last one open-ended: a draw of exactly `total` lands past its end
                    if (g > total - 1) g = total - 1;
                    rows[(size_t)t] = (uint32_t)g;
                }
                VIX_TRY(to_device(d_idx.ptr, rows));
                SubSrc sub = all;
                sub.idx = d_idx.ptr;
                VIX_TRY(launch_sub_assign(sub, eval_n, Cj, ks, 0, nullptr, d_md.ptr));
                std::vector<float> md_h;
                VIX_TRY(to_host(md_h, d_md.ptr, (size_t)eval_n));
                std::vector<OrdT> o((size_t)eval_n);
                for (int64_t t = 0; t < eval_n; ++t) o[(size_t)t] = OrdT{md_h[(size_t)t], t};
                std::stable_sort(o.begin(), o.end(), ord_less);
                std::vector<int64_t> src_rows;
                std::vector<int> ksl;
                for (size_t r = 0; r < empties.size() && (int64_t)r < eval_n; ++r) {
                    src_rows.push_back((int64_t)rows[(size_t)o[r].i]);
                    ksl.push_back(empties[r]);
                    gcounts[(size_t)empties[r]] = 1;
                }
                VIX_TRY(copy_raw_rows(X, d, j * dsub, dsub, src_rows, ksl, Cj));
            }
        }
    }
    VIX_CUDA(cudaStreamSynchronize(s));
    if (norms_out) {
        std::vector<float> cb;
        VIX_TRY(to_host(cb, codebooks_out, (size_t)m * ks * dsub));
        std::vector<float> nr((size_t)m * ks);
        for (size_t r = 0; r < nr.size(); ++r) {
            float acc = 0.0f;
            for (int u = 0; u < dsub; ++u) { const float v = cb[r * dsub + u]; acc = acc + v * v; }
            nr[r] = acc;
        }
        VIX_TRY(to_device(norms_out, nr));
    }
    return VIX_OK;
}

}  // namespace vix
