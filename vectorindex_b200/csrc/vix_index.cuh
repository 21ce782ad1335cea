// vix_index.cuh -- the device-resident index handle shared by vix_index.cu (single GPU) and vix_sharded.cu (the
// multi-GPU search / build steps around it).
#pragma once

#include "vix_common.cuh"

#include <mutex>
#include <vector>

namespace vix {

// entry points of the other translation units
int pq_encode_device(const float* x, int64_t n, int d, int m, int ks, const float* cb, const float* csq,
                     const float* coarse, const int32_t* assign, uint8_t* codes, int use_dot, int layout,
                     int B, int g, int u4);
int flat_search_device(const float* q, int64_t nq, const float* xb, int64_t n, int d, int metric, int k,
                       const float* xb_norm, float* out_dist, int64_t* out_ids, bool raw_scores);
int flat_search_masked_device(const float* q, int64_t nq, const float* xb, int64_t n, int d, int metric, int k,
                              const uint64_t* disabled_rows, float* out_dist, int64_t* out_ids);
int flat_search_auto_device(const float* q, int64_t nq, const float* xb, int64_t n, int d, int metric, int k,
                            const float* xb_norm, float* out_dist, int64_t* out_ids, bool raw_scores);
int probe_select_device(const float* q, int64_t nq, const float* c, int kc, int d, int metric, int nprobe,
                        const float* cnorm, const uint64_t* disabled, int32_t* out_idx, float* out_scores);
int ivf_assign_device(const float* x, int64_t n, int d, const float* c, int kc, int32_t* assign, float* dist);
int ivf_assign_auto_device(const float* x, int64_t n, int d, const float* c, int kc, int32_t* assign, float* dist);
int ivf_assign_metric_device(const float* x, int64_t n, int d, const float* c, int kc, int metric,
                             const float* cnorm, int32_t* assign);
int row_norms_device(const float* x, int64_t n, int d, float* out);
int train_coarse_device(const float* x, int64_t n, int d, int kc, int metric, const vix_kmeans_cfg* cfg,
                        float* centroids_out);
int train_pq_device(const float* x, int64_t n, int d, int m, int ks, const float* coarse, const int32_t* assign,
                    const vix_pq_train_cfg* cfg, float* codebooks_out, float* norms_out);
int kmeans_parity_device(const float* x, int64_t n, int d, int kc, const float* init, const vix_kmeans_cfg* cfg,
                         float* centroids_out, int32_t* assign_out);
int pq_train_parity_device(const float* x, int64_t n, int d, int m, int ks, const float* coarse, const int32_t* assign,
                           const vix_pq_train_cfg* cfg, float* codebooks_out, float* norms_out);
int centroid_batch_score_cosine_device(const float* q, int64_t nq, const float* c, int kc, int d, const float* cnorm,
                                       float* out);
int row_select_device(const float* scores, int64_t rows, int n, int k, const uint64_t* disabled, int32_t* out_idx,
                      float* out_scores);
int probe_select_fast_device(const float* q, int64_t nq, const float* c, int kc, int d, int metric, int nprobe,
                             const float* cnorm, int32_t* out_idx, float* out_scores, const float* cnorm_max_sqrt);
int max_sqrt_device(const float* x, int64_t n, float* out);


// ------------------------------------------------------------------------------------------------
// growable device buffer
// ------------------------------------------------------------------------------------------------
template <typename T>
struct DevBuf {
    T* ptr = nullptr;
    size_t size = 0, cap = 0;
    int reserve(size_t n, bool keep) {
        if (n <= cap) return VIX_OK;
        size_t ncap = cap ? cap : 1024;
        while (ncap < n) ncap = ncap + ncap / 2 + 1024;
        T* np = nullptr;
        VIX_CUDA(cudaMalloc(reinterpret_cast<void**>(&np), ncap * sizeof(T)));
        if (ptr) {
            cudaError_t e = cudaSuccess;
            if (keep && size) e = cudaMemcpyAsync(np, ptr, size * sizeof(T), cudaMemcpyDeviceToDevice, ctx().stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(ctx().stream);
            if (e != cudaSuccess) { cudaFree(np); VIX_CUDA(e); }          // keep the old buffer, drop the new one
            cudaFree(ptr);
        }
        ptr = np; cap = ncap;
        return VIX_OK;
    }
    int resize(size_t n, bool keep = true) {
        VIX_TRY(reserve(n, keep));
        size = n;
        return VIX_OK;
    }
    int assign_from(const T* src, size_t n) {   // src: host or device
        VIX_TRY(resize(n, false));
        if (n) VIX_CUDA(cudaMemcpyAsync(ptr, src, n * sizeof(T), cudaMemcpyDefault, ctx().stream));
        return VIX_OK;
    }
    void free_all() { if (ptr) cudaFree(ptr); ptr = nullptr; size = cap = 0; }
    // take over a cudaMalloc'ed array of n elements (the old one is freed)
    void adopt(T* p, size_t n) { free_all(); ptr = p; size = cap = n; }
    ~DevBuf() { free_all(); }
};

}  // namespace vix

struct vix_index {
    template <typename T> using DevBuf = vix::DevBuf<T>;
    vix_index_params p;
    std::mutex mu;
    // bytes of one stored PQ code: m (ks = 256) or m / 2 (ks = 16: two codes per byte, low nibble = even sub-quantiser,
    // pq_encode.c:594-596)
    int code_bytes() const { return p.ks == 16 ? p.m / 2 : p.m; }
    int kc = 0;                         // trained coarse centroids (nlist clamped to the training set)
    DevBuf<float> coarse, coarse_norms; // [kc x d], Norms.l2NormSquared per row
    DevBuf<float> coarse_norm_max;      // [1] sqrt(max coarse_norms): error-bound scale of the tensor-core shortlist
    DevBuf<float> codebooks, cb_norms;  // [m x ks x dsub], [m x ks]
    bool has_coarse = false, has_pq = false;
    // rows in add order
    int64_t n = 0;
    int64_t next_auto_id = 0;           // first id of an add without ids: grows with every add, equals n until a removal
    DevBuf<float> vecs;                 // FLAT / IVF_FLAT: [n x d]
    DevBuf<int64_t> ids;                // [n]
    DevBuf<int32_t> assign;             // IVF: [n]
    DevBuf<uint8_t> codes;              // IVF_PQ: [n x m] AoS (the reference's interchange format)
    // inverted lists, rebuilt lazily after adds and removals ("slots": rows sorted by list, list starts 32-aligned)
    bool dirty = true;
    int64_t nslots = 0;
    DevBuf<int64_t> list_off;           // [kc + 1] slot offsets (32-aligned)
    DevBuf<int32_t> list_len;           // [kc]
    DevBuf<int32_t> slot_row;           // [nslots] add-order row of a slot, -1 for padding
    DevBuf<uint8_t> slot_codes;         // [nslots x m] scan layout (vix_scan.cuh)
    DevBuf<uint8_t> tc_codes;           // [nslots x m] the list-major scan's decode layout of the same codes (vix_scan.cuh),
                                        // only when the index can take that path (tc_codes_shape)
    DevBuf<float> slot_tx;              // [nslots]  ||r^||^2 + 2<c, r^>  (L2) / 0 (IP)
    DevBuf<int64_t> slot_ids;           // [nslots]
    DevBuf<float> slot_vecs;            // IVF_FLAT: [nslots x d]
    DevBuf<float> codebooks_t;          // [ks x m x dsub] code-major copy of the codebooks
    DevBuf<uint32_t> tc_table;          // the list-major scan's decode table of these codebooks (vix_scan.cuh), when the
    DevBuf<float> tc_meta;              // shape takes that path; rebuilt with codebooks_t
    int align = 32;                     // list granularity in slots (ScanLayout::align)
    // search_ex(stats): events and counter are created once per handle
    cudaEvent_t ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};   // stage boundaries + the dominant scan kernel
    DevBuf<unsigned long long> scanned;
    // vix_index_trace(): per-call stage events recorded WITHOUT synchronising (read back afterwards)
    std::vector<cudaEvent_t> trace_ev;  // 5 per traced call
    DevBuf<unsigned long long> trace_scanned;
    int trace_cap = 0, trace_n = 0;
    std::vector<int> trace_path;        // IVF-PQ scan path of each traced call
};


namespace vix {

struct FilterArgs { const uint64_t* words = nullptr; int64_t cap = 0; int deny = 0; };

// one search of an index whose mutex the caller holds (all pointers host or device; see vix_index.cu)
int index_search_locked(vix_index* h, const float* queries, int64_t nq, int k, int nprobe, float* out_dist,
                        int64_t* out_ids, int32_t* out_probes, vix_search_stats* stats,
                        const int32_t* given_probes = nullptr, const FilterArgs* filter = nullptr);
// list assignment under the index's metric (device pointers)
int assign_lists_device(vix_index* h, const float* x, int64_t n, int32_t* assign);
// number of assignments outside [0, kc) in a device array (synchronises the stream)
int count_invalid_assign(const int32_t* assign, int64_t n, int kc, unsigned long long* out);
// append already encoded rows (device or host pointers) to an IVF-PQ index whose mutex the caller holds
int index_add_encoded_locked(vix_index* h, const int32_t* assign, const uint8_t* codes, const int64_t* ids, int64_t n);
int build_lists(vix_index* h);
// residual PQ codes (u8, or packed u4 when ks = 16) of rows whose list assignments are known (device pointers)
int encode_rows_device(vix_index* h, const float* x, int64_t n, const int32_t* assign, uint8_t* codes);

}  // namespace vix
