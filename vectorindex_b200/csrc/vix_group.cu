// vix_group.cu -- grouping rows by a small integer key (vix_group.cuh): the radix sorts and prefix sums of the build side,
// key histograms and offsets, and the small copy kernels the builders share.
#include "vix_group.cuh"

#include <cub/cub.cuh>

namespace vix {

namespace {

template <typename T>
__global__ void sequence_kernel(T* a, int64_t n, T start) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) a[i] = start + (T)i;
}

template <typename T>
__global__ void fill_kernel(T* a, int64_t n, T v) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) a[i] = v;
}

// one CTA per row
template <typename I>
__global__ void gather_rows_kernel(const float* __restrict__ x, int d, const I* __restrict__ rows, int64_t n,
                                   float* __restrict__ out) {
    const int64_t i = blockIdx.x;
    if (i >= n) return;
    const float* src = x + (int64_t)rows[i] * d;
    for (int e = threadIdx.x; e < d; e += blockDim.x) out[i * d + e] = src[e];
}

__global__ void seq_norms_kernel(const float* __restrict__ c, int64_t rows, int dsub, float* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows) return;
    float s = 0.0f;
    for (int e = 0; e < dsub; ++e) s = fadd(s, fmul(c[i * dsub + e], c[i * dsub + e]));
    out[i] = s;
}

__global__ void key_hist_kernel(const int32_t* __restrict__ keys, int64_t n, int nkeys, int32_t* __restrict__ counts) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        const int k = keys[i];
        if (k >= 0 && k < nkeys) atomicAdd(counts + k, 1);
    }
}

// single CTA: off[l+1] = off[l] + roundup(len[l], align); also unpadded offsets (CSR of the sorted rows) when off_raw != 0
__global__ void offsets_kernel(const int32_t* __restrict__ len, int kc, int align, int64_t* __restrict__ off,
                               int64_t* __restrict__ off_raw) {
    __shared__ int64_t s_pad[1024], s_raw[1024];
    __shared__ int64_t carry_pad, carry_raw;
    if (threadIdx.x == 0) { carry_pad = 0; carry_raw = 0; off[0] = 0; if (off_raw) off_raw[0] = 0; }
    __syncthreads();
    for (int base = 0; base < kc; base += 1024) {
        int l = base + threadIdx.x;
        int64_t v = (l < kc) ? len[l] : 0;
        int64_t vp = (v + align - 1) / align * align;
        s_pad[threadIdx.x] = vp; s_raw[threadIdx.x] = v;
        __syncthreads();
        for (int o = 1; o < 1024; o <<= 1) {     // Hillis-Steele inclusive scan
            int64_t a = 0, b = 0;
            if ((int)threadIdx.x >= o) { a = s_pad[threadIdx.x - o]; b = s_raw[threadIdx.x - o]; }
            __syncthreads();
            s_pad[threadIdx.x] += a; s_raw[threadIdx.x] += b;
            __syncthreads();
        }
        if (l < kc) { off[l + 1] = carry_pad + s_pad[threadIdx.x]; if (off_raw) off_raw[l + 1] = carry_raw + s_raw[threadIdx.x]; }
        __syncthreads();
        if (threadIdx.x == 1023) { carry_pad += s_pad[1023]; carry_raw += s_raw[1023]; }
        __syncthreads();
    }
}

inline unsigned blocks_256(int64_t n) { return (unsigned)((n + 255) / 256); }

// CUB's two phases: query the temporary storage, allocate it (stream-ordered), run
template <typename Call>
int cub_run(Call call) {
    size_t bytes = 0;
    VIX_CUDA(call(nullptr, bytes));
    Scratch<unsigned char> tmp;
    VIX_TRY(tmp.alloc(bytes + 16));
    VIX_CUDA(call(tmp.ptr, bytes));
    ctx().launches += 1;
    return VIX_OK;
}

}  // namespace

template <typename K>
int sort_pairs(const K* keys_in, K* keys_out, const int32_t* vals_in, int32_t* vals_out, int64_t n, int bits) {
    return cub_run([&](void* tmp, size_t& bytes) {
        return cub::DeviceRadixSort::SortPairs(tmp, bytes, keys_in, keys_out, vals_in, vals_out, (int)n, 0, bits, ctx().stream);
    });
}
template int sort_pairs<int32_t>(const int32_t*, int32_t*, const int32_t*, int32_t*, int64_t, int);
template int sort_pairs<uint32_t>(const uint32_t*, uint32_t*, const int32_t*, int32_t*, int64_t, int);

int sort_keys(const uint32_t* keys_in, uint32_t* keys_out, int64_t n) {
    return cub_run([&](void* tmp, size_t& bytes) {
        return cub::DeviceRadixSort::SortKeys(tmp, bytes, keys_in, keys_out, (int)n, 0, 32, ctx().stream);
    });
}

int exclusive_sum(const int32_t* in, int32_t* out, int64_t n) {
    return cub_run([&](void* tmp, size_t& bytes) {
        return cub::DeviceScan::ExclusiveSum(tmp, bytes, in, out, (int)n, ctx().stream);
    });
}

int order_by_key(const int32_t* keys, int64_t n, int nkeys, int32_t* order, int32_t* keys_sorted) {
    Scratch<int32_t> rows, sorted;
    VIX_TRY(rows.alloc((size_t)n));
    if (!keys_sorted) { VIX_TRY(sorted.alloc((size_t)n)); keys_sorted = sorted.ptr; }
    VIX_TRY(iota<int32_t>(rows.ptr, n, 0));
    int bits = 1;
    while ((1LL << bits) < nkeys) ++bits;
    return sort_pairs<int32_t>(keys, keys_sorted, rows.ptr, order, n, bits);
}

int key_offsets(const int32_t* keys, int64_t n, int nkeys, int32_t* counts, int64_t* off, int align, int64_t* off_raw) {
    cudaStream_t s = ctx().stream;
    VIX_CUDA(cudaMemsetAsync(counts, 0, (size_t)nkeys * 4, s));
    if (n > 0) {
        key_hist_kernel<<<blocks_256(n), 256, 0, s>>>(keys, n, nkeys, counts);
        VIX_LAUNCH_CHECK();
    }
    return offsets_from_counts(counts, nkeys, align, off, off_raw);
}

int offsets_from_counts(const int32_t* counts, int nkeys, int align, int64_t* off, int64_t* off_raw) {
    offsets_kernel<<<1, 1024, 0, ctx().stream>>>(counts, nkeys, align, off, off_raw);
    VIX_LAUNCH_CHECK();
    return VIX_OK;
}

template <typename T>
int iota(T* a, int64_t n, T start) {
    if (n <= 0) return VIX_OK;
    sequence_kernel<T><<<blocks_256(n), 256, 0, ctx().stream>>>(a, n, start);
    VIX_LAUNCH_CHECK();
    return VIX_OK;
}
template int iota<int32_t>(int32_t*, int64_t, int32_t);
template int iota<int64_t>(int64_t*, int64_t, int64_t);

template <typename T>
int fill(T* a, int64_t n, T v) {
    if (n <= 0) return VIX_OK;
    fill_kernel<T><<<blocks_256(n), 256, 0, ctx().stream>>>(a, n, v);
    VIX_LAUNCH_CHECK();
    return VIX_OK;
}
template int fill<float>(float*, int64_t, float);
template int fill<int32_t>(int32_t*, int64_t, int32_t);

template <typename I>
int gather_rows(const float* x, int d, const I* rows, int64_t n, float* out) {
    if (n <= 0) return VIX_OK;
    gather_rows_kernel<I><<<(unsigned)n, 128, 0, ctx().stream>>>(x, d, rows, n, out);
    VIX_LAUNCH_CHECK();
    return VIX_OK;
}
template int gather_rows<int32_t>(const float*, int, const int32_t*, int64_t, float*);
template int gather_rows<int64_t>(const float*, int, const int64_t*, int64_t, float*);

int seq_norms(const float* c, int64_t rows, int dsub, float* out) {
    if (rows <= 0) return VIX_OK;
    seq_norms_kernel<<<(unsigned)((rows + 127) / 128), 128, 0, ctx().stream>>>(c, rows, dsub, out);
    VIX_LAUNCH_CHECK();
    return VIX_OK;
}

}  // namespace vix
