// vix_common.cuh -- shared host/device helpers for libvindex_b200 (sm_100a only).
//
// Arithmetic contract: every "exact" path reproduces the reference's fp32 operation order with
// separate multiply and add (no FMA).  All such code goes through fmul()/fadd()/fsub() below
// (__f*_rn intrinsics are never contracted by nvcc), and the translation units are additionally
// compiled with -fmad=false.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>

#include <string>

#include "../../include/vindex_cuda.h"

namespace vix {

// ------------------------------------------------------------------------------------------------
// Errors
// ------------------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);
int  cuda_fail(cudaError_t e, const char* what, const char* file, int line);

#define VIX_CUDA(expr)                                                                     \
    do {                                                                                   \
        cudaError_t _e = (expr);                                                           \
        if (_e != cudaSuccess) return ::vix::cuda_fail(_e, #expr, __FILE__, __LINE__);     \
    } while (0)

#define VIX_TRY(expr)                      \
    do {                                   \
        int _s = (expr);                   \
        if (_s != VIX_OK) return _s;       \
    } while (0)

#define VIX_REQUIRE(cond, code, ...)       \
    do {                                   \
        if (!(cond)) {                     \
            ::vix::set_error(__VA_ARGS__); \
            return (code);                 \
        }                                  \
    } while (0)

// ------------------------------------------------------------------------------------------------
// Execution context (thread-local): stream + sync policy
// ------------------------------------------------------------------------------------------------
struct Ctx {
    cudaStream_t stream = 0;   // legacy default stream unless vix_set_stream() was called
    bool async = false;        // true: entry points return without synchronising device outputs
    int64_t launches = 0;      // kernels launched by this thread since the last reset
};
Ctx& ctx();
int ensure_device();           // fails loudly (VIX_ERR_NO_DEVICE) when no CUDA device is usable
int num_sms();

#define VIX_LAUNCH_CHECK()                                   \
    do {                                                     \
        ::vix::ctx().launches += 1;                          \
        VIX_CUDA(cudaGetLastError());                        \
    } while (0)

// ------------------------------------------------------------------------------------------------
// Host/device pointer staging.  Entry points accept host OR device pointers; host inputs are
// copied in, host outputs are copied back (and the stream synchronised) before returning.
// ------------------------------------------------------------------------------------------------
bool is_device_ptr(const void* p);

template <typename T>
struct In {
    const T* dev = nullptr;
    void* owned = nullptr;
    int stage(const T* p, size_t count) {
        release();
        if (p == nullptr || count == 0) { dev = p; return VIX_OK; }
        if (is_device_ptr(p)) { dev = p; return VIX_OK; }
        cudaStream_t s = ctx().stream;
        VIX_CUDA(cudaMallocAsync(&owned, count * sizeof(T), s));
        VIX_CUDA(cudaMemcpyAsync(owned, p, count * sizeof(T), cudaMemcpyHostToDevice, s));
        dev = static_cast<const T*>(owned);
        return VIX_OK;
    }
    void release() {
        if (owned) { cudaFreeAsync(owned, ctx().stream); owned = nullptr; }
        dev = nullptr;
    }
    ~In() { release(); }
};

template <typename T>
struct Out {
    T* dev = nullptr;
    T* host = nullptr;
    void* owned = nullptr;
    size_t count = 0;
    int stage(T* p, size_t n) {
        release();
        count = n;
        if (p == nullptr || n == 0) { dev = p; return VIX_OK; }
        if (is_device_ptr(p)) { dev = p; return VIX_OK; }
        VIX_CUDA(cudaMallocAsync(&owned, n * sizeof(T), ctx().stream));
        dev = static_cast<T*>(owned);
        host = p;
        return VIX_OK;
    }
    // copy back (async on the context stream); caller synchronises via finish()
    int commit() {
        if (host && owned && count)
            VIX_CUDA(cudaMemcpyAsync(host, owned, count * sizeof(T), cudaMemcpyDeviceToHost, ctx().stream));
        return VIX_OK;
    }
    bool is_host() const { return host != nullptr; }
    void release() {
        if (owned) { cudaFreeAsync(owned, ctx().stream); owned = nullptr; }
        dev = nullptr; host = nullptr; count = 0;
    }
    ~Out() { release(); }
};

// scratch device buffer (stream-ordered)
template <typename T>
struct Scratch {
    T* ptr = nullptr;
    int alloc(size_t n) {
        release();
        if (n == 0) return VIX_OK;
        VIX_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&ptr), n * sizeof(T), ctx().stream));
        return VIX_OK;
    }
    void release() {
        if (ptr) { cudaFreeAsync(ptr, ctx().stream); ptr = nullptr; }
    }
    ~Scratch() { release(); }
};

// synchronise when any output lives on the host or the context is synchronous
int finish(bool any_host_output);
int* pipeline_error_flag();    // mapped pinned host int, device-writable (nullptr if it cannot be allocated)
int check_pipeline_error();    // VIX_ERR_CUDA once after a tensor-core pipeline timed out

// ------------------------------------------------------------------------------------------------
// Device helpers
// ------------------------------------------------------------------------------------------------
#ifdef __CUDACC__

__device__ __forceinline__ float fmul(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float fadd(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float fsub(float a, float b) { return __fsub_rn(a, b); }
// ((v0+v1)+v2)+v3 -- the reference's SIMD4 horizontal sum everywhere (SURVEY Appendix A)
__device__ __forceinline__ float hsum4(float a, float b, float c, float d) {
    return fadd(fadd(fadd(a, b), c), d);
}

// Total-order keys.  key = (orderable(score) << 32) | id ; smaller key == better candidate.
// Mirrors HeapOrdering of /root/reference/Sources/VectorIndex/Operations/Selection/TopK.swift:8-31:
// .min => smaller score first, .max => larger score first, ties => smaller id.  NaN => worst.
typedef unsigned long long u64;
constexpr u64 kEmptyKey = 0xFFFFFFFFFFFFFFFFull;

__device__ __forceinline__ uint32_t f32_orderable(float f) {
    uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float f32_from_orderable(uint32_t u) {
    uint32_t v = (u & 0x80000000u) ? (u & 0x7FFFFFFFu) : ~u;
    return __uint_as_float(v);
}
__device__ __forceinline__ u64 make_key(float score, uint32_t id, int order_max) {
    float s = fadd(score, 0.0f);            // -0 -> +0 so that -0 == +0 ties fall to the id
    uint32_t u = f32_orderable(s);
    if (order_max) u = ~u;
    if (s != s) u = 0xFFFFFFFFu;
    return ((u64)u << 32) | (u64)id;
}
__device__ __forceinline__ float key_score(u64 key, int order_max) {
    uint32_t u = (uint32_t)(key >> 32);
    if (order_max) u = ~u;
    return f32_from_orderable(u);
}
__device__ __forceinline__ uint32_t key_id(u64 key) { return (uint32_t)(key & 0xFFFFFFFFull); }
// A CentroidBatchScore value (probe selection) of centroid c as the selection returns it.  make_key folds -0 into +0; the
// sign of a zero score follows from the metric: IP is -s with s summed from +0 in round-to-nearest (never -0), so a zero
// is -0; L2 is -2 s + ||c||^2, a zero is ||c||^2 itself when that is a zero (s = +0, -2 s = -0) and +0 otherwise (exact
// cancellation).
__device__ __forceinline__ float cbs_signed_zero(float s, uint32_t c, int metric, const float* cnorm) {
    if (s != 0.0f) return s;
    if (metric != VIX_METRIC_L2) return -0.0f;
    const float cn = cnorm ? cnorm[c] : 0.0f;
    return cn == 0.0f ? cn : 0.0f;
}

// idFilterPass (Operations/Filtering/IDFilter.swift:115-135): out-of-range ids are dropped in either mode
__device__ __forceinline__ bool id_filter_pass(const uint64_t* __restrict__ words, int64_t cap, int deny, int64_t id) {
    if (id < 0 || id >= cap) return false;
    const bool bit = (__ldg(words + (id >> 6)) >> (id & 63)) & 1ull;
    return deny ? !bit : bit;
}

#endif  // __CUDACC__

}  // namespace vix
