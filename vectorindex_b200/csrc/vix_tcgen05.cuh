// vix_tcgen05.cuh -- the PTX of the tensor-core pipelines (tc_score_kernel in vix_gemm.cu, pq_tc_encode_kernel in
// vix_pq_tc.cu, tc_scan_kernel in vix_ivfpq_tc.cu): mbarriers, TMA, TMEM, tcgen05.mma and their descriptors.
// Every mbarrier wait is bounded: after ~4e9 clocks (~2 s at 2 GHz), or once another thread has given up, the waiting
// thread raises the error flag and the wait returns false, so a stuck pipeline ends with an error instead of hanging the GPU.
#pragma once

#include <cuda.h>
#include <stdint.h>

namespace vix {

// ---------------------------------------------------------------------------------------------- mbarriers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
// after the mbar_init of a CTA's barriers, before the barrier that publishes them to the other threads
__device__ __forceinline__ void mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
// the same with a suspend-time hint: the thread sleeps in hardware until the phase completes or ~`ns` have passed
__device__ __forceinline__ bool mbar_try_wait_sleep(uint64_t* bar, uint32_t parity, uint32_t ns) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity), "r"(ns) : "memory");
    return ok != 0;
}
// raise the device flag (every other waiting thread of the launch polls it) and the optional mapped host copy (raised once,
// never polled by the device)
__device__ __forceinline__ void pipeline_give_up(int* error, int* error_host) {
    atomicExch(error, 1);
    if (error_host) { *reinterpret_cast<volatile int*>(error_host) = 1; __threadfence_system(); }
}
// Two policies, which run at different speeds (each kernel keeps the one it was measured with):
//   mbar_wait        spins, looking at the clock and the (global) error flag on every try: tc_score_kernel, pq_tc_encode_kernel.
//   mbar_wait_sleep  suspends in hardware between tries and looks at the clock and the flag only every 64th try: for kernels
//                    whose waiting warps share the schedulers with warps that set the pace (tc_scan_kernel: 23 warps, four
//                    schedulers, the decoders' issue slots) and whose pipeline hands over so often that a global load per
//                    try (~600 clocks) would slow every hand-over.
__device__ __forceinline__ bool mbar_wait(uint64_t* bar, uint32_t parity, int* error, int* error_host) {
    if (mbar_try_wait(bar, parity)) return true;
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > 4000000000LL || *reinterpret_cast<volatile int*>(error) != 0) {
            pipeline_give_up(error, error_host);
            return false;
        }
    }
    return true;
}
// `waited`: VIX_TCS_DIAG builds add the clocks this wait took (the per-role wait diagnostics of tc_scan_kernel)
__device__ __forceinline__ bool mbar_wait_sleep(uint64_t* bar, uint32_t parity, int* error, int* error_host,
                                                unsigned long long& waited) {
#ifdef VIX_TCS_DIAG
    const long long w0 = clock64();
    struct Acc { unsigned long long& w; long long t; __device__ ~Acc() { w += (unsigned long long)(clock64() - t); } } acc{waited, w0};
#endif
    if (mbar_try_wait(bar, parity)) return true;
    const long long t0 = clock64();
    for (uint32_t spins = 1;; ++spins) {
        if (mbar_try_wait_sleep(bar, parity, 4000u)) return true;
        if ((spins & 63u) == 0 && (clock64() - t0 > 4000000000LL || *reinterpret_cast<volatile int*>(error) != 0)) {
            pipeline_give_up(error, error_host);
            return false;
        }
    }
}

// ---------------------------------------------------------------------------------------------- TMA, TMEM
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(ncols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(ncols));
}
__device__ __forceinline__ void fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// generic-proxy writes to shared memory (st.shared, cp.async) made visible to the async proxy (tcgen05.mma operands)
__device__ __forceinline__ void fence_async_proxy() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// tcgen05.ld is asynchronous: `issue` starts the load of 32 columns into r, `wait` makes them readable.  The wait names
// every register of the load as an in/out operand, so the compiler cannot schedule a use of r in front of it.
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld32_wait(uint32_t (&r)[32]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]),
                   "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]), "+r"(r[16]),
                   "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]), "+r"(r[24]),
                   "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
                 :: "memory");
}
// two loads in flight, one wait: q is pinned right behind it (an empty asm that names q as in/out operands), so no use
// of q is scheduled in front of the wait either
__device__ __forceinline__ void tmem_ld32_wait(uint32_t (&r)[32], uint32_t (&q)[32]) {
    tmem_ld32_wait(r);
    asm volatile(""
                 : "+r"(q[0]), "+r"(q[1]), "+r"(q[2]), "+r"(q[3]), "+r"(q[4]), "+r"(q[5]), "+r"(q[6]), "+r"(q[7]), "+r"(q[8]),
                   "+r"(q[9]), "+r"(q[10]), "+r"(q[11]), "+r"(q[12]), "+r"(q[13]), "+r"(q[14]), "+r"(q[15]), "+r"(q[16]),
                   "+r"(q[17]), "+r"(q[18]), "+r"(q[19]), "+r"(q[20]), "+r"(q[21]), "+r"(q[22]), "+r"(q[23]), "+r"(q[24]),
                   "+r"(q[25]), "+r"(q[26]), "+r"(q[27]), "+r"(q[28]), "+r"(q[29]), "+r"(q[30]), "+r"(q[31])
                 :: "memory");
}
// 16 columns, load and wait in one
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
// .16x128b.x4: register 2 k + e of thread 4 i + c goes to TMEM lane i + 8 e, column 4 k + c (16 lanes x 16 columns)
__device__ __forceinline__ void tmem_st16x128_x4(uint32_t taddr, const uint32_t (&r)[8]) {
    asm volatile(
        "tcgen05.st.sync.aligned.16x128b.x4.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
        ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
        : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---------------------------------------------------------------------------------------------- MMA, descriptors
// Instruction descriptor of tcgen05.mma (kind::tf32 / kind::f16, dense, no negation, A and B K-major): D format at bit 4,
// A and B formats at bits 7 and 10, N >> 3 at bit 17, M >> 4 at bit 24.
constexpr uint32_t kFmtDF32 = 1;                        // D: fp32
constexpr uint32_t kFmtF16 = 0, kFmtTF32 = 2;           // A, B: fp16 (kind::f16), tf32 (kind::tf32)
__host__ __device__ constexpr uint32_t make_idesc(uint32_t d_fmt, uint32_t ab_fmt, int m, int n) {
    return (d_fmt << 4) | (ab_fmt << 7) | (ab_fmt << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
__host__ __device__ constexpr uint32_t idesc_tf32(int m, int n) { return make_idesc(kFmtDF32, kFmtTF32, m, n); }
__host__ __device__ constexpr uint32_t idesc_f16(int m, int n) { return make_idesc(kFmtDF32, kFmtF16, m, n); }

// K-major operand tile [rows][128 B] with 128B swizzle (8-row atoms of 1024 B); the leading byte offset (bit 16) is unused
__device__ __forceinline__ uint64_t make_desc_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);        // start address
    d |= (uint64_t)(1024 >> 4) << 32;                  // stride byte offset: one atom
    d |= (uint64_t)1 << 46;                            // descriptor version (Blackwell)
    d |= (uint64_t)2 << 61;                            // SWIZZLE_128B
    return d;
}

// A and B from shared memory
__device__ __forceinline__ void mma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// A operand in TMEM (rows = lanes, 32-bit columns of two halves), B from shared memory
__device__ __forceinline__ void mma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrives on `bar` when every tcgen05.mma this thread issued before it has completed
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

namespace tc {  // host side, defined in vix_gemm.cu
// TMA map of a rows x d fp32 row-major operand: boxes of 32 columns (128 B) x box_rows rows, 128B swizzle, zero fill
int make_map_rows(CUtensorMap* map, const float* ptr, int64_t rows, int d, int box_rows);
// whether tc_score_kernel takes A [nA x d] and B [nB x d] (sizes, 16-byte alignment, the driver's TMA encoder)
bool supported(int64_t nA, int64_t nB, int d, const float* A, const float* B);
}  // namespace tc

}  // namespace vix
