// Shared device/host helpers for the b2dt kernels (sm_100a only).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "b2dt.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ != 1000)
#error "b2dt kernels are written for sm_100a (B200) only"
#endif

// ---------------------------------------------------------------------------------------------
// error plumbing: every C-ABI entry returns an int status and records a message (thread local)
// ---------------------------------------------------------------------------------------------
void b2_set_error(const char* fmt, ...);

#define B2_CUDA(expr)                                                                          \
    do {                                                                                       \
        cudaError_t _e = (expr);                                                               \
        if (_e != cudaSuccess) {                                                               \
            b2_set_error("%s:%d: %s failed: %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
            return B2_ERR_CUDA;                                                                \
        }                                                                                      \
    } while (0)

#define B2_REQUIRE(cond, ...)                                                                  \
    do {                                                                                       \
        if (!(cond)) {                                                                         \
            b2_set_error(__VA_ARGS__);                                                         \
            return B2_ERR_ARG;                                                                 \
        }                                                                                      \
    } while (0)

static inline int b2_ceil_div(int a, int b) { return (a + b - 1) / b; }
int b2_num_sms();

// ---------------------------------------------------------------------------------------------
// small device utilities
// ---------------------------------------------------------------------------------------------
#ifdef __CUDACC__
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ float silu_f(float x) { return __fdividef(x, 1.0f + __expf(-x)); }
__device__ __forceinline__ float ex2_ftz(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
// Programmatic dependent launch (sm_90+): a kernel launched with cudaLaunchAttributeProgrammaticStreamSerialization may start
// (prologue: barrier init, TMEM allocation, weight preload) while its predecessor in the stream still runs its last tiles;
// pdl_wait() returns once the predecessor grid has completed and its writes are visible, pdl_launch_dependents() lets the
// successor's CTAs be scheduled as soon as SM resources free up.  Both are no-ops for launches without the attribute.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// exp(f - m), f <= m, for the DFL softmax: one FFMA + one MUFU (ml = m * log2 e).  decode_kernel and the fused Detect
// epilogue of conv_tc_kernel both use it, so the two paths give the same bits.
constexpr float kLog2e = 1.4426950408889634f;
__device__ __forceinline__ float dfl_exp(float f, float ml) { return ex2_ftz(fmaf(f, kLog2e, -ml)); }
// SiLU(x) = h + h tanh(h), h = x / 2: ONE MUFU op (tanh.approx.f32, max relative error 2^-11 on the tanh) and two FP32 ops.
// Absolute error <= |h| * 2^-11 (reached on the negative lobe, |SiLU| <= 0.28 there): below the bf16 rounding of the stored
// activation for every x > -1.5 and <= 1.2e-3 absolute beyond; the epilogues were MUFU / issue bound with the two-MUFU form.
__device__ __forceinline__ float silu_fast(float x) {
    const float h = 0.5f * x;
    float t;
    asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
    return fmaf(h, t, h);
}

// the same with h = x / 2 already formed (epilogues fold the halving into the bias FFMA)
__device__ __forceinline__ float silu_half(float h) {
    float t;
    asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
    return fmaf(h, t, h);
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float bf16_lo(uint32_t v) { return __uint_as_float(v << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t v) { return __uint_as_float(v & 0xFFFF0000u); }

__device__ __forceinline__ uint4 ldg_nc_v4(const void* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}

// ---- mbarrier -------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// B2_MBAR_NS: suspend-time hint of try_wait in ns (0: the plain form).  A waiting warp runs ~17 iterations of the spin loop per
// tile; the hint lets the hardware hold the thread a little longer per attempt.  Measured (one box, tools/ab_chain.py alone and
// tools/sustained.py under the power cap): 1 us and 20 us hints wake the waiter late -- chained convs 1-3 % slower alone, 0.5 %
// faster sustained; 200 ns is neutral-to-better on both (+0.3 % / +0.3 %) and is the default.
#ifndef B2_MBAR_NS
#define B2_MBAR_NS 200u
#endif
constexpr uint32_t kMbarSuspendNs = B2_MBAR_NS;
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
#if B2_MBAR_NS
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}" : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity), "r"(kMbarSuspendNs) : "memory");
#else
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}" : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
#endif
    return ok != 0;
}
// Bounded spin: a pipeline bug must trap instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        if (++spins > (1u << 22)) {
            printf("b2dt: mbarrier wait timed out (block %d thread %d)\n", blockIdx.x, threadIdx.x);
            __trap();
        }
    }
}

// Warp-collective wait: every lane polls and a vote makes the loop condition warp-uniform, so the compiler may keep the
// caller's loop state in uniform registers across the wait (a per-lane spin loop is a divergent region: everything live
// across it falls back to vector registers + R2UR, which made the MMA issue loops 2x slower than the tensor pipe).
__device__ __forceinline__ void mbar_wait_uniform(uint64_t* bar, uint32_t parity) {
    uint32_t spins = 0;
    while (!__any_sync(0xffffffffu, mbar_try_wait(bar, parity))) {
        if (++spins > (1u << 22)) {
            if ((threadIdx.x & 31) == 0) printf("b2dt: mbarrier wait timed out (block %d thread %d)\n", blockIdx.x, threadIdx.x);
            __trap();
        }
    }
}

// ---- TMA (tiled tensor maps) ------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(m) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(smem_u32(smem_dst)), "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
                 ::"r"(smem_u32(smem_dst)), "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}

__device__ __forceinline__ void tma_load_5d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2, int c3, int c4) {
    asm volatile("cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
                 ::"r"(smem_u32(smem_dst)), "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4) : "memory");
}

// ---- tcgen05 / TMEM ---------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() { asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, bf16 inputs, fp32 accumulate, M=128 (cta_group::1)
__device__ __forceinline__ void tc_mma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
// Same instructions predicated on a per-lane flag inside the asm, so that the surrounding code stays warp-converged
// (operands then live in uniform registers and no per-instruction election loop is generated).
__device__ __forceinline__ void tc_mma_bf16_if(uint32_t issue, uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p, q;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "setp.ne.b32 q, %5, 0;\n\t"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate), "r"(issue) : "memory");
}
__device__ __forceinline__ void tc_commit_if(uint32_t issue, uint64_t* bar) {
    asm volatile(
        "{\n\t"
        ".reg .pred q;\n\t"
        "setp.ne.b32 q, %1, 0;\n\t"
        "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t"
        "}" ::"r"(smem_u32(bar)), "r"(issue) : "memory");
}
// 32 lanes x 16 consecutive fp32 columns -> 16 registers per thread (thread t <-> lane base+t)
__device__ __forceinline__ void tmem_ld16(uint32_t addr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(addr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
#endif  // __CUDACC__
