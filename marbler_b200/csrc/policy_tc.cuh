// tcgen05 / TMEM / bulk-copy building blocks of the persistent policy kernel (policy_tc2.cuh): mbarrier and
// cp.async.bulk wrappers, UMMA shared-memory / instruction descriptors, tcgen05.mma / commit / ld wrappers, the SFU
// gate functions.
//
// Canonical K-major layout, no swizzle (CUTLASS cute/atom/mma_traits_sm100.hpp "LayoutType::INTERLEAVE:
// ((8,n),2):((1,SBO),LBO)" in 16-byte units): element (row r, k) of an operand with R rows lives at
//     (k / 8) * LBO + (r / 8) * SBO + (r % 8) * 16 + (k % 8) * 2   bytes,   SBO = 128,
// i.e. 8 rows x 8 halves form one contiguous 128-byte core matrix.  Weights use LBO = R / 8 * 128 (dense);
// the activation buffers use LBO = 2064 so that the row-wise staging stores do not all hit one bank group.
// Every wait on an mbarrier is bounded and traps instead of hanging the GPU.
#pragma once
#include <cuda_fp16.h>

#include "common.cuh"

namespace mrb {
namespace tc {

constexpr int kRows = 128, kH = 128;                       // envs per tile; hidden width this path is built for
constexpr int kActLBO = 2048 + 16;                         // activation buffers: padded k-chunk stride
constexpr int kActBytes = 16 * kActLBO;                    // 128 rows x 128 k
constexpr int kMaxKp1 = 64;                                // fc1 input width (padded to 16)
constexpr int kBiasFloats = kH + 3 * kH + 3 * kH + 32;     // b1 | b_ih | b_hh | b2

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
    uint32_t done = 0, spins = 0;
    while (!done) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(bar), "r"(parity) : "memory");
        if (!done && ++spins > (1u << 22)) __trap();      // never hang the device on a protocol bug
    }
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// shared-memory matrix descriptor: start address, LBO, SBO in 16-byte units, version 1 (sm_100), no swizzle
__device__ __forceinline__ uint64_t make_desc(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes)
{
    return (uint64_t)((addr >> 4) & 0x3fff) | ((uint64_t)((lbo_bytes >> 4) & 0x3fff) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3fff) << 32) | (1ull << 46);
}
// instruction descriptor, kind::f16: D = F32, A = B = F16, both K-major, M = 128, N = n
__host__ __device__ constexpr uint32_t make_idesc(int n) { return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24); }
__device__ __forceinline__ void umma(uint32_t d_tmem, uint64_t a, uint64_t b, uint32_t idesc, uint32_t accumulate)
{
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(d_tmem), "l"(a), "l"(b), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t addr, float (&v)[16])
{
    uint32_t r[16];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(addr));
#pragma unroll
    for (int i = 0; i < 16; i++) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ uint32_t h2(float lo, float hi)
{
    const __half2 v = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<const uint32_t *>(&v);
}
__device__ __forceinline__ float ex2a(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rcpa(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float sigm(float x) { return rcpa(1.f + ex2a(-1.4426950408889634f * x)); }
__device__ __forceinline__ float tanh_(float x) { return fmaf(2.f, rcpa(1.f + ex2a(-2.8853900817779268f * x)), -1.f); }

}  // namespace tc
}  // namespace mrb
