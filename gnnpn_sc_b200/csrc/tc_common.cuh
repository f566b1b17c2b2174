// sm_100a building blocks written as inline PTX: mbarrier, TMA (cp.async.bulk.tensor), tcgen05
// (TMEM alloc / mma / commit / ld), UMMA shared-memory + instruction descriptors.
// Bit layouts follow the PTX ISA "tcgen05" descriptors (as also encoded in CUTLASS's
// cute/arch/mma_sm100_desc.hpp, consulted for the field positions only).
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace gnnpn {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ----------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra WAIT_DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "WAIT_DONE:\n\t"
      "}" ::"r"(bar), "r"(parity) : "memory");
}

// ----------------------------------------------------------------- 256-bit global accesses
// sm_100: one full 32-byte sector per thread per instruction
__device__ __forceinline__ void ldg256(const float* p, float* v) {
  asm volatile("ld.global.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7])
               : "l"(p));
}
__device__ __forceinline__ void stg256(float* p, const float* v) {
  asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]),
               "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]) : "memory");
}

// ----------------------------------------------------------------- TMA
__device__ __forceinline__ void tma_load_2d(uint32_t smem_dst, const CUtensorMap* map, uint32_t bar, int c0,
                                            int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_dst), "l"(map), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

// ----------------------------------------------------------------- tcgen05
__device__ __forceinline__ void tmem_alloc(uint32_t smem_result, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_result), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem], fp32 accumulate, tf32 inputs, issued by ONE thread.
__device__ __forceinline__ void mma_tf32_ss(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// same with fp16 inputs (K = 16 per instruction): twice the MAC rate of tf32 and half the operand bytes
__device__ __forceinline__ void mma_f16_ss(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                           uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// mbarrier arrives once every previously issued tcgen05.mma of this thread has completed.
__device__ __forceinline__ void mma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// 32 lanes x 32 consecutive fp32 columns -> 32 registers per thread (thread i = TMEM lane base+i).
// Split into issue + wait so independent global loads can be put in flight between the two; the wait
// names the registers as read-write operands so no use of them can be scheduled above it.
__device__ __forceinline__ void tmem_ld_32x32_issue(uint32_t taddr, float* v) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait(float* v) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.wait::ld.sync.aligned;"
      : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
        "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]),
        "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]),
        "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
      :
      : "memory");
}

// ----------------------------------------------------------------- activations for the epilogue
// MUFU-based, ~1e-7 absolute error (same order as fp32 rounding of O(1) values); the libm-accurate
// expf/tanhf/IEEE-divide versions cost ~3x the instructions and made the epilogue the bottleneck.
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float rcp_refined(float d) {        // MUFU.RCP + one Newton step
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(d));
  return fmaf(r, fmaf(-d, r, 1.0f), r);
}
__device__ __forceinline__ float sigmoid_mufu(float x) {
  const float t = ex2_approx(fminf(-1.4426950408889634f * x, 80.0f));     // e^-x, clamped so 1+t stays finite
  return rcp_refined(1.0f + t);
}
__device__ __forceinline__ float tanh_mufu(float x) {
  const float ax = fabsf(x);
  // |x| >= 0.55 : 1 - 2/(e^{2|x|} + 1)
  const float t = ex2_approx(fminf(2.8853900817779268f * ax, 80.0f));
  const float big = fmaf(-2.0f, rcp_refined(t + 1.0f), 1.0f);
  // |x| <  0.55 : x + x^3 * P(x^2), degree-4 Chebyshev interpolant of (tanh(x)/x - 1)/x^2 (max rel err 7.3e-8)
  const float u = ax * ax;
  float p = -6.542542018e-03f;
  p = fmaf(p, u, 2.127274871e-02f);
  p = fmaf(p, u, -5.390334874e-02f);
  p = fmaf(p, u, 1.333308220e-01f);
  p = fmaf(p, u, -3.333333135e-01f);
  const float small = fmaf(p * u, ax, ax);
  return copysignf(ax < 0.55f ? small : big, x);
}

// ----------------------------------------------------------------- descriptors
// K-major operand tile, 128-byte rows (32 fp32), 128B swizzle, 8-row groups 1024 B apart, tile 1024B-aligned.
__device__ __forceinline__ uint64_t smem_desc_k_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);   // [0,14)  start address >> 4
  d |= (uint64_t)1 << 16;                         // [16,30) leading byte offset >> 4 (unused: swizzled K-major)
  d |= (uint64_t)(1024 >> 4) << 32;               // [32,46) stride byte offset >> 4
  d |= (uint64_t)1 << 46;                         // [46,48) descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;                         // [61,64) SWIZZLE_128B
  return d;
}

// kind::tf32, fp32 accumulate, A and B K-major, shape M x N (K = 8 per instruction).
__host__ __device__ inline uint32_t idesc_tf32(int M, int N) {
  return (1u << 4)                 // [4,6)   D format: F32
         | (2u << 7)               // [7,10)  A format: TF32
         | (2u << 10)              // [10,13) B format: TF32
         | ((uint32_t)(N >> 3) << 17)   // [17,23) N >> 3
         | ((uint32_t)(M >> 4) << 24);  // [24,29) M >> 4
}

// kind::f16 with fp16 A/B (format 0), fp32 accumulate, K-major operands (K = 16 per instruction).
__host__ __device__ inline uint32_t idesc_f16(int M, int N) {
  return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// round-to-nearest split  a = hi + lo,  hi exactly representable in tf32 (low 13 mantissa bits zero)
__device__ __forceinline__ void split_tf32(float a, float& hi, float& lo) {
  uint32_t h;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(h) : "f"(a));
  hi = __uint_as_float(h);
  lo = a - hi;
}

// fp16 split: hi = fp16(a) (11 significant bits), lo = fp16(a - hi).  For |a| <= 1 the pair represents a with
// absolute error <= 2^-25 (lo falls into fp16 subnormals for small |a|), relative ~2^-22 otherwise.
__device__ __forceinline__ void split_f16(float a, __half& hi, __half& lo) {
  hi = __float2half_rn(a);
  lo = __float2half_rn(a - __half2float(hi));
}

}  // namespace tc
}  // namespace gnnpn
