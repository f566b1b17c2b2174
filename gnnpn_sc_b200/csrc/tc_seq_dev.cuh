// Device-side helpers shared by the persistent tcgen05 LSTM scan kernels (tc_seq.cu: a CTA pair, 128 instances per
// CTA; tc_colsplit.cu: the gate columns of 128 instances split over a cluster of 8 CTAs).
#pragma once
#include <cuda_fp16.h>
#include "tc_common.cuh"
#include "tc_lstm.cuh"

namespace gnnpn {
namespace seq {

using namespace tc;

constexpr float kLog2e = 1.4426950408889634f;
constexpr float kClampT = 30.0f;           // exponentials are clamped to 2^30 so products of three stay finite
constexpr int XROW_BYTES = 32;             // x block: 16 halfs per row, 32-byte swizzle layout
constexpr int BM = 128;                    // instances per CTA (column-split: per cluster) = UMMA M = TMEM lanes
constexpr int KB_H = kH / 64;              // 4 k-blocks of 64 halfs (128-byte swizzle rows)
constexpr int BLK_BYTES = 128 * 128;       // one [128 rows x 64 halfs] block
constexpr int EPI_WARPS = 16;
constexpr int THREADS = 128 + 32 * EPI_WARPS;

// K-major operand block with 32-byte rows (16 halfs), 32B swizzle, 8-row groups 256 B apart
__device__ __forceinline__ uint64_t smem_desc_k_sw32(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(256 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)6 << 61;                         // SWIZZLE_32B
  return d;
}

// ---- thread-block-cluster helpers (CTA pair, cta_group::2)
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `addr` (a shared::cta address of this CTA) in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_rank(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  // default semantics (.release.cta): a .release.cluster arrive compiles to MEMBAR.ALL.GPU, which also waits for
  // every global store this thread has in flight (c scratch / h rows) -- ~10% of the epilogue warps' time.  What
  // the leader's MMAs consume is ordered by tcgen05.fence::before_thread_sync (TMEM reads) and
  // fence.proxy.async (shared-memory operand writes) issued before the arrive.
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAITC_LOOP:\n\t"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra WAITC_DONE;\n\t"
      "bra WAITC_LOOP;\n\t"
      "WAITC_DONE:\n\t"
      "}" ::"r"(bar), "r"(parity) : "memory");
}
// TMA load whose completion is signalled on a barrier that may live in the peer CTA of the pair
__device__ __forceinline__ void tma_load_2d_cg2(uint32_t smem_dst, const CUtensorMap* map, uint32_t bar_cluster, int c0,
                                                int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_dst), "l"(map), "r"(bar_cluster), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void mma_f16_ss_cg2(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// the same with A read from tensor memory: lane = row (each CTA of the pair holds its 128 rows at a_tmem), 32-bit
// column c = halfs 2c (low 16 bits) and 2c+1 of the K-major row
__device__ __forceinline__ void mma_f16_ts_cg2(uint32_t tmem_d, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t"
      "}" ::"r"(tmem_d), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// arrives (once all previously issued MMAs retire) on the barrier at this CTA-relative offset in BOTH CTAs of the pair
__device__ __forceinline__ void mma_commit_cg2(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"((uint16_t)3) : "memory");
}
__device__ __forceinline__ void tmem_alloc_cg2(uint32_t smem_result, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_result), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_cg2(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// 1 in exactly one lane of a fully active warp
__device__ __forceinline__ uint32_t elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}" : "=r"(pred));
  return pred;
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void tmem_st_32x32_x4(uint32_t taddr, const uint32_t* r) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};" ::"r"(taddr), "r"(r[0]), "r"(r[1]),
               "r"(r[2]), "r"(r[3]) : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* map, uint32_t smem_src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(map),
               "r"(smem_src), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ float4 ldg128(const float* p) {
  float4 r;
  asm volatile("ld.global.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ void stg128(float* p, float a, float b, float c, float d) {
  asm volatile("st.global.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
__device__ __forceinline__ uint32_t pack_h2(float a, float b) {       // {lo16 = a, hi16 = b}
  const __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&h);
}
__device__ __forceinline__ float2 unpack_h2(uint32_t u) {
  return __half22float2(*reinterpret_cast<const __half2*>(&u));
}

// fp16 hi/lo split of 8 floats: hi[j] = fp16 pair (v[2j], v[2j+1]), lo[j] = the pair's rounding remainders
__device__ __forceinline__ void split_f16x8(const float* v, uint32_t* hi, uint32_t* lo) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    hi[j] = pack_h2(v[2 * j], v[2 * j + 1]);
    const float2 bk = unpack_h2(hi[j]);
    lo[j] = pack_h2(v[2 * j] - bk.x, v[2 * j + 1] - bk.y);
  }
}

// One 32-byte x-block row in shared memory: [x hi (8 halfs) | same again] at hi_addr, the same for lo at lo_addr.  The
// weight block has zeros in halfs 8..15, so the duplicate makes the 32B swizzle pattern irrelevant on the A side.
__device__ __forceinline__ void st_x_row(uint32_t hi_addr, uint32_t lo_addr, const uint32_t* hi, const uint32_t* lo) {
  st_shared_v4(hi_addr, hi[0], hi[1], hi[2], hi[3]);
  st_shared_v4(hi_addr + 16, hi[0], hi[1], hi[2], hi[3]);
  st_shared_v4(lo_addr, lo[0], lo[1], lo[2], lo[3]);
  st_shared_v4(lo_addr + 16, lo[0], lo[1], lo[2], lo[3]);
}

// Encoder x block of step t for the 128 instances from m_first (rows lane + 32i, i < 4 of the calling warp): the raw
// input rows, zeros past n and past F.  P: either scan's parameter struct.
template <class P>
__device__ __forceinline__ void load_x_rows(const P& p, int64_t m_first, int t, int lane, float (*xv)[8]) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t m = m_first + lane + 32 * i;
#pragma unroll
    for (int f = 0; f < 8; ++f)
      xv[i][f] = (m < p.n && f < p.F) ? __ldg(p.inputs + m * p.x_inst_ld + (int64_t)t * p.F + f) : 0.f;
  }
}
// xv from load_x_rows as fp16 hi/lo rows lane + 32i of the x block at ax_hi / ax_lo
__device__ __forceinline__ void write_x_rows(uint32_t ax_hi, uint32_t ax_lo, int lane, const float (*xv)[8]) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const uint32_t o = (uint32_t)(lane + 32 * i) * XROW_BYTES;
    uint32_t hi[4], lo[4];
    split_f16x8(xv[i], hi, lo);
    st_x_row(ax_hi + o, ax_lo + o, hi, lo);
  }
}

// byte offset of the 16-byte chunk holding halfs [8*c16, 8*c16+8) of row r inside a 128B-swizzled block
__device__ __forceinline__ uint32_t sw128_off(int r, int c16) {
  return (uint32_t)((r >> 3) * 1024 + (r & 7) * 128 + ((c16 ^ (r & 7)) << 4));
}

// LSTM cell for 8 hidden units from their 32 gate accumulators (columns 4u+{i,f,g,o}).
// bias4[u] = (-log2e*b_i, -log2e*b_f, -2log2e*b_g, -log2e*b_o); acc = 16 * (pre-activation without bias).
// One reciprocal serves sigm(f), sigm(i) and tanh(g); a second one sigm(o) and tanh(c'):
//   c' = [c(1+Ei)(1+Eg) + (1-Eg)(1+Ef)] / [(1+Ei)(1+Ef)(1+Eg)],   h' = (1-Ec) / [(1+Eo)(1+Ec)]
// with Ex = 2^min(t_x, 30) = e^-x (e^-2x for the tanh arguments).  MUFU.EX2 / MUFU.RCP + one Newton step.
// `gates`, if not null, receives the post-activation gates (training saves: the BPTT reads sigm(i), sigm(f), tanh(g),
// sigm(o)):
//   sigm(i) = d g r, sigm(f) = a g r, tanh(g) = (1 - Eg) a d r, sigm(o) = (1 + Ec) r2     (r, r2 as above)
// It may be v itself: gates 4u..4u+3 are written after v[4u..4u+3] is read.
__device__ __forceinline__ void lstm_cell8(const float* v, const float4* bias4, const float* c_old, float* c_new,
                                           float* h_new, float* gates = nullptr) {
  constexpr float S1 = -kLog2e / kW16Scale, S2 = -2.0f * kLog2e / kW16Scale;
#pragma unroll
  for (int u = 0; u < 8; ++u) {
    const float4 b = bias4[u];
    const float Ei = ex2_approx(fminf(fmaf(v[4 * u + 0], S1, b.x), kClampT));
    const float Ef = ex2_approx(fminf(fmaf(v[4 * u + 1], S1, b.y), kClampT));
    const float Eg = ex2_approx(fminf(fmaf(v[4 * u + 2], S2, b.z), kClampT));
    const float Eo = ex2_approx(fminf(fmaf(v[4 * u + 3], S1, b.w), kClampT));
    const float a = 1.0f + Ei, d = 1.0f + Ef, g = 1.0f + Eg;
    const float ag = a * g;
    const float r = rcp_refined(ag * d);
    const float cn = fmaf(1.0f - Eg, d, c_old[u] * ag) * r;
    const float Ec = ex2_approx(fminf(cn * (-2.0f * kLog2e), kClampT));
    const float r2 = rcp_refined((1.0f + Eo) * (1.0f + Ec));
    c_new[u] = cn;
    h_new[u] = (1.0f - Ec) * r2;
    if (gates) {
      gates[4 * u + 0] = d * g * r;
      gates[4 * u + 1] = ag * r;
      gates[4 * u + 2] = (1.0f - Eg) * (a * d) * r;
      gates[4 * u + 3] = (1.0f + Ec) * r2;
    }
  }
}

}  // namespace seq
}  // namespace gnnpn
