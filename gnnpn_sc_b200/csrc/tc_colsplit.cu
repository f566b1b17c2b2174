// Column-split persistent tcgen05 LSTM scan for SMALL batches (latency mode).
//
// tc_seq.cu gives every CTA (pair) 128 instances and all 4H = 1024 gate columns: a time step costs ~31k cycles no
// matter how few instances there are, so a batch of n <= ~4k instances (the reference's own batch is 128; the
// scale-up configuration fits ~1.5k instances of L = 100,000 in HBM) leaves most of the 148 SMs idle while the L
// dependent steps run.  Here a CLUSTER of 8 CTAs shares one group of 128 instances and splits the gate columns:
// CTA r owns hidden units [32r, 32r+32) = gate columns [128r, 128r+128) for the whole scan.
//   * its slice of the folded weights (fp16 hi/lo, 136 KB) is loaded ONCE and stays resident in shared memory;
//   * its cell state lives in REGISTERS (thread = instance row x 8 units) for the whole scan;
//   * per step it issues 51 MMAs (M=128, N=128, K=16; 3xFP16 split, fp32 accumulate in TMEM) instead of 408;
//   * h'(t) is exchanged through an L2-resident scratch: every CTA writes its [128 x 32] slice as fp16 hi/lo rows,
//     publishes it with remote mbarrier arrives to the 8 CTAs of the cluster (one barrier per 64-unit k-block and
//     step parity), and every CTA pulls the full [128 x 256] operand back with TMA (128B swizzle = UMMA layout)
//     through a 5-slot ring, k-block by k-block, as soon as the two CTAs that produce that k-block have arrived.
//     (DSMEM stores were not used for the exchange: ~21 B/cycle per SM would cost ~6k cycles per step.)
// Reference semantics: nn.LSTM cell, gate order i,f,g,o (modelPN.py:157,191); same packed weights, same cell
// epilogue (lstm_cell8) as tc_seq.cu.
#include <stdio.h>
#include <cuda_fp16.h>
#include "tc_common.cuh"
#include "common.cuh"
#include "internal.cuh"
#include "lstm_step.cuh"
#include "tc_lstm.cuh"
#include "tc_seq.cuh"
#include "tc_seq_dev.cuh"
#include "pointer.cuh"

namespace gnnpn {
namespace cs {

using namespace tc;
using namespace seq;

constexpr int CL = 8;                      // CTAs per cluster = column slices
constexpr int TILE_N = kG / CL;            // 128 gate columns per CTA
constexpr int UNITS = kH / CL;             // 32 hidden units per CTA

// G = instance groups of 128 per cluster.  G = 1: lowest latency.  G = 2 (encoder only): two independent groups share the
// resident weights and are software-pipelined against each other -- while one group's h' is in flight through the exchange
// (cell epilogue -> publish -> TMA pull, ~8.7k of the 12k cycles of a step) the tensor pipe and the epilogue warps work
// on the other one.
template <int G> struct Layout {
  static constexpr int NSLOT = G == 1 ? 5 : 4;         // A ring slots (one per k-block half: lo or hi)
  static constexpr uint32_t OFF_W_HI = 0;
  static constexpr uint32_t OFF_W_LO = OFF_W_HI + KB_H * BLK_BYTES;
  static constexpr uint32_t OFF_WX_HI = OFF_W_LO + KB_H * BLK_BYTES;
  static constexpr uint32_t OFF_WX_LO = OFF_WX_HI + TILE_N * XROW_BYTES;
  static constexpr uint32_t OFF_AX = OFF_WX_LO + TILE_N * XROW_BYTES;       // per group: hi | lo x block
  static constexpr uint32_t AX_BYTES = 2 * BM * XROW_BYTES;
  static constexpr uint32_t OFF_RING = OFF_AX + G * AX_BYTES;
  static constexpr uint32_t OFF_BIAS = OFF_RING + NSLOT * BLK_BYTES;
  static constexpr uint32_t OFF_BAR = OFF_BIAS + 2 * TILE_N * 4;
  static constexpr int BAR_BYTES = G <= 2 ? 256 : 512;
  static constexpr int SMEM_BYTES = OFF_BAR + BAR_BYTES + 1024;
  static constexpr int TMEM_COLS = G * TILE_N <= 128 ? 128 : (G * TILE_N <= 256 ? 256 : 512);    // power of two
  static_assert(SMEM_BYTES <= 232448, "exceeds the 227 KB per-CTA shared memory limit");
  static_assert(8 * (1 + 2 * NSLOT + G * (3 + 2 * KB_H)) + 4 <= BAR_BYTES, "barrier block overflow");
  static_assert(G * TILE_N <= 512, "accumulators exceed TMEM");
};
constexpr uint32_t W_BYTES = 2 * KB_H * BLK_BYTES + 2 * TILE_N * XROW_BYTES;

struct Params {
  int64_t n;
  int steps, F, L;
  const float* inputs; int64_t x_inst_ld;
  const float* bias0;      // [kG] gate-interleaved bias of step 0 (decoder: start-token bias)
  const float* bias;       // [kG] bias of steps >= 1
  const float* c;          // [n, kH] decoder: initial cell state
  float* c_out;            // [n, kH] final cell state, or nullptr (rollout launches: c is shared by the rollouts)
  // Rollout launches (decoder, as in tc_seq.cu): cluster -> (instance groups, rollout) with the rollouts of one set of
  // groups adjacent; rollout r has its own dec_h slice and exchange scratch.  1 for every other launch.
  int rollouts;
  const float* sampled;    // [rollouts-1, K, n] uniforms of rollouts 1.. (pointer.cuh::rollout_args)
  const float* h0; int64_t h0_ld;          // decoder: initial hidden rows
  float* h_out; int64_t h_out_inst_ld;     // step t of instance m at h_out + m*ld + t*kH (enc_out / dec_h)
  __half* scratch;         // [groups][parity 2][hi|lo][128][kH] halfs
  PointerStepArgs pa;      // decoder only
  unsigned long long* prof;
  float* save_gates;       // training: [steps, n, kG] post-activation gates (columns 4j + {i,f,g,o}) or nullptr
  float* save_c;           // training: [steps, n, kH] cell state after every step or nullptr
};

__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }
// remote arrive that releases this thread's prior writes at cluster scope (compiles to a GPU-scope membar + arrive;
// cumulative: it also covers the writes of the other lanes that reached the preceding __syncwarp)
__device__ __forceinline__ void mbar_arrive_release_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void stg128_u(void* p, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.global.v4.b32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void st_cluster_v4(uint32_t cluster_addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared::cluster.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(cluster_addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

// Publish index of h'(t): the decoder also publishes its initial hidden state (index 0), so h'(t) has index t+1 there.
// Index j lives in scratch parity j & 1 and completes phase (j >> 1) & 1 of the a_rdy[group][j & 1][*] barriers.
template <bool DEC, int G>
__global__ void __launch_bounds__(THREADS, 1)
lstm_colsplit_kernel(const __grid_constant__ CUtensorMap map_wh_hi, const __grid_constant__ CUtensorMap map_wh_lo,
                     const __grid_constant__ CUtensorMap map_wx_hi, const __grid_constant__ CUtensorMap map_wx_lo,
                     const __grid_constant__ CUtensorMap map_scr, const __grid_constant__ Params p) {
  static_assert(!DEC || G <= 2, "the fused decoder runs one or two groups per cluster");
  using LY = Layout<G>;
  constexpr int NSLOT = LY::NSLOT;
  constexpr int SET_WARPS = EPI_WARPS;                 // every epilogue warp serves every group
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* sgen = smem_raw + (sbase - smem_u32(smem_raw));
  const uint32_t bar0 = sbase + LY::OFF_BAR;
  const uint32_t w_full = bar0;
  auto full_bar = [&](int s) { return bar0 + 8u * (1 + s); };
  auto empty_bar = [&](int s) { return bar0 + 8u * (1 + NSLOT + s); };
  const uint32_t gbar0 = bar0 + 8u * (1 + 2 * NSLOT);                      // per group: tfull, tempty, x_rdy, a_rdy[2][4]
  auto tfull = [&](int g) { return gbar0 + 8u * (g * (3 + 2 * KB_H)); };
  auto tempty = [&](int g) { return tfull(g) + 8u; };
  auto x_rdy = [&](int g) { return tfull(g) + 16u; };
  auto a_rdy = [&](int g, int par, int kb) { return tfull(g) + 24u + 8u * (par * KB_H + kb); };
  const uint32_t tmem_slot = gbar0 + 8u * (G * (3 + 2 * KB_H));
  auto ax_hi_off = [&](int g) { return sbase + LY::OFF_AX + (uint32_t)g * LY::AX_BYTES; };
  auto ax_lo_off = [&](int g) { return ax_hi_off(g) + BM * XROW_BYTES; };
  const uint32_t rank = cluster_ctarank();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t cluster = blockIdx.x / CL;
  const int roll = (int)(cluster % p.rollouts);
  const int64_t group0 = (cluster / p.rollouts) * G;                      // first instance group of this cluster
  const int64_t sgroup0 = cluster * G;                                    // its first group of the exchange scratch
  float* sbias = reinterpret_cast<float*>(sgen + LY::OFF_BIAS);
  constexpr int PUB0 = DEC ? 1 : 0;                    // publish index of h'(t) = t + PUB0

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_wh_hi); tma_prefetch_desc(&map_wh_lo);
    tma_prefetch_desc(&map_wx_hi); tma_prefetch_desc(&map_wx_lo); tma_prefetch_desc(&map_scr);
  }
  if (warp == 1 && lane == 0) {
    mbar_init(w_full, 1);
    for (int s = 0; s < NSLOT; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int g = 0; g < G; ++g) {
      mbar_init(tfull(g), 1);
      mbar_init(tempty(g), SET_WARPS);
      mbar_init(x_rdy(g), DEC ? CL * EPI_WARPS : 1);   // decoder: one arrival per instance of the group (its pointer warp)
      for (int par = 0; par < 2; ++par)
        for (int kb = 0; kb < KB_H; ++kb) mbar_init(a_rdy(g, par, kb), 2 * SET_WARPS);   // the two CTAs producing this k-block
    }
    fence_mbar_init();
  }
  if (warp == 2) tmem_alloc(tmem_slot, LY::TMEM_COLS);
  // transformed biases of this CTA's 128 gate columns (two sets: step 0, steps >= 1): (i,f,o) * -log2e, g * -2log2e
  for (int i = threadIdx.x; i < 2 * TILE_N; i += THREADS) {
    const int col = i & (TILE_N - 1);
    const float b = __ldg((i < TILE_N ? p.bias0 : p.bias) + rank * TILE_N + col);
    sbias[i] = b * ((col & 3) == 2 ? -2.0f * kLog2e : -kLog2e);
  }

  // load_x_rows is called through this lambda, as in tc_seq.cu: calling it directly changes the generated code
  auto load_inputs = [&](int g, int t, float (*xv)[8]) { load_x_rows(p, (group0 + g) * BM, t, lane, xv); };
  if (!DEC && warp == 3) {
    for (int g = 0; g < G; ++g) {
      float xv[4][8];
      load_inputs(g, 0, xv);
      write_x_rows(ax_hi_off(g), ax_lo_off(g), lane, xv);
    }
  }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncwarp();
  cluster_sync_all();                       // barrier inits visible cluster-wide before any remote arrive
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
  const bool prof = p.prof != nullptr;

  if (warp == 0) {
    // ================= TMA: resident weight slice once; then the A operand of every (step, group) from the exchange scratch
    if (lane == 0) {
      const int col0 = (int)rank * TILE_N;
      mbar_arrive_expect_tx(w_full, W_BYTES);
      for (int kb = 0; kb < KB_H; ++kb) {
        tma_load_2d(sbase + LY::OFF_W_HI + kb * BLK_BYTES, &map_wh_hi, w_full, kb * 64, col0);
        tma_load_2d(sbase + LY::OFF_W_LO + kb * BLK_BYTES, &map_wh_lo, w_full, kb * 64, col0);
      }
      tma_load_2d(sbase + LY::OFF_WX_HI, &map_wx_hi, w_full, kH, col0);
      tma_load_2d(sbase + LY::OFF_WX_LO, &map_wx_lo, w_full, kH, col0);
      int s = 0; uint32_t ph = 0;
      long long w_rdy = 0;
      for (int t = DEC ? 0 : 1; t < p.steps; ++t) {
        const int j = t - 1 + PUB0;                                    // publish index consumed by step t
        const int par = j & 1;
        const uint32_t rph = (uint32_t)(j >> 1) & 1u;
        for (int g = 0; g < G; ++g) {
          const int row_base = (int)(((sgroup0 + g) * 2 + par) * 2) * BM;      // hi rows; lo rows follow BM later
          for (int kb = 0; kb < KB_H; ++kb) {
            const long long t0 = prof ? clock64() : 0;
            mbar_wait_cluster(a_rdy(g, par, kb), rph);                   // both producers of units [64kb, 64kb+64) have published
            if (prof) w_rdy += clock64() - t0;
            fence_proxy_async_all();
#pragma unroll
            for (int part = 0; part < 2; ++part) {                       // lo first: its 4 MMAs free the slot early
              mbar_wait(empty_bar(s), ph ^ 1u);
              mbar_arrive_expect_tx(full_bar(s), BLK_BYTES);
              tma_load_2d(sbase + LY::OFF_RING + s * BLK_BYTES, &map_scr, full_bar(s), kb * 64, row_base + (part ? 0 : BM));
              if (++s == NSLOT) { s = 0; ph ^= 1u; }
            }
          }
        }
      }
      if (prof) p.prof[(size_t)blockIdx.x * 8 + 0] = (unsigned long long)w_rdy;
    }
  } else if (warp == 1) {
    // ================= MMA issuer =================
    const uint32_t leader = elect_one();
    const uint32_t idesc = idesc_f16(BM, TILE_N);
    const uint64_t wx_hi = smem_desc_k_sw32(sbase + LY::OFF_WX_HI), wx_lo = smem_desc_k_sw32(sbase + LY::OFF_WX_LO);
    mbar_wait(w_full, 0);
    tc_fence_after();
    int s = 0; uint32_t ph = 0;
    long long w_full_c = 0;
    const long long t_begin = clock64();
    for (int t = 0; t < p.steps; ++t) {
      for (int g = 0; g < G; ++g) {
        const uint32_t d = tmem_base + (uint32_t)(g * TILE_N);
        const uint64_t ax_hi = smem_desc_k_sw32(ax_hi_off(g)), ax_lo = smem_desc_k_sw32(ax_lo_off(g));
        mbar_wait(tempty(g), ((uint32_t)t & 1u) ^ 1u);
        tc_fence_after();
        // MMA order per step = tc_seq.cu's order per tile (h part k-block by k-block: a_lo.w_hi, a_hi.w_hi, a_hi.w_lo;
        // then the x part), so both scans produce the same bits and a batch can be sharded across them freely.
        uint32_t acc = 0u;                                     // the first MMA of a step overwrites the accumulator
        if (DEC || t > 0) {
          for (int kb = 0; kb < KB_H; ++kb) {
            const uint64_t w_hi = smem_desc_k_sw128(sbase + LY::OFF_W_HI + kb * BLK_BYTES);
            const uint64_t w_lo = smem_desc_k_sw128(sbase + LY::OFF_W_LO + kb * BLK_BYTES);
            long long t0 = prof ? clock64() : 0;
            mbar_wait(full_bar(s), ph);
            if (prof) w_full_c += clock64() - t0;
            tc_fence_after();
            const uint64_t a_lo = smem_desc_k_sw128(sbase + LY::OFF_RING + s * BLK_BYTES);
            if (leader) {
#pragma unroll
              for (int ks = 0; ks < 4; ++ks)
                mma_f16_ss(d, a_lo + (uint64_t)(ks * 2), w_hi + (uint64_t)(ks * 2), idesc, ks == 0 ? acc : 1u);
              mma_commit(empty_bar(s));
            }
            __syncwarp();
            acc = 1u;
            if (++s == NSLOT) { s = 0; ph ^= 1u; }
            t0 = prof ? clock64() : 0;
            mbar_wait(full_bar(s), ph);
            if (prof) w_full_c += clock64() - t0;
            tc_fence_after();
            const uint64_t a_hi = smem_desc_k_sw128(sbase + LY::OFF_RING + s * BLK_BYTES);
            if (leader) {
#pragma unroll
              for (int ks = 0; ks < 4; ++ks) mma_f16_ss(d, a_hi + (uint64_t)(ks * 2), w_hi + (uint64_t)(ks * 2), idesc, 1u);
#pragma unroll
              for (int ks = 0; ks < 4; ++ks) mma_f16_ss(d, a_hi + (uint64_t)(ks * 2), w_lo + (uint64_t)(ks * 2), idesc, 1u);
              mma_commit(empty_bar(s));
            }
            __syncwarp();
            if (++s == NSLOT) { s = 0; ph ^= 1u; }
          }
        }
        if (!DEC || t > 0) {
          // x part last.  Decoder: it is the raw row of the previous pick, so the pointer phase of step t-1 overlaps the
          // exchange and the h-part MMAs of step t.  Encoder: x_rdy was signalled long ago by the x producer.
          if (DEC) mbar_wait_cluster(x_rdy(g), (uint32_t)(t - 1) & 1u);
          else if (t > 0) mbar_wait(x_rdy(g), (uint32_t)(t - 1) & 1u);
          tc_fence_after();
          if (leader) {
            mma_f16_ss(d, ax_lo, wx_hi, idesc, acc);
            mma_f16_ss(d, ax_hi, wx_hi, idesc, 1u);
            mma_f16_ss(d, ax_hi, wx_lo, idesc, 1u);
          }
          __syncwarp();
        }
        if (leader) mma_commit(tfull(g));
        __syncwarp();
      }
    }
    if (prof && leader) {
      p.prof[(size_t)blockIdx.x * 8 + 1] = (unsigned long long)(clock64() - t_begin);
      p.prof[(size_t)blockIdx.x * 8 + 2] = (unsigned long long)w_full_c;
    }
  } else if (warp == 3) {
    // ================= x producer (encoder): raw input row of step t+1 -> fp16 hi/lo x block =================
    if (!DEC) {
      for (int t = 0; t + 1 < p.steps; ++t) {
        for (int g = 0; g < G; ++g) {
          float xv[4][8];
          load_inputs(g, t + 1, xv);
          mbar_wait(tfull(g), (uint32_t)t & 1u);          // the MMAs of step t no longer read the x block
          write_x_rows(ax_hi_off(g), ax_lo_off(g), lane, xv);
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) mbar_arrive(x_rdy(g));
        }
      }
    }
  } else if (warp >= 4) {
    // ================= epilogue: thread = one instance row x 8 hidden units, cell state in registers ===========
    // All 16 warps serve every group of the cluster in turn (G = 2: group 0 then group 1 of the same step), so a group's
    // cell epilogue always has the whole SM's MUFU throughput and its publish overlaps the other group's MMAs.
    const int q = warp & 3;
    const int grp = (warp - 4) >> 2;                       // 32-column chunk = 8 hidden units
    const int r = q * 32 + lane;
    const int u0 = (int)rank * UNITS + grp * 8;            // first hidden unit of this thread
    const uint32_t kb_mine = rank >> 1;
    const float4* const bias4_0 = reinterpret_cast<const float4*>(sbias) + grp * 8;
    const float4* const bias4_1 = reinterpret_cast<const float4*>(sbias + TILE_N) + grp * 8;
    auto row_of = [&](int g) { return (group0 + g) * BM + r; };
    float* const h_out = p.h_out + roll * p.n * p.h_out_inst_ld;      // this rollout's enc_out / dec_h
    // split 8 fp32 values to fp16 hi/lo and store them to scratch parity (j & 1) of group g
    auto stage = [&](int g, const float* hv, int j) {
      uint32_t pk[8];
      split_f16x8(hv, pk, pk + 4);
      __half* dst = p.scratch + (size_t)(sgroup0 + g) * (2 * 2 * BM * kH) + (size_t)(j & 1) * (2 * BM * kH) + (size_t)r * kH + u0;
      stg128_u(dst, pk[0], pk[1], pk[2], pk[3]);                    // hi rows
      stg128_u(dst + BM * kH, pk[4], pk[5], pk[6], pk[7]);          // lo rows
    };
    // publish index j of group g to the 8 CTAs: the warp's stores happen-before the release below through __syncwarp; ONE
    // cumulative release.cluster arrive per destination CTA (8 lanes in parallel) instead of a GPU-scope fence in every lane
    auto publish = [&](int g, int j) {
      __syncwarp();
      if (lane < CL) {
        fence_proxy_async_all();
        mbar_arrive_release_cluster(mapa_rank(a_rdy(g, j & 1, (int)kb_mine), (uint32_t)lane));
      }
      __syncwarp();
    };
    float c[G][8];
    if (DEC) {
#pragma unroll
      for (int g = 0; g < G; ++g) {
        const int64_t m = row_of(g);
        const bool ok = m < p.n;
        if (ok) ldg256(p.c + m * kH + u0, c[g]);
        else {
#pragma unroll
          for (int u = 0; u < 8; ++u) c[g][u] = 0.f;
        }
        float h0v[8];
        if (ok) ldg256(p.h0 + m * p.h0_ld + u0, h0v);
        else {
#pragma unroll
          for (int u = 0; u < 8; ++u) h0v[u] = 0.f;
        }
        stage(g, h0v, 0);
        publish(g, 0);
      }
    } else {
#pragma unroll
      for (int g = 0; g < G; ++g)
#pragma unroll
        for (int u = 0; u < 8; ++u) c[g][u] = 0.f;
    }
    long long w_tfull = 0, d_cell = 0, d_pub = 0, d_out = 0;
    for (int t = 0; t < p.steps; ++t) {
      const float4* bias4 = t == 0 ? bias4_0 : bias4_1;
#pragma unroll
      for (int g = 0; g < G; ++g) {
        const int64_t m = row_of(g);
        const bool ok = m < p.n;
        float* const h_dst = h_out + (ok ? m : 0) * p.h_out_inst_ld + (int64_t)t * kH + u0;
        const long long t0 = prof ? clock64() : 0;
        mbar_wait(tfull(g), (uint32_t)t & 1u);
        const long long t1 = prof ? clock64() : 0;
        if (prof && g == 0) w_tfull += t1 - t0;
        tc_fence_after();
        float v[32];
        tmem_ld_32x32_issue(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(g * TILE_N + grp * 32), v);
        tmem_ld_wait(v);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(tempty(g));                         // accumulator is in registers
        float cn[8], hn[8];
        // training forward: v becomes the post-activation gates; they are stored AFTER the publish (off the step's critical path)
        if (p.save_gates) lstm_cell8(v, bias4, c[g], cn, hn, v);
        else lstm_cell8(v, bias4, c[g], cn, hn);
        auto save_step = [&]() {
          // the BPTT's saves (gnnpn_pn_train_backward_f32): 128 + 32 contiguous bytes per thread
          if (p.save_gates && ok) {
            float* gd = p.save_gates + ((int64_t)t * p.n + m) * kG + 4 * u0;
#pragma unroll
            for (int i = 0; i < 4; ++i) stg256(gd + 8 * i, v + 8 * i);
            stg256(p.save_c + ((int64_t)t * p.n + m) * kH + u0, cn);
          }
        };
#pragma unroll
        for (int u = 0; u < 8; ++u) c[g][u] = cn[u];
        const long long t3 = prof ? clock64() : 0;
        if (prof && g == 0) d_cell += t3 - t1;
        if (DEC) {
          // the query of this step's pointer phase: fp32 h'(t) to dec_h BEFORE the publish (read by other CTAs after it)
          if (ok) stg256(h_dst, hn);
          stage(g, hn, t + 1);
          publish(g, t + 1);
          save_step();
          if (prof) d_pub += clock64() - t3;
          // ---- pointer step k = t for instance row 16 * rank + (warp - 4) of the group; the pick's raw row becomes the
          // x block row of ALL 8 CTAs for step t+1
          const long long t4 = prof ? clock64() : 0;
          const int pj = t + 1;
#pragma unroll
          for (int kb = 0; kb < KB_H; ++kb) mbar_wait_cluster(a_rdy(g, pj & 1, kb), (uint32_t)(pj >> 1) & 1u);   // all of h'(t) is in dec_h
          const int prow = (int)rank * (BM / CL) + (warp - 4);
          const int64_t b = (group0 + g) * BM + prow;
          int fed = 0;
          if (b < p.n) {                                                        // warp-uniform
            float4 q0, q1;
            ld_row8(h_out + b * p.h_out_inst_ld + (int64_t)t * kH, lane, q0, q1);
            fed = pointer_step_warp(rollout_args(p.pa, roll, p.steps, p.sampled), t, b, q0, q1, lane);
          }
          if (t + 1 < p.steps) {
            if (lane < CL) {
              float xv[8];
#pragma unroll
              for (int f = 0; f < 8; ++f)
                xv[f] = (b < p.n && f < p.F) ? __ldg(p.inputs + (b * p.L + fed) * (int64_t)p.F + f) : 0.f;
              uint32_t hi[4], lo[4];
              split_f16x8(xv, hi, lo);
              const uint32_t o = (uint32_t)prow * XROW_BYTES;
              const uint32_t dhi = mapa_rank(ax_hi_off(g) + o, (uint32_t)lane);
              const uint32_t dlo = mapa_rank(ax_lo_off(g) + o, (uint32_t)lane);
              st_cluster_v4(dhi, hi[0], hi[1], hi[2], hi[3]);
              st_cluster_v4(dhi + 16, hi[0], hi[1], hi[2], hi[3]);
              st_cluster_v4(dlo, lo[0], lo[1], lo[2], lo[3]);
              st_cluster_v4(dlo + 16, lo[0], lo[1], lo[2], lo[3]);
              fence_proxy_async_all();
              mbar_arrive_release_cluster(mapa_rank(x_rdy(g), (uint32_t)lane));
            }
            __syncwarp();
          }
          if (prof) d_out += clock64() - t4;
        } else {
          if (t + 1 < p.steps) {
            stage(g, hn, t);
            publish(g, t);
          }
          if (prof && g == 0) d_pub += clock64() - t3;
          const long long t4 = prof ? clock64() : 0;
          if (ok) stg256(h_dst, hn);
          save_step();
          if (prof && g == 0) d_out += clock64() - t4;
        }
      }
    }
#pragma unroll
    for (int g = 0; g < G; ++g) {
      const int64_t m = row_of(g);
      if (m < p.n && p.c_out) stg256(p.c_out + m * kH + u0, c[g]);
    }
    if (prof && warp == 4 && lane == 0) {
      unsigned long long* o = p.prof + (size_t)blockIdx.x * 8;
      o[3] = (unsigned long long)w_tfull; o[5] = (unsigned long long)d_cell;
      o[6] = (unsigned long long)d_pub; o[7] = (unsigned long long)d_out;
    }
  }
  __syncwarp();
  tc_fence_before();
  cluster_sync_all();
  if (warp == 2) tmem_dealloc(tmem_base, LY::TMEM_COLS);
}

}  // namespace cs

size_t tc_colsplit_scratch_bytes(int64_t n) {
  const int64_t groups = ceil_div(ceil_div(n, cs::BM), 6) * 6;             // 1 / 2 / 3 groups per cluster: whole clusters either way
  return (size_t)groups * 2 * 2 * cs::BM * kH * sizeof(__half);
}

// how many 8-CTA clusters of this kernel the device can hold at once (GPC packing decides; measured, not assumed)
int tc_colsplit_max_active_clusters() {
  static const int v = [] {
    using namespace cs;
    constexpr auto kern = lstm_colsplit_kernel<false, 1>;
    cudaLaunchConfig_t cfg;
    cudaLaunchAttribute attr;
    if (cluster_config<kern>(&cfg, &attr, CL * 64, CL, THREADS, Layout<1>::SMEM_BYTES, nullptr)) return 0;
    int nc = 0;
    if (cudaOccupancyMaxActiveClusters(&nc, kern, &cfg) != cudaSuccess) { cudaGetLastError(); return 0; }
    return nc;
  }();
  return v;
}

namespace cs {

template <bool DEC, int G>
static int launch(const float* packed, Params p, cudaStream_t st) {
  const int64_t clusters = ceil_div(ceil_div(p.n, BM), G) * p.rollouts;
  CUtensorMap maps[5];
  int rc = make_weight_maps(maps, packed, TILE_N);
  // exchange scratch as one 2-D fp16 tensor [groups * 2 parities * (hi|lo) * 128 rows, kH]; box = one k-block
  if (rc || (rc = make_map_2d(&maps[4], p.scratch, clusters * G * 4 * BM, kH, kH, BM, true))) return rc;
  const unsigned grid = (unsigned)(clusters * CL);
  if ((rc = prof_alloc(grid, 8, st, &p.prof))) return rc;
  rc = launch_cluster<lstm_colsplit_kernel<DEC, G>>(grid, CL, THREADS, Layout<G>::SMEM_BYTES, st, maps[0], maps[1], maps[2],
                                                    maps[3], maps[4], p);
  if (p.prof) {
    double acc[8];
    prof_collect(p.prof, grid, 8, st, acc);
    const double d = (double)grid * p.steps;
    fprintf(stderr, "[colsplit prof %s G=%d steps=%d grid=%u max_active_clusters=%d] per-step cycles: mma total %.0f (wait A full %.0f) | "
            "tma wait a_rdy %.0f | epi (group 0) wait tmem_full %.0f, tmem ld + cell %.0f, publish %.0f, %s %.0f\n", DEC ? "dec" : "enc", G,
            p.steps, grid, tc_colsplit_max_active_clusters(), acc[1] / d, acc[2] / d, acc[0] / d, acc[3] / d, acc[5] / d, acc[6] / d,
            DEC ? "pointer phase" : "h store", acc[7] / d);
  }
  return rc;
}

}  // namespace cs

int tc_colsplit_encode(const SeqEncodeArgs& a, int groups, cudaStream_t st) {
  cs::Params p{};
  p.n = a.n; p.steps = a.L; p.F = a.F; p.L = a.L;
  p.inputs = a.inputs; p.x_inst_ld = (int64_t)a.L * a.F;
  p.bias0 = p.bias = a.packed + kOffBias;
  p.c_out = a.c_state;
  p.rollouts = 1;
  p.h_out = a.enc_out; p.h_out_inst_ld = (int64_t)a.L * kH;
  p.scratch = reinterpret_cast<__half*>(a.c_scratch);
  p.save_gates = a.save_gates; p.save_c = a.save_c;
  switch (groups) {
    case 3: return cs::launch<false, 3>(a.packed, p, st);
    case 2: return cs::launch<false, 2>(a.packed, p, st);
    default: return cs::launch<false, 1>(a.packed, p, st);
  }
}

int tc_colsplit_decode(const SeqDecodeArgs& a, int groups, cudaStream_t st) {
  cs::Params p{};
  p.n = a.n; p.steps = a.K; p.F = a.F; p.L = a.L;
  p.inputs = a.inputs; p.x_inst_ld = (int64_t)a.L * a.F;
  p.bias0 = a.packed + kOffStart; p.bias = a.packed + kOffBias;
  p.c = a.c_state; p.c_out = a.rollouts ? nullptr : a.c_state;
  p.rollouts = a.rollouts ? a.rollouts : 1;
  p.sampled = a.sampled;
  p.h0 = a.enc_out + (int64_t)(a.L - 1) * kH; p.h0_ld = (int64_t)a.L * kH;
  p.h_out = a.dec_h; p.h_out_inst_ld = (int64_t)a.K * kH;
  p.scratch = reinterpret_cast<__half*>(a.c_scratch);
  p.pa = pointer_step_args(a.enc_out, a.latent_win, a.alpha, a.use_tanh, a.C, a.n, a.L, a.N, a.idx_out, a.win_logits,
                           a.win_probs, a.forced_idx, a.sample_uniform);
  p.save_gates = a.save_gates; p.save_c = a.save_c;
  return groups == 2 ? cs::launch<true, 2>(a.packed, p, st) : cs::launch<true, 1>(a.packed, p, st);
}

}  // namespace gnnpn
