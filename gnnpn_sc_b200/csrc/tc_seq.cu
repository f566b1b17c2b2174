// Persistent tcgen05 LSTM scan: one launch = one whole recurrence (encoder: L steps; decoder: K steps with
// the pointer step fused in between).  Reference semantics: nn.LSTM cell, gate order i,f,g,o
// (modelPN.py:157-158,191,205) and the decode loop modelPN.py:204-239.
//
// A CTA owns 128 composition instances for the whole scan, so the step-to-step dependency is CTA-local:
//   * A operand  [h | x]  as fp16 hi/lo pairs (error-compensated 3xFP16, fp32 accumulate:
//     a.w ~= a_lo.w_hi + a_hi.w_hi + a_hi.w_lo).  The h part is DOUBLE-BUFFERED: step t reads buffer t&1 and its
//     epilogue writes h'(t) straight into buffer (t+1)&1 -- h never goes through global memory between steps, and
//     nothing is staged or copied at the step boundary.  h_hi sits in TENSOR MEMORY (columns [256,384) and
//     [384,512), lane = instance, two halfs per column; the a_hi MMAs, 8 of every 12, read A from there), h_lo in
//     shared memory (two 64 KB blocks in the 128B-swizzled K-major UMMA layout).  The x block is single-buffered;
//   * B operand (the 4H x (H+F) folded weights, fp16 hi/lo, 1.1 MB, L2-resident) is streamed by TMA through a
//     ring of 8 slots; a slot holds one (N tile, k block, hi|lo) box, each CTA of the pair 8 KB = half its gate columns;
//   * accumulators: two 128-column TMEM buffers (N tile = 128 gate columns = 32 hidden units), so the
//     epilogue of tile j overlaps the MMAs of tile j+1;
//   * step t+1 starts one k-block at a time: k-block kb of h'(t) is complete once tiles 2kb and 2kb+1 of both CTAs
//     have been written, and tile 0 of step t+1 issues each k-block's 12 MMAs behind its own barrier, so k-blocks
//     0..2 run under the epilogue of tile 7.  Writing buffer (t+1)&1 needs no barrier of its own: the epilogue of
//     tile j of step t waits for that tile's commit, which retires after every MMA of step t-1, the buffer's last
//     readers.
// Warp roles: 0 = TMA producer, 1 = MMA issuer, 2 = TMEM allocator, 3 = x producer (encoder inputs),
// 4..19 = epilogue (TMEM lane quarter = warp & 3, column group = (warp - 4) / 4).
//
// Encodings layout (template parameter NR):
//   NR == 0  row-major enc_out [n, L, H] (GNNPN_ENC_ROWMAJOR).  Encoder: h' tiles leave by TMA store.  Decoder: a
//            separate pointer phase after each step's cell epilogue (each epilogue warp owns 8 instances, window rows
//            streamed per instance, pointer.cuh::pointer_steps_batched) -- the step is MMA phase + pointer phase.
//   NR >= 1  blocked encodings (GNNPN_ENC_BLOCKED128): per block of 128 instances
//            [L][8 tiles][4 groups][128 instances][8 floats], unit = 32*tile + 8*group + i -- exactly the
//            (thread = instance, 8 units per tile) ownership of the epilogue.  The encoder writes it with coalesced
//            256-bit stores.  In the decoder (NR = row capacity of the window, N <= NR) the pointer dot products are
//            FUSED INTO THE CELL EPILOGUE: when thread (instance r, group g) has produced the 8 h' units of tile nt
//            it multiplies them into the matching 8 floats of each of the N window rows of ITS instance (a warp's
//            load is 1 KB contiguous; the otherwise idle warp 3 bulk-prefetches every 16 KB (row, tile) slice into L2
//            two tiles ahead), in pointer.cuh's canonical order.  The window rows stream from HBM UNDER the step's MMAs; after the last tile the four group
//            partials are combined through shared memory and one thread per instance finishes the step (C*tanh,
//            latent, softmax, first-max pick / draw, next input row) while the tensor cores already run the h parts
//            of the next step's first two tiles.  No separate pointer phase remains.
// Cross-CTA mbarrier arrives use .release.cta semantics on purpose (see mbar_arrive_cluster).
#include <stdio.h>
#include <stdlib.h>
#include <algorithm>
#include <cuda_fp16.h>
#include <type_traits>
#include "tc_common.cuh"
#include "common.cuh"
#include "internal.cuh"
#include "lstm_step.cuh"
#include "tc_lstm.cuh"
#include "tc_seq.cuh"
#include "pointer.cuh"
#include "tc_seq_dev.cuh"
#include "options.cuh"

namespace gnnpn {
namespace seq {

using namespace tc;

constexpr int TILE_N = 128;                // gate columns per accumulator tile
constexpr int N_TILES = kG / TILE_N;       // 8
constexpr int RING = 8;                    // weight ring slots
constexpr int SLOT_ROWS = TILE_N / 2;      // each CTA of the pair loads half of a tile's gate columns
constexpr int SLOT_BYTES = BLK_BYTES / 2;  // [64 gate columns x 64 halfs]
constexpr int RING_BYTES = RING * SLOT_BYTES;
constexpr int TMEM_COLS = 512;             // [0,256): 2 accumulator buffers; [256,512): 2 h_hi buffers
constexpr int AHI_COL0 = 2 * TILE_N;
constexpr int AHI_COLS = kH / 2;           // 128: two halfs per 32-bit column

constexpr uint32_t A_LO_BYTES = KB_H * BLK_BYTES;                // one h_lo buffer, [128 rows x kH halfs]
constexpr uint32_t OFF_A_LO = 0;                                 // two h_lo buffers
constexpr uint32_t OFF_AX_HI = OFF_A_LO + 2 * A_LO_BYTES;
constexpr uint32_t OFF_AX_LO = OFF_AX_HI + BM * XROW_BYTES;
constexpr uint32_t OFF_RING = OFF_AX_LO + BM * XROW_BYTES;
constexpr uint32_t OFF_HBUF = OFF_RING + RING_BYTES;      // [128 rows x 32 fp32] h' tile for the TMA store
constexpr uint32_t OFF_BIAS = OFF_HBUF + BLK_BYTES;              // two transformed bias sets
constexpr uint32_t OFF_BAR = OFF_BIAS + 2 * kG * 4;
constexpr uint32_t SMEM_USED = OFF_BAR + 256;
constexpr int SMEM_BYTES = SMEM_USED + 1024;                     // + alignment slack
static_assert(SMEM_BYTES <= 232448, "exceeds the 227 KB per-CTA shared memory limit");


struct SeqParams {
  int64_t n;
  int steps;
  int L, F;
  const float* inputs; int64_t x_inst_ld;
  const float* bias0;      // [kG] gate-interleaved bias of step 0 (decoder: start-token bias)
  const float* bias;       // [kG] bias of steps >= 1
  const float* c;          // [n, kH] initial cell state (unless c_zero_init)
  float* c_out;            // [n, kH] final cell state, or nullptr (rollout launches: c is shared by the rollouts)
  int c_zero_init;
  // Rollout launches (decoder): clusters are ordered (instance pair block, rollout) with the rollouts of one block adjacent,
  // so they run in the same wave and their window-row reads meet in L2.  Rollout r writes its own dec_h slice
  // (h_out + r * n * h_out_inst_ld) and the pointer outputs of pointer.cuh::rollout_args.  1 for every other launch.
  int rollouts;
  const float* sampled;    // [rollouts-1, K, n] uniforms of rollouts 1.. (rollout_args)
  const float* h0; int64_t h0_ld;          // initial hidden rows or nullptr (zeros)
  float* h_out; int64_t h_out_inst_ld;     // step t of instance m at h_out + m*ld + t*kH
  PointerStepArgs pa;      // decoder only
  unsigned long long* prof; // debug (GNNPN_SEQ_PROF): per-CTA wait-cycle counters, 16 per CTA, or nullptr
  float* c_scr;            // blocked cell-state scratch, 128*kH floats per CTA (coalesced 128-bit accesses)
};

// mbar_wait that adds the cycles spent waiting to *acc (debug counters; acc lives in a register)
template <bool CLUSTER = false>
__device__ __forceinline__ void mbar_wait_t(uint32_t bar, uint32_t parity, bool prof, long long& acc) {
  const long long t0 = prof ? clock64() : 0;
  if (CLUSTER) mbar_wait_cluster(bar, parity); else mbar_wait(bar, parity);
  if (prof) acc += clock64() - t0;
}


// x block of the next decoder step: row rr, feature f -> halfs f and 8+f of the hi and lo 32-byte rows
__device__ __forceinline__ void store_ax(uint8_t* sgen, int rr, int f, float xv) {
  const __half hi = __float2half_rn(xv);
  const __half lo = __float2half_rn(xv - __half2float(hi));
  __half* ax_hi = reinterpret_cast<__half*>(sgen + OFF_AX_HI + rr * XROW_BYTES);
  __half* ax_lo = reinterpret_cast<__half*>(sgen + OFF_AX_LO + rr * XROW_BYTES);
  ax_hi[f] = hi; ax_hi[8 + f] = hi;
  ax_lo[f] = lo; ax_lo[8 + f] = lo;
}

// Pointer phase of decode step t for the 8 instances of one epilogue warp (rows rr0..rr0+7 of the CTA); see
// pointer_steps_batched in pointer.cuh.
__device__ __forceinline__ void pointer_phase(const SeqParams& p, const PointerStepArgs& pa, const float* h_out, int t,
                                              int rr0, int64_t m0, int lane, uint8_t* sgen) {
  const int64_t b0 = m0 + rr0;
  const int64_t left = p.n - b0;
  const int count = left <= 0 ? 0 : (left < BM / EPI_WARPS ? (int)left : BM / EPI_WARPS);
  const bool feed_next = t + 1 < p.steps;
  const float* q_base = h_out + (int64_t)t * kH;
  // the raw rows of the picks (next decoder inputs) of a whole pass are fetched together and written
  // to the x block after the last pass, so their latency is paid once
  float pend_x[kWarpInstances];
#pragma unroll
  for (int r = 0; r < kWarpInstances; ++r) pend_x[r] = 0.f;
  auto run = [&](auto seg_tag, auto ch_tag) {
    constexpr int SEG = decltype(seg_tag)::value, CH = decltype(ch_tag)::value;
    constexpr int IPP = 32 / SEG;
    auto feed = [&](int si, int64_t b, int fed, int j) {
      if (!feed_next) return;
      const float xv = (si < count && j < p.F) ? __ldg(p.inputs + (b * p.L + fed) * (int64_t)p.F + j) : 0.f;
#pragma unroll
      for (int r = 0; r < kWarpInstances / IPP; ++r)
        if (si / IPP == r) pend_x[r] = xv;
    };
    pointer_steps_batched<SEG, CH>(pa, t, b0, count, q_base, p.h_out_inst_ld, lane, feed
                                   );
    if (feed_next) {
      const int seg_i = lane / SEG, seg_j = lane % SEG;
#pragma unroll
      for (int r = 0; r < kWarpInstances / IPP; ++r) {
        const int si = r * IPP + seg_i;
        if (si < count && seg_j < 8) store_ax(sgen, rr0 + si, seg_j, pend_x[r]);
      }
    }
  };
  using std::integral_constant;
  const bool five = pa.N % 5 == 0;
  if (pa.N <= 8)       { if (five) run(integral_constant<int, 8>{}, integral_constant<int, 5>{});
                         else      run(integral_constant<int, 8>{}, integral_constant<int, 4>{}); }
  else if (pa.N <= 16) { if (five) run(integral_constant<int, 16>{}, integral_constant<int, 5>{});
                         else      run(integral_constant<int, 16>{}, integral_constant<int, 4>{}); }
  else                 run(integral_constant<int, 32>{}, integral_constant<int, 4>{});
}


// ---- blocked encodings (GNNPN_ENC_BLOCKED128) ------------------------------------------------------------------
// float offset of (block of 128 instances, position l, tile nt, group g); + row * 8 inside (8 consecutive units)
constexpr int64_t ENC_BLK_ROW = 8 * 4 * BM * 8;                  // floats between consecutive positions l (= BM * kH)
constexpr int ENC_BLK_TILE = 4 * BM * 8;                         // floats of one (position, tile): 16 KB, contiguous
__host__ __device__ inline int64_t enc_blk_off(int64_t block, int L, int64_t l, int nt, int g) {
  return (block * L + l) * ENC_BLK_ROW + (int64_t)(nt * 4 + g) * (BM * 8);
}
__device__ __forceinline__ void bulk_prefetch_l2(const void* p, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}
// L2 residency control.  The fused decoder streams 97 MB of window rows per step through L2 next to a 19 MB cell-state
// scratch that is re-read every step: the rows are loaded evict-first (read once), the scratch evict-last -- without
// the hints the scratch is evicted and costs 1.8 GB of extra DRAM traffic per launch (ncu, profiles/).
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ void ldg256_stream(const float* p, float4& a, float4& b, uint64_t pol) {
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8], %9;"
               : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w), "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w) : "l"(p), "l"(pol));
}
__device__ __forceinline__ float4 ldg128_hint(const float* p, uint64_t pol) {
  float4 r;
  asm volatile("ld.global.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p), "l"(pol));
  return r;
}
__device__ __forceinline__ void stg128_hint(float* p, float a, float b, float c, float d, uint64_t pol) {
  asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1,%2,%3,%4}, %5;" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d), "l"(pol)
               : "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int threads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory");
}


// ------------------------------------------------------------------------------------------------
// CTA pair (cluster of 2 = one TPC), cta_group::2 MMAs (M=256: 128 instances per CTA, N=128): each CTA streams only
// HALF of every weight tile (64 of the 128 gate columns) and the tensor cores read the other half from the peer --
// half the L2->SM weight traffic and B-operand shared-memory reads a lone CTA would need, and twice the ring depth.
// CTA rank 0 issues the MMAs for the pair; both CTAs run producer / epilogue.
template <bool DEC, int NR>
__global__ void __launch_bounds__(THREADS, 1)
lstm_seq_kernel(const __grid_constant__ CUtensorMap map_wh_hi, const __grid_constant__ CUtensorMap map_wh_lo,
                const __grid_constant__ CUtensorMap map_wx_hi, const __grid_constant__ CUtensorMap map_wx_lo,
                const __grid_constant__ CUtensorMap map_h, const __grid_constant__ SeqParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* sgen = smem_raw + (sbase - smem_u32(smem_raw));          // generic pointer to the aligned base
  const uint32_t bar0 = sbase + OFF_BAR;
  auto full_bar = [&](int s) { return bar0 + 8u * s; };
  auto empty_bar = [&](int s) { return bar0 + 8u * (RING + s); };
  auto tfull_bar = [&](int b) { return bar0 + 8u * (2 * RING + b); };
  auto tempty_bar = [&](int b) { return bar0 + 8u * (2 * RING + 2 + b); };
  const uint32_t a_ready_bar = bar0 + 8u * (2 * RING + 4);   // x(t+1) is in the x block
  const uint32_t mma_done_bar = bar0 + 8u * (2 * RING + 5);
  const uint32_t hfull_bar = bar0 + 8u * (2 * RING + 6);
  const uint32_t hempty_bar = bar0 + 8u * (2 * RING + 7);
  const uint32_t tmem_slot = bar0 + 8u * (2 * RING + 8);
  auto h_ready_bar = [&](int kb) { return bar0 + 8u * (2 * RING + 9 + kb); };   // k-block kb of h'(t) is in A
  const uint32_t rank = cluster_ctarank();
  // barriers the MMA issuer (rank 0) waits on collect arrivals from both CTAs of the pair
  const uint32_t a_ready_remote = mapa_rank(a_ready_bar, 0);
  float* sbias = reinterpret_cast<float*>(sgen + OFF_BIAS);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int cluster = (int)(blockIdx.x >> 1);
  const int roll = cluster % p.rollouts;
  const int blk = cluster / p.rollouts * 2 + (int)(blockIdx.x & 1);   // this CTA's block of 128 instances
  const int64_t m0 = (int64_t)blk * BM;
  constexpr bool BLK = NR > 0;                         // blocked encodings (see the file header)
  constexpr bool FUSED = DEC && BLK;                   // pointer dots fused into the cell epilogue
  const bool cta_ok = m0 < p.n;                        // a pair's second CTA may be all padding

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_wh_hi); tma_prefetch_desc(&map_wh_lo);
    tma_prefetch_desc(&map_wx_hi); tma_prefetch_desc(&map_wx_lo);
    if (!DEC && !BLK) tma_prefetch_desc(&map_h);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < RING; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(tfull_bar(b), 1); mbar_init(tempty_bar(b), 2 * EPI_WARPS); }
    mbar_init(a_ready_bar, DEC ? 2 * EPI_WARPS : 2);        // decoder: the epilogue writes x; encoder: warp 3
    for (int kb = 0; kb < KB_H; ++kb) mbar_init(h_ready_bar(kb), 2 * EPI_WARPS);
    mbar_init(mma_done_bar, 1);
    mbar_init(hfull_bar, EPI_WARPS);
    mbar_init(hempty_bar, 1);
    fence_mbar_init();
  }
  if (warp == 2) tmem_alloc_cg2(tmem_slot, TMEM_COLS);

  // ---- transformed biases: (i,f,o) * -log2e, g * -2log2e; x block of step 0 (h(-1) is written by the epilogue warps)
  for (int i = threadIdx.x; i < 2 * kG; i += THREADS) {
    const int col = i & (kG - 1);
    const float b = __ldg((i < kG ? p.bias0 : p.bias) + col);
    sbias[i] = b * ((col & 3) == 2 ? -2.0f * kLog2e : -kLog2e);
  }

  // load_x_rows is called through this lambda: calling it directly at the two sites changes the register allocation
  // of the encoder kernels' TMA producer
  auto load_inputs = [&](int t, float (*xv)[8]) { load_x_rows(p, m0, t, lane, xv); };
  if (warp == 3) {
    float xv[4][8];
    if (DEC) {
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int f = 0; f < 8; ++f) xv[i][f] = 0.f;
    } else {
      load_inputs(0, xv);
    }
    write_x_rows(sbase + OFF_AX_HI, sbase + OFF_AX_LO, lane, xv);
  }
  fence_proxy_async_smem();
  tc_fence_before();
  cluster_sync_all();                                       // barrier inits / TMEM / A operand visible pair-wide
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

  if (warp < 4) {
  if constexpr (FUSED) asm volatile("setmaxnreg.dec.sync.aligned.u32 32;");   // role warpgroup hands registers to the epilogue
  if (warp == 0) {
    // ================= TMA producer: weights, the same 72 boxes every step (each CTA of a pair loads its
    // half of the gate columns of every box and signals the leader's barrier) =================
    if (lane == 0) {
      int s = 0; uint32_t ph = 0;
      const int row_off = (int)rank * SLOT_ROWS;
      auto load_h = [&](int it) {                      // the 8 h-part boxes of tile `it` (hi, lo per k-block)
        const int nt = it;
        for (int kb = 0; kb < KB_H; ++kb) {
#pragma unroll
          for (int part = 0; part < 2; ++part) {
            mbar_wait(empty_bar(s), ph ^ 1u);
            const uint32_t dst = sbase + OFF_RING + s * SLOT_BYTES;
            if (rank == 0) mbar_arrive_expect_tx(full_bar(s), 2 * SLOT_BYTES);
            tma_load_2d_cg2(dst, part ? &map_wh_lo : &map_wh_hi, mapa_rank(full_bar(s), 0), kb * 64,
                            nt * TILE_N + row_off);
            if (++s == RING) { s = 0; ph ^= 1u; }
          }
        }
      };
      auto load_x = [&](int it) {                      // the x-part box (hi | lo) of tile `it`
        const int nt = it;
        mbar_wait(empty_bar(s), ph ^ 1u);
        const uint32_t dst = sbase + OFF_RING + s * SLOT_BYTES;
        if (rank == 0) mbar_arrive_expect_tx(full_bar(s), 2 * 2 * SLOT_ROWS * XROW_BYTES);
        const uint32_t fb = mapa_rank(full_bar(s), 0);
        tma_load_2d_cg2(dst, &map_wx_hi, fb, kH, nt * TILE_N + row_off);
        tma_load_2d_cg2(dst + SLOT_ROWS * XROW_BYTES, &map_wx_lo, fb, kH, nt * TILE_N + row_off);
        if (++s == RING) { s = 0; ph ^= 1u; }
      };
      for (int t = 0; t < p.steps; ++t) {
        // decoder: the h parts of tiles 0 and 1 come first (issued while the pointer phase still runs), see the MMA warp
        const int first = DEC ? 2 : 0;
        if (DEC) { load_h(0); load_h(1); load_x(0); load_x(1); }
        for (int it = first; it < N_TILES; ++it) { load_h(it); load_x(it); }
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer: the whole warp walks the pipeline (uniform control flow keeps the descriptors
    // in uniform registers); one elected lane issues tcgen05.mma / tcgen05.commit =================
    if (rank == 0) {
      const uint32_t leader = elect_one();
      const uint32_t idesc = idesc_f16(2 * BM, TILE_N);
      auto mma = [&](uint32_t d, uint64_t a, uint64_t b, uint32_t acc) { mma_f16_ss_cg2(d, a, b, idesc, acc); };
      auto mma_ts = [&](uint32_t d, uint32_t a, uint64_t b) { mma_f16_ts_cg2(d, a, b, idesc, 1u); };
      const uint64_t ax_hi = smem_desc_k_sw32(sbase + OFF_AX_HI), ax_lo = smem_desc_k_sw32(sbase + OFF_AX_LO);
      int s = 0; uint32_t ph = 0;
      uint32_t uses = 0;                                   // per-buffer use count = uses >> 1 (tiles alternate)
      const bool prof = p.prof != nullptr;
      long long w_aready = 0, w_tempty = 0, w_full = 0;
      const long long t_begin = clock64();
      // h part of one tile of step t: 8 ring slots, 48 MMAs.  The first tile of a step waits for each k-block of h(t-1).
      auto mma_h = [&](uint32_t d, int t, bool first) {
        const uint32_t hb = (uint32_t)t & 1u;
        for (int kb = 0; kb < KB_H; ++kb) {
          if (first) {
            mbar_wait_t<true>(h_ready_bar(kb), hb, prof, w_aready);
            tc_fence_after();
          }
          const uint32_t a_hi = tmem_base + (uint32_t)(AHI_COL0 + hb * AHI_COLS + kb * 32);   // 64 halfs = 32 columns
          const uint64_t a_lo = smem_desc_k_sw128(sbase + OFF_A_LO + hb * A_LO_BYTES + kb * BLK_BYTES);
          mbar_wait_t(full_bar(s), ph, prof, w_full);
          tc_fence_after();
          const uint64_t b_hi = smem_desc_k_sw128(sbase + OFF_RING + s * SLOT_BYTES);
          if (leader) {
#pragma unroll
            for (int ks = 0; ks < 4; ++ks)
              mma(d, a_lo + (uint64_t)(ks * 2), b_hi + (uint64_t)(ks * 2), (uint32_t)((kb | ks) != 0));
#pragma unroll
            for (int ks = 0; ks < 4; ++ks)
              mma_ts(d, a_hi + (uint32_t)(ks * 8), b_hi + (uint64_t)(ks * 2));
            mma_commit_cg2(empty_bar(s));
          }
          __syncwarp();
          if (++s == RING) { s = 0; ph ^= 1u; }
          mbar_wait_t(full_bar(s), ph, prof, w_full);
          tc_fence_after();
          const uint64_t b_lo = smem_desc_k_sw128(sbase + OFF_RING + s * SLOT_BYTES);
          if (leader) {
#pragma unroll
            for (int ks = 0; ks < 4; ++ks)
              mma_ts(d, a_hi + (uint32_t)(ks * 8), b_lo + (uint64_t)(ks * 2));
            mma_commit_cg2(empty_bar(s));
          }
          __syncwarp();
          if (++s == RING) { s = 0; ph ^= 1u; }
        }
      };
      auto mma_x = [&](uint32_t d, int buf, bool last) {  // x part of one tile, then hand the accumulator to the epilogue
        mbar_wait_t(full_bar(s), ph, prof, w_full);
        tc_fence_after();
        const uint64_t bx_hi = smem_desc_k_sw32(sbase + OFF_RING + s * SLOT_BYTES);
        const uint64_t bx_lo = smem_desc_k_sw32(sbase + OFF_RING + s * SLOT_BYTES + SLOT_ROWS * XROW_BYTES);
        if (leader) {
          mma(d, ax_lo, bx_hi, 1u);
          mma(d, ax_hi, bx_hi, 1u);
          mma(d, ax_hi, bx_lo, 1u);
          mma_commit_cg2(empty_bar(s));
          mma_commit_cg2(tfull_bar(buf));
          if (last) mma_commit_cg2(mma_done_bar);
        }
        __syncwarp();
        if (++s == RING) { s = 0; ph ^= 1u; }
      };
      for (int t = 0; t < p.steps; ++t) {
        int nt0 = 0;
        if (DEC) {
          // Only the K = 16 x part of a step depends on the pick.  TMEM has two accumulator buffers, so the h parts of
          // tiles 0 and 1 (96 of the step's 408 MMAs) are issued as soon as h'(t-1) is in A, i.e. while the
          // pointer phase of step t-1 still runs; their x parts follow once the picked rows are in the x block.
          for (int b = 0; b < 2; ++b) {
            mbar_wait_t<true>(tempty_bar(b), (((uses + b) >> 1) & 1u) ^ 1u, prof, w_tempty);
            tc_fence_after();
            mma_h(tmem_base + (uint32_t)(b * TILE_N), t, b == 0);
          }
          if (t > 0) {
            mbar_wait_t<true>(a_ready_bar, (uint32_t)(t - 1) & 1u, prof, w_aready);   // x(t) is in the x block
            tc_fence_after();
          }
          for (int b = 0; b < 2; ++b) mma_x(tmem_base + (uint32_t)(b * TILE_N), b, false);
          uses += 2;
          nt0 = 2;
        }
        for (int nt = nt0; nt < N_TILES; ++nt, ++uses) {
          const int buf = nt & 1;
          mbar_wait_t<true>(tempty_bar(buf), ((uses >> 1) & 1u) ^ 1u, prof, w_tempty);
          tc_fence_after();
          const uint32_t d = tmem_base + (uint32_t)(buf * TILE_N);
          mma_h(d, t, nt == 0);
          if (!DEC && nt == 0 && t > 0) {
            mbar_wait_t<true>(a_ready_bar, (uint32_t)(t - 1) & 1u, prof, w_aready);  // x(t) is in the x block
            tc_fence_after();
          }
          mma_x(d, buf, nt == N_TILES - 1);
        }
      }
      if (prof && leader) {
        unsigned long long* o = p.prof + (size_t)blockIdx.x * 16;
        o[0] = (unsigned long long)(clock64() - t_begin); o[1] = w_aready; o[2] = w_tempty; o[3] = w_full;
      }
    }
  } else if (warp == 2) {
    // ================= h' store issuer (encoder): one TMA store per tile, [128 instances x 32 units] -> enc_out ====
    if (!DEC && !BLK && lane == 0) {
      uint32_t g = 0;
      for (int t = 0; t < p.steps; ++t) {
        for (int it = 0; it < N_TILES; ++it, ++g) {
          const int nt = it;
          mbar_wait(hfull_bar, g & 1u);
          tma_store_3d(&map_h, sbase + OFF_HBUF, nt * 32, t, (int)m0);
          bulk_commit();
          bulk_wait_read0();                             // the tile has been read out of shared memory
          mbar_arrive(hempty_bar);
        }
      }
      bulk_wait0();
    }
  } else if (warp == 3) {
    if (FUSED) {
      // ================= L2 prefetcher (fused decoder): the 16 KB slice (window row j, tile nt) of this CTA's block is
      // contiguous; it is requested two tiles before the epilogue multiplies it, paced by the MMA's tile barriers
      if (lane == 0 && cta_ok) {
        // tiles ahead.  N = 5 (QWS): 1 tile ahead 40.1k cycles / step, 2: 39.7k, 3: 51.8k, none: 46.0k (profiles/).  Wider
        // windows keep the prefetched-but-unused footprint (dist x N x 16 KB per CTA) at the same ~24 MB: at N = 10 two tiles
        // ahead made the kernel re-read 35 % of the rows from DRAM (ncu: 13.1 GB for 9.7 GB algorithmic)
        const int dist = p.pa.N > 5 ? 1 : 2;
        const float* const rows = p.pa.enc_out + enc_blk_off(blk, p.L, 0, 0, 0);
        const int N = p.pa.N;
        for (int a = 0; a < dist; ++a)
          for (int j = 0; j < N; ++j) bulk_prefetch_l2(rows + (int64_t)j * ENC_BLK_ROW + a * ENC_BLK_TILE, ENC_BLK_TILE * 4);
        uint32_t uses = 0;
        for (int t = 0; t < p.steps; ++t) {
          for (int it = 0; it < N_TILES; ++it, ++uses) {
            mbar_wait(tfull_bar(it & 1), (uses >> 1) & 1u);      // tile `it` of step t is multiplied: the epilogue starts on it
            const int nt2 = (it + dist) & (N_TILES - 1);
            const int t2 = t + (it + dist >= N_TILES ? 1 : 0);
            if (t2 < p.steps)
              for (int j = 0; j < N; ++j)
                bulk_prefetch_l2(rows + ((int64_t)t2 * N + j) * ENC_BLK_ROW + nt2 * ENC_BLK_TILE, ENC_BLK_TILE * 4);
          }
        }
      }
    }
    // ================= x producer (encoder): raw input row of step t+1 -> fp16 hi/lo x block =================
    if (!DEC) {
      for (int t = 0; t + 1 < p.steps; ++t) {
        float xv[4][8];
        load_inputs(t + 1, xv);
        mbar_wait(mma_done_bar, (uint32_t)t & 1u);        // the MMAs of step t no longer read the x block
        write_x_rows(sbase + OFF_AX_HI, sbase + OFF_AX_LO, lane, xv);
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(a_ready_remote);
      }
    }
  }
  } else {
    // ================= epilogue: thread = one instance (TMEM lane), 32 gate columns = 8 hidden units per tile ====
    // (fused decoder: a chunk of window-row slices, 40 registers, is in flight next to the cell arithmetic)
    if constexpr (FUSED) asm volatile("setmaxnreg.inc.sync.aligned.u32 112;");
    const int q = warp & 3;
    const int grp = (warp - 4) >> 2;
    const int r = q * 32 + lane;                       // row inside the CTA
    const int64_t m = m0 + r;
    const bool ok = m < p.n;
    const uint32_t t_lane = tmem_base + ((uint32_t)(q * 32) << 16);
    const float* const c_row = p.c + (ok ? m : 0) * kH;
    float* const h_out = p.h_out ? p.h_out + roll * p.n * p.h_out_inst_ld : nullptr;     // this rollout's dec_h
    float* const h_row = h_out + (ok ? m : 0) * p.h_out_inst_ld;
    // blocked scratch: float4 index (((cta*8 + nt)*4 + grp)*2 + half)*128 + row  -> a warp touches 512 contiguous bytes
    float* const c_blk = p.c_scr + ((int64_t)blockIdx.x * (BM * kH) + (int64_t)grp * (2 * BM * 4) + r * 4);
    // blocked encodings of this thread (8 consecutive units): + position * ENC_BLK_ROW + nt * ENC_BLK_TILE
    const int64_t blk_thread = enc_blk_off(blk, p.L, 0, 0, grp) + r * 8;
    float* const e_out = BLK && !DEC ? p.h_out + blk_thread : nullptr;
    const float* const e_in = FUSED ? p.pa.enc_out + blk_thread : nullptr;
    const int N = DEC ? p.pa.N : 0;
    constexpr int NRA = NR > 0 ? NR : 1;
    constexpr int CHK = (NR % 5 == 0) ? 5 : 4;          // window rows in flight per thread (8 registers each)
    float acc[NRA];                                    // FUSED: running p[g] of the canonical dot, per window row
#pragma unroll
    for (int j = 0; j < NRA; ++j) acc[j] = 0.f;
    // FUSED: the first CHK window-row slices of the NEXT tile are requested as soon as the current tile's dots have
    // consumed the registers, i.e. a whole tile (barrier wait + cell arithmetic) before they are used
    float4 ea[CHK], eb[CHK];
    const uint64_t pol_stream = l2_policy_evict_first(), pol_keep = l2_policy_evict_last();
    const bool keep_c = FUSED;
    const bool do_dot = FUSED && cta_ok;
    auto request_rows = [&](int t_, int nt_) {
#pragma unroll
      for (int u = 0; u < CHK; ++u)
        if (u < N) ldg256_stream(e_in + ((int64_t)t_ * N + u) * ENC_BLK_ROW + nt_ * ENC_BLK_TILE, ea[u], eb[u], pol_stream);
    };
    // this thread's 8 units of tile nt -> h buffer nb: hi into TMEM (4 columns), lo into shared memory.  After the odd
    // tile of k-block kb the warp has written its whole part of the k-block, and says so to the MMA issuer.
    auto publish_h = [&](uint32_t nb, int nt, const float* hv) {
      uint32_t hi[4], lo[4];
      split_f16x8(hv, hi, lo);
      tmem_st_32x32_x4(t_lane + (uint32_t)(AHI_COL0 + nb * AHI_COLS + nt * 16 + grp * 4), hi);
      st_shared_v4(sbase + OFF_A_LO + nb * A_LO_BYTES + (uint32_t)(nt >> 1) * BLK_BYTES + sw128_off(r, (nt & 1) * 4 + grp),
                   lo[0], lo[1], lo[2], lo[3]);
      if (nt & 1) {
        tmem_st_wait();
        fence_proxy_async_smem();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(mapa_rank(h_ready_bar(nt >> 1), 0));
      }
    };
    // h(-1) into buffer 0: zeros for the encoder; the decoder starts from the encoder's last hidden state
    // (modelPN.py:191,205), with blocked encodings position L-1 of the block
    for (int nt = 0; nt < N_TILES; ++nt) {
      float hv[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      if (FUSED && cta_ok) ldg256(e_in + (int64_t)(p.L - 1) * ENC_BLK_ROW + nt * ENC_BLK_TILE, hv);
      else if (!FUSED && p.h0 && ok) ldg256(p.h0 + m * p.h0_ld + nt * 32 + grp * 8, hv);
      publish_h(0u, nt, hv);
    }
    if (do_dot) request_rows(0, 0);
    uint32_t uses = 0;
    const bool prof = p.prof != nullptr;
    long long w_tfull = 0, w_hempty = 0, w_ptr = 0;
    const long long t_begin = clock64();
    for (int t = 0; t < p.steps; ++t) {
      const float4* bias4 = reinterpret_cast<const float4*>(sbias + (t == 0 ? 0 : kG));
      const bool last = t == p.steps - 1;
      const float* const e_win = FUSED ? e_in + (int64_t)t * N * ENC_BLK_ROW : nullptr;     // window rows of step t
      for (int it = 0; it < N_TILES; ++it, ++uses) {
        const int buf = it & 1;
        const int nt = it;                             // which 128 gate columns this tile holds
        const int u0 = nt * 32 + grp * 8;              // first hidden unit of this thread's chunk
        float* const c_t = c_blk + nt * (4 * 2 * BM * 4);
        float c_old[8];
        if (t > 0) {
          const float4 a = keep_c ? ldg128_hint(c_t, pol_keep) : ldg128(c_t);
          const float4 b = keep_c ? ldg128_hint(c_t + BM * 4, pol_keep) : ldg128(c_t + BM * 4);
          c_old[0] = a.x; c_old[1] = a.y; c_old[2] = a.z; c_old[3] = a.w;
          c_old[4] = b.x; c_old[5] = b.y; c_old[6] = b.z; c_old[7] = b.w;
        } else if (ok && !p.c_zero_init) {
          ldg256(c_row + u0, c_old);
        } else {
#pragma unroll
          for (int u = 0; u < 8; ++u) c_old[u] = 0.f;
        }
        mbar_wait_t(tfull_bar(buf), (uses >> 1) & 1u, prof, w_tfull);
        tc_fence_after();
        float v[32];
        tmem_ld_32x32_issue(t_lane + (uint32_t)(buf * TILE_N + grp * 32), v);
        tmem_ld_wait(v);
        tc_fence_before();
        __syncwarp();
        // accumulators are in registers: MMA may reuse the buffer
        if (lane == 0) mbar_arrive_cluster(mapa_rank(tempty_bar(buf), 0));
        float cn[8], hn[8];
        lstm_cell8(v, bias4 + u0, c_old, cn, hn);
        if (!last) publish_h((uint32_t)(t + 1) & 1u, nt, hn);
        if (!last && keep_c) {
          stg128_hint(c_t, cn[0], cn[1], cn[2], cn[3], pol_keep);
          stg128_hint(c_t + BM * 4, cn[4], cn[5], cn[6], cn[7], pol_keep);
        } else if (!last) {
          stg128(c_t, cn[0], cn[1], cn[2], cn[3]);
          stg128(c_t + BM * 4, cn[4], cn[5], cn[6], cn[7]);
        } else if (ok && p.c_out) {
          stg256(p.c_out + m * kH + u0, cn);
        }
        if (DEC) {
          if (ok && p.h_out) stg256(h_row + (int64_t)t * kH + u0, hn);        // dec_h is optional in the fused decoder
        } else if (BLK) {
          // blocked encodings: the thread's 8 units of position t, coalesced across the warp (1 KB per store)
          if (cta_ok) stg256(e_out + (int64_t)t * ENC_BLK_ROW + nt * ENC_BLK_TILE, hn);
        } else {
          // fp32 h' -> 128B-swizzled [128 x 32] tile; the store issuer (warp 2) sends it to enc_out by TMA
          mbar_wait_t(hempty_bar, (uses & 1u) ^ 1u, prof, w_hempty);   // the previous tile's store has left shared memory
          const uint32_t hb = sbase + OFF_HBUF + (uint32_t)r * 128;
          st_shared_v4(hb + (uint32_t)(((2 * grp) ^ (r & 7)) << 4), __float_as_uint(hn[0]), __float_as_uint(hn[1]),
                       __float_as_uint(hn[2]), __float_as_uint(hn[3]));
          st_shared_v4(hb + (uint32_t)(((2 * grp + 1) ^ (r & 7)) << 4), __float_as_uint(hn[4]), __float_as_uint(hn[5]),
                       __float_as_uint(hn[6]), __float_as_uint(hn[7]));
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) mbar_arrive(hfull_bar);
        }
        if (do_dot) {
          // canonical dot (pointer.cuh): s[nt][g] = fma chain over the 8 units, p[g] sequential over the tiles
#pragma unroll
          for (int j0 = 0; j0 < NR; j0 += CHK) {
            if (j0 > 0) {
#pragma unroll
              for (int u = 0; u < CHK; ++u) {
                if (j0 + u < NR && j0 + u < N)
                  ldg256_stream(e_win + (int64_t)(j0 + u) * ENC_BLK_ROW + nt * ENC_BLK_TILE, ea[u], eb[u], pol_stream);
              }
            }
#pragma unroll
            for (int u = 0; u < CHK; ++u) {
              if (j0 + u < NR && j0 + u < N) {
                // dot8's operand order: row element first, query element second
                float sj = __fmul_rn(ea[u].x, hn[0]);
                sj = fmaf(ea[u].y, hn[1], sj); sj = fmaf(ea[u].z, hn[2], sj); sj = fmaf(ea[u].w, hn[3], sj);
                sj = fmaf(eb[u].x, hn[4], sj); sj = fmaf(eb[u].y, hn[5], sj); sj = fmaf(eb[u].z, hn[6], sj);
                sj = fmaf(eb[u].w, hn[7], sj);
                acc[j0 + u] = it == 0 ? sj : __fadd_rn(acc[j0 + u], sj);
              }
            }
          }
          if (it + 1 < N_TILES) request_rows(t, it + 1);
          else if (!last) request_rows(t + 1, 0);
        }
      }
      if (DEC && !FUSED) {
        // ---- pointer step k = t: query = h'(t) (just written to dec_h by this CTA), window rows of enc_out
        const long long tp0 = prof ? clock64() : 0;
        __threadfence_block();
        asm volatile("bar.sync 1, %0;" ::"n"(32 * EPI_WARPS) : "memory");
        pointer_phase(p, rollout_args(p.pa, roll, p.steps, p.sampled), h_out, t, (warp - 4) * (BM / EPI_WARPS), m0, lane,
                      sgen);
        if (prof) w_ptr += clock64() - tp0;
      }
      if (FUSED) {
        // ---- combine the four group partials of every instance and finish the step (one thread per instance)
        const long long tp0 = prof ? clock64() : 0;
        float* const part = reinterpret_cast<float*>(sgen + OFF_HBUF);      // [3 groups][NR][128 rows]
        if (grp > 0) {
#pragma unroll
          for (int j = 0; j < NR; ++j)
            if (j < N) part[((grp - 1) * NR + j) * BM + r] = acc[j];
        }
        named_bar_sync(1 + q, 128);                     // the four warps that own this quarter's rows
        if (grp == 0) {
          float d[NRA];
#pragma unroll
          for (int j = 0; j < NR; ++j)
            d[j] = j < N ? __fadd_rn(__fadd_rn(acc[j], part[(0 * NR + j) * BM + r]),
                                      __fadd_rn(part[(1 * NR + j) * BM + r], part[(2 * NR + j) * BM + r])) : 0.f;
          const int fed = pointer_finish_thread<NRA>(rollout_args(p.pa, roll, p.steps, p.sampled), t, m, ok, d);
          if (t + 1 < p.steps) {                        // the fed row is the x block row of the next step
            float xv[8];
#pragma unroll
            for (int f = 0; f < 8; ++f)
              xv[f] = (ok && f < p.F) ? __ldg(p.inputs + (m * p.L + fed) * (int64_t)p.F + f) : 0.f;
            uint32_t hi[4], lo[4];
            split_f16x8(xv, hi, lo);
            const uint32_t o = (uint32_t)r * XROW_BYTES;
            st_x_row(sbase + OFF_AX_HI + o, sbase + OFF_AX_LO + o, hi, lo);
          }
        }
        if (prof) w_ptr += clock64() - tp0;
      }
      if (DEC) {                                          // x(t+1) is in the x block
        fence_proxy_async_smem();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(a_ready_remote);
      }
    }
    if (prof && warp == 4 && lane == 0) {
      unsigned long long* o = p.prof + (size_t)blockIdx.x * 16;
      o[4] = (unsigned long long)(clock64() - t_begin); o[5] = w_tfull; o[6] = w_hempty; o[7] = w_ptr;
    }
  }
  tc_fence_before();
  cluster_sync_all();
  if (warp == 2) tmem_dealloc_cg2(tmem_base, TMEM_COLS);
}

template <bool DEC, int NR>
int launch_seq(const float* packed, SeqParams p, cudaStream_t st) {
  CUtensorMap maps[4];
  int rc = make_weight_maps(maps, packed, SLOT_ROWS);
  if (rc) return rc;
  CUtensorMap map_h = maps[0];                         // only the row-major encoder stores through it
  if (!DEC && NR == 0) {
    // h_out as a 3-D tensor {unit, step, instance}; box = 32 units x 1 step x 128 instances, 128B swizzle
    const int64_t T = p.h_out_inst_ld / kH;
    cuuint64_t dims[3] = {(cuuint64_t)kH, (cuuint64_t)T, (cuuint64_t)p.n};
    cuuint64_t strides[2] = {(cuuint64_t)kH * 4, (cuuint64_t)p.h_out_inst_ld * 4};
    cuuint32_t box[3] = {32, 1, (cuuint32_t)BM};
    cuuint32_t estr[3] = {1, 1, 1};
    if (encode_fn()(&map_h, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, (void*)p.h_out, dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
      return GNNPN_ESHAPE;
  }
  const unsigned grid = (unsigned)(ceil_div(p.n, 2 * BM) * 2 * p.rollouts);
  if ((rc = prof_alloc(grid, 16, st, &p.prof))) return rc;
  rc = launch_cluster<lstm_seq_kernel<DEC, NR>>(grid, 2, THREADS, SMEM_BYTES, st, maps[0], maps[1], maps[2], maps[3], map_h,
                                                p);
  if (p.prof) {
    double acc[8];
    unsigned leaders = prof_collect(p.prof, grid, 16, st, acc);     // the MMA-issuing CTAs write counter 0
    if (!leaders) leaders = 1;
    fprintf(stderr, "[seq prof %s nr=%d steps=%d grid=%u] per-step cycles: mma total %.0f (wait a_ready %.0f, tmem_empty %.0f, "
            "B full %.0f) | epi total %.0f (wait tmem_full %.0f, h buf %.0f, pointer %.0f)\n", DEC ? "dec" : "enc", NR,
            p.steps, grid, acc[0] / leaders / p.steps, acc[1] / leaders / p.steps, acc[2] / leaders / p.steps,
            acc[3] / leaders / p.steps, acc[4] / grid / p.steps, acc[5] / grid / p.steps, acc[6] / grid / p.steps,
            acc[7] / grid / p.steps);
  }
  return rc;
}

}  // namespace seq

int tc_seq_encode(const SeqEncodeArgs& a, int nr, cudaStream_t st) {
  seq::SeqParams p{};
  p.n = a.n; p.steps = a.L; p.L = a.L; p.F = a.F;
  p.inputs = a.inputs; p.x_inst_ld = (int64_t)a.L * a.F;
  p.bias0 = p.bias = a.packed + kOffBias;
  p.c = p.c_out = a.c_state; p.c_zero_init = 1;
  p.rollouts = 1;
  p.h0 = nullptr; p.h0_ld = 0;
  p.h_out = a.enc_out; p.h_out_inst_ld = (int64_t)a.L * kH;
  p.c_scr = a.c_scratch;
  return nr ? seq::launch_seq<false, 1>(a.packed, p, st) : seq::launch_seq<false, 0>(a.packed, p, st);
}

int tc_seq_decode(const SeqDecodeArgs& a, int nr, cudaStream_t st) {
  seq::SeqParams p{};
  p.n = a.n; p.steps = a.K; p.L = a.L; p.F = a.F;
  p.inputs = a.inputs; p.x_inst_ld = (int64_t)a.L * a.F;
  p.bias0 = a.packed + kOffStart; p.bias = a.packed + kOffBias;
  p.c = a.c_state; p.c_zero_init = 0;
  p.c_out = a.rollouts ? nullptr : a.c_state;
  p.rollouts = a.rollouts ? a.rollouts : 1;
  p.sampled = a.sampled;
  p.h_out = a.dec_h; p.h_out_inst_ld = (int64_t)a.K * kH;
  p.pa = pointer_step_args(a.enc_out, a.latent_win, a.alpha, a.use_tanh, a.C, a.n, a.L, a.N, a.idx_out, a.win_logits,
                           a.win_probs, a.forced_idx, a.sample_uniform);
  p.c_scr = a.c_scratch;
  // blocked encodings (nr > 0): the pointer dots ride in the cell epilogue, and h0 is read from the block's position
  // L-1 inside the kernel
  if (nr == 0) { p.h0 = a.enc_out + (int64_t)(a.L - 1) * kH; p.h0_ld = (int64_t)a.L * kH; }
  switch (nr) {
    case 5: return seq::launch_seq<true, 5>(a.packed, p, st);
    case 8: return seq::launch_seq<true, 8>(a.packed, p, st);
    case 10: return seq::launch_seq<true, 10>(a.packed, p, st);
    default: return seq::launch_seq<true, 0>(a.packed, p, st);
  }
}

// ================================================================================================================
// Host side shared by both scans (this file and tc_colsplit.cu): which kernel runs a batch, and their launch code.
namespace {

// Column-split groups of 128 instances per encoder cluster for a batch of n, or 0 when the CTA-pair scan runs it.
// Option "scan": -1 automatic, 0 CTA-pair, 1 column-split.  Automatic (measured on a B200 with 15 co-resident clusters,
// profiles/r01_colsplit_timing.jsonl, r01_pn_batch_sweep.jsonl): a column-split step costs ~6.6 us per wave (~7 us with
// two groups per cluster) against ~16.7 us (encoder) / ~37 us (fused decoder) for the CTA-pair scan at any batch up to
// 18,944.  So the column-split scan takes up to two waves of groups: one-group clusters up to one wave, two-group
// clusters up to 30 groups (one wave; two waves of them are slower than the pair scan).  Option "scan_groups": 0
// automatic, 1 / 2 / 3 forced; pipeline.low_high picks 3 for 15..21 groups so that PNLow's and PNHigh's encoders --
// 7 clusters each -- run side by side on the 15 cluster slots.  The decoder runs two groups per cluster whenever the
// encoder runs two or three (one wave of 8..15 clusters for 16..30 groups).
int colsplit_groups(int64_t n) {
  const int scan = options().scan.load(std::memory_order_relaxed);
  if (scan == 0) return 0;
  const int64_t groups = ceil_div(n, 128);
  if (scan != 1 && groups > 2 * (int64_t)tc_colsplit_max_active_clusters()) return 0;
  const int g = options().scan_groups.load(std::memory_order_relaxed);
  if (g >= 1 && g <= 3) return g;
  return groups > tc_colsplit_max_active_clusters() ? 2 : 1;
}

}  // namespace

// Option "persistent": bit 0 runs the encoder, bit 1 the decoder as one persistent launch (default 3); without its bit
// a recurrence runs one launch per step (kept for inputs wider than 8 columns, runs without a workspace and as the
// A/B reference).  The blocked encodings layout exists for the CTA-pair scan's fused decoder, so it is asked for only
// when both scans are persistent, the batch is not the column-split scan's, and the window fits the fused decoder's
// row capacity (N <= 10).  Encodings that are already blocked go to the CTA-pair scan before the column-split test.
// A rollout launch decodes n * rollouts rows from the encodings of n instances: the encoder's choice and the layout come
// from n, the decoder's from the n * rollouts rows and the layout the encoder wrote.
ScanPlan plan_scans(int64_t n, int F, int N, int layout, bool has_workspace, int rollouts, int persistent) {
  ScanPlan p{{ScanKind::kStep, 0}, {ScanKind::kStep, 0}, GNNPN_ENC_ROWMAJOR};
  if (!has_workspace || F < 1 || F > 8) return p;
  if (persistent < 0) persistent = options().persistent.load(std::memory_order_relaxed);
  const bool blocked = layout == GNNPN_ENC_BLOCKED128;
  const int g = colsplit_groups(n), g_dec = colsplit_groups(n * rollouts);
  if (persistent == 3 && N >= 1 && N <= 10 && g == 0) p.layout = GNNPN_ENC_BLOCKED128;
  if (persistent & 1) {
    if (blocked) p.enc = {ScanKind::kPair, 1};
    else if (g) p.enc = {ScanKind::kColsplit, g};
    else p.enc = {ScanKind::kPair, 0};
  }
  if (persistent & 2) {
    if (blocked && N > 10) p.dec = {ScanKind::kUnsupported, 0};
    else if (blocked) p.dec = {ScanKind::kPair, N == 5 ? 5 : (N <= 8 ? 8 : 10)};
    else if (g_dec) p.dec = {ScanKind::kColsplit, std::min(g_dec, 2)};
    else p.dec = {ScanKind::kPair, 0};
  }
  return p;
}

int make_weight_maps(CUtensorMap maps[4], const float* packed, int box_rows) {
  int rc = GNNPN_OK;
  for (int i = 0; i < 4 && !rc; ++i)           // i < 2: h part, 64 halfs per gate column; i >= 2: x part, 16 halfs
    rc = tc::make_map_2d(&maps[i], packed + ((i & 1) ? kOffTc16Lo : kOffTc16Hi), kG, kKp16, kKp16, box_rows, true,
                         i < 2 ? 64 : 16);
  return rc;
}

int prof_alloc(unsigned ctas, int per_cta, cudaStream_t st, unsigned long long** counters) {
  *counters = nullptr;
  if (!options().prof.load(std::memory_order_relaxed)) return GNNPN_OK;
  const size_t bytes = (size_t)ctas * per_cta * sizeof(unsigned long long);
  if (cudaMalloc(counters, bytes) != cudaSuccess) return GNNPN_EUNSUPPORTED;
  cudaMemsetAsync(*counters, 0, bytes, st);
  return GNNPN_OK;
}

unsigned prof_collect(unsigned long long* counters, unsigned ctas, int per_cta, cudaStream_t st, double sums[8]) {
  const size_t bytes = (size_t)ctas * per_cta * sizeof(unsigned long long);
  unsigned long long* h = (unsigned long long*)malloc(bytes);
  cudaStreamSynchronize(st);
  cudaMemcpy(h, counters, bytes, cudaMemcpyDeviceToHost);
  cudaFree(counters);
  unsigned wrote = 0;
  for (int i = 0; i < 8; ++i) sums[i] = 0;
  for (unsigned c = 0; c < ctas; ++c) {
    if (h[(size_t)c * per_cta]) ++wrote;
    for (int i = 0; i < 8; ++i) sums[i] += (double)h[(size_t)c * per_cta + i];
  }
  free(h);
  return wrote;
}

}  // namespace gnnpn
