// tcgen05 (5th-gen tensor core) kernels, fp32 results through error-compensated 3xTF32:
//     A.B^T  ~=  A_hi.B_hi^T + A_lo.B_hi^T + A_hi.B_lo^T       (hi = tf32(a), lo = a - hi; the dropped
//                                                                lo.lo term is ~2^-22 relative)
// accumulated in fp32 in TMEM.  One mainloop, two epilogues:
//   * GEMM             C = act((A.W^T + bias)*scale + shift) for the shapes node_transform.cu does not take (K or N
//                      > 256, K % 4 != 0, N % 16 != 0), split-K for the long-K weight gradients
//   * LSTM step        gates = [h|x].P^T + bias -> c', h'  (+ fp16 split of h' for the next step's A operand); its
//                      operands are fp16 hi/lo pairs (3xFP16, same three products), see Kind<true>
//
// CTA = one 128-row M tile; loops over `n_tiles` N tiles of BN <= 256 columns with two TMEM
// accumulator buffers so the epilogue of tile j overlaps the MMAs of tile j+1.
// Warp roles: 0 = TMA producer, 1 = MMA issuer, 2 = TMEM allocator, 4..19 = epilogue (TMEM lane quarter = warp&3;
// epilogue group g = (warp-4)/4 takes the 32-column chunks g, g+4, ... of a tile: four epilogue warps per SM
// sub-partition, which is what hides the global-memory latency of the per-row state loads/stores).
// smem ring: STAGES x { A_hi, A_lo [128 x 32 f32], B_hi, B_lo [BN x 32 f32] }, 128B-swizzled K-major tiles
// written by TMA and read by tcgen05.mma through UMMA descriptors.
#include <algorithm>
#include "tc_common.cuh"
#include "common.cuh"
#include "internal.cuh"
#include "lstm_step.cuh"
#include "tc_lstm.cuh"
#include "tc_seq.cuh"

namespace gnnpn {
namespace tc {

constexpr int BM = 128;            // rows per CTA = UMMA M = TMEM lanes
constexpr int BK = 32;             // fp32 per 128-byte swizzle row
constexpr int BN_MAX = 256;        // UMMA N limit
constexpr int STAGES = 2;
constexpr int A_TILE_BYTES = BM * BK * 4;          // 16 KiB
constexpr int B_TILE_BYTES = BN_MAX * BK * 4;      // 32 KiB
constexpr int STAGE_BYTES = 2 * A_TILE_BYTES + 2 * B_TILE_BYTES;
constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /*alignment slack*/ + 256 /*barriers*/ + 4096 /*epilogue*/;
constexpr int EPI_GROUPS = 4;
constexpr int EPI_WARPS = 4 * EPI_GROUPS;
constexpr int THREADS = 128 + 32 * EPI_WARPS;
constexpr int TMEM_COLS = 512;

struct GemmEpilogueParams {
  const float* bias; const float* scale; const float* shift; int act;
  float* C; int64_t ldc; int N;
  int64_t split_stride;     // split-K: floats between the partial outputs of consecutive k-splits (blockIdx.y), else 0
};

struct LstmEpilogueParams {
  const float* bias;        // [1024] gate-interleaved
  float* c;                 // [M,256] in/out
  float* h_out;             // exact fp32 h' rows, h_out_ld apart
  int64_t h_out_ld;
  __half* a_hi_next;        // [M, a_ld]  fp16 split of h' for the next step (+ x columns)
  __half* a_lo_next;
  int64_t a_ld;
  const float* x_next;      // raw inputs row of the NEXT step per instance (nullptr: none)
  int64_t x_inst_ld;
  int x_row_next;           // fixed row (encoder) ; <0 -> no x written here (decoder: pointer step writes it)
  int F;
  int first;                // c_old = 0
};

struct MainloopParams {
  int M;                    // valid rows
  int n_tiles;              // N tiles handled by each CTA
  int bn;                   // columns per N tile (multiple of 16, <= 256)
  int k_blocks;             // K / 32
  int last_block_ksteps;    // k-steps (of 8) actually non-zero in the last k block (1..4)
  int kb_per_split;         // split-K: k blocks per blockIdx.y (>= k_blocks: no split)
};

// Operand flavour of the mainloop: every smem tile row is 128 bytes either way.
template <bool F16> struct Kind;
template <> struct Kind<false> {                    // tf32-in-fp32: 32 elements / row, K = 8 per MMA
  static constexpr int BKE = 32;
  __device__ static uint32_t idesc(int n) { return idesc_tf32(BM, n); }
  __device__ static void mma(uint32_t d, uint64_t a, uint64_t b, uint32_t i, uint32_t acc) { mma_tf32_ss(d, a, b, i, acc); }
};
template <> struct Kind<true> {                     // fp16: 64 elements / row, K = 16 per MMA
  static constexpr int BKE = 64;
  __device__ static uint32_t idesc(int n) { return idesc_f16(BM, n); }
  __device__ static void mma(uint32_t d, uint64_t a, uint64_t b, uint32_t i, uint32_t acc) { mma_f16_ss(d, a, b, i, acc); }
};

// ------------------------------------------------------------------------------------------------
template <class Epilogue, class EpiParams, bool F16>
__global__ void __launch_bounds__(THREADS, 1)
tc_mainloop_kernel(const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
                   const __grid_constant__ CUtensorMap map_b_hi, const __grid_constant__ CUtensorMap map_b_lo,
                   const MainloopParams mp, const EpiParams ep) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = smem_base + STAGES * STAGE_BYTES;
  // barrier slots (8 B each): full[STAGES], empty[STAGES], tmem_full[2], tmem_empty[2]; then tmem ptr
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  auto tmem_full_bar = [&](int b) { return bar_base + 8u * (2 * STAGES + b); };
  auto tmem_empty_bar = [&](int b) { return bar_base + 8u * (2 * STAGES + 2 + b); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * STAGES + 4);
  float* epi_smem = reinterpret_cast<float*>(smem_raw + (bar_base + 256u - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m0 = blockIdx.x * BM;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_a_hi); tma_prefetch_desc(&map_a_lo);
    tma_prefetch_desc(&map_b_hi); tma_prefetch_desc(&map_b_lo);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(tmem_full_bar(b), 1); mbar_init(tmem_empty_bar(b), EPI_WARPS); }
    fence_mbar_init();
  }
  if (warp == 2) tmem_alloc(tmem_slot, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

  constexpr int BKE = Kind<F16>::BKE;                 // elements per 128-byte k-block row
  // split-K (weight-gradient GEMMs: few output tiles, very long K): blockIdx.y owns the k blocks [kb0, kb1)
  const int kb0 = (int)blockIdx.y * mp.kb_per_split;
  const int kb1 = min(mp.k_blocks, kb0 + mp.kb_per_split);
  const uint32_t stage_tx = 2u * A_TILE_BYTES + 2u * (uint32_t)mp.bn * 128u;

  if (warp == 0) {
    // ================= TMA producer =================
    if (lane == 0) {
      int s = 0; uint32_t ph = 0;
      for (int nt = 0; nt < mp.n_tiles; ++nt) {
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(empty_bar(s), ph ^ 1u);
          mbar_arrive_expect_tx(full_bar(s), stage_tx);
          const uint32_t st = smem_base + s * STAGE_BYTES;
          tma_load_2d(st, &map_a_hi, full_bar(s), kb * BKE, m0);
          tma_load_2d(st + A_TILE_BYTES, &map_a_lo, full_bar(s), kb * BKE, m0);
          tma_load_2d(st + 2 * A_TILE_BYTES, &map_b_hi, full_bar(s), kb * BKE, nt * mp.bn);
          tma_load_2d(st + 2 * A_TILE_BYTES + B_TILE_BYTES, &map_b_lo, full_bar(s), kb * BKE, nt * mp.bn);
          if (++s == STAGES) { s = 0; ph ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer (one thread) =================
    if (lane == 0) {
      const uint32_t idesc = Kind<F16>::idesc(mp.bn);
      int s = 0; uint32_t ph = 0;
      for (int nt = 0; nt < mp.n_tiles; ++nt) {
        const int buf = nt & 1;
        const uint32_t use = (uint32_t)(nt >> 1);            // how many times this buffer was used before
        mbar_wait(tmem_empty_bar(buf), (use & 1u) ^ 1u);    // epilogue has drained it (passes on first use)
        tc_fence_after();
        const uint32_t d = tmem_base + (uint32_t)(buf * BN_MAX);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(full_bar(s), ph);
          tc_fence_after();
          const uint32_t st = smem_base + s * STAGE_BYTES;
          const uint64_t a_hi = smem_desc_k_sw128(st), a_lo = smem_desc_k_sw128(st + A_TILE_BYTES);
          const uint64_t b_hi = smem_desc_k_sw128(st + 2 * A_TILE_BYTES);
          const uint64_t b_lo = smem_desc_k_sw128(st + 2 * A_TILE_BYTES + B_TILE_BYTES);
          const int ksteps = (kb == mp.k_blocks - 1) ? mp.last_block_ksteps : 4;
          for (int ks = 0; ks < ksteps; ++ks) {
            const uint64_t adv = (uint64_t)(ks * 2);            // +32 B per k-step inside the 128-byte swizzle row
            const uint32_t acc0 = ((kb - kb0) | ks) != 0;
            Kind<F16>::mma(d, a_lo + adv, b_hi + adv, idesc, acc0);
            Kind<F16>::mma(d, a_hi + adv, b_lo + adv, idesc, 1u);
            Kind<F16>::mma(d, a_hi + adv, b_hi + adv, idesc, 1u);
          }
          mma_commit(empty_bar(s));                 // smem slot reusable once these MMAs retire
          if (kb == kb1 - 1) mma_commit(tmem_full_bar(buf));
          if (++s == STAGES) { s = 0; ph ^= 1u; }
        }
      }
    }
  } else if (warp >= 4) {
    // ================= epilogue: thread = one accumulator row, 32-column chunks =================
    const int q = warp & 3;
    const int grp = (warp - 4) >> 2;                 // chunk phase of this warp
    const int row = m0 + q * 32 + lane;
    Epilogue::stage_smem(ep, epi_smem, threadIdx.x - 128, 32 * EPI_WARPS);
    asm volatile("bar.sync 1, %0;" ::"n"(32 * EPI_WARPS) : "memory");     // epilogue warps only
    Epilogue epi(ep, epi_smem, row, row < mp.M, grp == 0);
    constexpr int MAX_CHUNKS = BN_MAX / (32 * EPI_GROUPS);     // chunks of one tile owned by a thread
    for (int nt = 0; nt < mp.n_tiles; ++nt) {
      const int buf = nt & 1;
      const uint32_t use = (uint32_t)(nt >> 1);
      // per-row state this thread needs for the tile does not depend on the accumulators: put those global
      // loads in flight before blocking on the MMA warp
#pragma unroll
      for (int i = 0; i < MAX_CHUNKS; ++i) {
        const int c0 = (grp + i * EPI_GROUPS) * 32;
        if (c0 < mp.bn) epi.prefetch(i, nt * mp.bn + c0);
      }
      mbar_wait(tmem_full_bar(buf), use & 1u);
      tc_fence_after();
      const uint32_t t0 = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * BN_MAX);
#pragma unroll
      for (int i = 0; i < MAX_CHUNKS; ++i) {
        const int c0 = (grp + i * EPI_GROUPS) * 32;
        if (c0 < mp.bn) {
          float v[32];
          tmem_ld_32x32_issue(t0 + (uint32_t)c0, v);
          tmem_ld_wait(v);
          epi.chunk(i, nt * mp.bn + c0, min(32, mp.bn - c0), v);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tmem_empty_bar(buf));
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem_base, TMEM_COLS);
}

// ------------------------------------------------------------------------------------------------
struct GemmEpilogue {
  const GemmEpilogueParams& p; int64_t row; bool ok;
  __device__ static void stage_smem(const GemmEpilogueParams&, float*, int, int) {}
  __device__ GemmEpilogue(const GemmEpilogueParams& p_, const float*, int row_, bool ok_, bool)
      : p(p_), row(row_), ok(ok_) {}
  __device__ void prefetch(int, int) {}
  __device__ void chunk(int, int col0, int ncols, const float* v) {
    if (!ok) return;
    float* out = p.C + (int64_t)blockIdx.y * p.split_stride + row * p.ldc;
    // a thread owns 32 consecutive columns of ONE row: with 8-float-aligned rows it writes whole 32-byte sectors (one
    // 256-bit store per 8 columns); scalar stores put 32 different rows into every warp-wide store instruction -- 8x the
    // L2 write transactions (the [18,944 x 2,507] readout of the ML stage: 0.43 -> 0.1x ms)
    const bool vec = (p.ldc & 7) == 0 && (reinterpret_cast<uintptr_t>(p.C) & 31u) == 0 && (p.split_stride & 7) == 0;
#pragma unroll
    for (int j0 = 0; j0 < 32; j0 += 8) {
      float r8[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int n = col0 + j0 + j;
        float r = v[j0 + j];
        if (j0 + j < ncols && n < p.N) {
          bias_bn_act<1>(&r, p.bias, p.scale, p.shift, p.act, [&](const float* a, float* x) { x[0] = __ldg(a + n); });
        }
        r8[j] = r;
      }
      const int n0 = col0 + j0;
      if (vec && j0 + 8 <= ncols && n0 + 8 <= p.N) {
        asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(out + n0), "f"(r8[0]), "f"(r8[1]), "f"(r8[2]),
                     "f"(r8[3]), "f"(r8[4]), "f"(r8[5]), "f"(r8[6]), "f"(r8[7]) : "memory");
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j)
          if (j0 + j < ncols && n0 + j < p.N) out[n0 + j] = r8[j];
      }
    }
  }
};

struct LstmEpilogue {
  const LstmEpilogueParams& p; int64_t row; bool ok;
  const float* sbias;            // the 1024 gate biases, staged once per CTA
  float c_pre[BN_MAX / (32 * EPI_GROUPS)][8];   // prefetched cell state: 8 hidden units per owned chunk
  __device__ static void stage_smem(const LstmEpilogueParams& p, float* smem, int tid, int nthreads) {
    for (int i = tid; i < kG; i += nthreads) smem[i] = __ldg(p.bias + i);
  }
  __device__ LstmEpilogue(const LstmEpilogueParams& p_, const float* smem, int row_, bool ok_, bool primary)
      : p(p_), row(row_), ok(ok_), sbias(smem) {
    if (ok && primary && p.x_next && p.x_row_next >= 0) {   // stage the next step's raw input as A columns 256..
      const float* x = p.x_next + row * p.x_inst_ld + (int64_t)p.x_row_next * p.F;
      for (int f = 0; f < p.F; ++f) stage_x_f16(p.a_hi_next, p.a_lo_next, p.a_ld, row, f, __ldg(x + f));
    }
  }
  __device__ void prefetch(int slot, int col0) {
    if (ok && !p.first) {
      ldg256(p.c + row * kH + (col0 >> 2), c_pre[slot]);
    } else {
#pragma unroll
      for (int u = 0; u < 8; ++u) c_pre[slot][u] = 0.f;
    }
  }
  // 32 gate columns = 8 hidden units x (i,f,g,o)
  __device__ void chunk(int slot, int col0, int /*ncols*/, const float* v) {
    if (!ok) return;
    const int j0 = col0 >> 2;
    float hv[8], cv[8];
    const float4* bias4 = reinterpret_cast<const float4*>(sbias + col0);
    constexpr float kAccScale = 1.0f / kW16Scale;      // fp16 weights are stored pre-scaled
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const float4 b = bias4[u];
      const float gi = fmaf(v[4 * u + 0], kAccScale, b.x), gf = fmaf(v[4 * u + 1], kAccScale, b.y);
      const float gg = fmaf(v[4 * u + 2], kAccScale, b.z), go = fmaf(v[4 * u + 3], kAccScale, b.w);
      const float cn = fmaf(sigmoid_mufu(gf), c_pre[slot][u], sigmoid_mufu(gi) * tanh_mufu(gg));
      cv[u] = cn;
      hv[u] = sigmoid_mufu(go) * tanh_mufu(cn);
    }
    stg256(p.c + row * kH + j0, cv);
    stg256(p.h_out + row * p.h_out_ld + j0, hv);
    __half2 hh[4], hl[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      __half a0, l0, a1, l1;
      split_f16(hv[2 * u], a0, l0);
      split_f16(hv[2 * u + 1], a1, l1);
      hh[u] = __halves2half2(a0, a1);
      hl[u] = __halves2half2(l0, l1);
    }
    *reinterpret_cast<uint4*>(p.a_hi_next + row * p.a_ld + j0) = *reinterpret_cast<uint4*>(hh);
    *reinterpret_cast<uint4*>(p.a_lo_next + row * p.a_ld + j0) = *reinterpret_cast<uint4*>(hl);
  }
};

// ------------------------------------------------------------------------------------------------
// elementwise tf32 split with zero padding of K up to Kpad (also used for the weights)
__global__ void split_tf32_kernel(const float* __restrict__ src, int64_t ld, int64_t rows, int K, int Kpad,
                                  float* __restrict__ hi, float* __restrict__ lo) {
  const int64_t total = rows * Kpad;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total;
       e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = e / Kpad;
    const int k = (int)(e % Kpad);
    float h = 0.f, l = 0.f;
    if (k < K) split_tf32(src[r * ld + k], h, l);
    hi[e] = h;
    lo[e] = l;
  }
}

// ------------------------------------------------------------------------------------------------
// host side: tensor maps through the driver entry point (no link-time libcuda dependency)
EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  }
  return fn;
}

int make_map_2d(CUtensorMap* m, const void* base, int64_t rows, int64_t cols, int64_t ld, int box_rows, bool f16,
                int box_cols) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return GNNPN_EUNSUPPORTED;
  const int esz = f16 ? 2 : 4;
  if (!box_cols) box_cols = 128 / esz;
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * esz};
  cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(m, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)base, dims,
                  strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  box_cols * esz == 32 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? GNNPN_OK : GNNPN_ESHAPE;
}

template <class Epi, class EpiParams, bool F16>
int launch_mainloop(const CUtensorMap maps[4], const MainloopParams& mp, const EpiParams& ep, cudaStream_t st, int splits = 1) {
  auto kern = tc_mainloop_kernel<Epi, EpiParams, F16>;
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
    if (e != cudaSuccess) return (int)e;
    configured = true;
  }
  const unsigned grid = (unsigned)ceil_div(mp.M, BM);
  MainloopParams mpd = mp;
  if (mpd.kb_per_split <= 0) mpd.kb_per_split = mpd.k_blocks;
  kern<<<dim3(grid, (unsigned)splits), THREADS, SMEM_BYTES, st>>>(maps[0], maps[1], maps[2], maps[3], mpd, ep);
  return after_launch();
}

}  // namespace tc

// ------------------------------------------------------------------------------------------------
// 3xTF32 GEMM through tcgen05.  Workspace holds the tf32 splits of A and W.
// split-K factor of the GEMM: only when the output has few row tiles and K is long (weight gradients of the REINFORCE
// replay: [4H, T*n] x [T*n, H+16] = 8 row tiles, 940 k blocks of 32).  Two reasons: (1) 8 CTAs on 148 SMs; (2) the tensor
// cores' fp32 accumulation loses ~0.5 ulp per MMA, so one 11,000-MMA chain is 1e-4 off where the element-wise bound of
// this entry is 1e-5 -- chains of 8 k blocks (96 MMAs) summed by fp32 adds in split order stay inside it.  The partial
// outputs are capped at 256 MB.
static int tc_gemm_splits(int64_t M, int N, int K) {
  const int64_t row_tiles = ceil_div(M, tc::BM);
  const int k_blocks = round_up(K, tc::BK) / tc::BK;
  if (row_tiles * 2 > kNumSMs || k_blocks < 64) return 1;
  int64_t s_max = (256ll << 20) / (M * (int64_t)N * 4);
  if (s_max > 128) s_max = 128;
  if (s_max < 2) return 1;
  const int kps = (int)std::max<int64_t>(8, ceil_div(k_blocks, s_max));
  return (int)ceil_div(k_blocks, kps);
}

size_t tc_gemm_workspace_bytes(int64_t M, int N, int K) {
  const int64_t Kp = round_up(K, tc::BK);
  const int S = tc_gemm_splits(M, N, K);
  return (size_t)(2 * (M + N) * Kp) * sizeof(float) + 1024 + (S > 1 ? (size_t)S * M * N * sizeof(float) + 256 : 0);
}

namespace {
// C = epilogue(sum over the k-splits, in split order): deterministic
__global__ void splitk_reduce_kernel(const float* __restrict__ part, int S, int64_t M, int N, const float* __restrict__ bias,
                                     const float* __restrict__ scale, const float* __restrict__ shift, int act,
                                     float* __restrict__ C, int64_t ldc) {
  const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e >= M * N) return;
  const int n = (int)(e % N);
  float r = part[e];
  for (int s = 1; s < S; ++s) r += part[(int64_t)s * M * N + e];
  bias_bn_act<1>(&r, bias, scale, shift, act, [&](const float* p, float* x) { x[0] = __ldg(p + n); });
  C[(e / N) * ldc + n] = r;
}
}  // namespace

int launch_gemm_tc(const float* A, int64_t lda, const float* W, int64_t ldw, const float* bias, const float* scale,
                   const float* shift, int act, float* C, int64_t ldc, int64_t M, int N, int K, void* workspace,
                   cudaStream_t st) {
  using namespace tc;
  const int Kp = round_up(K, BK);
  float* ws = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
  float* a_hi = ws;
  float* a_lo = a_hi + M * Kp;
  float* w_hi = a_lo + M * Kp;
  float* w_lo = w_hi + (int64_t)N * Kp;
  split_tf32_kernel<<<kNumSMs * 4, 256, 0, st>>>(A, lda, M, K, Kp, a_hi, a_lo);
  int rc = after_launch();
  if (rc) return rc;
  split_tf32_kernel<<<kNumSMs * 4, 256, 0, st>>>(W, ldw, N, K, Kp, w_hi, w_lo);
  if ((rc = after_launch())) return rc;
  int bn = N >= BN_MAX ? BN_MAX : round_up(N, 16);
  const int n_tiles = (int)ceil_div(N, bn);
  CUtensorMap maps[4];
  if ((rc = make_map_2d(&maps[0], a_hi, M, Kp, Kp, BM))) return rc;
  if ((rc = make_map_2d(&maps[1], a_lo, M, Kp, Kp, BM))) return rc;
  if ((rc = make_map_2d(&maps[2], w_hi, N, Kp, Kp, bn))) return rc;
  if ((rc = make_map_2d(&maps[3], w_lo, N, Kp, Kp, bn))) return rc;
  const int S = tc_gemm_splits(M, N, K);
  if (S > 1) {
    float* part = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(w_lo + (int64_t)N * Kp) + 255) & ~uintptr_t(255));
    const int kps = (int)ceil_div(Kp / BK, S);
    const int S_eff = (int)ceil_div(Kp / BK, kps);               // every split owns at least one k block (S_eff <= S)
    MainloopParams mp{(int)M, n_tiles, bn, Kp / BK, BK / 8, kps};
    GemmEpilogueParams ep{nullptr, nullptr, nullptr, GNNPN_ACT_NONE, part, N, N, (int64_t)M * N};
    if ((rc = launch_mainloop<GemmEpilogue, GemmEpilogueParams, false>(maps, mp, ep, st, S_eff))) return rc;
    splitk_reduce_kernel<<<(unsigned)ceil_div(M * (int64_t)N, 256), 256, 0, st>>>(part, S_eff, M, N, bias, scale, shift, act, C,
                                                                               ldc);
    return after_launch();
  }
  MainloopParams mp{(int)M, n_tiles, bn, Kp / BK, BK / 8, Kp / BK};
  GemmEpilogueParams ep{bias, scale, shift, act, C, ldc, N, 0};
  return launch_mainloop<GemmEpilogue, GemmEpilogueParams, false>(maps, mp, ep, st);
}

// ------------------------------------------------------------------------------------------------
// LSTM recurrence, one launch per step
namespace {

__global__ void stage_x_kernel(const float* __restrict__ inputs, int64_t x_inst_ld, int row, int F, int64_t n,
                               __half* __restrict__ hi, __half* __restrict__ lo, int ld) {
  const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e >= n * F) return;
  const int64_t m = e / F;
  const int f = (int)(e % F);
  stage_x_f16(hi, lo, ld, m, f, inputs[m * x_inst_ld + (int64_t)row * F + f]);
}

// rows of fp32 h (ld apart) -> fp16 hi/lo rows of kKp16 columns, padding zeroed
__global__ void split_f16_rows_kernel(const float* __restrict__ src, int64_t ld, int64_t rows, int K, int Kpad,
                                      __half* __restrict__ hi, __half* __restrict__ lo) {
  const int64_t total = rows * Kpad;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total;
       e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = e / Kpad;
    const int k = (int)(e % Kpad);
    __half h = __float2half_rn(0.f), l = h;
    if (k < K) tc::split_f16(src[r * ld + k], h, l);
    hi[e] = h;
    lo[e] = l;
  }
}

int tc_zero(const TcLstmPlan& plan, int which, cudaStream_t st) {
  // hi[which] and lo[which] are adjacent in the workspace
  cudaError_t e = cudaMemsetAsync(plan.hi[which], 0, (size_t)2 * plan.n * kKp16 * sizeof(__half), st);
  return e == cudaSuccess ? GNNPN_OK : (int)e;
}

// one tcgen05 step on [h | x] (h only when !use_x) of buffer cur; the epilogue writes h' into buffer cur ^ 1
int tc_step(const TcLstmPlan& plan, int cur, bool use_x, tc::LstmEpilogueParams ep, cudaStream_t st) {
  using namespace tc;
  const CUtensorMap maps[4] = {plan.a_hi[cur], plan.a_lo[cur], plan.b_hi, plan.b_lo};
  MainloopParams mp;
  mp.M = (int)plan.n;
  mp.n_tiles = kG / BN_MAX;
  mp.bn = BN_MAX;
  mp.k_blocks = kH / 64 + (use_x ? 1 : 0);
  mp.last_block_ksteps = use_x ? (ep.F + 15) / 16 : 4;
  mp.kb_per_split = mp.k_blocks;
  ep.a_hi_next = plan.hi[cur ^ 1]; ep.a_lo_next = plan.lo[cur ^ 1]; ep.a_ld = kKp16;
  return launch_mainloop<LstmEpilogue, LstmEpilogueParams, true>(maps, mp, ep, st);
}

int ffma_step(LstmStepArgs& a, const LstmRecurrence& r, const LstmStepSaves* saves, cudaStream_t st) {
  a.P = r.packed;
  a.M = (int)r.n;
  a.c = saves ? saves->c : r.c;
  a.c_in = saves ? saves->c_in : nullptr;
  a.gates_out = saves ? saves->gates : nullptr;
  return launch_lstm_step(a, st);
}

}  // namespace

size_t tc_lstm_workspace_bytes(int64_t n) {
  const size_t step = (size_t)4 * n * kKp16 * sizeof(__half) + 1024;
  const size_t seq = tc_seq_scratch_floats(n) * sizeof(float) + 1024;
  const size_t colsplit = tc_colsplit_scratch_bytes(n) + 1024;
  const size_t m = step > seq ? step : seq;
  return m > colsplit ? m : colsplit;
}

int lstm_recurrence_init(LstmRecurrence* r, const float* packed, const float* inputs, int64_t n, int L, int F,
                         float* c_state, void* workspace, size_t workspace_bytes) {
  r->packed = packed; r->inputs = inputs; r->n = n; r->L = L; r->F = F; r->c = c_state;
  r->tc = workspace != nullptr;
  if (!r->tc) return GNNPN_OK;
  if (workspace_bytes < tc_lstm_workspace_bytes(n)) return GNNPN_EWORKSPACE;
  // two ping-pong [n, kKp16] hi/lo pairs
  TcLstmPlan& p = r->plan;
  __half* ws = align_ws<__half>(workspace);
  const size_t one = (size_t)n * kKp16;       // halfs, a multiple of 64 bytes
  p.n = n;
  p.hi[0] = ws; p.lo[0] = ws + one; p.hi[1] = ws + 2 * one; p.lo[1] = ws + 3 * one;
  int rc;
  for (int b = 0; b < 2; ++b) {
    if ((rc = tc::make_map_2d(&p.a_hi[b], p.hi[b], n, kKp16, kKp16, tc::BM, true))) return rc;
    if ((rc = tc::make_map_2d(&p.a_lo[b], p.lo[b], n, kKp16, kKp16, tc::BM, true))) return rc;
  }
  if ((rc = tc::make_map_2d(&p.b_hi, packed + kOffTc16Hi, kG, kKp16, kKp16, tc::BN_MAX, true))) return rc;
  return tc::make_map_2d(&p.b_lo, packed + kOffTc16Lo, kG, kKp16, kKp16, tc::BN_MAX, true);
}

int lstm_encoder_step(const LstmRecurrence& r, int t, float* enc_out, const LstmStepSaves* saves, cudaStream_t st) {
  const int64_t x_inst_ld = (int64_t)r.L * r.F, h_ld = (int64_t)r.L * kH;
  float* h_out = enc_out + (int64_t)t * kH;
  if (r.tc) {
    if (saves) return GNNPN_EUNSUPPORTED;
    int rc;
    if (t == 0) {                // h = 0 and x = raw row 0 in buffer 0; zero padding in both buffers
      if ((rc = tc_zero(r.plan, 0, st)) || (rc = tc_zero(r.plan, 1, st))) return rc;
      stage_x_kernel<<<(unsigned)ceil_div(r.n * r.F, 256), 256, 0, st>>>(r.inputs, x_inst_ld, 0, r.F, r.n, r.plan.hi[0],
                                                                          r.plan.lo[0], kKp16);
      if ((rc = after_launch())) return rc;
    }
    tc::LstmEpilogueParams ep{};
    ep.bias = r.packed + kOffBias; ep.c = r.c; ep.h_out = h_out; ep.h_out_ld = h_ld;
    ep.x_next = r.inputs; ep.x_inst_ld = x_inst_ld; ep.x_row_next = t + 1 < r.L ? t + 1 : -1; ep.F = r.F;
    ep.first = t == 0;
    return tc_step(r.plan, t & 1, true, ep, st);
  }
  LstmStepArgs a{};
  a.h_in = t == 0 ? nullptr : h_out - kH; a.h_in_ld = h_ld;
  a.x = r.inputs; a.x_inst_ld = x_inst_ld; a.x_row = t; a.F = r.F; a.use_x = 1;
  a.bias = r.packed + kOffBias; a.h_out = h_out; a.h_out_ld = h_ld; a.first = t == 0;
  return ffma_step(a, r, saves, st);
}

int lstm_decoder_step(const LstmRecurrence& r, int k, const float* enc_out, float* dec_h, int K, const int32_t* fed,
                      const LstmStepSaves* saves, cudaStream_t st) {
  // the decoder state starts from the encoder's last hidden state (modelPN.py:191,205)
  const float* h_last = enc_out + (int64_t)(r.L - 1) * kH;
  const float* bias = r.packed + (k == 0 ? kOffStart : kOffBias);
  const int64_t h_ld = (int64_t)K * kH;
  float* h_out = dec_h + (int64_t)k * kH;
  if (r.tc) {
    if (saves) return GNNPN_EUNSUPPORTED;
    int rc;
    if (k == 0) {
      split_f16_rows_kernel<<<kNumSMs * 4, 256, 0, st>>>(h_last, (int64_t)r.L * kH, r.n, kH, kKp16, r.plan.hi[0],
                                                         r.plan.lo[0]);
      if ((rc = after_launch()) || (rc = tc_zero(r.plan, 1, st))) return rc;
    }
    tc::LstmEpilogueParams ep{};
    ep.bias = bias; ep.c = r.c; ep.h_out = h_out; ep.h_out_ld = h_ld; ep.x_row_next = -1; ep.F = r.F;
    return tc_step(r.plan, k & 1, k != 0, ep, st);
  }
  LstmStepArgs a{};
  a.h_in = k == 0 ? h_last : h_out - kH; a.h_in_ld = k == 0 ? (int64_t)r.L * kH : h_ld;
  a.x = r.inputs; a.x_inst_ld = (int64_t)r.L * r.F; a.x_row = -1; a.gather = k == 0 ? nullptr : fed + (int64_t)(k - 1) * r.n;
  a.F = r.F; a.use_x = k != 0; a.bias = bias; a.h_out = h_out; a.h_out_ld = h_ld; a.first = 0;
  return ffma_step(a, r, saves, st);
}

LstmXSlot lstm_decoder_x_slot(const LstmRecurrence& r, int k) {
  if (!r.tc) return LstmXSlot{nullptr, nullptr, 0};
  return LstmXSlot{r.plan.hi[(k + 1) & 1], r.plan.lo[(k + 1) & 1], kKp16};
}

}  // namespace gnnpn
