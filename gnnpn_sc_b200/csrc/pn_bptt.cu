// Persistent BPTT of one LSTM (the REINFORCE backward, trainPNLow.py:88-96 via torch autograd in the reference): ALL T
// dependent backward steps in ONE launch instead of two launches per step.
//
// A cluster of 8 CTAs owns a block of 16 instances for the whole scan; CTA rank r owns hidden units [32r, 32r + 32):
//   * its slice W_hh[:, 32r : 32r + 32] ([4H x 32] fp32, 128 KB) is loaded ONCE and stays in shared memory;
//   * per step it (a) turns dh(t), dc(t+1) and the saved gates / cell states of ITS (instance, unit) pairs into the gate
//     gradients dG(t) -- thread = (instance, 2 units), dc lives in registers for the whole scan -- and writes them to the
//     transposed block dG_T [4H, T*n] that the weight-gradient GEMM reads anyway; (b) after ONE cluster barrier pulls the
//     block's complete dG(t) [4H x 16] back from L2 into shared memory; (c) computes its [16 x 32] tile of
//     dh(t-1) = dG(t) . W_hh with FFMAs (8 warps = 4 k-slices x 2 unit halves, 2 x 4 register tile, partial sums combined
//     in k-slice order: deterministic).
// The exchange goes through dG_T itself (64-byte segments, L2-resident between the write and the read), so the scan adds no
// traffic beyond what the per-step kernels wrote; the cluster barrier (release / acquire at cluster scope) orders it.
// Same formulas as lstm_cell_bwd_kernel (pn_train.cu); strict fp32.
#include <math.h>
#include "internal.cuh"
#include "lstm_step.cuh"
#include "options.cuh"

namespace gnnpn {
namespace bptt {

constexpr int CL = 8;                 // CTAs per cluster = unit tiles
constexpr int BI = 16;                // instances per cluster
constexpr int UT = kH / CL;           // 32 units per CTA
constexpr int THREADS = 256;
constexpr int KS = 4;                 // k-slices of the dh GEMM (kG / KS = 256 gate rows each)
constexpr uint32_t SMEM_W = (uint32_t)kG * UT * 4;          // 128 KB
constexpr uint32_t SMEM_A = (uint32_t)kG * BI * 4;          // 64 KB
constexpr uint32_t SMEM_RED = (uint32_t)KS * BI * UT * 4;   // 8 KB
constexpr uint32_t SMEM_BYTES = SMEM_W + SMEM_A + SMEM_RED;

struct Args {
  const float* gates;     // [T, n, 4H] saved post-activation gates, columns 4j + {i,f,g,o}
  const float* c;         // [T, n, H] cell state after every step
  const float* c_init;    // [n, H] cell state before step 0, or nullptr (zeros)
  const float* dh_ext;    // external gradient w.r.t. h(t): element (m, t, j) at dh_ext + m*ld_m + t*kH + j
  int64_t dh_ld_m;
  const float* dh_init;   // [n, H] gradient w.r.t. h(T-1) from downstream (added to dh_ext), or nullptr
  const float* dc_init;   // [n, H] gradient w.r.t. c(T-1) from downstream, or nullptr
  const float* w_hh;      // [4H, H] torch layout
  float* dG_T;            // [4H, T*n] gate gradients, torch gate order rows
  float* dh_out;          // [n, H] gradient w.r.t. the hidden state before step 0, or nullptr (not needed)
  float* dc_out;          // [n, H] same for the cell state, or nullptr
  int64_t n;
  int T;
};

__device__ __forceinline__ void cluster_arrive_release() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait_acquire() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
__device__ __forceinline__ uint32_t cluster_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}

__global__ void __launch_bounds__(THREADS, 1) lstm_bptt_cluster_kernel(const Args a) {
  extern __shared__ __align__(16) float smem[];
  float* Ws = smem;                                  // [kG][UT]
  float* As = smem + kG * UT;                        // [kG][BI]   dG(t) of the block's 16 instances, all gate rows
  float* red = As + kG * BI;                         // [KS][BI][UT] partial dh tiles; also the dG transpose stage [4][UT][BI]
  const int tid = threadIdx.x;
  const uint32_t rank = cluster_rank();
  const int64_t m0 = (int64_t)(blockIdx.x / CL) * BI;
  const int u0 = (int)rank * UT;
  const int64_t Tn = (int64_t)a.T * a.n;

  // resident weight slice: Ws[r][j] = W_hh[r][u0 + j]
  for (int i = tid; i < kG * (UT / 4); i += THREADS) {
    const int r = i / (UT / 4), c4 = i % (UT / 4);
    reinterpret_cast<float4*>(Ws + r * UT)[c4] = __ldg(reinterpret_cast<const float4*>(a.w_hh + (int64_t)r * kH + u0) + c4);
  }
  // cell phase ownership: instance ci, units cu, cu + 1 (of this CTA's 32)
  const int ci = tid >> 4, cu = (tid & 15) * 2;
  const int64_t m = m0 + ci;
  const bool ok = m < a.n;
  const int ju = u0 + cu;                            // global unit index of the first element
  float dc[2] = {0.f, 0.f}, dh_rec[2] = {0.f, 0.f};
  if (ok && a.dc_init) { dc[0] = a.dc_init[m * kH + ju]; dc[1] = a.dc_init[m * kH + ju + 1]; }
  if (ok && a.dh_init) { dh_rec[0] = a.dh_init[m * kH + ju]; dh_rec[1] = a.dh_init[m * kH + ju + 1]; }
  // GEMM phase ownership
  const int warp = tid >> 5, lane = tid & 31;
  const int ks = warp >> 1, uh = warp & 1;
  const int ip = lane >> 2, uq = lane & 3;
  __syncthreads();

  // saved operands of the cell phase of one step (14 registers): requested one step ahead, under the dh GEMM
  struct CellOps { float4 g0, g1; float2 ct, cp, de; };
  auto load_ops = [&](int t) {
    CellOps o;
    o.g0 = o.g1 = make_float4(0.f, 0.f, 0.f, 0.f);
    o.ct = o.cp = o.de = make_float2(0.f, 0.f);
    if (ok && t >= 0) {
      const float* gp = a.gates + ((int64_t)t * a.n + m) * kG + 4 * ju;
      o.g0 = *reinterpret_cast<const float4*>(gp);
      o.g1 = *reinterpret_cast<const float4*>(gp + 4);
      o.ct = *reinterpret_cast<const float2*>(a.c + ((int64_t)t * a.n + m) * kH + ju);
      if (t > 0) o.cp = *reinterpret_cast<const float2*>(a.c + ((int64_t)(t - 1) * a.n + m) * kH + ju);
      else if (a.c_init) o.cp = *reinterpret_cast<const float2*>(a.c_init + m * kH + ju);
      o.de = *reinterpret_cast<const float2*>(a.dh_ext + m * a.dh_ld_m + (int64_t)t * kH + ju);
    }
    return o;
  };
  CellOps nxt = load_ops(a.T - 1);
  for (int t = a.T - 1; t >= 0; --t) {
    // ---- (a) gate gradients of step t for this thread's two (instance, unit) elements
    const CellOps cur = nxt;
    float dG[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
    if (ok) {
      const float gi[2] = {cur.g0.x, cur.g1.x}, gf[2] = {cur.g0.y, cur.g1.y}, gg[2] = {cur.g0.z, cur.g1.z}, go[2] = {cur.g0.w, cur.g1.w};
      const float ctv[2] = {cur.ct.x, cur.ct.y}, cpv[2] = {cur.cp.x, cur.cp.y}, dev[2] = {cur.de.x, cur.de.y};
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const float tc = tanhf(ctv[e]);
        const float dh = dev[e] + dh_rec[e];
        const float d_o = dh * tc;
        const float dcv = dh * go[e] * (1.0f - tc * tc) + dc[e];
        dG[e][0] = dcv * gg[e] * gi[e] * (1.0f - gi[e]);
        dG[e][1] = dcv * cpv[e] * gf[e] * (1.0f - gf[e]);
        dG[e][2] = dcv * gi[e] * (1.0f - gg[e] * gg[e]);
        dG[e][3] = d_o * go[e] * (1.0f - go[e]);
        dc[e] = dcv * gf[e];
      }
    }
    // transpose through shared memory: stage[g][unit][instance] -> rows of dG_T, 16 instances = 64 contiguous bytes
    float* stage = red;
#pragma unroll
    for (int e = 0; e < 2; ++e)
#pragma unroll
      for (int g = 0; g < 4; ++g) stage[(g * UT + cu + e) * BI + ci] = dG[e][g];
    __syncthreads();
    for (int i = tid; i < 4 * UT * (BI / 4); i += THREADS) {
      const int row = i / (BI / 4), q4 = i % (BI / 4);       // row = g * UT + unit
      const int g = row / UT, u = row % UT;
      const float4 v = *reinterpret_cast<const float4*>(stage + row * BI + q4 * 4);
      float* dst = a.dG_T + (int64_t)(g * kH + u0 + u) * Tn + (int64_t)t * a.n + m0 + q4 * 4;
      if (m0 + q4 * 4 + 3 < a.n && ((reinterpret_cast<uintptr_t>(dst) & 15u) == 0)) {
        *reinterpret_cast<float4*>(dst) = v;
      } else {
        const float vv[4] = {v.x, v.y, v.z, v.w};
        for (int k = 0; k < 4; ++k) if (m0 + q4 * 4 + k < a.n) dst[k] = vv[k];
      }
    }
    if (t == 0 && !a.dh_out) break;                         // the gradient w.r.t. the initial state is not needed
    // ---- (b) every CTA of the cluster has written its rows of dG(t): pull the block's [4H x 16] back
    cluster_arrive_release();
    cluster_wait_acquire();
    {
      constexpr int PER = kG * (BI / 4) / THREADS;           // 16 float4 per thread, all in flight together
      float4 v[PER];
      // every 4-instance segment inside the batch and 16-byte aligned
      const bool vec_ok = (a.n & 3) == 0 && m0 + BI <= a.n && (reinterpret_cast<uintptr_t>(a.dG_T) & 15u) == 0;
#pragma unroll
      for (int j = 0; j < PER; ++j) {
        const int i = tid + j * THREADS;
        const int r = i / (BI / 4), q4 = i % (BI / 4);
        const float* src = a.dG_T + (int64_t)r * Tn + (int64_t)t * a.n + m0 + q4 * 4;
        if (vec_ok) {
          v[j] = __ldcg(reinterpret_cast<const float4*>(src));
        } else {
          float vv[4] = {0.f, 0.f, 0.f, 0.f};
          for (int k = 0; k < 4; ++k) if (m0 + q4 * 4 + k < a.n) vv[k] = __ldcg(src + k);
          v[j] = make_float4(vv[0], vv[1], vv[2], vv[3]);
        }
      }
      nxt = load_ops(t - 1);                                 // next step's saves: their latency hides under the GEMM
#pragma unroll
      for (int j = 0; j < PER; ++j) {
        const int i = tid + j * THREADS;
        *reinterpret_cast<float4*>(As + (i / (BI / 4)) * BI + (i % (BI / 4)) * 4) = v[j];
      }
    }
    __syncthreads();
    // ---- (c) dh(t-1)[16 x 32] = dG(t)[16 x 4H] . Ws[4H x 32]: this warp's k-slice and unit half, 2 instances x 4 units / lane
    float acc[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
    const float* Ap = As + (ks * (kG / KS)) * BI + ip * 2;
    const float* Wp = Ws + (ks * (kG / KS)) * UT + uh * 16 + uq * 4;
#pragma unroll 8
    for (int k = 0; k < kG / KS; ++k) {
      const float2 av = *reinterpret_cast<const float2*>(Ap + k * BI);
      const float4 wv = *reinterpret_cast<const float4*>(Wp + k * UT);
      acc[0][0] = fmaf(av.x, wv.x, acc[0][0]); acc[0][1] = fmaf(av.x, wv.y, acc[0][1]);
      acc[0][2] = fmaf(av.x, wv.z, acc[0][2]); acc[0][3] = fmaf(av.x, wv.w, acc[0][3]);
      acc[1][0] = fmaf(av.y, wv.x, acc[1][0]); acc[1][1] = fmaf(av.y, wv.y, acc[1][1]);
      acc[1][2] = fmaf(av.y, wv.z, acc[1][2]); acc[1][3] = fmaf(av.y, wv.w, acc[1][3]);
    }
#pragma unroll
    for (int e = 0; e < 2; ++e)
      *reinterpret_cast<float4*>(red + ((ks * BI) + ip * 2 + e) * UT + uh * 16 + uq * 4) =
          make_float4(acc[e][0], acc[e][1], acc[e][2], acc[e][3]);
    __syncthreads();
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      float s = red[(0 * BI + ci) * UT + cu + e];
#pragma unroll
      for (int q = 1; q < KS; ++q) s += red[(q * BI + ci) * UT + cu + e];      // k-slice order
      dh_rec[e] = s;
    }
    __syncthreads();                                         // red is reused as the transpose stage of the next step
  }
  if (a.dh_out && ok) {
    a.dh_out[m * kH + ju] = dh_rec[0]; a.dh_out[m * kH + ju + 1] = dh_rec[1];
    if (a.dc_out) { a.dc_out[m * kH + ju] = dc[0]; a.dc_out[m * kH + ju + 1] = dc[1]; }
  }
  // no CTA may exit while a peer could still be waiting on the cluster barrier: every CTA executes the same number of
  // barrier phases (the loop bounds are cluster-uniform), so nothing more is needed here
}

}  // namespace bptt

// BPTT through one LSTM; see bptt::Args.  n_max_per_launch is unlimited (clusters are independent).
int launch_bptt_scan(const float* gates, const float* c, const float* c_init, const float* dh_ext, int64_t dh_ld_m,
                     const float* dh_init, const float* dc_init, const float* w_hh, float* dG_T, float* dh_out,
                     float* dc_out, int64_t n, int T, float* scratch, cudaStream_t st) {
  using namespace bptt;
  (void)scratch;
  if (n <= 0 || T <= 0) return GNNPN_OK;
  const Args a{gates, c, c_init, dh_ext, dh_ld_m, dh_init, dc_init, w_hh, dG_T, dh_out, dc_out, n, T};
  return launch_cluster<lstm_bptt_cluster_kernel>((unsigned)(ceil_div(n, BI) * CL), CL, THREADS, (int)SMEM_BYTES, st, a);
}

}  // namespace gnnpn
