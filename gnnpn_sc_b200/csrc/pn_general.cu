// General pointer-network decode: every variant of PointerNet.forward's decode loop (modelPN.py:204-239) that the
// fused fast paths (pn.cu / tc_seq.cu: Dot attention, no glimpses, window <= 32, <= 8 raw columns) do not cover:
//   * attention "Bahdanau" (modelPN.py:83-91,103-109):  u_l = V . tanh(W_query q + W_ref ref_l),
//     with E = W_ref ref + b_ref computed ONCE per forward (the reference recomputes the 1x1 conv every step);
//   * n_glimpses > 0 (modelPN.py:208-211): q <- sum_l softmax_l(glimpse logits, visited -> -inf) * ref'_l over ALL L
//     positions (ref' = enc_out for Dot, the glimpse's own W_ref conv output for Bahdanau);
//   * any window width N (scale-up: N = 1000) and up to 32 raw input columns (embedding_size = 20).
// One launch per piece and per step (LSTM cell, [query GEMM, glimpse] x n_glimpses, query GEMM, pointer); one CTA
// per composition instance in the attention kernels.  For Dot / no glimpse / N <= 32 the pointer arithmetic is the
// pointer.cuh's (canonical dot, then the shared logit / softmax / pick / draw rules) -> bit-identical picks / logits.
#include <math.h>
#include <cuda_fp16.h>
#include "internal.cuh"
#include "lstm_step.cuh"
#include "tc_lstm.cuh"
#include "pointer.cuh"

namespace gnnpn {
namespace {

constexpr int kAttThreads = 256, kAttWarps = kAttThreads / 32;
constexpr size_t kAttBlockFloats = 2 * (size_t)kH * kH + 3 * kH;   // [W_query | b_query | W_ref | b_ref | V]
constexpr size_t kOffWq = 0, kOffBq = (size_t)kH * kH, kOffWr = kOffBq + kH, kOffBr = kOffWr + (size_t)kH * kH,
                 kOffV = kOffBr + kH;

// sum over the lane's 8 elements of V * tanh(qw + r): explicit fma chain (fixed rounding order)
__device__ __forceinline__ float bahdanau8(const float4 r0, const float4 r1, const float4 w0, const float4 w1,
                                           const float4 v0, const float4 v1) {
  float s = v0.x * tanhf(w0.x + r0.x);
  s = fmaf(v0.y, tanhf(w0.y + r0.y), s); s = fmaf(v0.z, tanhf(w0.z + r0.z), s); s = fmaf(v0.w, tanhf(w0.w + r0.w), s);
  s = fmaf(v1.x, tanhf(w1.x + r1.x), s); s = fmaf(v1.y, tanhf(w1.y + r1.y), s); s = fmaf(v1.z, tanhf(w1.z + r1.z), s);
  s = fmaf(v1.w, tanhf(w1.w + r1.w), s);
  return s;
}

struct GeneralArgs {
  const float* rows;         // [n, L, kH]  enc_out (Dot) or E = W_ref enc_out + b_ref (Bahdanau)
  const float* q;            // [n] rows q_ld apart: the query (Dot) or W_query q + b_query (Bahdanau)
  int64_t q_ld;
  const float* V;            // [kH] (Bahdanau)
  const int32_t* fed;        // [K, n] picks the visited mask follows (forced picks when teacher forcing) -- steps < k
  int64_t n;
  int L, k;
};

// ---------------------------------------------------------------------------------------------------------
// glimpse (modelPN.py:208-211): one CTA per instance, online softmax over all L rows, 8 warps stride the rows
// ---------------------------------------------------------------------------------------------------------
template <bool BAHD>
__global__ void __launch_bounds__(kAttThreads) glimpse_step_kernel(const GeneralArgs a, float* __restrict__ q_out,
                                                                   int64_t q_out_ld) {
  extern __shared__ uint32_t smem_u[];
  uint32_t* visited = smem_u;                              // bitmap of L bits
  const int words = (a.L + 31) / 32;
  const int words4 = (words + 3) & ~3;                     // keep the float4 accesses below 16-byte aligned
  float* red_ms = reinterpret_cast<float*>(smem_u + words4);           // [8 warps][2] running max, sum
  float* red_acc = red_ms + 4 * kAttWarps;                               // [8 warps][kH] weighted row sums
  const int64_t b = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < words; i += kAttThreads) visited[i] = 0u;
  __syncthreads();
  for (int j = threadIdx.x; j < a.k; j += kAttThreads) {
    const int pos = a.fed[(int64_t)j * a.n + b];
    if (pos >= 0 && pos < a.L) atomicOr(&visited[pos >> 5], 1u << (pos & 31));
  }
  __syncthreads();
  const float4* qp = reinterpret_cast<const float4*>(a.q + b * a.q_ld);
  const float4 q0 = qp[lane], q1 = qp[32 + lane];
  float4 v0 = make_float4(0, 0, 0, 0), v1 = v0;
  if (BAHD) { v0 = __ldg(reinterpret_cast<const float4*>(a.V) + lane); v1 = __ldg(reinterpret_cast<const float4*>(a.V) + 32 + lane); }
  float m = -INFINITY, s = 0.f;
  float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  const float* base = a.rows + b * (int64_t)a.L * kH;
  for (int l = warp; l < a.L; l += kAttWarps) {
    if (visited[l >> 5] & (1u << (l & 31))) continue;      // exp(-inf) = 0: contributes nothing
    const float4* rp = reinterpret_cast<const float4*>(base + (int64_t)l * kH);
    const float4 r0 = __ldg(rp + lane), r1 = __ldg(rp + 32 + lane);
    const float u = warp_sum(BAHD ? bahdanau8(r0, r1, q0, q1, v0, v1) : dot8(r0, r1, q0, q1));   // glimpse: no C*tanh
    const float nm = fmaxf(m, u);
    const float sc = expf(m - nm), p = expf(u - nm);       // m = -inf on the first row: sc = 0
    s = fmaf(s, sc, p);
    acc[0] = fmaf(acc[0], sc, p * r0.x); acc[1] = fmaf(acc[1], sc, p * r0.y);
    acc[2] = fmaf(acc[2], sc, p * r0.z); acc[3] = fmaf(acc[3], sc, p * r0.w);
    acc[4] = fmaf(acc[4], sc, p * r1.x); acc[5] = fmaf(acc[5], sc, p * r1.y);
    acc[6] = fmaf(acc[6], sc, p * r1.z); acc[7] = fmaf(acc[7], sc, p * r1.w);
    m = nm;
  }
  if (lane == 0) { red_ms[2 * warp] = m; red_ms[2 * warp + 1] = s; }
  // lane owns hidden elements 4*lane..+3 and 128+4*lane..+3 (float4 index lane and 32+lane)
  reinterpret_cast<float4*>(red_acc + warp * kH)[lane] = make_float4(acc[0], acc[1], acc[2], acc[3]);
  reinterpret_cast<float4*>(red_acc + warp * kH)[32 + lane] = make_float4(acc[4], acc[5], acc[6], acc[7]);
  __syncthreads();
  float M = -INFINITY;
  for (int w = 0; w < kAttWarps; ++w) M = fmaxf(M, red_ms[2 * w]);
  float S = 0.f;
  for (int w = 0; w < kAttWarps; ++w) {
    const float mw = red_ms[2 * w];
    if (mw > -INFINITY) S += red_ms[2 * w + 1] * expf(mw - M);
  }
  for (int h = threadIdx.x; h < kH; h += kAttThreads) {
    float o = 0.f;
    for (int w = 0; w < kAttWarps; ++w) {
      const float mw = red_ms[2 * w];
      if (mw > -INFINITY) o = fmaf(red_acc[w * kH + h], expf(mw - M), o);
    }
    q_out[b * q_out_ld + h] = o / S;
  }
}

// ---------------------------------------------------------------------------------------------------------
// pointer on window k, any N: one CTA per instance
// ---------------------------------------------------------------------------------------------------------
struct PointerGeneralArgs {
  PointerStepArgs s;         // s.enc_out: the rows the query scores, enc_out (Dot) or E (Bahdanau), [n, L, kH]
  int k;
  const float* q;            // [n] rows q_ld apart: the query (Dot) or W_query q + b_query (Bahdanau)
  int64_t q_ld;
  const float* V;            // [kH] (Bahdanau)
  const float* inputs;       // [n, L, F]
  int F;
  LstmXSlot x_next;          // tensor-core LSTM path: where the fed row goes (hi == nullptr: the FFMA step gathers it)
};

template <bool BAHD>
__global__ void __launch_bounds__(kAttThreads) pointer_general_kernel(const PointerGeneralArgs p) {
  extern __shared__ float smem_f[];
  const PointerStepArgs& a = p.s;
  const int N = a.N, k = p.k;
  float* sw = smem_f;                  // [N] masked working logits
  float* se = smem_f + N;              // [N] exp(w - max)
  __shared__ float red_v[kAttWarps];
  __shared__ int red_i[kAttWarps];
  __shared__ float s_bcast[2];
  __shared__ int s_pick;
  const int64_t b = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // Dot: canonical pointer dot (pointer.cuh), lane owns floats [8*lane, 8*lane+8); Bahdanau: float4 lane / 32+lane
  const float4* qp = reinterpret_cast<const float4*>(p.q + b * p.q_ld);
  const int i0 = BAHD ? lane : 2 * lane, i1 = BAHD ? 32 + lane : 2 * lane + 1;
  const float4 q0 = qp[i0], q1 = qp[i1];
  float4 v0 = make_float4(0, 0, 0, 0), v1 = v0;
  if (BAHD) { v0 = __ldg(reinterpret_cast<const float4*>(p.V) + lane); v1 = __ldg(reinterpret_cast<const float4*>(p.V) + 32 + lane); }
  const int64_t wbase = b * (int64_t)a.L + (int64_t)k * N;
  const float* base = a.enc_out + wbase * kH;                            // row-major rows: enc_inst_ld = L * kH
  for (int j = warp; j < N; j += kAttWarps) {
    const float4* rp = reinterpret_cast<const float4*>(base + (int64_t)j * kH);
    const float4 r0 = ldg_stream(rp + i0), r1 = ldg_stream(rp + i1);
    const float d = BAHD ? warp_sum(bahdanau8(r0, r1, q0, q1, v0, v1)) : dot_reduce(dot8(r0, r1, q0, q1), lane);
    if (lane == 0) {
      const float l = window_logit(a.use_tanh, a.C, d);
      a.win_logits[wbase + j] = l;
      sw[j] = work_logit(a, l, a.latent_win ? __ldg(a.latent_win + wbase + j) : 0.f);
    }
  }
  __syncthreads();
  // max (exact, order-free)
  float mx = -INFINITY;
  for (int j = threadIdx.x; j < N; j += kAttThreads) mx = fmaxf(mx, sw[j]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if (lane == 0) red_v[warp] = mx;
  __syncthreads();
  if (threadIdx.x == 0) {
    float m2 = red_v[0];
    for (int w = 1; w < kAttWarps; ++w) m2 = fmaxf(m2, red_v[w]);
    s_bcast[0] = m2;
  }
  __syncthreads();
  mx = s_bcast[0];
  for (int j = threadIdx.x; j < N; j += kAttThreads) se[j] = expf(sw[j] - mx);
  __syncthreads();
  if (threadIdx.x == 0) {                    // sequential sum in candidate order (same order as the fused kernels)
    float s = 0.f;
    for (int j = 0; j < N; ++j) s += se[j];
    s_bcast[1] = s;
  }
  __syncthreads();
  const float s = s_bcast[1];
  // probabilities + first maximal probability: per thread, then per warp, then across the warps
  FirstMax m{-1.f, 0x7fffffff};
  for (int j = threadIdx.x; j < N; j += kAttThreads) {
    const float pj = se[j] / s;
    a.win_probs[wbase + j] = pj;
    se[j] = pj;
    m.add(j, pj);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m.merge(__shfl_xor_sync(0xffffffffu, m.best, o), __shfl_xor_sync(0xffffffffu, m.j, o));
  if (lane == 0) { red_v[warp] = m.best; red_i[warp] = m.j; }
  __syncthreads();
  if (threadIdx.x == 0) {
    FirstMax cta{red_v[0], red_i[0]};
    for (int w = 1; w < kAttWarps; ++w) cta.merge(red_v[w], red_i[w]);
    int pick = cta.j;
    if (a.uniform) {
      const float u = __ldg(a.uniform + (int64_t)k * a.n + b);
      InverseCdf draw;
      for (int j = 0; j < N; ++j) draw.add(j, se[j], u);
      pick = draw.result();
    }
    s_pick = record_pick(a, k, b, pick, true, forced_pick(a, k, b));
  }
  __syncthreads();
  if (p.x_next.hi && threadIdx.x < p.F) {
    const int f = threadIdx.x;
    stage_x_f16(p.x_next.hi, p.x_next.lo, p.x_next.ld, b, f, __ldg(p.inputs + (b * a.L + s_pick) * (int64_t)p.F + f));
  }
}

// Dense logits (prev_logits, modelPN.py:213-214,239): out[k, b, l] = the window logit of row l against query k, -inf at
// the picks of steps < k.  Dot: rows = enc_out, q = dec_h, canonical dot (pointer.cuh); Bahdanau: rows = E, q = qw,
// V . tanh(qw + E).  One CTA per (instance, 32-row slab of L), the instance's K queries in shared memory.
template <bool BAHD>
__global__ void __launch_bounds__(256) full_logits_kernel(
    const float* __restrict__ rows, const float* __restrict__ q, const float* __restrict__ V,
    const int32_t* __restrict__ idx, int use_tanh, float C, int64_t n, int L, int K, float* __restrict__ out) {
  extern __shared__ float sq[];                // [K][kH]
  const int64_t b = blockIdx.x;
  const int l0 = blockIdx.y * 32;
  const float4* qsrc = reinterpret_cast<const float4*>(q + b * (int64_t)K * kH);
  for (int i = threadIdx.x; i < K * kH / 4; i += blockDim.x) reinterpret_cast<float4*>(sq)[i] = __ldg(qsrc + i);
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // Dot: lane owns floats [8*lane, 8*lane+8); Bahdanau: float4 lane / 32+lane
  const int i0 = BAHD ? lane : 2 * lane, i1 = BAHD ? 32 + lane : 2 * lane + 1;
  float4 v0 = make_float4(0, 0, 0, 0), v1 = v0;
  if (BAHD) { v0 = __ldg(reinterpret_cast<const float4*>(V) + lane); v1 = __ldg(reinterpret_cast<const float4*>(V) + 32 + lane); }
  for (int l = l0 + warp; l < min(L, l0 + 32); l += 8) {
    const float4* rp = reinterpret_cast<const float4*>(rows + (b * L + l) * (int64_t)kH);
    const float4 r0 = __ldg(rp + i0), r1 = __ldg(rp + i1);
    for (int k = 0; k < K; ++k) {
      const float4 a0 = reinterpret_cast<const float4*>(sq + k * kH)[i0];
      const float4 a1 = reinterpret_cast<const float4*>(sq + k * kH)[i1];
      const float d = BAHD ? warp_sum(bahdanau8(r0, r1, a0, a1, v0, v1)) : dot_reduce(dot8(r0, r1, a0, a1), lane);
      if (lane == 0) out[((int64_t)k * n + b) * L + l] = window_logit(use_tanh, C, d);
    }
  }
  // cumulative visited mask: step k sees -inf at the picks of steps 0..k-1 (modelPN.py:165-173)
  __syncthreads();
  for (int pair = threadIdx.x; pair < K * K; pair += blockDim.x) {
    const int k = pair / K, jprev = pair % K;
    if (jprev >= k) continue;
    const int pos = idx[(int64_t)jprev * n + b];
    if (pos >= l0 && pos < l0 + 32 && pos < L) out[((int64_t)k * n + b) * L + pos] = -INFINITY;
  }
}

template <bool BAHD>
int launch_full_logits(const float* rows, const float* q, const float* V, const int32_t* idx, int use_tanh, float C,
                       int64_t n, int L, int K, float* out, cudaStream_t st) {
  const size_t smem = (size_t)K * kH * sizeof(float);
  GNNPN_REQUIRE(smem <= 200 * 1024, GNNPN_ESHAPE);
  GNNPN_REQUIRE(n < 65536ll * 32768ll, GNNPN_ERANGE);
  if (n == 0) return GNNPN_OK;
  cudaError_t e = cudaFuncSetAttribute(full_logits_kernel<BAHD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  dim3 grid((unsigned)n, (unsigned)ceil_div(L, 32));
  full_logits_kernel<BAHD><<<grid, 256, smem, st>>>(rows, q, V, idx, use_tanh, C, n, L, K, out);
  return after_launch();
}

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct GeneralWs {
  size_t tc, e_p, e_g, qw, qw_all, total;
};
GeneralWs general_ws(int64_t n, int L, int K, int attention, int n_glimpses, int use_tc) {
  GeneralWs w{};
  size_t off = 0;
  w.tc = off; off += use_tc ? align_up(tc_lstm_workspace_bytes(n), 1024) : 0;
  const size_t big = align_up((size_t)n * L * kH * sizeof(float), 1024);
  w.e_p = off; off += attention == GNNPN_ATT_BAHDANAU ? big : 0;
  w.e_g = off; off += (attention == GNNPN_ATT_BAHDANAU && n_glimpses > 0) ? big : 0;
  w.qw = off; off += align_up((size_t)n * kH * sizeof(float), 1024);
  w.qw_all = off; off += attention == GNNPN_ATT_BAHDANAU ? align_up((size_t)n * K * kH * sizeof(float), 1024) : 0;
  w.total = off + 1024;
  return w;
}

}  // namespace
}  // namespace gnnpn

using namespace gnnpn;

extern "C" {

size_t gnnpn_pn_att_block_floats(int hidden) { return hidden == kH ? kAttBlockFloats : 0; }

size_t gnnpn_pn_decode_general_workspace_bytes(int64_t n, int L, int K, int hidden, int attention, int n_glimpses,
                                               int use_tc) {
  if (hidden != kH || n < 0 || L < 1 || K < 1) return 0;
  return general_ws(n, L, K, attention, n_glimpses, use_tc).total;
}

int gnnpn_pn_decode_general_f32(const float* inputs, const float* enc_out, float* c_state, const float* latent_win,
                                float alpha, const float* packed, int attention, const float* att_params,
                                int n_glimpses, int use_tanh, float C, int64_t n, int L, int in_features, int hidden,
                                int K, int N, float* dec_h, float* dec_q, float* qw_pointer, int32_t* idx_out,
                                float* win_logits, float* win_probs, const int32_t* forced_idx,
                                const float* sample_uniform, int use_tc, void* workspace, size_t workspace_bytes,
                                void* stream) {
  GNNPN_REQUIRE(inputs && enc_out && c_state && packed && dec_h && dec_q && idx_out && win_logits && win_probs &&
                    workspace, GNNPN_ENULL);
  GNNPN_REQUIRE(hidden == kH && in_features >= 1 && in_features <= kXPad, GNNPN_ESHAPE);
  GNNPN_REQUIRE(K >= 1 && N >= 1 && (int64_t)K * N == L && n_glimpses >= 0, GNNPN_ESHAPE);
  GNNPN_REQUIRE((size_t)N * 2 * sizeof(float) <= 160 * 1024 && (size_t)L / 8 <= 160 * 1024, GNNPN_ESHAPE);
  GNNPN_REQUIRE(n >= 0 && n < (1ll << 31), GNNPN_ERANGE);
  GNNPN_REQUIRE(attention == GNNPN_ATT_DOT || attention == GNNPN_ATT_BAHDANAU, GNNPN_EUNSUPPORTED);
  const bool bahd = attention == GNNPN_ATT_BAHDANAU;
  GNNPN_REQUIRE(!bahd || (att_params && qw_pointer), GNNPN_ENULL);
  GNNPN_REQUIRE(n_glimpses == 0 || dec_q != dec_h, GNNPN_ESHAPE);
  GNNPN_REQUIRE(aligned16(enc_out) && aligned16(dec_h) && aligned16(dec_q) && aligned16(c_state) && aligned16(packed) &&
                    (!att_params || aligned16(att_params)), GNNPN_EALIGN);
  if (n == 0) return GNNPN_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const GeneralWs wsl = general_ws(n, L, K, attention, n_glimpses, use_tc);
  GNNPN_REQUIRE(workspace_bytes >= wsl.total, GNNPN_EWORKSPACE);
  uint8_t* ws = align_ws(workspace);
  float* e_p = reinterpret_cast<float*>(ws + wsl.e_p);
  float* e_g = reinterpret_cast<float*>(ws + wsl.e_g);
  float* qw = reinterpret_cast<float*>(ws + wsl.qw);
  const float* att_p = att_params;                                   // pointer block
  const float* att_g = att_params ? att_params + kAttBlockFloats : nullptr;   // glimpse block (follows)
  int rc;
  if (bahd) {
    // E = W_ref . enc_out + b_ref for all positions, once (Conv1d(H,H,1) == a row-wise Linear, modelPN.py:87,105)
    if ((rc = launch_gemm_ffma(enc_out, kH, att_p + kOffWr, kH, att_p + kOffBr, nullptr, nullptr, GNNPN_ACT_NONE, e_p,
                               kH, n * (int64_t)L, kH, kH, st))) return rc;
    if (n_glimpses > 0 &&
        (rc = launch_gemm_ffma(enc_out, kH, att_g + kOffWr, kH, att_g + kOffBr, nullptr, nullptr, GNNPN_ACT_NONE, e_g,
                               kH, n * (int64_t)L, kH, kH, st))) return rc;
  }
  LstmRecurrence r;
  if ((rc = lstm_recurrence_init(&r, packed, inputs, n, L, in_features, c_state, use_tc ? ws + wsl.tc : nullptr,
                                 tc_lstm_workspace_bytes(n)))) return rc;
  const int32_t* fed_all = forced_idx ? forced_idx : idx_out;
  const size_t glimpse_smem = (size_t)((((L + 31) / 32) + 3) & ~3) * 4 + (size_t)kAttWarps * (4 + kH) * 4;
  const size_t ptr_smem = (size_t)N * 2 * sizeof(float);
  if (glimpse_smem > 48 * 1024) {
    cudaFuncSetAttribute(glimpse_step_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)glimpse_smem);
    cudaFuncSetAttribute(glimpse_step_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)glimpse_smem);
  }
  if (ptr_smem > 48 * 1024) {
    cudaFuncSetAttribute(pointer_general_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ptr_smem);
    cudaFuncSetAttribute(pointer_general_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ptr_smem);
  }
  PointerGeneralArgs pa{};
  pa.s = pointer_step_args(bahd ? e_p : enc_out, latent_win, alpha, use_tanh, C, n, L, N, idx_out, win_logits, win_probs,
                           forced_idx, sample_uniform);
  pa.q_ld = (int64_t)K * kH;
  pa.V = bahd ? att_p + kOffV : nullptr;
  pa.inputs = inputs;
  pa.F = in_features;
  for (int k = 0; k < K; ++k) {
    // ---- decoder LSTM cell (modelPN.py:205)
    if ((rc = lstm_decoder_step(r, k, enc_out, dec_h, K, fed_all, nullptr, st))) return rc;
    // ---- glimpses (modelPN.py:208-211)
    const float* q_cur = dec_h + (int64_t)k * kH;
    for (int g = 0; g < n_glimpses; ++g) {
      GeneralArgs ga{};
      ga.fed = fed_all; ga.n = n; ga.L = L; ga.k = k;
      if (bahd) {
        if ((rc = launch_gemm_ffma(q_cur, (int64_t)K * kH, att_g + kOffWq, kH, att_g + kOffBq, nullptr, nullptr,
                                   GNNPN_ACT_NONE, qw, kH, n, kH, kH, st))) return rc;
        ga.rows = e_g; ga.q = qw; ga.q_ld = kH; ga.V = att_g + kOffV;
        glimpse_step_kernel<true><<<(unsigned)n, kAttThreads, glimpse_smem, st>>>(ga, dec_q + (int64_t)k * kH,
                                                                                  (int64_t)K * kH);
      } else {
        ga.rows = enc_out; ga.q = q_cur; ga.q_ld = (int64_t)K * kH; ga.V = nullptr;
        glimpse_step_kernel<false><<<(unsigned)n, kAttThreads, glimpse_smem, st>>>(ga, dec_q + (int64_t)k * kH,
                                                                                   (int64_t)K * kH);
      }
      if ((rc = after_launch())) return rc;
      q_cur = dec_q + (int64_t)k * kH;
    }
    if (n_glimpses == 0 && dec_q != dec_h) {
      if (cudaMemcpy2DAsync(dec_q + (int64_t)k * kH, (size_t)K * kH * 4, dec_h + (int64_t)k * kH, (size_t)K * kH * 4,
                            (size_t)kH * 4, (size_t)n, cudaMemcpyDeviceToDevice, st) != cudaSuccess)
        return (int)cudaGetLastError();
    }
    // ---- pointer on window k (modelPN.py:213-228)
    pa.k = k;
    pa.x_next = lstm_decoder_x_slot(r, k);
    if (bahd) {
      float* qwp = qw_pointer + (int64_t)k * kH;                 // [n, K, kH]: kept for the dense-logits kernel
      if ((rc = launch_gemm_ffma(q_cur, (int64_t)K * kH, att_p + kOffWq, kH, att_p + kOffBq, nullptr, nullptr,
                                 GNNPN_ACT_NONE, qwp, (int64_t)K * kH, n, kH, kH, st))) return rc;
      pa.q = qwp;
      pointer_general_kernel<true><<<(unsigned)n, kAttThreads, ptr_smem, st>>>(pa);
    } else {
      pa.q = q_cur;
      pointer_general_kernel<false><<<(unsigned)n, kAttThreads, ptr_smem, st>>>(pa);
    }
    if ((rc = after_launch())) return rc;
  }
  return GNNPN_OK;
}

int gnnpn_pn_ref_transform_f32(const float* enc_out, const float* att_block, int64_t rows, int hidden, float* E,
                               void* stream) {
  GNNPN_REQUIRE(enc_out && att_block && E, GNNPN_ENULL);
  GNNPN_REQUIRE(hidden == kH && rows >= 0, GNNPN_ESHAPE);
  if (rows == 0) return GNNPN_OK;
  return launch_gemm_ffma(enc_out, kH, att_block + kOffWr, kH, att_block + kOffBr, nullptr, nullptr, GNNPN_ACT_NONE, E,
                          kH, rows, kH, kH, (cudaStream_t)stream);
}

int gnnpn_pn_query_transform_f32(const float* q, int64_t q_ld, const float* att_block, int64_t rows, int hidden,
                                 float* qw, int64_t qw_ld, void* stream) {
  GNNPN_REQUIRE(q && att_block && qw, GNNPN_ENULL);
  GNNPN_REQUIRE(hidden == kH && rows >= 0 && q_ld >= kH && qw_ld >= kH, GNNPN_ESHAPE);
  if (rows == 0) return GNNPN_OK;
  return launch_gemm_ffma(q, q_ld, att_block + kOffWq, kH, att_block + kOffBq, nullptr, nullptr, GNNPN_ACT_NONE, qw,
                          qw_ld, rows, kH, kH, (cudaStream_t)stream);
}

int gnnpn_pn_full_logits_f32(const float* enc_out, const float* dec_h, const int32_t* idx,
                             int attention, const float* att_params, int use_tanh, float C,
                             int64_t n, int L, int hidden, int K, float* logits_full, void* stream) {
  GNNPN_REQUIRE(enc_out && dec_h && idx && logits_full, GNNPN_ENULL);
  GNNPN_REQUIRE(hidden == kH && K >= 1 && L >= 1, GNNPN_ESHAPE);
  GNNPN_REQUIRE(attention == GNNPN_ATT_DOT, GNNPN_EUNSUPPORTED);
  (void)att_params;
  return launch_full_logits<false>(enc_out, dec_h, nullptr, idx, use_tanh, C, n, L, K, logits_full, (cudaStream_t)stream);
}

int gnnpn_pn_full_logits_bahdanau_f32(const float* E, const float* qw, const float* att_block, const int32_t* idx,
                                      int use_tanh, float C, int64_t n, int L, int hidden, int K, float* logits_full,
                                      void* stream) {
  GNNPN_REQUIRE(E && qw && att_block && idx && logits_full, GNNPN_ENULL);
  GNNPN_REQUIRE(hidden == kH && K >= 1 && L >= 1, GNNPN_ESHAPE);
  return launch_full_logits<true>(E, qw, att_block + kOffV, idx, use_tanh, C, n, L, K, logits_full,
                                  (cudaStream_t)stream);
}

}  // extern "C"
