// REINFORCE backward of the pointer network (src/models/trainPNLow.py:77-106, trainPNHigh.py:77-112: the reference
// back-propagates sum_k log p_k(a_k) through its K-step python graph with torch autograd).  Here the differentiable
// replay of a sampled decode runs on this library's kernels:
//   forward  (gnnpn_pn_train_forward_f32, pn.cu): the sampled decode itself on the column-split scan, or a replay of the
//            sampled picks on the strict-fp32 FFMA LSTM steps + pointer steps, saving per step the post-activation gates
//            and the cell state;
//   backward (this file): window-softmax / C*tanh / dot-attention backward in one launch, then BPTT through the decoder
//            (K steps) and the encoder (L steps): one persistent cluster scan per LSTM (pn_bptt.cu), or per step one cell
//            kernel (gate derivatives, written row-major for the recurrence and TRANSPOSED [4H, T*n] for the
//            weight-gradient GEMMs) and one GEMM dh(t-1) = dG(t) . W_hh (launch_bptt_steps below, option "bptt" = 0).
// The weight gradients are then contractions over all (step, instance) pairs, dW_hh = dG^T . h(t-1), dM = dG^T . x(t)
// (M = the folded W_ih . W_embed input block), which the caller runs through gnnpn_gemm_f32_bias_act.
// Dot attention, no glimpses, embedding_size = 0 (what every reference call site trains).
#include <math.h>
#include "internal.cuh"
#include "lstm_step.cuh"
#include "pointer.cuh"
#include "options.cuh"

namespace gnnpn {
namespace {

// split-K of dh(t-1) = dG(t) . W_hh (dh_splitk_kernel): 16 chunks of 64 gate rows
constexpr int SK_S = 16, SK_KC = kG / SK_S, SK_COLS = 32, SK_ROWS = 128;

// ---- attention backward: one warp per (instance b, step k)
//   p_kj = softmax_j(w_kj), w = l + alpha * latent, l = C * tanh(u) (or u), u_kj = <enc[b, kN+j], q_k>
//   given gp = dLoss/dp_k[a_k]:   dLoss/dw_kj = gp * p_ka * (delta_ja - p_kj)
//   g_kj = dLoss/du_kj = dLoss/dw_kj * C * (1 - (l/C)^2)
//   dq_k = sum_j g_kj * enc[b, kN+j],    d_enc[b, kN+j] = g_kj * q_k     (windows partition L: every row written once)
__global__ void __launch_bounds__(256) attention_bwd_kernel(
    const float* __restrict__ enc_out, const float* __restrict__ dec_h, const float* __restrict__ win_logits,
    const float* __restrict__ win_probs, const int32_t* __restrict__ idx, const float* __restrict__ grad_p, int use_tanh,
    float C, int64_t n, int L, int K, int N, float* __restrict__ dq, float* __restrict__ d_enc) {
  const int lane = threadIdx.x & 31;
  const int64_t wid = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (wid >= n * K) return;
  const int64_t b = wid / K;
  const int k = (int)(wid % K);
  const int a = idx[(int64_t)k * n + b] - k * N;
  const float gp = grad_p[(int64_t)k * n + b];
  const float pa = win_probs[b * L + (int64_t)k * N + a];
  const float4* qp = reinterpret_cast<const float4*>(dec_h + (b * K + k) * (int64_t)kH);
  const float4 q0 = qp[2 * lane], q1 = qp[2 * lane + 1];
  float4 s0 = make_float4(0.f, 0.f, 0.f, 0.f), s1 = s0;
  for (int j = 0; j < N; ++j) {
    const int64_t pos = b * L + (int64_t)k * N + j;
    const float p = win_probs[pos];
    float g = gp * pa * ((j == a ? 1.0f : 0.0f) - p);
    if (use_tanh) {
      const float th = win_logits[pos] / C;
      g *= C * (1.0f - th * th);
    }
    const float4* ep = reinterpret_cast<const float4*>(enc_out + pos * kH);
    const float4 e0 = ep[2 * lane], e1 = ep[2 * lane + 1];
    s0.x = fmaf(g, e0.x, s0.x); s0.y = fmaf(g, e0.y, s0.y); s0.z = fmaf(g, e0.z, s0.z); s0.w = fmaf(g, e0.w, s0.w);
    s1.x = fmaf(g, e1.x, s1.x); s1.y = fmaf(g, e1.y, s1.y); s1.z = fmaf(g, e1.z, s1.z); s1.w = fmaf(g, e1.w, s1.w);
    float4* dp = reinterpret_cast<float4*>(d_enc + pos * kH);
    dp[2 * lane] = make_float4(g * q0.x, g * q0.y, g * q0.z, g * q0.w);
    dp[2 * lane + 1] = make_float4(g * q1.x, g * q1.y, g * q1.z, g * q1.w);
  }
  float4* op = reinterpret_cast<float4*>(dq + (b * K + k) * (int64_t)kH);
  op[2 * lane] = s0;
  op[2 * lane + 1] = s1;
}

// ---- LSTM cell backward for one step: thread = (instance m, hidden unit j)
//   dh = dh_ext + dh_rec;  do = dh * tanh(c_t);  dc = dc_next + dh * o * (1 - tanh(c_t)^2)
//   di = dc * g, df = dc * c_prev, dg = dc * i, dc_prev = dc * f
//   dG = (di*i(1-i), df*f(1-f), dg*(1-g^2), do*o(1-o))   -> row-major [n, 4H] in TORCH gate order r = gate*H + j (the A
//   operand of dh(t-1) = dG . W_hh) and transposed dG_T[r][t*n + m] (the A operand of the weight-gradient GEMMs)
struct CellBwdArgs {
  const float* gates;      // [n, 4H] saved post-activation gates of this step, columns 4j + {i,f,g,o}
  const float* c_t;        // [n, H] cell state after this step
  const float* c_prev;     // [n, H] cell state before this step, or nullptr (zeros)
  const float* dh_ext;     // external gradient w.r.t. h_t (attention), rows dh_ext_ld apart, or nullptr
  int64_t dh_ext_ld;
  const float* dh_init;    // [n, H] gradient w.r.t. h_t from downstream (last step only), added after dh_ext, or nullptr
  const float* dh_rec;     // [SK_S][n, H] split-K partials of the gradient from step t+1 (dG(t+1) . W_hh), or nullptr
  const float* dc_next;    // [n, H] or nullptr
  float* dc_prev;          // [n, H]
  float* dG;               // [n, 4H] torch gate order
  float* dG_T;             // [4H, T*n] base pointer of the transposed block
  int64_t t_off;           // t * n
  int64_t Tn;              // T * n
  int64_t n;
};

// block = 32 x 8 threads on a [32 instances x 32 units] tile: loads and the row-major dG stores are coalesced along the
// unit index, the transposed dG_T stores along the instance index (through a shared-memory tile)
__global__ void __launch_bounds__(256) lstm_cell_bwd_kernel(const CellBwdArgs a) {
  __shared__ float tile[4][32][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int64_t m0 = (int64_t)blockIdx.x * 32;
  const int j0 = blockIdx.y * 32;
  const int j = j0 + tx;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int ml = ty + 8 * i;
    const int64_t m = m0 + ml;
    float dGi = 0.f, dGf = 0.f, dGg = 0.f, dGo = 0.f;
    if (m < a.n) {
      const float4 g4 = *reinterpret_cast<const float4*>(a.gates + m * kG + 4 * j);
      const float gi = g4.x, gf = g4.y, gg = g4.z, go = g4.w;
      const float tc = tanhf(a.c_t[m * kH + j]);
      float dh = 0.f;
      if (a.dh_ext) dh += a.dh_ext[m * a.dh_ext_ld + j];
      if (a.dh_init) dh += a.dh_init[m * kH + j];
      if (a.dh_rec) {
        float rsum = a.dh_rec[m * kH + j];
#pragma unroll
        for (int sidx = 1; sidx < SK_S; ++sidx) rsum += a.dh_rec[(int64_t)sidx * a.n * kH + m * kH + j];   // chunk order
        dh += rsum;
      }
      const float d_o = dh * tc;
      float dc = dh * go * (1.0f - tc * tc);
      if (a.dc_next) dc += a.dc_next[m * kH + j];
      const float cp = a.c_prev ? a.c_prev[m * kH + j] : 0.f;
      dGi = dc * gg * gi * (1.0f - gi);
      dGf = dc * cp * gf * (1.0f - gf);
      dGg = dc * gi * (1.0f - gg * gg);
      dGo = d_o * go * (1.0f - go);
      a.dc_prev[m * kH + j] = dc * gf;
      float* row = a.dG + m * kG;
      row[j] = dGi; row[kH + j] = dGf; row[2 * kH + j] = dGg; row[3 * kH + j] = dGo;
    }
    tile[0][ml][tx] = dGi; tile[1][ml][tx] = dGf; tile[2][ml][tx] = dGg; tile[3][ml][tx] = dGo;
  }
  __syncthreads();
  const int64_t m = m0 + tx;
  if (m < a.n) {
#pragma unroll
    for (int g = 0; g < 4; ++g)
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int jl = ty + 8 * i;
        a.dG_T[(int64_t)(g * kH + j0 + jl) * a.Tn + a.t_off + m] = tile[g][tx][jl];
      }
  }
}

// ---- dh(t-1) = dG(t) . W_hh for a small batch: split-K so that a batch of 128 fills the machine.
// grid (S = 16 chunks of 64 gate rows, H / 32 column tiles, ceil(n / 128)); CTA = [128 instances x 32 units] partial over
// its k chunk -> part[s][n][H]; the consumer adds the S partials in chunk order (deterministic).
__global__ void __launch_bounds__(256) dh_splitk_kernel(const float* __restrict__ dG, const float* __restrict__ w_hh,
                                                        int64_t n, float* __restrict__ part) {
  __shared__ __align__(16) float As[SK_KC][SK_ROWS + 4];      // transposed: [k][row]
  __shared__ __align__(16) float Bs[SK_KC][SK_COLS];
  const int tid = threadIdx.x;
  const int k0 = blockIdx.x * SK_KC, c0 = blockIdx.y * SK_COLS;
  const int64_t m0 = (int64_t)blockIdx.z * SK_ROWS;
  for (int i = tid; i < SK_ROWS * (SK_KC / 4); i += 256) {
    const int r = i / (SK_KC / 4), k4 = i % (SK_KC / 4);
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (m0 + r < n) v = *reinterpret_cast<const float4*>(dG + (m0 + r) * kG + k0 + k4 * 4);
    As[k4 * 4 + 0][r] = v.x; As[k4 * 4 + 1][r] = v.y; As[k4 * 4 + 2][r] = v.z; As[k4 * 4 + 3][r] = v.w;
  }
  for (int i = tid; i < SK_KC * (SK_COLS / 4); i += 256) {
    const int k = i / (SK_COLS / 4), c4 = i % (SK_COLS / 4);
    reinterpret_cast<float4*>(&Bs[k][0])[c4] = __ldg(reinterpret_cast<const float4*>(w_hh + (int64_t)(k0 + k) * kH + c0) + c4);
  }
  __syncthreads();
  const int rg = tid >> 3, cg = tid & 7;                      // 4 rows x 4 columns per thread
  float acc[4][4] = {};
#pragma unroll 8
  for (int k = 0; k < SK_KC; ++k) {
    const float4 av = *reinterpret_cast<const float4*>(&As[k][rg * 4]);
    const float4 bv = *reinterpret_cast<const float4*>(&Bs[k][cg * 4]);
    const float a4[4] = {av.x, av.y, av.z, av.w}, b4[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a4[i], b4[j], acc[i][j]);
  }
  float* dst = part + (int64_t)blockIdx.x * n * kH;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t m = m0 + rg * 4 + i;
    if (m < n) *reinterpret_cast<float4*>(dst + m * kH + c0 + cg * 4) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
  }
}

// dst [n, H] = sum of the SK_S split-K partials in src (chunk order, as lstm_cell_bwd_kernel adds them)
__global__ void sum_partials_kernel(float* __restrict__ dst, const float* __restrict__ src, int64_t n) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n * kH) return;
  float s = src[e];
  for (int sidx = 1; sidx < SK_S; ++sidx) s += src[(int64_t)sidx * n * kH + e];
  dst[e] = s;
}

// scratch of launch_bptt_steps: dG [n, 4H] + 2 x dh split-K partials [SK_S][n, H] + 2 x dc [n, H]
size_t bptt_steps_scratch_floats(int64_t n) { return (size_t)n * kG + (2 * SK_S + 2) * (size_t)n * kH; }

// BPTT through one LSTM with two launches per step (the A/B reference of the cluster scan); the arguments of
// launch_bptt_scan (internal.cuh) and bptt_steps_scratch_floats(n) floats of scratch.
int launch_bptt_steps(const float* gates, const float* c, const float* c_init, const float* dh_ext, int64_t dh_ld_m,
                      const float* dh_init, const float* dc_init, const float* w_hh, float* dG_T, float* dh_out,
                      float* dc_out, int64_t n, int T, float* scratch, cudaStream_t st) {
  if (n <= 0 || T <= 0) return GNNPN_OK;
  const size_t nh = (size_t)n * kH;
  float* dG = scratch;
  float* dh_rec[2] = {dG + (size_t)n * kG, dG + (size_t)n * kG + SK_S * nh};
  float* dc[2] = {dh_rec[1] + SK_S * nh, dh_rec[1] + SK_S * nh + nh};
  int cur = 0, rc;
  for (int t = T - 1; t >= 0; --t) {
    CellBwdArgs a{};
    a.gates = gates + (size_t)t * n * kG;
    a.c_t = c + (size_t)t * nh;
    a.c_prev = t > 0 ? c + (size_t)(t - 1) * nh : c_init;
    a.dh_ext = dh_ext + (size_t)t * kH; a.dh_ext_ld = dh_ld_m;
    a.dh_init = t == T - 1 ? dh_init : nullptr;
    a.dh_rec = t == T - 1 ? nullptr : dh_rec[cur];
    a.dc_next = t == T - 1 ? dc_init : dc[cur];
    a.dc_prev = t == 0 && dc_out ? dc_out : dc[cur ^ 1];
    a.dG = dG; a.dG_T = dG_T; a.t_off = (int64_t)t * n; a.Tn = (int64_t)T * n; a.n = n;
    lstm_cell_bwd_kernel<<<dim3((unsigned)ceil_div(n, 32), kH / 32), 256, 0, st>>>(a);
    if ((rc = after_launch())) return rc;
    if (t > 0 || dh_out) {                                    // dh(t-1) = dG . W_hh (split-K partials)
      dh_splitk_kernel<<<dim3(SK_S, kH / SK_COLS, (unsigned)ceil_div(n, SK_ROWS)), 256, 0, st>>>(dG, w_hh, n, dh_rec[cur ^ 1]);
      if ((rc = after_launch())) return rc;
    }
    cur ^= 1;
  }
  if (!dh_out) return GNNPN_OK;
  sum_partials_kernel<<<(unsigned)ceil_div(n * kH, 256), 256, 0, st>>>(dh_out, dh_rec[cur], n);
  return after_launch();
}

}  // namespace
}  // namespace gnnpn

using namespace gnnpn;

extern "C" {

size_t gnnpn_pn_train_backward_workspace_floats(int64_t n, int L, int K, int hidden) {
  if (hidden != kH || n < 0) return 0;
  // dq [n,K,H] + d_enc [n,L,H] + the decoder's dh / dc w.r.t. its initial state [n,H] each + launch_bptt_steps' scratch
  return (size_t)n * K * kH + (size_t)n * L * kH + 2 * (size_t)n * kH + bptt_steps_scratch_floats(n);
}

int gnnpn_pn_train_backward_f32(const float* enc_out, const float* gates_e, const float* c_e, const float* dec_h,
                                const float* gates_d, const float* c_d, const float* win_logits, const float* win_probs,
                                const int32_t* idx, const float* grad_p, const float* w_hh_enc, const float* w_hh_dec,
                                int use_tanh, float C, int64_t n, int L, int hidden, int K, int N, float* dG_enc_T,
                                float* dG_dec_T, float* workspace, size_t workspace_floats, void* stream) {
  GNNPN_REQUIRE(enc_out && gates_e && c_e && dec_h && gates_d && c_d && win_logits && win_probs && idx && grad_p &&
                    w_hh_enc && w_hh_dec && dG_enc_T && dG_dec_T && workspace, GNNPN_ENULL);
  GNNPN_REQUIRE(hidden == kH && K >= 1 && N >= 1 && (int64_t)K * N == L && n >= 0, GNNPN_ESHAPE);
  GNNPN_REQUIRE(workspace_floats >= gnnpn_pn_train_backward_workspace_floats(n, L, K, hidden), GNNPN_EWORKSPACE);
  GNNPN_REQUIRE(aligned16(enc_out) && aligned16(dec_h) && aligned16(gates_e) && aligned16(gates_d) && aligned16(workspace),
                GNNPN_EALIGN);
  if (n == 0) return GNNPN_OK;
  cudaStream_t st = (cudaStream_t)stream;
  float* dq = workspace;
  float* d_enc = dq + (size_t)n * K * kH;
  float* dh0 = d_enc + (size_t)n * L * kH;
  float* dc0 = dh0 + (size_t)n * kH;
  float* scratch = dc0 + (size_t)n * kH;
  int rc;
  attention_bwd_kernel<<<(unsigned)ceil_div(n * K, 8), 256, 0, st>>>(enc_out, dec_h, win_logits, win_probs, idx, grad_p,
                                                                    use_tanh, C, n, L, K, N, dq, d_enc);
  if ((rc = after_launch())) return rc;
  const auto bptt = options().bptt.load(std::memory_order_relaxed) ? launch_bptt_scan : launch_bptt_steps;
  // the decoder started from the encoder's last state: its dh / dc w.r.t. that state enter the encoder at t = L-1
  const float* c_last_e = c_e + (size_t)(L - 1) * n * kH;
  if ((rc = bptt(gates_d, c_d, c_last_e, dq, (int64_t)K * kH, nullptr, nullptr, w_hh_dec, dG_dec_T, dh0, dc0, n, K,
                 scratch, st)))
    return rc;
  return bptt(gates_e, c_e, nullptr, d_enc, (int64_t)L * kH, dh0, dc0, w_hh_enc, dG_enc_T, nullptr, nullptr, n, L, scratch,
              st);
}

}  // extern "C"
