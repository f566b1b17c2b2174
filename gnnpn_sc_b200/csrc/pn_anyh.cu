// Pointer network for ANY hidden size (environment.ini's hidden_size is a free parameter, trainPNLow.py:204; every shipped
// section uses 256, which the tcgen05 / packed-layout kernels are specialised for).  Strict fp32, one launch pair per
// recurrence step: the step GEMM  gates = [h | x] . Wcat^T + b  on the library's FFMA GEMM, then a cell kernel; the decode
// adds one pointer-step kernel per step (Dot attention, window mask, C*tanh, latent, softmax, first-max pick / inverse-CDF
// draw, next-input gather: modelPN.py:204-239).  Same folded weights as the H = 256 path: embedding2 is folded into the
// LSTM input block on the host (Wx = W_ih . W_emb, b = b_ih + b_hh + W_ih . b_emb; decoder start token: b0 = b_ih + b_hh +
// W_ih . start), torch gate order (i, f, g, o) as row blocks of Wcat [4H, H + F].
#include <math.h>
#include "common.cuh"
#include "internal.cuh"
#include "pointer.cuh"

namespace gnnpn {
namespace {

inline unsigned init_grid(int64_t elems) {
  const int64_t b = ceil_div(elems, 256);
  return (unsigned)(b < 8 * kNumSMs ? b : 8 * kNumSMs);
}

// A_cat [n, H + F]: h part <- h0 rows (or zeros), x part <- the raw row x_row of every instance (or zeros)
__global__ void anyh_init_kernel(float* __restrict__ a_cat, int64_t n, int H, int F, const float* __restrict__ h0,
                                 int64_t h0_ld, const float* __restrict__ inputs, int64_t x_inst_ld, int x_row) {
  const int W = H + F;
  const int64_t total = n * W;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t m = e / W;
    const int j = (int)(e % W);
    float v = 0.f;
    if (j < H) { if (h0) v = h0[m * h0_ld + j]; }
    else if (inputs && x_row >= 0) v = inputs[m * x_inst_ld + (int64_t)x_row * F + (j - H)];
    a_cat[e] = v;
  }
}

// LSTM cell (nn.LSTM, gate order i,f,g,o: modelPN.py:157-158): thread = (instance m, unit j)
//   c' = sigm(f) c + sigm(i) tanh(g),  h' = sigm(o) tanh(c')
// h' goes to h_out (enc_out / dec_h row of this step) and into the h part of A_cat for the next step; the encoder also
// places the next raw row into the x part (next_row >= 0).
__global__ void anyh_cell_kernel(const float* __restrict__ gates, float* __restrict__ c, int c_zero, float* __restrict__ h_out,
                                 int64_t h_out_ld, float* __restrict__ a_cat, int64_t n, int H, int F,
                                 const float* __restrict__ inputs, int64_t x_inst_ld, int next_row) {
  const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e >= n * H) return;
  const int64_t m = e / H;
  const int j = (int)(e % H);
  const float* g = gates + m * 4 * (int64_t)H;
  const float gi = sigmoid_accurate(g[j]), gf = sigmoid_accurate(g[H + j]);
  const float gg = tanhf(g[2 * H + j]), go = sigmoid_accurate(g[3 * H + j]);
  const float c_old = c_zero ? 0.f : c[e];
  const float cn = fmaf(gf, c_old, gi * gg);
  const float hn = go * tanhf(cn);
  c[e] = cn;
  h_out[m * h_out_ld + j] = hn;
  a_cat[m * (H + F) + j] = hn;
  if (next_row >= 0 && j < F) a_cat[m * (H + F) + H + j] = inputs[m * x_inst_ld + (int64_t)next_row * F + j];
}

// Pointer step k for one instance per warp (N <= 32, a.enc_inst_ld = L * H): lane j forms d_j with the H-generic dot
// and pointer_finish_lanes finishes candidate j.
__global__ void __launch_bounds__(256) anyh_pointer_kernel(const PointerStepArgs a, int k, int H, const float* __restrict__ q,
                                                           int64_t q_ld, const float* __restrict__ inputs, int F,
                                                           float* __restrict__ a_cat, int feed_next) {
  const int lane = threadIdx.x & 31;
  const int64_t b = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (b >= a.n) return;
  const int N = a.N;
  const float* qb = q + b * q_ld;
  const float* rows = a.enc_out + b * a.enc_inst_ld + (int64_t)k * N * H;
  float d = 0.f;
  for (int j = 0; j < N; ++j) {
    const float* row = rows + (int64_t)j * H;
    float s = 0.f;
    for (int u = lane; u < H; u += 32) s = fmaf(row[u], qb[u], s);
    s = warp_sum(s);                                    // xor butterfly: every lane holds the same sum
    if (lane == j) d = s;
  }
  const float lat = a.latent_win && lane < N ? a.latent_win[b * a.L + (int64_t)k * N + lane] : 0.f;
  const int fed = pointer_finish_lanes<32>(a, k, b, true, d, lat, lane, N <= 8 ? 4 : 16);
  if (feed_next && lane < F) a_cat[b * (H + F) + H + lane] = inputs[(b * a.L + fed) * (int64_t)F + lane];
}

// prev_logits materialised (modelPN.py:213-214,239): warp = (instance b, position l), loop over the K steps
__global__ void __launch_bounds__(256) anyh_full_logits_kernel(
    const float* __restrict__ enc_out, const float* __restrict__ dec_h, const int32_t* __restrict__ idx, int use_tanh,
    float C, int64_t n, int L, int H, int K, float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t w = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (w >= n * L) return;
  const int64_t b = w / L;
  const int l = (int)(w % L);
  const float* row = enc_out + w * (int64_t)H;
  bool visited = false;
  for (int k = 0; k < K; ++k) {
    const float* qb = dec_h + (b * K + k) * (int64_t)H;
    float s = 0.f;
    for (int u = lane; u < H; u += 32) s = fmaf(row[u], qb[u], s);
    s = warp_sum(s);
    if (lane == 0) out[((int64_t)k * n + b) * L + l] = visited ? -INFINITY : (use_tanh ? C * tanhf(s) : s);
    if (idx[(int64_t)k * n + b] == l) visited = true;   // masked from the next step on
  }
}

}  // namespace
}  // namespace gnnpn

using namespace gnnpn;

extern "C" {

size_t gnnpn_pn_anyh_workspace_floats(int64_t n, int hidden, int in_features) {
  if (n < 0 || hidden < 1 || in_features < 1) return 0;
  return (size_t)n * (hidden + in_features) + (size_t)n * 4 * hidden;      // A_cat + gate pre-activations
}

int gnnpn_lstm_encode_anyh_f32(const float* inputs, int64_t n, int L, int in_features, int hidden, const float* w_cat,
                               const float* bias, float* enc_out, float* c_state, float* workspace,
                               size_t workspace_floats, void* stream) {
  GNNPN_REQUIRE(inputs && w_cat && bias && enc_out && c_state && workspace, GNNPN_ENULL);
  GNNPN_REQUIRE(hidden >= 1 && in_features >= 1 && in_features <= 32 && L >= 1 && n >= 0, GNNPN_ESHAPE);
  GNNPN_REQUIRE(workspace_floats >= gnnpn_pn_anyh_workspace_floats(n, hidden, in_features), GNNPN_EWORKSPACE);
  GNNPN_REQUIRE(n * (int64_t)hidden < (1ll << 31) * 256, GNNPN_ERANGE);
  if (n == 0) return GNNPN_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const int H = hidden, F = in_features, W = H + F;
  float* a_cat = workspace;
  float* gates = workspace + (size_t)n * W;
  const int64_t x_ld = (int64_t)L * F;
  int rc;
  anyh_init_kernel<<<init_grid(n * W), 256, 0, st>>>(a_cat, n, H, F, nullptr, 0,
                                                                                             inputs, x_ld, 0);
  if ((rc = after_launch())) return rc;
  for (int t = 0; t < L; ++t) {
    if ((rc = launch_gemm_ffma(a_cat, W, w_cat, W, bias, nullptr, nullptr, GNNPN_ACT_NONE, gates, 4 * (int64_t)H, n, 4 * H,
                               W, st)))
      return rc;
    anyh_cell_kernel<<<(unsigned)ceil_div(n * H, 256), 256, 0, st>>>(gates, c_state, t == 0, enc_out + (int64_t)t * H,
                                                                     (int64_t)L * H, a_cat, n, H, F, inputs, x_ld,
                                                                     t + 1 < L ? t + 1 : -1);
    if ((rc = after_launch())) return rc;
  }
  return GNNPN_OK;
}

int gnnpn_pn_decode_anyh_f32(const float* inputs, const float* enc_out, float* c_state, const float* latent_win,
                             float alpha, const float* w_cat, const float* bias, const float* bias0, int use_tanh,
                             float C, int64_t n, int L, int in_features, int hidden, int K, int N, float* dec_h,
                             int32_t* idx_out, float* win_logits, float* win_probs, const int32_t* forced_idx,
                             const float* sample_uniform, float* workspace, size_t workspace_floats, void* stream) {
  GNNPN_REQUIRE(inputs && enc_out && c_state && w_cat && bias && bias0 && dec_h && idx_out && win_logits && win_probs &&
                    workspace, GNNPN_ENULL);
  GNNPN_REQUIRE(hidden >= 1 && in_features >= 1 && in_features <= 32 && K >= 1 && N >= 1 && N <= kMaxWindow &&
                    (int64_t)K * N == L && n >= 0, GNNPN_ESHAPE);
  GNNPN_REQUIRE(workspace_floats >= gnnpn_pn_anyh_workspace_floats(n, hidden, in_features), GNNPN_EWORKSPACE);
  if (n == 0) return GNNPN_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const int H = hidden, F = in_features, W = H + F;
  float* a_cat = workspace;
  float* gates = workspace + (size_t)n * W;
  int rc;
  // h(-1) = the encoder's last hidden state, no input term at step 0 (the start token lives in bias0)
  anyh_init_kernel<<<init_grid(n * W), 256, 0, st>>>(
      a_cat, n, H, F, enc_out + (int64_t)(L - 1) * H, (int64_t)L * H, nullptr, 0, -1);
  if ((rc = after_launch())) return rc;
  const PointerStepArgs pa{enc_out, (int64_t)L * H, latent_win, alpha, use_tanh, C, n, L, N, idx_out, win_logits,
                          win_probs, forced_idx, sample_uniform};
  for (int k = 0; k < K; ++k) {
    if ((rc = launch_gemm_ffma(a_cat, W, w_cat, W, k == 0 ? bias0 : bias, nullptr, nullptr, GNNPN_ACT_NONE, gates,
                               4 * (int64_t)H, n, 4 * H, W, st)))
      return rc;
    anyh_cell_kernel<<<(unsigned)ceil_div(n * H, 256), 256, 0, st>>>(gates, c_state, 0, dec_h + (int64_t)k * H,
                                                                     (int64_t)K * H, a_cat, n, H, F, nullptr, 0, -1);
    if ((rc = after_launch())) return rc;
    anyh_pointer_kernel<<<(unsigned)ceil_div(n, 8), 256, 0, st>>>(pa, k, H, dec_h + (int64_t)k * H, (int64_t)K * H, inputs,
                                                                  F, a_cat, k + 1 < K);
    if ((rc = after_launch())) return rc;
  }
  return GNNPN_OK;
}

int gnnpn_pn_full_logits_anyh_f32(const float* enc_out, const float* dec_h, const int32_t* idx, int use_tanh, float C,
                                  int64_t n, int L, int hidden, int K, float* logits_full, void* stream) {
  GNNPN_REQUIRE(enc_out && dec_h && idx && logits_full, GNNPN_ENULL);
  GNNPN_REQUIRE(hidden >= 1 && K >= 1 && L >= 1 && n >= 0, GNNPN_ESHAPE);
  GNNPN_REQUIRE(n * (int64_t)L < (1ll << 31) * 8, GNNPN_ERANGE);
  if (n == 0) return GNNPN_OK;
  anyh_full_logits_kernel<<<(unsigned)ceil_div(n * L, 8), 256, 0, (cudaStream_t)stream>>>(enc_out, dec_h, idx, use_tanh, C, n,
                                                                                         L, hidden, K, logits_full);
  return after_launch();
}

}  // extern "C"
