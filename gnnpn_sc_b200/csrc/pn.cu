// Pointer-network entry points: weight packing, encoder scan, fused greedy decode and its rollouts, composition
// objective / reward and the best rollout (the dense logits are in pn_general.cu).
#include <math.h>
#include <cuda_fp16.h>
#include "lstm_step.cuh"
#include "tc_lstm.cuh"
#include "tc_seq.cuh"
#include "pointer.cuh"

namespace gnnpn {
namespace {

// ---------------------------------------------------------------------------
// weight packing (fp64 accumulate, once per model)
// ---------------------------------------------------------------------------
__device__ float folded_weight(const float* __restrict__ w_ih, const float* __restrict__ w_hh,
                               const float* __restrict__ w_e, int H, int F, int r, int k) {
  // column k of the "[h | x]" operand for torch gate row r:  k < H -> W_hh ; H <= k < H+F -> (W_ih . W_e)[:, k-H]
  if (k < H) return w_hh[(int64_t)r * H + k];
  const int f = k - H;
  if (f >= F) return 0.f;
  double s = 0.0;
  for (int i = 0; i < H; ++i) s += (double)w_ih[(int64_t)r * H + i] * (double)w_e[(int64_t)i * F + f];
  return (float)s;
}

__global__ void pack_lstm_kernel(const float* __restrict__ w_ih, const float* __restrict__ w_hh,
                                 const float* __restrict__ b_ih, const float* __restrict__ b_hh,
                                 const float* __restrict__ w_e, const float* __restrict__ b_e,
                                 const float* __restrict__ start, int H, int F, int Fpad,
                                 float* __restrict__ packed) {
  const int G = 4 * H;
  const int rows = H + Fpad + 2;  // + bias row + start row
  const int64_t ffma_total = (int64_t)rows * G;
  const int64_t tc16_total = (int64_t)G * kKp16;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < ffma_total + tc16_total;
       e += (int64_t)gridDim.x * blockDim.x) {
    if (e >= ffma_total) {                         // fp16-split tcgen05 operand: [4H][kKp16] halfs, weights x 2^4
      const int64_t t = e - ffma_total;
      const int nn = (int)(t / kKp16), k = (int)(t % kKp16);
      const int r = (nn & 3) * H + (nn >> 2);
      const float w = kW16Scale * folded_weight(w_ih, w_hh, w_e, H, F, r, k);
      const __half hi = __float2half_rn(w);
      __half* base = reinterpret_cast<__half*>(packed + ffma_total);
      base[t] = hi;
      base[tc16_total + t] = __float2half_rn(w - __half2float(hi));
      continue;
    }
    const int k = (int)(e / G), nn = (int)(e % G);
    const int j = nn >> 2, g = nn & 3;
    const int r = g * H + j;                       // torch row: gate-major
    float out = 0.f;
    if (k < H + Fpad) {
      out = folded_weight(w_ih, w_hh, w_e, H, F, r, k);
    } else if (k == H + Fpad) {                    // bias = b_ih + b_hh + W_ih . b_e
      double s = (double)b_ih[r] + (double)b_hh[r];
      for (int i = 0; i < H; ++i) s += (double)w_ih[(int64_t)r * H + i] * (double)b_e[i];
      out = (float)s;
    } else {                                       // start = b_ih + b_hh + W_ih . start_input
      if (start) {
        double s = (double)b_ih[r] + (double)b_hh[r];
        for (int i = 0; i < H; ++i) s += (double)w_ih[(int64_t)r * H + i] * (double)start[i];
        out = (float)s;
      }
    }
    packed[e] = out;
  }
}

// ---------------------------------------------------------------------------
// pointer step (Dot attention, pointer.cuh): one warp per instance
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) pointer_step_dot_kernel(
    const PointerStepArgs pa, int k, const float* __restrict__ q, int64_t q_ld, const float* __restrict__ inputs, int F,
    const LstmXSlot x_next) {
  const int lane = threadIdx.x & 31;
  const int64_t b = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (b >= pa.n) return;
  const float4* qp = reinterpret_cast<const float4*>(q + b * q_ld);
  const float4 q0 = __ldg(qp + 2 * lane), q1 = __ldg(qp + 2 * lane + 1);     // the lane's floats [8*lane, 8*lane+8)
  const int fed = pointer_step_warp(pa, k, b, q0, q1, lane);
  if (x_next.hi && lane < F)     // tensor-core path: the fed candidate's raw row is the next step's input
    stage_x_f16(x_next.hi, x_next.lo, x_next.ld, b, lane, __ldg(inputs + (b * pa.L + fed) * (int64_t)F + lane));
}

// The K steps of a per-step decode: before_step(k) (the decoder's LSTM step, or nothing), then the pointer step on the
// query dec_h[:, k].  With a tensor-core recurrence r the pointer step stages the fed row as r's next input.
template <class BeforeStep>
int launch_pointer_steps(const PointerStepArgs& pa, int K, const float* dec_h, const float* inputs, int F,
                         const LstmRecurrence* r, cudaStream_t st, BeforeStep before_step) {
  for (int k = 0; k < K; ++k) {
    int rc = before_step(k);
    if (rc) return rc;
    pointer_step_dot_kernel<<<(unsigned)ceil_div(pa.n, 8), 256, 0, st>>>(
        pa, k, dec_h + (int64_t)k * kH, (int64_t)K * kH, inputs, F, r ? lstm_decoder_x_slot(*r, k) : LstmXSlot{nullptr, nullptr, 0});
    if ((rc = after_launch())) return rc;
  }
  return GNNPN_OK;
}

// ---------------------------------------------------------------------------
// composition objective (calc / reward): one thread per instance, fp32 sequential products
// and numpy's float32 pairwise-sum order for sum(q0) so results are bit-identical to the CPU path
// ---------------------------------------------------------------------------
constexpr int kMaxTasks = 512;

struct Reward {
  int viol;        // violated global constraints (the "Low" reward)
  float obj;       // objFunc
  float high;      // float32(round(viol + obj, 5)) (the "High" reward)
};
// the objective of instance b's picks idx[k * n + b]
__device__ __forceinline__ Reward composition_reward(const float* __restrict__ inputs, const int32_t* __restrict__ idx,
                                                     int64_t n, int64_t b, int L, int F, int K, int tag) {
  float q0s[kMaxTasks];
  float prod[2] = {1.f, 1.f};
  float min_q1 = INFINITY;
  int used = 0;
  float lo[2] = {0, 0}, hi[2] = {0, 0};
  for (int k = 0; k < K; ++k) {
    const float* row = inputs + (b * L + idx[(int64_t)k * n + b]) * (int64_t)F + tag;
    const float q0 = row[0], q1 = row[1];
    q0s[k] = q0;
    used += q0 > 0.f;
    min_q1 = fminf(min_q1, q1);
    prod[0] = k == 0 ? row[2] : __fmul_rn(prod[0], row[2]);
    prod[1] = k == 0 ? row[3] : __fmul_rn(prod[1], row[3]);
    if (k == 0) { lo[0] = row[4]; hi[0] = row[5]; lo[1] = row[6]; hi[1] = row[7]; }
  }
  int viol = 0;
  for (int i = 0; i < 2; ++i) viol += (prod[i] < lo[i] || prod[i] > hi[i]) ? 1 : 0;
  const float s = numpy_sum<kMaxTasks>(q0s, K);
  float obj = __fdiv_rn(s, (float)used);
  obj = __fadd_rn(obj, 1.0f);
  obj = __fsub_rn(obj, min_q1);
  obj = __fdiv_rn(obj, 2.0f);
  const double v = (double)viol + (double)obj;            // python: round(violate + objFunc, 5)
  return Reward{viol, obj, (float)(rint(v * 1e5) / 1e5)};
}

__global__ void reward_kernel(const float* __restrict__ inputs, const int32_t* __restrict__ idx, int64_t n,
                              int L, int F, int K, int tag, int32_t* __restrict__ viol_out,
                              float* __restrict__ obj_out, float* __restrict__ rew_out) {
  const int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (b >= n) return;
  const Reward r = composition_reward(inputs, idx, n, b, L, F, K, tag);
  if (viol_out) viol_out[b] = r.viol;
  if (obj_out) obj_out[b] = r.obj;
  if (rew_out) rew_out[b] = r.high;
}

// Best of R rollouts idx [R, K, n] per instance: the lowest reward of `level` (0: Low, 1: High), the lowest rollout on a tie
__global__ void best_rollout_kernel(const float* __restrict__ inputs, const int32_t* __restrict__ idx, int64_t n, int L,
                                    int F, int K, int tag, int level, int R, int32_t* __restrict__ best_idx,
                                    float* __restrict__ best_reward, int32_t* __restrict__ best_rollout,
                                    float* __restrict__ rollout_rewards) {
  const int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (b >= n) return;
  float best = 0.f;
  int best_r = 0;
  for (int r = 0; r < R; ++r) {
    const Reward rw = composition_reward(inputs, idx + (int64_t)r * K * n, n, b, L, F, K, tag);
    const float s = level ? rw.high : (float)rw.viol;
    if (rollout_rewards) rollout_rewards[(int64_t)r * n + b] = s;
    if (r == 0 || s < best) { best = s; best_r = r; }
  }
  const int32_t* src = idx + (int64_t)best_r * K * n;
  for (int k = 0; k < K; ++k) best_idx[(int64_t)k * n + b] = src[(int64_t)k * n + b];
  best_reward[b] = best;
  best_rollout[b] = best_r;
}

// raw input range check: *flag |= 1 if any value is NaN / inf or has |x| >= limit
__global__ void check_inputs_kernel(const float* __restrict__ x, int64_t count, float limit, int32_t* __restrict__ flag) {
  bool bad = false;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x)
    bad |= !(fabsf(__ldg(x + i)) < limit);
  if (bad) atomicOr(flag, 1);
}

// blocked encodings -> row-major [n, L, kH]; one thread per float4 of the output (coalesced writes)
__global__ void enc_unblock_kernel(const float* __restrict__ blk, int64_t n, int L, float* __restrict__ out) {
  const int64_t total = n * L * (kH / 4);
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int c4 = (int)(e % (kH / 4));
    const int64_t bl = e / (kH / 4);
    const int l = (int)(bl % L);
    const int64_t b = bl / L;
    const int u = c4 * 4, nt = u >> 5, g = (u >> 3) & 3;
    const int64_t src = ((((b >> 7) * L + l) * 8 + nt) * 4 + g) * 1024 + (b & 127) * 8 + (u & 7);
    reinterpret_cast<float4*>(out)[e] = __ldg(reinterpret_cast<const float4*>(blk + src));
  }
}

// The kernels of gnnpn_pn_train_forward_f32: of the scans only the column-split scan has the saves, whatever the
// "persistent" option says; it runs when a workspace is given and it takes the batch (the reference trains with 128).
// Otherwise forced picks are replayed on the strict-fp32 FFMA per-step kernels (kStep); free-running is kUnsupported.
ScanPlan plan_train_forward(int64_t n, int F, int N, bool has_workspace, bool forced) {
  ScanPlan p = plan_scans(n, F, N, GNNPN_ENC_ROWMAJOR, has_workspace, 1, 3);
  if (p.enc.kind != ScanKind::kColsplit) p.enc = p.dec = {forced ? ScanKind::kStep : ScanKind::kUnsupported, 0};
  return p;
}

}  // namespace
}  // namespace gnnpn

using namespace gnnpn;

extern "C" {

size_t gnnpn_pn_packed_lstm_floats(int hidden, int in_features) {
  (void)in_features;
  return hidden == kH ? kPackedFloats : 0;
}

size_t gnnpn_pn_workspace_bytes(int64_t n, int hidden) {
  return hidden == kH && n >= 0 ? tc_lstm_workspace_bytes(n) : 0;
}

int gnnpn_pn_pack_lstm_f32(const float* w_ih, const float* w_hh, const float* b_ih, const float* b_hh,
                           const float* w_embed, const float* b_embed, const float* start_input,
                           int hidden, int in_features, float* packed, void* stream) {
  GNNPN_REQUIRE(w_ih && w_hh && b_ih && b_hh && w_embed && b_embed && packed, GNNPN_ENULL);
  GNNPN_REQUIRE(hidden == kH && in_features >= 1 && in_features <= kXPad, GNNPN_ESHAPE);
  pack_lstm_kernel<<<kNumSMs * 4, 256, 0, (cudaStream_t)stream>>>(w_ih, w_hh, b_ih, b_hh, w_embed, b_embed,
                                                                  start_input, hidden, in_features, kXPad, packed);
  return after_launch();
}

float gnnpn_pn_input_limit(void) { return 65504.0f; }

int gnnpn_pn_check_inputs_f32(const float* inputs, int64_t count, int32_t* flag, void* stream) {
  GNNPN_REQUIRE(inputs && flag, GNNPN_ENULL);
  GNNPN_REQUIRE(count >= 0, GNNPN_ESHAPE);
  if (count == 0) return GNNPN_OK;
  const int64_t blocks = ceil_div(count, 256 * 8);
  check_inputs_kernel<<<(unsigned)(blocks < 8 * kNumSMs ? blocks : 8 * kNumSMs), 256, 0, (cudaStream_t)stream>>>(
      inputs, count, gnnpn_pn_input_limit(), flag);
  return after_launch();
}

int gnnpn_pn_enc_layout(int64_t n, int L, int in_features, int K, int N, int has_workspace) {
  (void)L; (void)K;
  return plan_scans(n, in_features, N, GNNPN_ENC_ROWMAJOR, has_workspace != 0).layout;
}

size_t gnnpn_pn_enc_out_floats(int64_t n, int L, int hidden, int layout) {
  if (n < 0 || L < 1 || hidden != kH) return 0;
  const int64_t rows = layout == GNNPN_ENC_BLOCKED128 ? (n + 127) / 128 * 128 : n;
  return (size_t)rows * L * kH;
}

int gnnpn_pn_enc_to_rowmajor_f32(const float* enc_blocked, int64_t n, int L, int hidden, float* enc_out, void* stream) {
  GNNPN_REQUIRE(enc_blocked && enc_out, GNNPN_ENULL);
  GNNPN_REQUIRE(hidden == kH && L >= 1 && n >= 0, GNNPN_ESHAPE);
  GNNPN_REQUIRE(aligned16(enc_blocked) && aligned16(enc_out), GNNPN_EALIGN);
  if (n == 0) return GNNPN_OK;
  enc_unblock_kernel<<<kNumSMs * 8, 256, 0, (cudaStream_t)stream>>>(enc_blocked, n, L, enc_out);
  return after_launch();
}

int gnnpn_lstm_encode_f32(const float* inputs, int64_t n, int L, int in_features, int hidden,
                          const float* packed, float* enc_out, float* c_state, void* workspace,
                          size_t workspace_bytes, int enc_layout, void* stream) {
  GNNPN_REQUIRE(enc_layout == GNNPN_ENC_ROWMAJOR || enc_layout == GNNPN_ENC_BLOCKED128, GNNPN_ESHAPE);
  GNNPN_REQUIRE(inputs && packed && enc_out && c_state, GNNPN_ENULL);
  GNNPN_REQUIRE(hidden == kH && in_features >= 1 && in_features <= kXPad && L >= 1 && n >= 0, GNNPN_ESHAPE);
  GNNPN_REQUIRE(n < (1ll << 31), GNNPN_ERANGE);
  GNNPN_REQUIRE(aligned16(enc_out) && aligned16(c_state) && aligned16(packed), GNNPN_EALIGN);
  if (n == 0) return GNNPN_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const ScanChoice scan = plan_scans(n, in_features, /*N: no window*/ 0, enc_layout, workspace != nullptr).enc;
  if (scan.kind == ScanKind::kStep) {
    GNNPN_REQUIRE(enc_layout == GNNPN_ENC_ROWMAJOR, GNNPN_EUNSUPPORTED);
    LstmRecurrence r;
    int rc = lstm_recurrence_init(&r, packed, inputs, n, L, in_features, c_state, workspace, workspace_bytes);
    for (int t = 0; t < L && !rc; ++t) rc = lstm_encoder_step(r, t, enc_out, nullptr, st);
    return rc;
  }
  // ---- persistent tcgen05 scan: one launch for all L steps
  GNNPN_REQUIRE(aligned32(enc_out) && aligned32(c_state), GNNPN_EALIGN);
  GNNPN_REQUIRE(workspace_bytes >= tc_lstm_workspace_bytes(n), GNNPN_EWORKSPACE);
  SeqEncodeArgs sa{inputs, n, L, in_features, packed, enc_out, c_state, align_ws<float>(workspace)};
  if (scan.kind == ScanKind::kColsplit) return tc_colsplit_encode(sa, scan.variant, st);
  return tc_seq_encode(sa, scan.variant, st);
}

int gnnpn_pn_decode_greedy_f32(const float* inputs, const float* enc_out, float* c_state,
                               const float* latent_win, float alpha, const float* packed,
                               int attention, const float* att_params, int use_tanh, float C,
                               int64_t n, int L, int in_features, int hidden, int K, int N,
                               float* dec_h, int32_t* idx_out, float* win_logits, float* win_probs,
                               const int32_t* forced_idx, const float* sample_uniform, void* workspace,
                               size_t workspace_bytes, int enc_layout, void* stream) {
  GNNPN_REQUIRE(enc_layout == GNNPN_ENC_ROWMAJOR || enc_layout == GNNPN_ENC_BLOCKED128, GNNPN_ESHAPE);
  GNNPN_REQUIRE(inputs && enc_out && c_state && packed && idx_out && win_logits && win_probs, GNNPN_ENULL);
  GNNPN_REQUIRE(dec_h || enc_layout == GNNPN_ENC_BLOCKED128, GNNPN_ENULL);   // optional only in the fused decoder
  GNNPN_REQUIRE(hidden == kH && in_features >= 1 && in_features <= kXPad, GNNPN_ESHAPE);
  GNNPN_REQUIRE(K >= 1 && N >= 1 && N <= kMaxWindow && (int64_t)K * N == L, GNNPN_ESHAPE);
  GNNPN_REQUIRE(n >= 0 && n < (1ll << 31), GNNPN_ERANGE);
  GNNPN_REQUIRE(attention == GNNPN_ATT_DOT, GNNPN_EUNSUPPORTED);
  (void)att_params;
  GNNPN_REQUIRE(aligned16(enc_out) && aligned16(dec_h) && aligned16(c_state) && aligned16(packed), GNNPN_EALIGN);   // NULL dec_h passes
  if (n == 0) return GNNPN_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const ScanChoice scan = plan_scans(n, in_features, N, enc_layout, workspace != nullptr).dec;
  if (scan.kind == ScanKind::kStep) {
    GNNPN_REQUIRE(enc_layout == GNNPN_ENC_ROWMAJOR, GNNPN_EUNSUPPORTED);
    LstmRecurrence r;
    const int rc = lstm_recurrence_init(&r, packed, inputs, n, L, in_features, c_state, workspace, workspace_bytes);
    if (rc) return rc;
    const PointerStepArgs pa = pointer_step_args(enc_out, latent_win, alpha, use_tanh, C, n, L, N, idx_out, win_logits,
                                                 win_probs, forced_idx, sample_uniform);
    return launch_pointer_steps(pa, K, dec_h, inputs, in_features, &r, st, [&](int k) {
      return lstm_decoder_step(r, k, enc_out, dec_h, K, forced_idx ? forced_idx : idx_out, nullptr, st);
    });
  }
  GNNPN_REQUIRE(aligned32(enc_out) && aligned32(c_state) && aligned32(dec_h), GNNPN_EALIGN);
  GNNPN_REQUIRE(workspace_bytes >= tc_lstm_workspace_bytes(n), GNNPN_EWORKSPACE);
  SeqDecodeArgs sa{inputs, enc_out, c_state, latent_win, alpha, packed, use_tanh, C, n, L, in_features, K, N,
                   dec_h, idx_out, win_logits, win_probs, forced_idx, sample_uniform, align_ws<float>(workspace)};
  if (scan.kind == ScanKind::kColsplit) return tc_colsplit_decode(sa, scan.variant, st);
  return scan.kind == ScanKind::kPair ? tc_seq_decode(sa, scan.variant, st) : GNNPN_EUNSUPPORTED;
}

size_t gnnpn_pn_rollouts_workspace_bytes(int64_t n, int hidden, int rollouts) {
  return hidden == kH && n >= 0 && rollouts >= 1 ? tc_seq_rollouts_workspace_bytes(n, rollouts) : 0;
}

// The decode of gnnpn_pn_decode_greedy_f32 `rollouts` times per instance in one launch of the persistent scan that
// plan_scans picks for the n * rollouts rows; the encodings, c_state and latent are read by every rollout.
int gnnpn_pn_decode_rollouts_f32(const float* inputs, const float* enc_out, const float* c_state,
                                 const float* latent_win, float alpha, const float* packed,
                                 int attention, const float* att_params, int use_tanh, float C,
                                 int64_t n, int L, int in_features, int hidden, int K, int N,
                                 float* dec_h, int32_t* idx_out, float* win_logits, float* win_probs,
                                 const float* sample_uniform, void* workspace, size_t workspace_bytes,
                                 int enc_layout, int rollouts, void* stream) {
  GNNPN_REQUIRE(enc_layout == GNNPN_ENC_ROWMAJOR || enc_layout == GNNPN_ENC_BLOCKED128, GNNPN_ESHAPE);
  GNNPN_REQUIRE(rollouts >= 1 && hidden == kH && in_features >= 1 && in_features <= 8, GNNPN_ESHAPE);
  GNNPN_REQUIRE(K >= 1 && N >= 1 && N <= kMaxWindow && (int64_t)K * N == L, GNNPN_ESHAPE);
  GNNPN_REQUIRE(inputs && enc_out && c_state && packed && idx_out && win_logits && win_probs, GNNPN_ENULL);
  GNNPN_REQUIRE(dec_h || enc_layout == GNNPN_ENC_BLOCKED128, GNNPN_ENULL);   // optional only in the fused decoder
  GNNPN_REQUIRE(sample_uniform || rollouts == 1, GNNPN_ENULL);
  GNNPN_REQUIRE(n >= 0 && n * rollouts < (1ll << 31), GNNPN_ERANGE);
  GNNPN_REQUIRE(attention == GNNPN_ATT_DOT, GNNPN_EUNSUPPORTED);
  (void)att_params;
  GNNPN_REQUIRE(aligned32(enc_out) && aligned32(dec_h) && aligned32(c_state) && aligned16(packed), GNNPN_EALIGN);
  if (n == 0) return GNNPN_OK;
  const ScanChoice scan = plan_scans(n, in_features, N, enc_layout, workspace != nullptr, rollouts).dec;
  GNNPN_REQUIRE(scan.kind == ScanKind::kPair || scan.kind == ScanKind::kColsplit, GNNPN_EUNSUPPORTED);
  GNNPN_REQUIRE(workspace_bytes >= tc_seq_rollouts_workspace_bytes(n, rollouts), GNNPN_EWORKSPACE);
  SeqDecodeArgs sa{inputs, enc_out, const_cast<float*>(c_state), latent_win, alpha, packed, use_tanh, C, n, L,
                   in_features, K, N, dec_h, idx_out, win_logits, win_probs, nullptr, nullptr, align_ws<float>(workspace)};
  sa.rollouts = rollouts;                    // c_state is read, not written
  sa.sampled = sample_uniform;
  cudaStream_t st = (cudaStream_t)stream;
  return scan.kind == ScanKind::kColsplit ? tc_colsplit_decode(sa, scan.variant, st) : tc_seq_decode(sa, scan.variant, st);
}

size_t gnnpn_pn_train_forward_workspace_bytes(int64_t n, int L, int in_features, int hidden, int K, int N) {
  (void)L; (void)K;
  if (hidden != kH || n < 0) return 0;
  const ScanPlan plan = plan_train_forward(n, in_features, N, true, false);
  return plan.enc.kind == ScanKind::kColsplit ? tc_lstm_workspace_bytes(n) : 0;
}

// Differentiable replay, forward half (see pn_train.cu): the decode, saving the post-activation gates and the cell state
// of every step for the backward pass, on the kernels plan_train_forward picks.
int gnnpn_pn_train_forward_f32(const float* inputs, const float* packed_enc, const float* packed_dec,
                               const int32_t* forced_idx, const float* sample_uniform, const float* latent_win,
                               float alpha, int use_tanh, float C, int64_t n, int L, int in_features, int hidden, int K,
                               int N, float* enc_out, float* gates_e, float* c_e, float* dec_h, float* gates_d,
                               float* c_d, float* win_logits, float* win_probs, int32_t* idx_out, void* workspace,
                               size_t workspace_bytes, void* stream) {
  GNNPN_REQUIRE(inputs && packed_enc && packed_dec && enc_out && gates_e && c_e && dec_h && gates_d && c_d && win_logits &&
                    win_probs && idx_out, GNNPN_ENULL);
  GNNPN_REQUIRE(hidden == kH && in_features >= 1 && in_features <= 8 && K >= 1 && N >= 1 && N <= kMaxWindow &&
                    (int64_t)K * N == L && n >= 0 && n < (1ll << 31), GNNPN_ESHAPE);
  GNNPN_REQUIRE(aligned16(enc_out) && aligned16(dec_h) && aligned16(gates_e) && aligned16(gates_d), GNNPN_EALIGN);
  const ScanPlan plan = plan_train_forward(n, in_features, N, workspace != nullptr, forced_idx != nullptr);
  GNNPN_REQUIRE(plan.enc.kind != ScanKind::kUnsupported, GNNPN_EUNSUPPORTED);
  if (plan.enc.kind == ScanKind::kColsplit) {
    GNNPN_REQUIRE(aligned16(c_e) && aligned16(c_d), GNNPN_EALIGN);
    GNNPN_REQUIRE(workspace_bytes >= tc_lstm_workspace_bytes(n), GNNPN_EWORKSPACE);
  }
  if (n == 0) return GNNPN_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const size_t nh = (size_t)n * kH;
  if (plan.enc.kind == ScanKind::kStep) {
    // strict-fp32 FFMA steps + pointer steps, teacher-forced on forced_idx
    LstmRecurrence r;
    int rc = lstm_recurrence_init(&r, packed_enc, inputs, n, L, in_features, nullptr, nullptr, 0);
    for (int t = 0; t < L && !rc; ++t) {
      const LstmStepSaves sv{gates_e + t * n * kG, c_e + t * nh, t == 0 ? nullptr : c_e + (t - 1) * nh};
      rc = lstm_encoder_step(r, t, enc_out, &sv, st);
    }
    if (rc || (rc = lstm_recurrence_init(&r, packed_dec, inputs, n, L, in_features, nullptr, nullptr, 0))) return rc;
    const PointerStepArgs pa = pointer_step_args(enc_out, latent_win, alpha, use_tanh, C, n, L, N, idx_out, win_logits,
                                                 win_probs, forced_idx, nullptr);
    return launch_pointer_steps(pa, K, dec_h, inputs, in_features, &r, st, [&](int k) {
      const LstmStepSaves sv{gates_d + k * n * kG, c_d + k * nh, k == 0 ? c_e + (L - 1) * nh : c_d + (k - 1) * nh};
      return lstm_decoder_step(r, k, enc_out, dec_h, K, forced_idx, &sv, st);
    });
  }
  // column-split scans with saves, free-running or teacher-forced
  float* scr = align_ws<float>(workspace);
  float* c_last_e = c_e + (size_t)(L - 1) * nh;          // the encoder's final cell state = its last save
  float* c_last_d = c_d + (size_t)(K - 1) * nh;          // decoder: in (copy of c_last_e) / out (= its last save)
  SeqEncodeArgs ea{inputs, n, L, in_features, packed_enc, enc_out, c_last_e, scr};
  ea.save_gates = gates_e; ea.save_c = c_e;
  int rc = tc_colsplit_encode(ea, plan.enc.variant, st);
  if (rc) return rc;
  cudaError_t ce = cudaMemcpyAsync(c_last_d, c_last_e, nh * sizeof(float), cudaMemcpyDeviceToDevice, st);
  if (ce != cudaSuccess) return (int)ce;
  SeqDecodeArgs da{inputs, enc_out, c_last_d, latent_win, alpha, packed_dec, use_tanh, C, n, L, in_features, K, N, dec_h,
                   idx_out, win_logits, win_probs, forced_idx, sample_uniform, scr};
  da.save_gates = gates_d; da.save_c = c_d;
  return tc_colsplit_decode(da, plan.dec.variant, st);
}

// The attention of the decode loop alone (modelPN.py:213-228 restricted to the windows): for given decoder states
// dec_h [n, K, H] every step's window logits / probabilities / first-max picks.  One launch of the stand-alone pointer
// kernel per step; reads every encoding row exactly once.  Used to re-derive window logits for saved states and as the
// attention-only roofline point of bench.py (no LSTM step in the launches).
int gnnpn_pn_attention_windows_f32(const float* enc_out, const float* dec_h, const float* latent_win, float alpha,
                                   int use_tanh, float C, int64_t n, int L, int hidden, int K, int N, int32_t* idx_out,
                                   float* win_logits, float* win_probs, void* stream) {
  GNNPN_REQUIRE(enc_out && dec_h && idx_out && win_logits && win_probs, GNNPN_ENULL);
  GNNPN_REQUIRE(hidden == kH && K >= 1 && N >= 1 && N <= kMaxWindow && (int64_t)K * N == L && n >= 0, GNNPN_ESHAPE);
  GNNPN_REQUIRE(aligned16(enc_out) && aligned16(dec_h), GNNPN_EALIGN);
  if (n == 0) return GNNPN_OK;
  const PointerStepArgs pa = pointer_step_args(enc_out, latent_win, alpha, use_tanh, C, n, L, N, idx_out, win_logits,
                                               win_probs, nullptr, nullptr);
  return launch_pointer_steps(pa, K, dec_h, nullptr, 0, nullptr, (cudaStream_t)stream, [](int) { return GNNPN_OK; });
}

int gnnpn_pn_reward_f32(const float* inputs, const int32_t* idx, int64_t n, int L, int in_features,
                        int K, int tag, int32_t* viol_out, float* obj_out, float* reward_high_out,
                        void* stream) {
  GNNPN_REQUIRE(inputs && idx, GNNPN_ENULL);
  GNNPN_REQUIRE(K >= 1 && K <= kMaxTasks && (tag == 0 || tag == 1) && in_features >= tag + 8, GNNPN_ESHAPE);
  if (n == 0) return GNNPN_OK;
  reward_kernel<<<(unsigned)ceil_div(n, 128), 128, 0, (cudaStream_t)stream>>>(
      inputs, idx, n, L, in_features, K, tag, viol_out, obj_out, reward_high_out);
  return after_launch();
}

int gnnpn_pn_best_rollout_f32(const float* inputs, const int32_t* idx, int64_t n, int L, int in_features, int K, int tag,
                              int level, int rollouts, int32_t* best_idx, float* best_reward, int32_t* best_rollout,
                              float* rollout_rewards, void* stream) {
  GNNPN_REQUIRE(rollouts >= 1 && (level == 0 || level == 1), GNNPN_ESHAPE);
  GNNPN_REQUIRE(K >= 1 && K <= kMaxTasks && (tag == 0 || tag == 1) && in_features >= tag + 8, GNNPN_ESHAPE);
  GNNPN_REQUIRE(inputs && idx && best_idx && best_reward && best_rollout, GNNPN_ENULL);
  GNNPN_REQUIRE(n >= 0, GNNPN_ESHAPE);
  if (n == 0) return GNNPN_OK;
  best_rollout_kernel<<<(unsigned)ceil_div(n, 128), 128, 0, (cudaStream_t)stream>>>(
      inputs, idx, n, L, in_features, K, tag, level, rollouts, best_idx, best_reward, best_rollout, rollout_rewards);
  return after_launch();
}

}  // extern "C"
