// Packed LSTM block layout and the per-step LSTM recurrence driver (implemented in tc_kernels.cu).
#pragma once
#include <cuda.h>
#include "lstm_step.cuh"
#include "tc_common.cuh"

namespace gnnpn {

// float offsets inside one packed LSTM block (see gnnpn_pn_packed_lstm_floats): FFMA block [kH + kXPad][kG], bias,
// start, then the fp16-split tensor-core operand blocks [4H][kKp16] halfs (hi, lo), weights pre-scaled by kW16Scale
constexpr size_t kOffBias = (size_t)(kH + kXPad) * kG;
constexpr size_t kOffStart = kOffBias + kG;
constexpr int kKp16 = kH + 64;   // [h | x | zero pad] as 5 k-blocks of 64 halfs (128-byte swizzle rows)
constexpr float kW16Scale = 16.0f;   // |w| <~ 0.06 would push the fp16 "lo" parts into subnormals; 2^4 is exact to undo
constexpr size_t kOffTc16Hi = kOffStart + kG;
constexpr size_t kOffTc16Lo = kOffTc16Hi + (size_t)kG * kKp16 / 2;
constexpr size_t kPackedFloats = kOffTc16Lo + (size_t)kG * kKp16 / 2;

// Where a raw input row is staged for the tensor-core step: columns [kH, kH + F) of the fp16 hi/lo [h | x] operand
// rows, ld halfs apart.  hi == nullptr: the FFMA step, which gathers its input row itself.
struct LstmXSlot {
  __half* hi;
  __half* lo;
  int64_t ld;
};
__device__ __forceinline__ void stage_x_f16(__half* hi, __half* lo, int64_t ld, int64_t m, int f, float v) {
  __half h, l;
  tc::split_f16(v, h, l);
  hi[m * ld + kH + f] = h;
  lo[m * ld + kH + f] = l;
}

// the tensor-core step's two ping-pong [n, kKp16] hi/lo operand buffers and their TMA descriptors
struct TcLstmPlan {
  CUtensorMap a_hi[2], a_lo[2], b_hi, b_lo;
  __half* hi[2];
  __half* lo[2];
  int64_t n;
};

// scratch of the tensor-core recurrences (per-step operands, persistent scans' cell state, column-split exchange)
size_t tc_lstm_workspace_bytes(int64_t n);

// One LSTM recurrence run one launch per step over n instances: the tcgen05 step kernel when a workspace is given
// (3xFP16 split of [h | x] kept in the workspace between steps), else the strict-fp32 FFMA step kernel.
struct LstmRecurrence {
  const float* packed;     // packed LSTM block
  const float* inputs;     // raw rows [n, L, F]
  int64_t n;
  int L, F;
  float* c;                // [n, kH] cell state, updated in place
  bool tc;
  TcLstmPlan plan;         // tc only
};
// training replay (FFMA only): the step writes its cell state to c and its post-activation gates to gates, and reads
// the previous cell state from c_in
struct LstmStepSaves {
  float* gates;            // [n, kG]
  float* c;                // [n, kH]
  const float* c_in;       // [n, kH]
};
int lstm_recurrence_init(LstmRecurrence* r, const float* packed, const float* inputs, int64_t n, int L, int F,
                         float* c_state, void* workspace, size_t workspace_bytes);
// encoder step t (from h = c = 0 at t = 0) on raw row t: h -> enc_out[:, t, :] ([n, L, kH])
int lstm_encoder_step(const LstmRecurrence& r, int t, float* enc_out, const LstmStepSaves* saves, cudaStream_t st);
// decoder step k: k = 0 starts from h = enc_out[:, L-1, :] with the start-token bias and no input; k > 0 feeds the raw
// row fed[(k-1) * n + m] (the FFMA step gathers it, the tensor-core step reads what the pointer step staged in
// lstm_decoder_x_slot(r, k - 1)).  h -> dec_h[:, k, :] ([n, K, kH])
int lstm_decoder_step(const LstmRecurrence& r, int k, const float* enc_out, float* dec_h, int K, const int32_t* fed,
                      const LstmStepSaves* saves, cudaStream_t st);
// where the pointer step after decoder step k stages the row it feeds to step k + 1
LstmXSlot lstm_decoder_x_slot(const LstmRecurrence& r, int k);

}  // namespace gnnpn
