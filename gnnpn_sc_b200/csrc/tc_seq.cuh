// Host-side interface of the persistent tcgen05 LSTM sequence kernels: the CTA-pair scan (tc_seq.cu), the column-split
// cluster scan (tc_colsplit.cu) and which of them runs a batch (tc_seq.cu).
//
// One launch runs a whole LSTM scan (encoder: L steps; decoder: K steps with the pointer step fused
// between them).  A CTA owns 128 composition instances for the whole scan; the recurrence is CTA-local
// (h never leaves the SM between steps), so there is no grid-wide synchronisation.
#pragma once
#include <cuda.h>
#include "lstm_step.cuh"
#include "tc_lstm.cuh"

namespace gnnpn {

// ---- which kernel runs a recurrence (tc_seq.cu) -------------------------------------------------------------------
enum class ScanKind {
  kStep,          // one launch per step (lstm_recurrence_*)
  kPair,          // CTA-pair scan lstm_seq_kernel<DEC, NR>
  kColsplit,      // column-split cluster scan lstm_colsplit_kernel<DEC, G>
  kUnsupported,   // blocked encodings with a window the fused decoder cannot hold (N > 10); a free-running forward with
                  // saves outside the column-split scan (pn.cu)
};
struct ScanChoice {
  ScanKind kind;
  int variant;    // kPair: NR (encoder 0 row-major / 1 blocked; decoder 0 / 5 / 8 / 10); kColsplit: G (1 / 2 / 3)
};
struct ScanPlan {
  ScanChoice enc, dec;
  int layout;     // the encodings layout gnnpn_pn_enc_layout reports for the batch
};
// Encoder and decoder choice for n instances with F input columns and windows of N candidates, whose encodings are in
// `layout`, under the current "scan" and "scan_groups" options and the "persistent" bits (-1: the option); the decoder of
// a rollout launch runs `rollouts` rows per instance.  A step choice with blocked encodings is GNNPN_EUNSUPPORTED for
// the caller.
ScanPlan plan_scans(int64_t n, int F, int N, int layout, bool has_workspace, int rollouts = 1, int persistent = -1);

// ---- host launch code shared by the two scans (tc_seq.cu) ---------------------------------------------------------
// The packed block's fp16 hi/lo weights as TMA maps, boxes of `box_rows` gate columns: {h hi, h lo} (64 halfs,
// 128B swizzle) and {x hi, x lo} (16 halfs, 32B swizzle)
int make_weight_maps(CUtensorMap maps[4], const float* packed, int box_rows);
// "prof" option: `ctas * per_cta` zeroed device counters that the kernel adds clock64() cycles to, or nullptr when
// the option is off
int prof_alloc(unsigned ctas, int per_cta, cudaStream_t st, unsigned long long** counters);
// waits for the stream, copies the counters back and frees them (debug only); sums[i] = counter i (< 8) summed over the
// CTAs.  Returns how many CTAs wrote counter 0.
unsigned prof_collect(unsigned long long* counters, unsigned ctas, int per_cta, cudaStream_t st, double sums[8]);

// ---- the scans -----------------------------------------------------------------------------------------------------
// cell-state scratch of the persistent kernels: 128 x kH floats per CTA (blocked layout), CTAs launched in pairs
inline size_t tc_seq_scratch_floats(int64_t n) { return (size_t)((n + 255) / 256) * 256 * kH; }

struct SeqEncodeArgs {
  const float* inputs;     // [n, L, F]
  int64_t n;
  int L;
  int F;                   // <= 8
  const float* packed;     // packed LSTM block (uses the bias and the fp16 hi/lo operand blocks)
  float* enc_out;          // [n, L, kH], or the blocked layout (gnnpn_pn_enc_out_floats) for tc_seq_encode's nr = 1
  float* c_state;          // [n, kH] out
  float* c_scratch;        // the 1024-byte aligned workspace: cell-state scratch of the CTA-pair scan
                           // (tc_seq_scratch_floats(n) floats), h' exchange of the column-split scan (tc_colsplit_scratch_bytes(n))
  // training (column-split scan only): per-step saves for the BPTT, or nullptr
  float* save_gates;       // [L, n, 4H] post-activation gates, columns 4j + {i,f,g,o}
  float* save_c;           // [L, n, H] cell state after every step
};
// nr: 0 row-major, 1 blocked encodings
int tc_seq_encode(const SeqEncodeArgs& a, int nr, cudaStream_t st);

// Small-batch (latency) variant, tc_colsplit.cu: a cluster of 8 CTAs shares G groups of 128 instances and splits the
// gate columns.
int tc_colsplit_max_active_clusters();
size_t tc_colsplit_scratch_bytes(int64_t n);
int tc_colsplit_encode(const SeqEncodeArgs& a, int groups, cudaStream_t st);
struct SeqDecodeArgs;
int tc_colsplit_decode(const SeqDecodeArgs& a, int groups, cudaStream_t st);

struct SeqDecodeArgs {
  const float* inputs;     // [n, L, F]
  const float* enc_out;    // [n, L, kH], or blocked for tc_seq_decode's nr > 0
  float* c_state;          // [n, kH] in/out
  const float* latent_win; // [n, L] or nullptr
  float alpha;
  const float* packed;     // decoder block
  int use_tanh;
  float C;
  int64_t n;
  int L, F, K, N;
  float* dec_h;            // [n, K, kH]
  int32_t* idx_out;        // [K, n]
  float* win_logits;       // [n, L]
  float* win_probs;        // [n, L]
  const int32_t* forced_idx;     // [K, n] or nullptr
  const float* sample_uniform;   // [K, n] or nullptr
  float* c_scratch;              // as SeqEncodeArgs::c_scratch
  float* save_gates;             // training (column-split scan only): [K, n, 4H] post-activation gates, or nullptr
  float* save_c;                 // [K, n, H] cell state after every step, or nullptr
  // rollout launch (gnnpn_pn_decode_rollouts_f32), 0 for a plain decode: `rollouts` decodes of every instance, c_state
  // read only; dec_h [rollouts, n, K, H], idx_out [rollouts, K, n], win_logits / win_probs [rollouts, n, L]; rollout 0
  // greedy, rollout r >= 1 drawn with sampled[r-1] (sample_uniform is NULL).  The workspace c_scratch lies in is
  // tc_seq_rollouts_workspace_bytes(n, rollouts) long.
  int rollouts;
  const float* sampled;          // [rollouts-1, K, n]
};
// nr: 0 row-major encodings; 5 / 8 / 10 blocked encodings, window row capacity of the fused decoder (N <= nr)
int tc_seq_decode(const SeqDecodeArgs& a, int nr, cudaStream_t st);

// Workspace of a rollout launch: every rollout has the per-CTA scratch of a decode of n instances (the CTA-pair scan's
// cell state, the column-split scan's h' exchange), so it is sized from rollouts * n rows padded to whole pair blocks.
inline size_t tc_seq_rollouts_workspace_bytes(int64_t n, int rollouts) {
  return tc_lstm_workspace_bytes(rollouts * ((n + 255) / 256) * 256);
}

}  // namespace gnnpn
