/*
 * gnnpn_b200.h -- C ABI of libgnnpn_b200.so: the B200 (sm_100a) hot path of GNNPN-SC.
 *
 * The reference (wangxiaohit/GNNPN-SC) is pure Python and has no FFI of its own;
 * each entry point below names the reference interface it replaces (file:line in
 * the reference tree) -- these are the calls a maintainer binds with ctypes from
 * the reference's src/models modules (see INTEGRATION.md).
 *
 * Conventions (SURVEY 8b)
 *  - every pointer is a DEVICE pointer unless the name ends in _host;
 *  - tensors are caller-allocated, row-major, fp32 / int32 / int64 as declared;
 *    the library never allocates, frees or retains a pointer past return;
 *    scratch is sized by the matching *_workspace_bytes() query;
 *  - `stream` is a cudaStream_t passed as void*; all work is enqueued on it and
 *    the call returns without synchronising (except *_host entry points);
 *  - return 0 on success, a negative GNNPN_E* for an argument error detected
 *    before any launch, or a positive cudaError_t from the launch.  Nothing
 *    throws across the ABI.  There is no CPU fallback.
 */
#ifndef GNNPN_B200_H_
#define GNNPN_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GNNPN_ABI_VERSION 12

#if defined(__GNUC__)
#define GNNPN_API __attribute__((visibility("default")))
#else
#define GNNPN_API
#endif

enum {
  GNNPN_OK = 0,
  GNNPN_ENULL = -1,      /* required pointer is NULL */
  GNNPN_ESHAPE = -2,     /* unsupported size (e.g. hidden_size != 256) */
  GNNPN_EALIGN = -3,     /* pointer / leading dimension not 16-byte aligned */
  GNNPN_EWORKSPACE = -4, /* workspace too small */
  GNNPN_ERANGE = -5,     /* size exceeds the int32 index range used internally */
  GNNPN_EUNSUPPORTED = -6
};

enum { GNNPN_ATT_DOT = 0, GNNPN_ATT_BAHDANAU = 1 };
enum { GNNPN_ACT_NONE = 0, GNNPN_ACT_RELU = 1, GNNPN_ACT_SIGMOID = 2 };
enum { GNNPN_CSR_PLAIN = 0, GNNPN_CSR_GCN_NORM = 1 };

GNNPN_API int gnnpn_abi_version(void);
GNNPN_API const char* gnnpn_error_string(int code);
/* number of kernels this library has launched in the calling process (bench.py's gpu_launches) */
GNNPN_API uint64_t gnnpn_launch_count(void);

/* Process-wide run-time options (dispatch overrides for tests / benches / profiling; defaults need no call):
 *   "scan"         -1 auto by batch size (default) | 0 CTA-pair scan | 1 column-split cluster scan
 *   "scan_groups"   0 auto | 1 | 2 | 3 instance groups per column-split encoder cluster
 *   "persistent"    bit 0: encoder, bit 1: decoder run as one persistent launch (default 3; 0 = one launch per step)
 *   "bptt"          1: REINFORCE backward as two persistent cluster scans (default) | 0: two launches per step
 *   "prof"          1: in-kernel wait-cycle counters printed to stderr (debug; makes the call synchronous)
 * Initial values are taken once, at load time, from GNNPN_COLSPLIT / GNNPN_COLSPLIT_G / GNNPN_SEQ / GNNPN_BPTT /
 * GNNPN_SEQ_PROF.
 * Unknown name -> GNNPN_EUNSUPPORTED. */
GNNPN_API int gnnpn_set_option(const char* name, int value);
GNNPN_API int gnnpn_get_option(const char* name, int* value);

/* ---------------------------------------------------------------------------
 * Pointer network  (reference: src/models/modelPN.py)
 * ------------------------------------------------------------------------- */

/* Size in floats of one packed LSTM ("[h | x] -> 4H gates") weight block for hidden size H and
 * `in_features` raw input columns: 624,640 for H = 256.  Layout (Kp = H + 64):
 *   [ (H + 32) x 4H   k-major block for the strict-fp32 FFMA step kernel ]
 *   [ 4H bias ] [ 4H start ]
 *   [ 4H x Kp  fp16 "hi" part of 16 w, gate-column-major (K contiguous), for the tcgen05 kernels ]
 *   [ 4H x Kp  fp16 "lo" part ( = fp16(16 w - hi) ) ]   (each fp16 block is 4H * Kp / 2 floats long)
 * ABI version 8 changed this layout (version 7 also held tf32 hi/lo blocks): re-pack blocks stored by older versions,
 * e.g. the host copies passed to gnnpn_pn_greedy_low_high_host. */
GNNPN_API size_t gnnpn_pn_packed_lstm_floats(int hidden, int in_features);

/* Fold nn.Linear(F,H) `embedding2` (modelPN.py:155,190) into an nn.LSTM's input weights
 * (modelPN.py:157-158) and lay the result out for the step kernel:
 *   packed[k][4*j+g]            k <  H : W_hh[g*H+j][k]
 *   packed[H+f][4*j+g]          f <  F : sum_i W_ih[g*H+j][i] * W_e[i][f]      (fp64 accumulate)
 *   bias[4*j+g]   = b_ih + b_hh + W_ih . b_e
 *   start[4*j+g]  = b_ih + b_hh + W_ih . start_input   (decoder_start_input, modelPN.py:162,202; may be NULL)
 * Gate order i,f,g,o as in torch.  All inputs fp32 device pointers. */
GNNPN_API int gnnpn_pn_pack_lstm_f32(const float* w_ih, const float* w_hh, const float* b_ih, const float* b_hh,
                           const float* w_embed, const float* b_embed, const float* start_input,
                           int hidden, int in_features, float* packed, void* stream);

/* Layout of the encodings buffer handed from gnnpn_lstm_encode_f32 to gnnpn_pn_decode_greedy_f32.
 *   GNNPN_ENC_ROWMAJOR    fp32 [n, L, H] (what modelPN.py:191 returns; every other entry point takes this one)
 *   GNNPN_ENC_BLOCKED128  blocks of 128 instances, fp32 [ceil(n/128)][L][8 tiles][4 groups][128 instances][8] with hidden
 *                         unit = 32*tile + 8*group + i: the ownership (thread = instance, 8 units per
 *                         accumulator tile) of the persistent CTA-pair scan's epilogue.  The encoder writes it with
 *                         coalesced 128-bit stores and the decoder folds the pointer dot products into its cell
 *                         epilogue, so the window rows stream from HBM under the step's MMAs (no separate attention
 *                         phase).  Only valid for the pair (encode, decode_greedy) on the same n.
 * gnnpn_pn_enc_layout() returns the layout the dispatcher wants for a batch (blocked for batches that run on the
 * CTA-pair scan: F <= 8, window N <= 10, workspace given, more instances than the column-split cluster scan takes);
 * gnnpn_pn_enc_out_floats() the buffer size; gnnpn_pn_enc_to_rowmajor_f32() converts a blocked buffer to [n, L, H]
 * (for callers that want modelPN.py:191's tensor, e.g. the dense logits of gnnpn_pn_full_logits_f32). */
#define GNNPN_ENC_ROWMAJOR 0
#define GNNPN_ENC_BLOCKED128 1
GNNPN_API int gnnpn_pn_enc_layout(int64_t n, int L, int in_features, int K, int N, int has_workspace);
GNNPN_API size_t gnnpn_pn_enc_out_floats(int64_t n, int L, int hidden, int layout);
GNNPN_API int gnnpn_pn_enc_to_rowmajor_f32(const float* enc_blocked, int64_t n, int L, int hidden, float* enc_out,
                                 void* stream);

/* Input range of the tensor-core LSTM kernels: the raw rows are split into fp16 hi/lo pairs, so |x| must stay below
 * gnnpn_pn_input_limit() (65504; min-max-normalised QoS values are in [0, 1]).  gnnpn_pn_check_inputs_f32 ORs 1 into the
 * device word *flag (caller zeroes it) when any of `count` values is NaN, infinite or at / above the limit; the
 * Python modules call it on every batch and raise instead of decoding garbage (GNNPN_ERANGE semantics, asynchronous). */
GNNPN_API float gnnpn_pn_input_limit(void);
GNNPN_API int gnnpn_pn_check_inputs_f32(const float* inputs, int64_t count, int32_t* flag, void* stream);

/* Encoder: embedding2 + nn.LSTM over L steps (modelPN.py:190-191).
 *   inputs  fp32 [n, L, F]          (F = in_features, 8 when embedding_size == 0)
 *   enc_out fp32 [n, L, H]          every hidden state (or the blocked layout, gnnpn_pn_enc_out_floats() floats)
 *   c_state fp32 [n, H]             final cell state (also scratch during the scan)
 * The final hidden state is enc_out[:, L-1, :].  enc_layout = GNNPN_ENC_BLOCKED128 needs a workspace and F <= 8
 * (else GNNPN_EUNSUPPORTED). */
GNNPN_API int gnnpn_lstm_encode_f32(const float* inputs, int64_t n, int L, int in_features, int hidden,
                          const float* packed_encoder, float* enc_out, float* c_state,
                          void* workspace, size_t workspace_bytes, int enc_layout, void* stream);

/* Scratch for the tensor-core (tcgen05, 3xFP16) recurrences: at least the fp16 hi/lo split of [h | x] of the
 * current and next step, 4 * n * (H + 64) halfs, and the persistent scans' cell-state and exchange buffers.  Passing
 * workspace == NULL to encode/decode selects the strict-fp32 FFMA step kernel instead (same results to ~1e-6, ~5x
 * slower). */
GNNPN_API size_t gnnpn_pn_workspace_bytes(int64_t n, int hidden);

/* Fused greedy pointer decode: K x { decoder LSTM cell -> pointer logits on window k ->
 * C*tanh -> (+ alpha*latent) -> window/visited mask -> softmax -> first-max index -> gather
 * next decoder input }  (modelPN.py:204-239 with sample="greedy"), batched over n instances.
 *   enc_out      fp32 [n, L, H]     from gnnpn_lstm_encode_f32, in the layout `enc_layout` names
 *   c_state      fp32 [n, H]        in: encoder final cell state; out: decoder final cell state
 *   latent_win   fp32 [n, L] or NULL   PNLow's step-(l/N) logit at position l (only the window
 *                                   slice of latent[k] can influence a pick, SURVEY 3.4)
 *   att_params   unused: Dot attention only (Bahdanau runs through gnnpn_pn_decode_general_f32 with a block of
 *                                   gnnpn_pn_att_block_floats() floats, as ops.att_block lays it out)
 *   dec_h        fp32 [n, K, H]     out: decoder hidden state (= attention query) of every step; may be NULL with
 *                                   enc_layout = GNNPN_ENC_BLOCKED128 (the fused decoder does not need it in memory)
 *   idx_out      int32 [K, n]       out: selected position in [k*N, (k+1)*N)
 *   win_logits   fp32 [n, L]        out: this network's pointer logit at position l taken at step l/N
 *   win_probs    fp32 [n, L]        out: softmax probability at position l at step l/N
 *   forced_idx   int32 [K, n] or NULL: teacher forcing -- feed these picks to the next step
 *                                   while idx_out still records the free choice
 *   sample_uniform fp32 [K, n] or NULL: sample="sample" (modelPN.py:227-228) -- with uniforms in [0,1)
 *                                   the pick is an inverse-CDF draw from the window distribution instead
 *                                   of the first maximum (same distribution as torch.multinomial, not the
 *                                   same random stream)
 */
GNNPN_API int gnnpn_pn_decode_greedy_f32(const float* inputs, const float* enc_out, float* c_state,
                               const float* latent_win, float alpha, const float* packed_decoder,
                               int attention, const float* att_params, int use_tanh, float C,
                               int64_t n, int L, int in_features, int hidden, int K, int N,
                               float* dec_h, int32_t* idx_out, float* win_logits, float* win_probs,
                               const int32_t* forced_idx, const float* sample_uniform,
                               void* workspace, size_t workspace_bytes, int enc_layout, void* stream);

/* Best-of-R sampled decoding ("Sampling" inference of a REINFORCE-trained pointer network): R rollouts of every instance
 * decoded from ONE set of encodings (encoder run once, each extra rollout costs one decoder pass), then the rollout with
 * the best objective.  Scope: the fused configuration above (H = 256, Dot attention, in_features <= 8, N <= 32).
 *
 * gnnpn_pn_decode_rollouts_f32: the arguments of gnnpn_pn_decode_greedy_f32 without forced_idx, plus `rollouts` = R >= 1.
 * Rollout r of instance b is row r * n + b.  Rollout 0 is the greedy decode (first-max picks); rollout r >= 1 draws with
 * sample_uniform[r-1] as gnnpn_pn_decode_greedy_f32 draws with its sample_uniform, so every rollout is bit for bit the
 * single decode with those inputs.  The rollouts of an instance share enc_out, c_state (read only: not updated),
 * latent_win and the input rows.
 *   sample_uniform fp32 [R-1, K, n]  (may be NULL when R = 1)
 *   dec_h          fp32 [R, n, K, H] or NULL with enc_layout = GNNPN_ENC_BLOCKED128
 *   idx_out        int32 [R, K, n];  win_logits, win_probs  fp32 [R, n, L]
 *   workspace      gnnpn_pn_rollouts_workspace_bytes(n, H, R) bytes (per-rollout scan scratch); required
 * The launch is the persistent scan plan for n * R decoder rows (the CTA-pair scan, fused with blocked encodings, or the
 * column-split scan); without a workspace, or with the "persistent" option's decoder bit off, GNNPN_EUNSUPPORTED.  The
 * CTAs of an instance block's rollouts are scheduled next to each other, so their encodings reads coincide in L2.
 * GNNPN_ESHAPE for R < 1 or shapes outside the scope. */
GNNPN_API size_t gnnpn_pn_rollouts_workspace_bytes(int64_t n, int hidden, int rollouts);
GNNPN_API int gnnpn_pn_decode_rollouts_f32(const float* inputs, const float* enc_out, const float* c_state,
                                 const float* latent_win, float alpha, const float* packed_decoder,
                                 int attention, const float* att_params, int use_tanh, float C,
                                 int64_t n, int L, int in_features, int hidden, int K, int N,
                                 float* dec_h, int32_t* idx_out, float* win_logits, float* win_probs,
                                 const float* sample_uniform, void* workspace, size_t workspace_bytes,
                                 int enc_layout, int rollouts, void* stream);

/* gnnpn_pn_best_rollout_f32: scores every rollout idx int32 [R, K, n] with gnnpn_pn_reward_f32's arithmetic (one device
 * function serves both) -- level 0 ("Low"): the violations as fp32, level 1 ("High"): float32(round(viol + obj, 5)) --
 * and keeps the lowest score; ties go to the lowest rollout, so the greedy rollout 0 wins them and the result is never
 * worse than greedy.
 *   best_idx int32 [K, n] (the chosen rollout's picks), best_reward fp32 [n], best_rollout int32 [n],
 *   rollout_rewards fp32 [R, n] or NULL (every rollout's score)
 * GNNPN_ESHAPE for R < 1, a level other than 0 / 1, or gnnpn_pn_reward_f32's shape errors. */
GNNPN_API int gnnpn_pn_best_rollout_f32(const float* inputs, const int32_t* idx, int64_t n, int L, int in_features, int K,
                              int tag, int level, int rollouts, int32_t* best_idx, float* best_reward,
                              int32_t* best_rollout, float* rollout_rewards, void* stream);

/* ---- REINFORCE training: differentiable replay of a sampled decode (src/models/trainPNLow.py:77-106,
 * trainPNHigh.py:77-112 back-propagate sum_k log p_k(a_k) with torch autograd through the K-step python graph).
 * Dot attention, no glimpses, embedding_size = 0, N <= 32 (what every reference call site trains).
 *
 * forward: the decode, free-running (greedy, or sampled with sample_uniform: modelPN.py:227-228) or teacher-forced on
 *   forced_idx int32 [K, n], saving for the backward
 *   enc_out [n,L,H], gates_e [L,n,4H] (post-activation, columns 4j+{i,f,g,o}), c_e [L,n,H], dec_h [n,K,H],
 *   gates_d [K,n,4H], c_d [K,n,H], win_logits / win_probs [n,L]; idx_out int32 [K,n] receives the free picks (the fed
 *   picks when free-running, so a sampled decode needs no replay forward).  It runs on
 *   - the tensor-core column-split cluster scan (tcgen05, 3xFP16 split: the kernels of the small-batch inference path
 *     with the per-step saves enabled) when a workspace of gnnpn_pn_train_forward_workspace_bytes() bytes is given and
 *     that size is not 0, i.e. the scan takes the batch (n <= ~3,840 on a B200; the reference trains with 128);
 *   - else, with forced_idx, the strict-fp32 per-step kernels (FFMA LSTM steps + pointer steps; sample_uniform unused);
 *   - else nothing: GNNPN_EUNSUPPORTED before any launch.
 * backward: grad_p fp32 [K,n] = dLoss/dp_k[idx_k] ->
 *   dG_enc_T [4H, L*n], dG_dec_T [4H, K*n]: gradients w.r.t. the gate pre-activations, TORCH gate order (row = gate*H +
 *   unit), column = step*n + instance.  The weight gradients are contractions of these with the step inputs
 *   (dW_hh = dG_T . h(t-1), d(W_ih.W_embed) = dG_T . x(t), db = row sums), run by the caller through
 *   gnnpn_gemm_f32_bias_act.  w_hh_* = weight_hh_l0 as torch stores it, fp32 [4H, H].
 *   workspace: gnnpn_pn_train_backward_workspace_floats(n, L, K, H) floats, 16-byte aligned. */
GNNPN_API size_t gnnpn_pn_train_forward_workspace_bytes(int64_t n, int L, int in_features, int hidden, int K, int N);
GNNPN_API int gnnpn_pn_train_forward_f32(const float* inputs, const float* packed_encoder, const float* packed_decoder,
                               const int32_t* forced_idx, const float* sample_uniform, const float* latent_win,
                               float alpha, int use_tanh, float C, int64_t n, int L, int in_features, int hidden,
                               int K, int N, float* enc_out, float* gates_e, float* c_e, float* dec_h, float* gates_d,
                               float* c_d, float* win_logits, float* win_probs, int32_t* idx_out, void* workspace,
                               size_t workspace_bytes, void* stream);
GNNPN_API size_t gnnpn_pn_train_backward_workspace_floats(int64_t n, int L, int K, int hidden);
GNNPN_API int gnnpn_pn_train_backward_f32(const float* enc_out, const float* gates_e, const float* c_e, const float* dec_h,
                                const float* gates_d, const float* c_d, const float* win_logits,
                                const float* win_probs, const int32_t* idx, const float* grad_p,
                                const float* w_hh_enc, const float* w_hh_dec, int use_tanh, float C, int64_t n,
                                int L, int hidden, int K, int N, float* dG_enc_T, float* dG_dec_T, float* workspace,
                                size_t workspace_floats, void* stream);

/* ---- general decode: every PointerNet variant outside the fused fast path above --------------------------
 * Attention parameter block (gnnpn_pn_att_block_floats(H) floats per Attention module, modelPN.py:83-91):
 *   [ W_query.weight H x H (out, in) | W_query.bias H | W_ref.weight H x H (Conv1d kernel 1 -> out, in) | W_ref.bias H | V H ]
 * `att_params` = the pointer's block, followed by the glimpse's block when n_glimpses > 0 (Bahdanau only; NULL for Dot). */
GNNPN_API size_t gnnpn_pn_att_block_floats(int hidden);

/* Decode loop modelPN.py:204-239 with attention Dot or Bahdanau, n_glimpses >= 0, any window width N, up to 32 raw
 * input columns.  Same outputs as gnnpn_pn_decode_greedy_f32 plus
 *   dec_q       fp32 [n, K, H]   the pointer's query of every step (= dec_h when n_glimpses == 0; must be a distinct
 *                                buffer when n_glimpses > 0)
 *   qw_pointer  fp32 [n, K, H]   Bahdanau: W_query.q + b of every step (input of gnnpn_pn_full_logits_bahdanau_f32); NULL for Dot
 * use_tc != 0 runs the LSTM cell on tcgen05 (3xFP16 split), 0 on the strict-fp32 FFMA kernel.
 * Workspace: gnnpn_pn_decode_general_workspace_bytes(); for Bahdanau it holds E = W_ref.enc_out + b_ref for every
 * position, computed once per call (the reference re-runs the 1x1 convolution at every step, modelPN.py:105). */
GNNPN_API size_t gnnpn_pn_decode_general_workspace_bytes(int64_t n, int L, int K, int hidden, int attention,
                                                         int n_glimpses, int use_tc);
GNNPN_API int gnnpn_pn_decode_general_f32(const float* inputs, const float* enc_out, float* c_state,
                                const float* latent_win, float alpha, const float* packed_decoder, int attention,
                                const float* att_params, int n_glimpses, int use_tanh, float C,
                                int64_t n, int L, int in_features, int hidden, int K, int N,
                                float* dec_h, float* dec_q, float* qw_pointer, int32_t* idx_out, float* win_logits,
                                float* win_probs, const int32_t* forced_idx, const float* sample_uniform, int use_tc,
                                void* workspace, size_t workspace_bytes, void* stream);

/* Building blocks of Attention.forward for name == 'Bahdanau' (modelPN.py:103-109):
 *   E  [rows, H] = W_ref . enc_out[rows, H] + b_ref          (the Conv1d(H, H, 1))
 *   qw [rows, H] = W_query . q + b_query
 *   logits_full [K, n, L] = C*tanh( V . tanh(qw[b,k,:] + E[b,l,:]) ), -inf at the picks of steps < k */
GNNPN_API int gnnpn_pn_ref_transform_f32(const float* enc_out, const float* att_block, int64_t rows, int hidden,
                               float* E, void* stream);
GNNPN_API int gnnpn_pn_query_transform_f32(const float* q, int64_t q_ld, const float* att_block, int64_t rows,
                                 int hidden, float* qw, int64_t qw_ld, void* stream);
GNNPN_API int gnnpn_pn_full_logits_bahdanau_f32(const float* E, const float* qw, const float* att_block,
                                      const int32_t* idx, int use_tanh, float C, int64_t n, int L, int hidden,
                                      int K, float* logits_full, void* stream);

/* ---- any hidden size (the ini's hidden_size is free: src/models/trainPNLow.py:204, environment.ini:24,39; the kernels above
 * are specialised for the shipped value 256 and return GNNPN_ESHAPE otherwise).  Strict fp32, one GEMM + one cell launch per
 * recurrence step, one pointer-step launch per decode step (Dot attention, no glimpses, N <= 32, in_features <= 32).
 *   w_cat  fp32 [4H, H + F]   rows in torch gate order (i, f, g, o blocks of H); columns [W_hh | W_ih . W_emb]
 *   bias   fp32 [4H]          b_ih + b_hh + W_ih . b_emb;   bias0 (decoder step 0): b_ih + b_hh + W_ih . decoder_start_input
 *   workspace: gnnpn_pn_anyh_workspace_floats(n, H, F) floats.  Encodings are row-major [n, L, H]; dec_h [n, K, H] is required.
 * Same meaning of every other argument as gnnpn_lstm_encode_f32 / gnnpn_pn_decode_greedy_f32 / gnnpn_pn_full_logits_f32
 * (modelPN.py:183-239). */
GNNPN_API size_t gnnpn_pn_anyh_workspace_floats(int64_t n, int hidden, int in_features);
GNNPN_API int gnnpn_lstm_encode_anyh_f32(const float* inputs, int64_t n, int L, int in_features, int hidden,
                               const float* w_cat, const float* bias, float* enc_out, float* c_state,
                               float* workspace, size_t workspace_floats, void* stream);
GNNPN_API int gnnpn_pn_decode_anyh_f32(const float* inputs, const float* enc_out, float* c_state, const float* latent_win,
                             float alpha, const float* w_cat, const float* bias, const float* bias0, int use_tanh,
                             float C, int64_t n, int L, int in_features, int hidden, int K, int N, float* dec_h,
                             int32_t* idx_out, float* win_logits, float* win_probs, const int32_t* forced_idx,
                             const float* sample_uniform, float* workspace, size_t workspace_floats, void* stream);
GNNPN_API int gnnpn_pn_full_logits_anyh_f32(const float* enc_out, const float* dec_h, const int32_t* idx, int use_tanh,
                                  float C, int64_t n, int L, int hidden, int K, float* logits_full, void* stream);

/* The attention of the decode loop alone (modelPN.py:213-228 restricted to the windows) for GIVEN decoder states:
 *   enc_out fp32 [n, L, H] row-major, dec_h fp32 [n, K, H]  ->  win_logits / win_probs [n, L], idx_out int32 [K, n]
 * (first-max pick of every window; latent_win / alpha / use_tanh / C as in gnnpn_pn_decode_greedy_f32).  K launches of the
 * stand-alone pointer kernel, every encoding row read once: the attention-only roofline point of bench.py. */
GNNPN_API int gnnpn_pn_attention_windows_f32(const float* enc_out, const float* dec_h, const float* latent_win, float alpha,
                                   int use_tanh, float C, int64_t n, int L, int hidden, int K, int N, int32_t* idx_out,
                                   float* win_logits, float* win_probs, void* stream);

/* Interface-faithful materialisation of PointerNet.forward's prev_logits (modelPN.py:213-214,239):
 *   logits_full fp32 [K, n, L] = C*tanh(<enc_out[b,l,:], dec_h[b,k,:]>) with -inf at the positions
 *   chosen at steps < k (the cumulative visited mask, modelPN.py:165-173). */
GNNPN_API int gnnpn_pn_full_logits_f32(const float* enc_out, const float* dec_h, const int32_t* idx,
                             int attention, const float* att_params, int use_tanh, float C,
                             int64_t n, int L, int hidden, int K, float* logits_full, void* stream);

/* reward()/calc() (modelPN.py:15-72; also src/ML2PN.py:6-12):
 *   inputs fp32 [n, L, F], idx int32 [K, n]; tag = 1 if the rows carry a leading category column.
 *   viol_out int32 [n]  number of violated global constraints (level "Low" reward)
 *   obj_out  fp32 [n]   objFunc = (sum q0 / #(q0>0) + 1 - min q1) / 2
 *   reward_high_out fp32 [n]  float32(round(viol + objFunc, 5))   (any out pointer may be NULL) */
GNNPN_API int gnnpn_pn_reward_f32(const float* inputs, const int32_t* idx, int64_t n, int L, int in_features,
                        int K, int tag, int32_t* viol_out, float* obj_out, float* reward_high_out,
                        void* stream);

/* ESWOA fitness (src/baselines/WOA.py:87-105 `ESWOA.calc`, used at :59,78,119,151) for a batch of P whale positions:
 * float64, every operation in numpy's order (sequential cumprod, np.sum's pairwise scheme), so fitness values and the
 * search's `bestFitness > fitness` comparisons are bit-identical to the reference's.
 *   qos    f64 [n_services, 4]  q0..q3 of every candidate service the positions can select
 *   idx    int32 [P, idx_ld]    row of `qos` chosen for task k of position p (k < klen[p])
 *   klen   int32 [P] or NULL    tasks per position (NULL: Kmax for all); Kmax <= 512
 *   bounds f64 [P, 4]           lo1, hi1, lo2, hi2: the instance's two global constraints (loadData.py:279-283)
 *   viol_out int32 [P], obj_out f64 [P], fit_out f64 [P] = viol + obj   (any may be NULL) */
GNNPN_API int gnnpn_woa_fitness_f64(const double* qos, int64_t n_services, const int32_t* idx, int64_t idx_ld,
                          const int32_t* klen, const double* bounds, int64_t P, int Kmax,
                          int32_t* viol_out, double* obj_out, double* fit_out, void* stream);

/* `ML2PN.calc` (src/ML2PN.py:6-12) for a batch of compositions, float64 in numpy's operation order: same layout as
 * gnnpn_woa_fitness_f64, but the objective is 0.5*(np.average(q0) + 1 - np.min(q1)) -- the mean runs over ALL klen[p]
 * picks, not over those with q0 > 0 -- and score = obj with 1.0 added once per violated global constraint, constraint 1
 * first (as `obj += 1` in ML2PN.calc; with both violated, (obj + 1) + 1 can differ from obj + 2 in the last bit).
 * obj_out is the objective before the violations. */
GNNPN_API int gnnpn_ml2pn_score_f64(const double* qos, int64_t n_rows, const int32_t* idx, int64_t idx_ld,
                          const int32_t* klen, const double* bounds, int64_t P, int Kmax,
                          int32_t* viol_out, double* obj_out, double* score_out, void* stream);

/* Device-resident ESWOA search (src/baselines/WOA.py:107-162): one CTA per instance, one thread per whale, all
 * `iters` iterations in one launch, same sequential semantics as the reference's loop (in-order best-so-far replay,
 * speculative local phase committed up to the first improvement, bestPops aliasing).  Random numbers are counter-based
 * Philox4x32-10: key = seeds[I], counter = (slot, whale, phase, iteration), phase 0 = global (slots q / task / candidate),
 * 1 = exploration skip, 2 = local (slots r / l / p); uniform = ((x0 >> 5) * 2^26 + (x1 >> 6)) / 2^53; integers are
 * floor(u * n).  The caller initialises the population and the best state (WOA.py:50-85).
 *   base, size  int32 [I, Kmax]      first `qos` row / length of every task's candidate list (klen[I] tasks used)
 *   pops        int32 [I, popSize, Kmax] in/out   local candidate index per task (Python index semantics)
 *   best_fit f64 [I], best_ref int32 [I] (whale whose row IS the best position, or -1), best_vec int32 [I, Kmax]  in/out
 *   traj        f64 [I, iters]       best fitness after every iteration (`ESWOA.bestFitnesses`)
 * popSize <= 128, Kmax <= 128. */
GNNPN_API int gnnpn_woa_search_f64(const double* qos, int64_t n_services, const int32_t* base, const int32_t* size,
                         const int32_t* klen, const double* bounds, int32_t* pops, double* best_fit,
                         int32_t* best_ref, int32_t* best_vec, const uint64_t* seeds, double* traj,
                         int64_t n_instances, int popSize, int Kmax, int iters, void* stream);

/* Everything gnnpn_woa_search_f64 needs, built on the device from request data and PNHigh's picks, exactly as the host
 * path computes it before its search (gnnpn_sc_b200/WOA.py: loadDataOther + _add_s, the seed rows of WOA.start,
 * _Instance.__init__, _Engine._init_population).  One CTA per instance.
 *  Candidate lists: for every requested task in request order, the services of its category in position order with
 *   lo_cost <= q2 <= hi_cost and lo_q <= q3 <= hi_q (float64); with reduct != 0 thinned by _add_s's running front
 *   (sentinel entry, index bookkeeping and protected seed rows included).  Empty lists are dropped.
 *  Seed: the picks whose float64 sum ((q0+q1)+q2)+q3 is not 3, in category order.  With at least one, every candidate row
 *   is rounded to 5 decimals (svc_round), the seed rows too, six of them patched as the reference does; seed row l is
 *   looked up in list l (first exact match) or appended to it.  Without one the rows stay unrounded and the best
 *   fitness starts at 3.
 *  Population: pops[i, k] = floor(u * size_before_append[k]), u = Philox(seeds[I]) at (slot k, whale i, phase 3, t 0);
 *   the seed is evaluated first, then whales 0..popSize-1, accepted on a strictly lower fitness.
 *   svc_raw, svc_round f64 [n_services, 4]  q0..q3 of every service (JSON values) and the same rounded (Python round)
 *   cat_ptr      int32 [K+1]          service range of every category (category-major service ids), K <= 128
 *   req_cat      int32 [I, K]         category (0-based) of task j in request-node order, j < n_req[I]
 *   n_req        int32 [I]
 *   local_bounds f64 [I, K, 4]        lo_cost, hi_cost, lo_q, hi_q of the task node of every category
 *   global_bounds f64 [I, 4]          lo1, hi1, lo2, hi2 of the global-constraint node (the search's `bounds`)
 *   seed_rows    fp32 [I, K, 4]       q0..q3 of PNHigh's pick per category; seed_ids int32 [I, K] its service id
 *   seeds        uint64 [I]           Philox key of every instance (the search takes the same array)
 *   reduct       0 (plain lists) or the _add_s threshold (0.55 in the Normal ini sections)
 * Outputs, in the layouts gnnpn_woa_search_f64 takes with Kmax = K:
 *   qos f64 [gnnpn_woa_prepare_rows(I, n_services, K), 4] candidate rows; ids int32 [same rows] service id of every row
 *   base, size int32 [I, K] (size after the seed appends; base 0, size 1 past klen); klen int32 [I] number of lists
 *   list_cat int32 [I, K]             category of every list (-1 past klen)
 *   pops int32 [I, popSize, K], best_fit f64 [I], best_ref int32 [I], best_vec int32 [I, K]
 *   flags int32 [I]   0, or why the instance has no result.  The host path raises for bits 0, 1, 2 and 4: bit 0 more
 *                     seed rows than lists, bit 1 the front replaces past the end of its list, bit 2 no list at all,
 *                     bit 4 fewer seed rows than lists.  Bit 3 is input this entry does not take: a category outside
 *                     [0, K), or one requested twice (the host path gives both tasks the same list object, so a seed
 *                     row appended to one shows in the other).  Results of a flagged instance are meaningless.
 * popSize <= 128; GNNPN_ESHAPE when I * (n_services + K) reaches 2^31 rows. */
GNNPN_API int gnnpn_woa_prepare_f64(const double* svc_raw, const double* svc_round, const int32_t* cat_ptr,
                          int64_t n_services, int K, const int32_t* req_cat, const int32_t* n_req,
                          const double* local_bounds, const double* global_bounds, const float* seed_rows,
                          const int32_t* seed_ids, const uint64_t* seeds, int64_t n_instances, int popSize,
                          double reduct, double* qos, int32_t* ids, int32_t* base, int32_t* size, int32_t* klen,
                          int32_t* list_cat, int32_t* pops, double* best_fit, int32_t* best_ref, int32_t* best_vec,
                          int32_t* flags, void* stream);
/* rows of gnnpn_woa_prepare_f64's qos / ids: n_instances * (n_services + K), one slot of (size + 1) rows per category */
GNNPN_API int64_t gnnpn_woa_prepare_rows(int64_t n_instances, int64_t n_services, int K);

/* Host-buffer convenience for non-torch callers: PNLow greedy -> latent -> PNHigh greedy
 * (src/models/trainPNHigh.py:131-144) on pageable or pinned HOST memory; allocates its own device
 * scratch, copies in and out, synchronises.  idx_high_host int32 [K, n]; reward_high_host fp32 [n]. */
GNNPN_API int gnnpn_pn_greedy_low_high_host(const float* inputs_host, int64_t n, int L, int in_features, int hidden,
                                  int K, int N, const float* packed_low_host, const float* packed_high_host,
                                  int use_tanh, float C, float alpha,
                                  int32_t* idx_low_host, int32_t* idx_high_host, float* reward_high_host);

/* ---------------------------------------------------------------------------
 * Between the stages: ML ranking -> pointer-network input rows  (reference: src/loadData.py:99-150, loadDataPN)
 * ------------------------------------------------------------------------- */

/* Per instance b and category c: the first N services of category c in descending-score order that satisfy the
 * task's local bounds (lo2 <= q2 <= hi2 and lo3 <= q3 <= hi3, loadData.py:120-124), padded to N by cyclic
 * self-duplication (loadData.py:137-138); categories the request does not use, or with no feasible service, become
 * N neutral rows [0,1,1,1] (loadData.py:148).  Ranking order is kept (the reference's unseeded shuffle,
 * loadData.py:135, is not reproduced); score ties go to the lower service id.
 *   scores        fp32 [n, >=S] rows scores_ld apart   Net.forward output (modelML.py:176)
 *   svc_qos       fp32 [S, 4]    q0..q3 of every service, service-id (= category-major) order, 16-byte aligned
 *   cat_ptr       int32 [K+1]    service-id range of every category
 *   local_bounds  fp32 [n, K, 4] lo2, hi2, lo3, hi3 of the task node of category c (loadData.py:112-113)
 *   used          uint8 [n, K]   1 when the request has a task of category c
 *   global_bounds fp32 [n, 4]    bounds of the global-constraint node (loadData.py:109-110): tail of category 0's rows
 *   rows          fp32 [n, K*N, 8 (+1 leading category column when with_category)]   the PN input
 *   picked        int32 [n, K*N] service id per row, -1 for neutral rows (may be NULL) */
GNNPN_API int gnnpn_select_candidates_f32(const float* scores, int64_t scores_ld, const float* svc_qos,
                                const int32_t* cat_ptr, int max_category_size, const float* local_bounds,
                                const uint8_t* used, const float* global_bounds, int64_t n, int K, int N,
                                int with_category, float* rows, int32_t* picked, void* stream);

/* ---------------------------------------------------------------------------
 * ML stage: graph message passing  (reference: src/models/modelML.py + PyG 1.7.0 ops)
 * ------------------------------------------------------------------------- */

/* edge_index -> destination-major CSR, stable in edge order (replaces the per-forward, per-layer
 * re-normalisation inside GCNConv, modelML.py:153, and the scatter index handling of GINConv :140).
 *   mode GNNPN_CSR_PLAIN   : rows = edge_index[1] (target), cols = edge_index[0] (source), val = weight or absent
 *   mode GNNPN_CSR_GCN_NORM: add_remaining_self_loops(fill 1) then val = deg^-1/2[src] * w * deg^-1/2[dst]
 *   rowptr int64 [n_nodes+1]; col int32 [nnz]; val fp32 [nnz] (NULL allowed for PLAIN without weights);
 *   nnz_out int64 [1] device.  Capacity of col/val must be n_edges (PLAIN) or n_edges + n_nodes (GCN). */
GNNPN_API int gnnpn_csr_build_workspace_bytes(int64_t n_nodes, int64_t n_edges, int mode, size_t* bytes);
GNNPN_API int gnnpn_csr_build(const int64_t* edge_index, const float* edge_weight, int64_t n_edges, int64_t n_nodes,
                    int mode, int64_t* rowptr, int32_t* col, float* val, int64_t* nnz_out,
                    void* workspace, size_t workspace_bytes, void* stream);

/* NodeEncoder + concat (modelML.py:22-29,134-137,145-149): column 0 of x (a category id stored as float)
 * selects a row of the [table_rows, embed_dim] embedding table, the remaining n_cols-1 float columns are
 * appended, the row is zero-padded to ld_out (a multiple of 4 so the aggregation can use 128-bit loads). */
GNNPN_API int gnnpn_embed_concat_f32(const float* x, int64_t n, int n_cols, const float* table, int table_rows,
                           int embed_dim, float* out, int64_t ld_out, void* stream);

/* Neighbour aggregation as CSR segment-reduce, one warp (or sub-warp) per destination row,
 * sequential in CSR order per feature (deterministic; equals CPU index_add_ in edge order):
 *   y[i,:] = act( ( self_scale * x[i,:] + sum_e val[e] * x[col[e],:] ) / (mean ? max(rowlen,1) : 1)
 *                 [+ bias] [* scale + shift] )
 * Covers GINConv's sum + (1+eps)*x (self_scale = 1+eps), GCNConv's normalised sum + bias with the
 * following eval-mode BatchNorm + ReLU folded in, and scatter(reduce='mean') (modelML.py:166,172).
 * F must be a multiple of 4; x, y 16-byte aligned with leading dimensions ldx, ldy (floats).  `nnz` is rowptr[n_rows]
 * or any upper bound of it (known to the caller, not read from the device).
 * LONG-ROW SPLITTING for skewed in-degree distributions (hub destinations: the service co-usage graph of
 * src/loadData.py:55-65 gives popular services rows of 10^4..10^5 edges): rows with more than T edges are cut into
 * chunks of max(256, T / 8) consecutive edges (longer for a row that would otherwise have more than 4096 chunks), each
 * chunk is summed by one lane group like a short row, and the chunk sums are added in chunk order: deterministic, no
 * atomics in the arithmetic.  Rows of at most T edges are bit-identical to the sequential index_add_ order; split rows
 * differ from the strictly sequential sum by re-association only.
 *   long_row_threshold < 0 : the library chooses T from nnz and F (no split below 2^22 edges)
 *                      0   : never split: every row in index_add_ order
 *                   >= 32  : T = long_row_threshold (1..31: GNNPN_ESHAPE)
 * workspace: gnnpn_spmm_csr_workspace_bytes(nnz, F, long_row_threshold) bytes, 256-byte aligned.  The query returns 0
 * when the call does not split; workspace may then be NULL. */
GNNPN_API size_t gnnpn_spmm_csr_workspace_bytes(int64_t nnz, int F, int64_t long_row_threshold);
GNNPN_API int gnnpn_spmm_csr_f32(const int64_t* rowptr, const int32_t* col, const float* val, const float* x,
                                 int64_t ldx, float* y, int64_t ldy, int64_t n_rows, int64_t nnz, int F,
                                 float self_scale, int mean, const float* bias, const float* scale, const float* shift,
                                 int act, int64_t long_row_threshold, void* workspace, size_t workspace_bytes,
                                 void* stream);

/* Train-mode BatchNorm1d (+ optional fused ReLU) for the ML stage's training path (torch.nn.BatchNorm1d in training mode,
 * src/models/modelML.py:75-93,98-104 under TrainML.train, trainML.py:34-47).
 * forward : batch mean / biased variance per channel over the M rows of y [M, C] (two passes), out = act((y - mean) * rstd
 *           * gamma + beta); save_mean / save_rstd [C] for the backward; running_mean / running_var (may be NULL) updated
 *           with `momentum` and the unbiased variance, as torch does.
 * backward: dout masked by the ReLU (out > 0), dgamma = sum dout * xhat, dbeta = sum dout,
 *           dx = gamma * rstd * (dout - dbeta / M - xhat * dgamma / M).  Deterministic (fixed-order reductions). */
GNNPN_API int gnnpn_bn_train_forward_f32(const float* y, int64_t ldy, int64_t M, int C, const float* gamma, const float* beta,
                               float eps, float momentum, int relu, float* out, int64_t ldo, float* save_mean,
                               float* save_rstd, float* running_mean, float* running_var, void* stream);
GNNPN_API int gnnpn_bn_train_backward_f32(const float* y, int64_t ldy, const float* out, int64_t ldo, const float* dout,
                                int64_t ldd, int64_t M, int C, const float* gamma, const float* save_mean,
                                const float* save_rstd, int relu, float* dx, int64_t ldx, float* dgamma, float* dbeta,
                                void* stream);

/* Node transform: C[M,N] = act( (A[M,K] . W[N,K]^T + bias[N]) * scale[N] + shift[N] )
 * (nn.Linear / GCNConv's X.W, modelML.py:77-93,98-106,164-165; bias/scale/shift may be NULL).
 * fp32 in/out.  One of three kernels runs:
 *   - workspace == NULL: strict fp32 FFMA (the small request-graph shapes);
 *   - K, N <= 256, K % 4 == 0, N % 16 == 0, A 16-byte aligned and lda % 4 == 0: the persistent tcgen05 node transform,
 *     error-compensated 3xFP16 with fp32 accumulate in TMEM; when an input is outside its fp16 range (|a| >= 4095, or
 *     not finite) a strict fp32 FFMA pass recomputes C on the device;
 *   - any other shape: tcgen05 error-compensated 3xTF32, split over K when the output has few row tiles and K is long.
 * A node-transform shape whose A is misaligned runs the FFMA kernel, which needs no workspace: the size
 * gnnpn_gemm_workspace_bytes(M, N, K) returns is enough for every A. */
GNNPN_API size_t gnnpn_gemm_workspace_bytes(int64_t M, int N, int K);
GNNPN_API int gnnpn_gemm_f32_bias_act(const float* A, int64_t lda, const float* W, int64_t ldw,
                            const float* bias, const float* scale, const float* shift, int act,
                            float* C, int64_t ldc, int64_t M, int N, int K,
                            void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GNNPN_B200_H_ */
