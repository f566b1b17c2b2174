// Pointer step for one composition instance, executed by one warp (Dot attention, modelPN.py:111-120,
// 213-228).  Shared by the stand-alone pointer kernel (pn.cu) and the persistent decode kernel (tc_seq.cu)
// so both round identically.
//   u_j   = <enc_out[b, kN+j, :], q[b,:]>            j in [0,N)
//   l_j   = use_tanh ? C*tanh(u_j) : u_j            -> win_logits[b, kN+j]
//   w_j   = l_j + alpha*latent[b, kN+j]
//   p     = softmax_j(w)  (exp(w-max)/sum, fp32)    -> win_probs[b, kN+j]
//   pick  = first j with maximal p                  -> idx_out[b] = kN + j
// Positions outside the window carry -inf after modelPN.py:220-222 and contribute exp(-inf)=0.
#pragma once
#include <math.h>
#include "common.cuh"
#include "lstm_step.cuh"

namespace gnnpn {

constexpr int kMaxWindow = 32;

struct PointerStepArgs {
  const float* enc_out;      // [n, L, kH]
  int64_t enc_inst_ld;
  const float* latent_win;   // [n, L] or nullptr
  float alpha;
  int use_tanh;
  float C;
  int64_t n;
  int L, N;
  int32_t* idx_out;          // [K, n]
  float* win_logits;         // [n, L]
  float* win_probs;          // [n, L]
  const int32_t* forced;     // [K, n] teacher-forced picks or nullptr
  const float* uniform;      // [K, n] uniforms (sample="sample") or nullptr
};
// The decode step k is passed separately so that the argument block itself can stay in constant memory.

// Rollout r of a rollout launch (gnnpn_pn_decode_rollouts_f32): the encodings, latent and input rows are the instance's,
// the outputs rollout r's slices of idx_out [R, K, n] and win_logits / win_probs [R, n, L].  Rollout 0 decodes with
// a.uniform (NULL in a rollout launch: greedy), rollout r >= 1 draws with the uniforms [r-1] of `sampled` [R-1, K, n].
// r = 0 leaves the block as it is, so a launch of one rollout is the plain decode.
__device__ __forceinline__ PointerStepArgs rollout_args(const PointerStepArgs& a, int r, int K, const float* sampled) {
  PointerStepArgs o = a;
  if (r > 0) {
    o.idx_out += (int64_t)r * K * a.n;
    o.win_logits += (int64_t)r * a.n * a.L;
    o.win_probs += (int64_t)r * a.n * a.L;
    o.uniform = sampled + (int64_t)(r - 1) * K * a.n;
  }
  return o;
}

// argument block of the pointer steps over row-major encodings [n, L, kH]
inline PointerStepArgs pointer_step_args(const float* enc_out, const float* latent_win, float alpha, int use_tanh, float C,
                                         int64_t n, int L, int N, int32_t* idx_out, float* win_logits, float* win_probs,
                                         const int32_t* forced, const float* uniform) {
  return PointerStepArgs{enc_out, (int64_t)L * kH, latent_win, alpha, use_tanh, C, n, L, N, idx_out, win_logits,
                         win_probs, forced, uniform};
}

// ---- canonical pointer-logit dot product ------------------------------------------------------------------
// Every kernel that forms a Dot pointer logit <row, q> rounds in THIS order, so window logits == the same entries of
// the dense logits == the fused decoders' values, bit for bit, whichever kernel a batch is dispatched to:
//   the 256 hidden units are indexed u = 32*nt + 8*g + i   (nt = 0..7 "tile", g = 0..3 "group", i = 0..7)
//   s[nt][g] = r_u0*q_u0, then fmaf over i = 1..7                       (8 consecutive units)
//   p[g]     = ((((s[0][g] + s[1][g]) + s[2][g]) + ... ) + s[7][g])     (sequential over the tiles)
//   dot      = (p[0] + p[1]) + (p[2] + p[3])
// It is the order the persistent tcgen05 decoder meets for free: its epilogue thread (instance, g) produces the h'
// units of accumulator tile nt as exactly those 8 consecutive values (tc_seq.cu).  A warp computes one row with lane
// l = 4*nt + g owning the 32 contiguous bytes [8l, 8l+8) of the row and of the query (one 256-bit load each).
__device__ __forceinline__ float dot8(const float4 r0, const float4 r1, const float4 q0, const float4 q1) {
  float s = __fmul_rn(r0.x, q0.x);
  s = fmaf(r0.y, q0.y, s); s = fmaf(r0.z, q0.z, s); s = fmaf(r0.w, q0.w, s);
  s = fmaf(r1.x, q1.x, s); s = fmaf(r1.y, q1.y, s); s = fmaf(r1.z, q1.z, s); s = fmaf(r1.w, q1.w, s);
  return s;
}
// s = this lane's s[nt][g] (lane = 4*nt + g)  ->  the canonical dot, in every lane
__device__ __forceinline__ float dot_reduce(float s, int lane) {
  const int g = lane & 3;
  float p = __shfl_sync(0xffffffffu, s, g);
#pragma unroll
  for (int nt = 1; nt < 8; ++nt) p = __fadd_rn(p, __shfl_sync(0xffffffffu, s, 4 * nt + g));
  const float a = __fadd_rn(p, __shfl_xor_sync(0xffffffffu, p, 1));          // p0+p1 | p2+p3 (commutative: both lanes agree)
  return __fadd_rn(a, __shfl_xor_sync(0xffffffffu, a, 2));
}
// the lane's 8 consecutive floats of a 256-float row: streaming (read-once) and coherent variants
__device__ __forceinline__ void ldg_row8_stream(const float* row, int lane, float4& a, float4& b) {
  asm volatile("ld.global.nc.L1::no_allocate.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w), "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w)
               : "l"(row + 8 * lane));
}
__device__ __forceinline__ void ld_row8(const float* row, int lane, float4& a, float4& b) {
  asm volatile("ld.global.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w), "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w)
               : "l"(row + 8 * lane) : "memory");
}

// ---- the rest of the step, from the pre-activations d_j = <row_j, q> -----------------------------------------------
// Each rule is written once, here.  The forms below (and the general kernels, pn_general.cu / pn_anyh.cu) only decide
// which lane, thread or CTA handles which candidate, so their window logits, probabilities and picks are bit-identical.

__device__ __forceinline__ float window_logit(int use_tanh, float C, float d) { return use_tanh ? C * tanhf(d) : d; }
// working logit: the window logit plus PNHigh's latent term
__device__ __forceinline__ float work_logit(const PointerStepArgs& a, float l, float lat) {
  return a.latent_win ? fmaf(a.alpha, lat, l) : l;
}

// first maximal probability (torch.max tie rule, modelPN.py:225-226): `add` takes candidates in ascending order,
// `merge` joins the result over another set of candidates
struct FirstMax {
  float best;
  int j;
  __device__ __forceinline__ void add(int c, float p) {
    if (p > best) { best = p; j = c; }
  }
  __device__ __forceinline__ void merge(float ob, int oj) {
    if (ob > best || (ob == best && oj < j)) { best = ob; j = oj; }
  }
};

// sample="sample" (modelPN.py:227-228): inverse-CDF draw from the window distribution with a caller-supplied uniform
// u in [0,1), candidates added in ascending order; falls back to the last candidate with non-zero probability when
// round-off leaves the cumulative sum at or below u
struct InverseCdf {
  float cum = 0.f;
  int pick = -1, last_pos = 0;
  __device__ __forceinline__ void add(int c, float p, float u) {
    cum += p;
    if (p > 0.f) last_pos = c;
    if (pick < 0 && u < cum) pick = c;
  }
  __device__ __forceinline__ int result() const { return pick < 0 ? last_pos : pick; }
};

// the teacher-forced position of step k for instance b, or -1
__device__ __forceinline__ int forced_pick(const PointerStepArgs& a, int k, int64_t b) {
  return a.forced ? a.forced[(int64_t)k * a.n + b] : -1;
}
// Records window candidate `pick` of step k (idx_out[k, b] = kN + pick, when `write`) and returns the position fed to
// the next decoder step: `forced` (forced_pick) when teacher forcing, else kN + pick.
__device__ __forceinline__ int record_pick(const PointerStepArgs& a, int k, int64_t b, int pick, bool write, int forced) {
  if (write) a.idx_out[(int64_t)k * a.n + b] = k * a.N + pick;
  return a.forced ? forced : k * a.N + pick;
}

// Lane form: one instance per segment of SEG lanes (8, 16 or 32).  Lane j (< N) of the segment holds d_j in `d` and,
// with a latent, latent[b, kN+j] in `lat`; `inst` is false in a segment without an instance (b must still be a valid
// index).  The butterflies start at offset `top`, a power of two with N <= 2 * top <= SEG: max and first maximum are
// exact, so the depth changes no result.  Writes win_logits / win_probs / idx_out and returns, in every lane of the
// segment, the position fed to the next decoder step.
template <int SEG>
__device__ __forceinline__ int pointer_finish_lanes(const PointerStepArgs& a, int k, int64_t b, bool inst, float d,
                                                    float lat, int j, int top) {
  const int N = a.N;
  const bool valid = inst && j < N;
  const float l = window_logit(a.use_tanh, a.C, d);
  const int64_t wpos = b * a.L + (int64_t)k * N + j;
  float w = -INFINITY;
  if (valid) {
    w = work_logit(a, l, lat);
    a.win_logits[wpos] = l;
  }
  float mx = w;
#pragma unroll
  for (int o = top; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  const float e = valid ? expf(w - mx) : 0.f;
  float s = 0.f;
  for (int c = 0; c < N; ++c) s += __shfl_sync(0xffffffffu, e, c, SEG);    // sequential, in candidate order
  const float p = e / s;
  if (valid) a.win_probs[wpos] = p;
  FirstMax m{valid ? p : -1.f, valid ? j : 0x7fffffff};
#pragma unroll
  for (int o = top; o > 0; o >>= 1) m.merge(__shfl_xor_sync(0xffffffffu, m.best, o), __shfl_xor_sync(0xffffffffu, m.j, o));
  int pick = __shfl_sync(0xffffffffu, m.j, 0, SEG);   // lanes at or past 2 * top took no part in the butterflies
  if (a.uniform) {
    const float u = __ldg(a.uniform + (int64_t)k * a.n + b);
    InverseCdf draw;
    for (int c = 0; c < N; ++c) draw.add(c, __shfl_sync(0xffffffffu, p, c, SEG), u);
    pick = draw.result();
  }
  return record_pick(a, k, b, pick, inst && j == 0, forced_pick(a, k, b));
}

// Serial form (the fused decoder, tc_seq.cu): ONE thread finishes the step of instance b from d[j] = d_j (j < N <= NR).
// Threads without an instance (ok == false) run the same code on instance 0 without writing.  Returns the position fed
// to the next decoder step.
template <int NR>
__device__ __forceinline__ int pointer_finish_thread(const PointerStepArgs& a, int k, int64_t b, bool ok,
                                                     const float (&d)[NR]) {
  const int N = a.N;
  if (!ok) b = 0;
  const int64_t wpos = b * a.L + (int64_t)k * N;
  float w[NR];
  float lat[NR];
#pragma unroll
  for (int j = 0; j < NR; ++j) lat[j] = (a.latent_win && j < N) ? __ldg(a.latent_win + wpos + j) : 0.f;
  const float u = a.uniform ? __ldg(a.uniform + (int64_t)k * a.n + b) : 0.f;
  const int forced = forced_pick(a, k, b);
  float mx = -INFINITY;
#pragma unroll
  for (int j = 0; j < NR; ++j) {
    w[j] = -INFINITY;
    if (j < N) {
      const float l = window_logit(a.use_tanh, a.C, d[j]);
      if (ok) a.win_logits[wpos + j] = l;
      w[j] = work_logit(a, l, lat[j]);
      mx = fmaxf(mx, w[j]);
    }
  }
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < NR; ++j) {
    if (j < N) { w[j] = expf(w[j] - mx); s += w[j]; }
  }
  InverseCdf draw;
  FirstMax m{-1.f, 0};
#pragma unroll
  for (int j = 0; j < NR; ++j) {
    if (j < N) {
      const float pj = w[j] / s;
      if (ok) a.win_probs[wpos + j] = pj;
      m.add(j, pj);
      draw.add(j, pj, u);
    }
  }
  return record_pick(a, k, b, a.uniform ? draw.result() : m.j, ok, forced);
}

// q0/q1: the lane's 8 query elements (floats [8*lane, 8*lane+8) of the 256-float query).
// Returns, in every lane, the position fed to the next decoder step (the pick, or forced[b]).
__device__ __forceinline__ int pointer_step_warp(const PointerStepArgs& a, int k, int64_t b, const float4 q0,
                                                 const float4 q1, int lane) {
  const int N = a.N;
  const float* base = a.enc_out + b * a.enc_inst_ld + (int64_t)k * N * kH;
  float my_d = 0.f;                            // lane j holds candidate j
  for (int j0 = 0; j0 < N; j0 += 4) {          // 4 rows in flight per iteration
    float part[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      part[u] = 0.f;
      if (j0 + u < N) {
        float4 r0, r1;
        ldg_row8_stream(base + (int64_t)(j0 + u) * kH, lane, r0, r1);
        part[u] = dot8(r0, r1, q0, q1);
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const float d = dot_reduce(part[u], lane);
      if (lane == j0 + u) my_d = d;
    }
  }
  float lat = 0.f;
  if (a.latent_win && lane < N) lat = __ldg(a.latent_win + b * a.L + (int64_t)k * N + lane);
  // windows of <= 8 candidates live in lanes 0..7: 3 butterfly levels instead of 5
  return pointer_finish_lanes<32>(a, k, b, true, my_d, lat, lane, N <= 8 ? 4 : 16);
}

// ---- form used by the fused decode kernel: one warp owns WI = 8 consecutive instances.
// Phase 1 streams the window rows: per instance one chunk of CH rows is in flight in registers and the next chunk is
// requested as soon as the dot products have consumed the current one, so the DRAM round trips of consecutive
// instances overlap the butterfly reductions.  The logit pre-activations are parked lane-wise: instance i,
// candidate j -> register i / IPP, lane (i % IPP) * SEG + j  (SEG = 8, 16 or 32 lanes per instance, IPP = 32 / SEG).
// Phase 2 then finishes IPP instances per pass with pointer_finish_lanes<SEG>.
// `feed(i, b, fed, j)` is called by every lane of a pass with the position fed to the next step for ITS instance
// (i = instance slot 0..7, j = lane index inside the segment); slots >= count must be ignored by the callee.
constexpr int kWarpInstances = 8;

template <int SEG, int CH, class Feed>
__device__ __forceinline__ void pointer_steps_batched(const PointerStepArgs& a, int k, int64_t b0, int count,
                                                      const float* q_base, int64_t q_ld, int lane, Feed feed
                                                      ) {
  constexpr int IPP = 32 / SEG;                    // instances per phase-2 pass
  constexpr int PASSES = kWarpInstances / IPP;
  if (count <= 0) return;
  const int N = a.N;
  const int seg_i = lane / SEG, seg_j = lane % SEG;

  // ---- phase 1: one exposed memory round trip per chunk (all CH rows + the query in flight together)
  float dv[PASSES];
#pragma unroll
  for (int r = 0; r < PASSES; ++r) dv[r] = 0.f;
  const float* rows = a.enc_out + b0 * a.enc_inst_ld + (int64_t)k * N * kH;
  const float* qrow = q_base + b0 * q_ld;
#pragma unroll 1
  for (int i = 0; i < count; ++i) {
    float4 q0, q1;
    ld_row8(qrow, lane, q0, q1);                                          // coherent loads: written earlier in this launch
    const int slot = i / IPP, base = (i % IPP) * SEG;
#pragma unroll 1
    for (int j0 = 0; j0 < N; j0 += CH) {
      float4 r0[CH], r1[CH];
#pragma unroll
      for (int u = 0; u < CH; ++u) {
        const int j = j0 + u < N ? j0 + u : N - 1;                        // clamp: every register is always written
        ldg_row8_stream(rows + (int64_t)j * kH, lane, r0[u], r1[u]);
      }
      float part[CH];
#pragma unroll
      for (int u = 0; u < CH; ++u) part[u] = dot8(r0[u], r1[u], q0, q1);
#pragma unroll
      for (int u = 0; u < CH; ++u) {
        const float d = dot_reduce(part[u], lane);
        const bool mine = j0 + u < N && lane == base + j0 + u;
#pragma unroll
        for (int r = 0; r < PASSES; ++r) dv[r] = (mine && slot == r) ? d : dv[r];   // selects: dv stays in registers
      }
    }
    rows += a.enc_inst_ld;
    qrow += q_ld;
  }

  float lat[PASSES];
#pragma unroll
  for (int r = 0; r < PASSES; ++r) {
    const int i = r * IPP + seg_i;
    lat[r] = (a.latent_win && i < count && seg_j < N)
                 ? __ldg(a.latent_win + (b0 + i) * a.L + (int64_t)k * N + seg_j) : 0.f;
  }
  // ---- phase 2
#pragma unroll
  for (int r = 0; r < PASSES; ++r) {
    const int si = r * IPP + seg_i;                // this lane's instance slot
    if (r * IPP >= count) break;                   // warp-uniform
    const bool inst_ok = si < count;
    const int64_t b = b0 + (inst_ok ? si : 0);
    feed(si, b, pointer_finish_lanes<SEG>(a, k, b, inst_ok, dv[r], lat[r], seg_j, SEG / 2), seg_j);
  }
}

}  // namespace gnnpn
