// Shared helpers for libgnnpn_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <atomic>
#include "gnnpn_b200.h"

namespace gnnpn {

extern std::atomic<uint64_t> g_launch_count;

inline int after_launch() {
  g_launch_count.fetch_add(1, std::memory_order_relaxed);
  cudaError_t e = cudaPeekAtLastError();
  return e == cudaSuccess ? GNNPN_OK : (int)cudaGetLastError();
}

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
inline bool aligned32(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 31u) == 0; }
inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }
inline int round_up(int a, int b) { return (a + b - 1) / b * b; }
// A workspace is used from its first 1024-byte boundary (TMA and swizzled operand alignment); the *_workspace_bytes
// sizes include that slack.
template <class T = uint8_t>
inline T* align_ws(void* workspace) {
  return reinterpret_cast<T*>((reinterpret_cast<uintptr_t>(workspace) + 1023) & ~uintptr_t(1023));
}

constexpr int kNumSMs = 148;  // B200: 2 dies x 74 SMs

__device__ __forceinline__ float sigmoid_accurate(float x) { return 1.0f / (1.0f + expf(-x)); }

// The fused tail of a GIN / GCN layer, act((r + b) * s + t): bias, eval-mode BatchNorm scale / shift, activation.  The
// FFMA and 3xTF32 GEMMs, the split-K reduction and the aggregation all end a layer with this one copy, so the layer
// gives the same bits whichever of them runs.  It updates N consecutive columns r[0..N) of a row in place.  Each kernel
// keeps its own loads: load(p, v) puts the N columns of the per-column array p into v; it runs only for the arrays the
// layer has, right before their use.  The add is __fadd_rn so that no call site can contract it into an FMA.
template <int N, class Load>
__device__ __forceinline__ void bias_bn_act(float* r, const float* bias, const float* scale, const float* shift, int act,
                                            Load load) {
  float v[N], w[N];
  if (bias) {
    load(bias, v);
#pragma unroll
    for (int i = 0; i < N; ++i) r[i] = __fadd_rn(r[i], v[i]);
  }
  if (scale) {
    load(scale, v);
    load(shift, w);
#pragma unroll
    for (int i = 0; i < N; ++i) r[i] = fmaf(r[i], v[i], w[i]);
  }
  if (act == GNNPN_ACT_RELU) {
#pragma unroll
    for (int i = 0; i < N; ++i) r[i] = fmaxf(r[i], 0.f);
  } else if (act == GNNPN_ACT_SIGMOID) {
#pragma unroll
    for (int i = 0; i < N; ++i) r[i] = sigmoid_accurate(r[i]);
  }
}

__device__ __forceinline__ float add_rn(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ double add_rn(double a, double b) { return __dadd_rn(a, b); }

// np.sum of a contiguous float32 / float64 vector, in numpy's order (pairwise_sum in
// numpy/core/src/umath/loops_utils.h.src): < 8 elements sequential, <= 128 elements eight running accumulators, above
// that a recursive split at n/2 rounded down to a multiple of 8.  The recursion is unrolled at compile time for
// n <= NMAX (a piece of n holds at most ceil(n/2) + 7 elements; NMAX = 512 unrolls three levels), so the kernel needs
// no device call stack.
template <int NMAX, class T>
__device__ __forceinline__ T numpy_sum(const T* a, int n) {
  if constexpr (NMAX > 128) {
    if (n > 128) {
      int n2 = n / 2;
      n2 -= n2 % 8;
      return add_rn(numpy_sum<NMAX / 2 + 8>(a, n2), numpy_sum<NMAX / 2 + 8>(a + n2, n - n2));
    }
  }
  if (n < 8) {
    T res = 0;
    for (int i = 0; i < n; ++i) res = add_rn(res, a[i]);
    return res;
  }
  T r[8];
  for (int j = 0; j < 8; ++j) r[j] = a[j];
  int i;
  for (i = 8; i < n - (n % 8); i += 8)
    for (int j = 0; j < 8; ++j) r[j] = add_rn(r[j], a[i + j]);
  T res = add_rn(add_rn(add_rn(r[0], r[1]), add_rn(r[2], r[3])), add_rn(add_rn(r[4], r[5]), add_rn(r[6], r[7])));
  for (; i < n; ++i) res = add_rn(res, a[i]);
  return res;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// 128-bit streaming load that does not allocate in L1 (read-once data).
__device__ __forceinline__ float4 ldg_stream(const float4* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}

}  // namespace gnnpn

#define GNNPN_REQUIRE(cond, code) \
  do {                            \
    if (!(cond)) return (code);   \
  } while (0)
