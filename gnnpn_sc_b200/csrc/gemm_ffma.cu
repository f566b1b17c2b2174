// Strict-fp32 FFMA node transform:  C = act((A . W^T + bias) * scale + shift).
// Parity anchor and small-shape path (request graphs have <= ~100 nodes per batch, K = 28/128/256), and the range
// guard of the node transform; the large service-side transforms go through the tcgen05 kernels in node_transform.cu
// and tc_kernels.cu (gnnpn_gemm_f32_bias_act in abi.cu picks the kernel).
#include "common.cuh"
#include "internal.cuh"

namespace gnnpn {
namespace {

constexpr int TM = 64, TN = 64, TK = 16, TPB = 256;

// One [TM x TN] output tile.  `only_if` != nullptr: the launch is a guarded fall-back -- the whole grid returns at once
// unless *only_if is non-zero (the tcgen05 node transform sets it when an input is outside the fp16-split range),
// and the (persistent) grid then walks all tiles.
template <bool GUARDED>
__global__ void __launch_bounds__(TPB) gemm_ffma_kernel(
    const float* __restrict__ A, int64_t lda, const float* __restrict__ W, int64_t ldw,
    const float* __restrict__ bias, const float* __restrict__ scale, const float* __restrict__ shift,
    int act, float* __restrict__ C, int64_t ldc, int64_t M, int N, int K, const int* __restrict__ only_if) {
  __shared__ float As[TK][TM + 1];
  __shared__ float Ws[TK][TN + 1];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  if (GUARDED && *only_if == 0) return;
  const int64_t tiles_m = (M + TM - 1) / TM, tiles_n = (N + TN - 1) / TN;
  for (int64_t tile = GUARDED ? blockIdx.x : 0; tile < (GUARDED ? tiles_m * tiles_n : 1); tile += gridDim.x) {
  const int64_t m0 = (GUARDED ? tile / tiles_n : (int64_t)blockIdx.x) * TM;
  const int n0 = (int)(GUARDED ? tile % tiles_n : blockIdx.y) * TN;
  const int lr = tid >> 2;          // 0..63: tile row loaded by this thread
  const int lk = (tid & 3) * 4;     // 0,4,8,12: first of 4 k-columns
  float acc[4][4] = {};
  for (int k0 = 0; k0 < K; k0 += TK) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int k = k0 + lk + i;
      const int64_t am = m0 + lr;
      const int wn = n0 + lr;
      As[lk + i][lr] = (am < M && k < K) ? __ldg(A + am * lda + k) : 0.f;
      Ws[lk + i][lr] = (wn < N && k < K) ? __ldg(W + (int64_t)wn * ldw + k) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < TK; ++kk) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { a[i] = As[kk][ty * 4 + i]; b[i] = Ws[kk][tx * 4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t m = m0 + ty * 4 + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int nn = n0 + tx * 4 + j;
      if (nn >= N) continue;
      float v = acc[i][j];
      bias_bn_act<1>(&v, bias, scale, shift, act, [&](const float* p, float* x) { x[0] = __ldg(p + nn); });
      C[m * ldc + nn] = v;
    }
  }
  if (GUARDED) __syncthreads();
  }
}

}  // namespace

int launch_gemm_ffma(const float* A, int64_t lda, const float* W, int64_t ldw, const float* bias,
                     const float* scale, const float* shift, int act, float* C, int64_t ldc, int64_t M, int N,
                     int K, cudaStream_t st) {
  dim3 grid((unsigned)ceil_div(M, TM), (unsigned)ceil_div(N, TN));
  gemm_ffma_kernel<false><<<grid, TPB, 0, st>>>(A, lda, W, ldw, bias, scale, shift, act, C, ldc, M, N, K, nullptr);
  return after_launch();
}

// Guarded fall-back (persistent grid): recomputes C with strict-fp32 FFMAs iff *only_if != 0, else returns immediately.
int launch_gemm_ffma_if(const int* only_if, const float* A, int64_t lda, const float* W, int64_t ldw, const float* bias,
                        const float* scale, const float* shift, int act, float* C, int64_t ldc, int64_t M, int N,
                        int K, cudaStream_t st) {
  const int64_t tiles = ceil_div(M, TM) * ceil_div(N, TN);
  const unsigned grid = (unsigned)(tiles < 8 * kNumSMs ? tiles : 8 * kNumSMs);
  gemm_ffma_kernel<true><<<grid, TPB, 0, st>>>(A, lda, W, ldw, bias, scale, shift, act, C, ldc, M, N, K, only_if);
  return after_launch();
}

}  // namespace gnnpn
