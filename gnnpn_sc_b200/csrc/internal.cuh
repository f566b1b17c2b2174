// Host functions that one .cu file of the library defines and another calls, declared once so that a signature change
// is a compile error instead of a silent mismatch at link time, and the host launch helpers they share.  (The LSTM and
// scan kernels keep theirs with their argument structs: lstm_step.cuh, tc_lstm.cuh, tc_seq.cuh.)
#pragma once
#include <cuda.h>
#include "common.cuh"

namespace gnnpn {

// gemm_ffma.cu: strict-fp32  C = act((A . W^T + bias) * scale + shift);  the _if form returns at once unless *only_if != 0
int launch_gemm_ffma(const float* A, int64_t lda, const float* W, int64_t ldw, const float* bias, const float* scale,
                     const float* shift, int act, float* C, int64_t ldc, int64_t M, int N, int K, cudaStream_t st);
int launch_gemm_ffma_if(const int* only_if, const float* A, int64_t lda, const float* W, int64_t ldw, const float* bias,
                        const float* scale, const float* shift, int act, float* C, int64_t ldc, int64_t M, int N, int K,
                        cudaStream_t st);

// tc_kernels.cu: the same contraction on tcgen05 as error-compensated 3xTF32
size_t tc_gemm_workspace_bytes(int64_t M, int N, int K);
int launch_gemm_tc(const float* A, int64_t lda, const float* W, int64_t ldw, const float* bias, const float* scale,
                   const float* shift, int act, float* C, int64_t ldc, int64_t M, int N, int K, void* workspace,
                   cudaStream_t st);

// node_transform.cu: persistent fp16-split node transform: K <= 256, N <= 256, N % 16 == 0, K % 4 == 0; A 16-byte
// aligned with lda % 4 == 0 (plan_gemm in abi.cu)
bool node_transform_supported(int64_t M, int N, int K);
size_t node_transform_workspace_bytes(int N, int K);
int launch_node_transform(const float* A, int64_t lda, const float* W, int64_t ldw, const float* bias,
                          const float* scale, const float* shift, int act, float* C, int64_t ldc, int64_t M, int N,
                          int K, void* workspace, cudaStream_t st);

// pn_bptt.cu: BPTT through one LSTM of T steps as one cluster scan (arguments: bptt::Args).  `scratch` is unused: the
// signature is that of launch_bptt_steps (pn_train.cu), the per-step reference, so that a caller picks one of the two.
int launch_bptt_scan(const float* gates, const float* c, const float* c_init, const float* dh_ext, int64_t dh_ld_m,
                     const float* dh_init, const float* dc_init, const float* w_hh, float* dG_T, float* dh_out,
                     float* dc_out, int64_t n, int T, float* scratch, cudaStream_t st);

namespace tc {
// cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time libcuda dependency); nullptr when the
// driver does not provide it
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_fn();
// row-major [rows, cols] fp32 (or fp16) with leading dimension ld (elements); box = {box_cols (default: 128 bytes of
// columns), box_rows}; 128B swizzle, or 32B for 32-byte box rows
int make_map_2d(CUtensorMap* m, const void* base, int64_t rows, int64_t cols, int64_t ld, int box_rows, bool f16 = false,
                int box_cols = 0);
}  // namespace tc

// Launch configuration of `Kern` for a 1-D grid of 1-D clusters of `cluster` CTAs, setting the kernel's dynamic
// shared-memory limit on first use.  `attr` receives the cluster-dimension attribute `cfg` points at.
template <auto Kern>
int cluster_config(cudaLaunchConfig_t* cfg, cudaLaunchAttribute* attr, unsigned grid, unsigned cluster, int threads,
                   int smem, cudaStream_t st) {
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(Kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return (int)e;
    configured = true;
  }
  attr->id = cudaLaunchAttributeClusterDimension;
  attr->val.clusterDim = {cluster, 1, 1};
  *cfg = cudaLaunchConfig_t{dim3(grid), dim3(threads), (size_t)smem, st, attr, 1};
  return GNNPN_OK;
}
template <auto Kern, class... Args>
int launch_cluster(unsigned grid, unsigned cluster, int threads, int smem, cudaStream_t st, const Args&... args) {
  cudaLaunchConfig_t cfg;
  cudaLaunchAttribute attr;
  const int rc = cluster_config<Kern>(&cfg, &attr, grid, cluster, threads, smem, st);
  if (rc) return rc;
  const cudaError_t e = cudaLaunchKernelEx(&cfg, Kern, args...);
  if (e != cudaSuccess) { cudaGetLastError(); return (int)e; }
  return after_launch();
}

}  // namespace gnnpn
