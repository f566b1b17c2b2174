// Library-wide C ABI plumbing: version, error strings, launch counter, GEMM dispatch,
// host-buffer convenience entry for the PNLow -> PNHigh greedy decode.
#include <stdlib.h>
#include <string.h>
#include <vector>
#include "common.cuh"
#include "internal.cuh"
#include "options.cuh"

namespace gnnpn {
std::atomic<uint64_t> g_launch_count{0};

// initial option values come from the environment, read once at load time
static void env_int(const char* name, std::atomic<int>& dst) {
  const char* e = getenv(name);
  if (e && *e) dst.store(atoi(e), std::memory_order_relaxed);
}
Options& options() {
  static Options* o = [] {
    Options* x = new Options();
    env_int("GNNPN_COLSPLIT", x->scan);
    env_int("GNNPN_COLSPLIT_G", x->scan_groups);
    env_int("GNNPN_SEQ", x->persistent);
    env_int("GNNPN_SEQ_PROF", x->prof);
    env_int("GNNPN_BPTT", x->bptt);
    return x;
  }();
  return *o;
}
static std::atomic<int>* option_slot(const char* name) {
  if (!name) return nullptr;
  Options& o = options();
  if (!strcmp(name, "scan")) return &o.scan;
  if (!strcmp(name, "scan_groups")) return &o.scan_groups;
  if (!strcmp(name, "persistent")) return &o.persistent;
  if (!strcmp(name, "prof")) return &o.prof;
  if (!strcmp(name, "bptt")) return &o.bptt;
  return nullptr;
}
}  // namespace gnnpn

using namespace gnnpn;

extern "C" {

int gnnpn_abi_version(void) { return GNNPN_ABI_VERSION; }

uint64_t gnnpn_launch_count(void) { return g_launch_count.load(std::memory_order_relaxed); }

int gnnpn_set_option(const char* name, int value) {
  std::atomic<int>* s = option_slot(name);
  if (!s) return GNNPN_EUNSUPPORTED;
  s->store(value, std::memory_order_relaxed);
  return GNNPN_OK;
}

int gnnpn_get_option(const char* name, int* value) {
  std::atomic<int>* s = option_slot(name);
  if (!s || !value) return s ? GNNPN_ENULL : GNNPN_EUNSUPPORTED;
  *value = s->load(std::memory_order_relaxed);
  return GNNPN_OK;
}

const char* gnnpn_error_string(int code) {
  switch (code) {
    case GNNPN_OK: return "ok";
    case GNNPN_ENULL: return "required pointer is NULL";
    case GNNPN_ESHAPE: return "unsupported shape";
    case GNNPN_EALIGN: return "pointer or leading dimension not 16-byte aligned";
    case GNNPN_EWORKSPACE: return "workspace too small";
    case GNNPN_ERANGE: return "size exceeds the supported index range";
    case GNNPN_EUNSUPPORTED: return "variant not implemented by the CUDA path";
    default: break;
  }
  if (code > 0) return cudaGetErrorString((cudaError_t)code);
  return "unknown gnnpn error";
}

// The kernel gnnpn_gemm_f32_bias_act runs.  A misaligned A of a node-transform shape runs the FFMA kernel, which needs
// no workspace, so the workspace size, planned for an aligned A (nullptr, lda = K), holds for every A.
enum class GemmKernel { kFfma, kNodeTransform, kTf32 };
static GemmKernel plan_gemm(int64_t M, int N, int K, const float* A, int64_t lda, bool has_workspace) {
  if (!has_workspace) return GemmKernel::kFfma;
  if (!node_transform_supported(M, N, K)) return GemmKernel::kTf32;
  return aligned16(A) && (lda & 3) == 0 ? GemmKernel::kNodeTransform : GemmKernel::kFfma;
}

size_t gnnpn_gemm_workspace_bytes(int64_t M, int N, int K) {
  if (M < 0 || N < 1 || K < 1) return 0;
  return plan_gemm(M, N, K, nullptr, K, true) == GemmKernel::kNodeTransform ? node_transform_workspace_bytes(N, K)
                                                                            : tc_gemm_workspace_bytes(M, N, K);
}

int gnnpn_gemm_f32_bias_act(const float* A, int64_t lda, const float* W, int64_t ldw, const float* bias,
                            const float* scale, const float* shift, int act, float* C, int64_t ldc, int64_t M,
                            int N, int K, void* workspace, size_t workspace_bytes, void* stream) {
  GNNPN_REQUIRE(A && W && C, GNNPN_ENULL);
  GNNPN_REQUIRE(M >= 0 && N >= 1 && K >= 1 && lda >= K && ldw >= K && ldc >= N, GNNPN_ESHAPE);
  GNNPN_REQUIRE((scale == nullptr) == (shift == nullptr), GNNPN_ENULL);
  GNNPN_REQUIRE(M < (1ll << 31) * 64, GNNPN_ERANGE);
  if (M == 0) return GNNPN_OK;
  const cudaStream_t st = (cudaStream_t)stream;
  switch (plan_gemm(M, N, K, A, lda, workspace != nullptr)) {
    case GemmKernel::kNodeTransform:
      GNNPN_REQUIRE(workspace_bytes >= node_transform_workspace_bytes(N, K), GNNPN_EWORKSPACE);
      return launch_node_transform(A, lda, W, ldw, bias, scale, shift, act, C, ldc, M, N, K, workspace, st);
    case GemmKernel::kTf32:
      GNNPN_REQUIRE(workspace_bytes >= tc_gemm_workspace_bytes(M, N, K), GNNPN_EWORKSPACE);
      GNNPN_REQUIRE(M < (1ll << 31), GNNPN_ERANGE);
      return launch_gemm_tc(A, lda, W, ldw, bias, scale, shift, act, C, ldc, M, N, K, workspace, st);
    case GemmKernel::kFfma:
      break;
  }
  return launch_gemm_ffma(A, lda, W, ldw, bias, scale, shift, act, C, ldc, M, N, K, st);
}

// ---------------------------------------------------------------------------------------------
// Host-buffer path (what a non-torch caller of the reference's validation loop would bind):
// trainPNHigh.py:131-144  latent = low(greedy); high(greedy, latent) -> actions -> reward.
// Instances are processed in chunks so device scratch stays bounded (enc_out is L*H*4 B/instance).
// ---------------------------------------------------------------------------------------------
#define CUDA_TRY(x)                          \
  do {                                       \
    cudaError_t _e = (x);                    \
    if (_e != cudaSuccess) { rc = (int)_e; goto done; } \
  } while (0)
#define RC_TRY(x)            \
  do {                       \
    rc = (x);                \
    if (rc) goto done;       \
  } while (0)

int gnnpn_pn_greedy_low_high_host(const float* inputs_host, int64_t n, int L, int F, int H, int K, int N,
                                  const float* packed_low_host, const float* packed_high_host, int use_tanh,
                                  float C, float alpha, int32_t* idx_low_host, int32_t* idx_high_host,
                                  float* reward_high_host) {
  GNNPN_REQUIRE(inputs_host && packed_low_host && packed_high_host && idx_high_host, GNNPN_ENULL);
  GNNPN_REQUIRE(H == 256 && (int64_t)K * N == L, GNNPN_ESHAPE);
  int rc = GNNPN_OK;
  const int64_t chunk = n < 8192 ? n : 8192;
  const size_t pfloats = gnnpn_pn_packed_lstm_floats(H, F);
  float *d_in = nullptr, *d_enc = nullptr, *d_c = nullptr, *d_dech = nullptr, *d_wl_lo = nullptr, *d_wl_hi = nullptr,
        *d_wp = nullptr, *d_rew = nullptr, *d_pk = nullptr;
  void* d_ws = nullptr;
  const size_t ws_bytes = gnnpn_pn_workspace_bytes(chunk, H);
  int32_t *d_idx_lo = nullptr, *d_idx_hi = nullptr;
  cudaStream_t st = nullptr;
  if (n == 0) return GNNPN_OK;
  CUDA_TRY(cudaStreamCreate(&st));
  CUDA_TRY(cudaMalloc(&d_pk, 4 * pfloats * sizeof(float)));   // enc/dec blocks of low and high
  CUDA_TRY(cudaMalloc(&d_in, chunk * L * F * sizeof(float)));
  CUDA_TRY(cudaMalloc(&d_enc, gnnpn_pn_enc_out_floats(chunk, L, H, GNNPN_ENC_BLOCKED128) * sizeof(float)));
  CUDA_TRY(cudaMalloc(&d_c, chunk * H * sizeof(float)));
  CUDA_TRY(cudaMalloc(&d_dech, chunk * (size_t)K * H * sizeof(float)));
  CUDA_TRY(cudaMalloc(&d_wl_lo, chunk * L * sizeof(float)));
  CUDA_TRY(cudaMalloc(&d_wl_hi, chunk * L * sizeof(float)));
  CUDA_TRY(cudaMalloc(&d_wp, chunk * L * sizeof(float)));
  CUDA_TRY(cudaMalloc(&d_rew, chunk * sizeof(float)));
  CUDA_TRY(cudaMalloc(&d_idx_lo, chunk * K * sizeof(int32_t)));
  CUDA_TRY(cudaMalloc(&d_idx_hi, chunk * K * sizeof(int32_t)));
  CUDA_TRY(cudaMalloc(&d_ws, ws_bytes));
  // packed_*_host = [encoder block | decoder block], each gnnpn_pn_packed_lstm_floats() long
  CUDA_TRY(cudaMemcpyAsync(d_pk, packed_low_host, 2 * pfloats * sizeof(float), cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaMemcpyAsync(d_pk + 2 * pfloats, packed_high_host, 2 * pfloats * sizeof(float),
                           cudaMemcpyHostToDevice, st));
  for (int64_t s = 0; s < n; s += chunk) {
    const int64_t m = (n - s) < chunk ? (n - s) : chunk;
    const int layout = gnnpn_pn_enc_layout(m, L, F, K, N, 1);
    CUDA_TRY(cudaMemcpyAsync(d_in, inputs_host + s * L * F, m * L * F * sizeof(float), cudaMemcpyHostToDevice, st));
    for (int level = 0; level < 2; ++level) {
      const float* pk = d_pk + (size_t)level * 2 * pfloats;
      RC_TRY(gnnpn_lstm_encode_f32(d_in, m, L, F, H, pk, d_enc, d_c, d_ws, ws_bytes, layout, st));
      RC_TRY(gnnpn_pn_decode_greedy_f32(d_in, d_enc, d_c, level ? d_wl_lo : nullptr, alpha, pk + pfloats,
                                        GNNPN_ATT_DOT, nullptr, use_tanh, C, m, L, F, H, K, N, d_dech,
                                        level ? d_idx_hi : d_idx_lo, level ? d_wl_hi : d_wl_lo, d_wp, nullptr,
                                        nullptr, d_ws, ws_bytes, layout, st));
    }
    RC_TRY(gnnpn_pn_reward_f32(d_in, d_idx_hi, m, L, F, K, 0, nullptr, nullptr, d_rew, st));
    // device layout is [K, m]; the host result is [K, n]: copy row by row
    for (int k = 0; k < K; ++k) {
      if (idx_low_host)
        CUDA_TRY(cudaMemcpyAsync(idx_low_host + (int64_t)k * n + s, d_idx_lo + (int64_t)k * m, m * sizeof(int32_t),
                                 cudaMemcpyDeviceToHost, st));
      CUDA_TRY(cudaMemcpyAsync(idx_high_host + (int64_t)k * n + s, d_idx_hi + (int64_t)k * m, m * sizeof(int32_t),
                               cudaMemcpyDeviceToHost, st));
    }
    if (reward_high_host)
      CUDA_TRY(cudaMemcpyAsync(reward_high_host + s, d_rew, m * sizeof(float), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
  }
done:
  cudaFree(d_pk); cudaFree(d_in); cudaFree(d_enc); cudaFree(d_c); cudaFree(d_dech); cudaFree(d_wl_lo);
  cudaFree(d_ws); cudaFree(d_wl_hi); cudaFree(d_wp); cudaFree(d_rew); cudaFree(d_idx_lo); cudaFree(d_idx_hi);
  if (st) cudaStreamDestroy(st);
  return rc;
}

}  // extern "C"
