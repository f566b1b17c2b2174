// ML stage graph kernels: edge_index -> CSR (+ gcn_norm), CSR segment-reduce aggregation.
#include <cub/device/device_radix_sort.cuh>
#include "common.cuh"

namespace gnnpn {
namespace {

// ------------------------------------------------------------------ CSR build
// Virtual edge list (PyG add_remaining_self_loops order): the E original edges, then one loop per
// node.  In GCN mode an original self loop is dropped (key = n_nodes sentinel) and its weight moves
// to the appended loop of that node (last one in edge order wins, as sequential index_put does).
__global__ void csr_keys_kernel(const int64_t* __restrict__ edge_index, int64_t E, int64_t Nn, int gcn,
                                int32_t* __restrict__ keys, int32_t* __restrict__ payload,
                                int32_t* __restrict__ loop_eid) {
  const int64_t total = E + (gcn ? Nn : 0);
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total;
       e += (int64_t)gridDim.x * blockDim.x) {
    payload[e] = (int32_t)e;
    if (e < E) {
      const int64_t s = edge_index[e], d = edge_index[E + e];
      if (gcn && s == d) {
        keys[e] = (int32_t)Nn;
        atomicMax(&loop_eid[s], (int32_t)e);      // integer max: order-independent, deterministic
      } else {
        keys[e] = (int32_t)d;
      }
    } else {
      keys[e] = (int32_t)(e - E);
    }
  }
}

__global__ void fill_i32_kernel(int32_t* p, int64_t n, int32_t v) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    p[i] = v;
}

// rowptr[i] = first sorted position whose key >= i  (no atomics; i in [0, Nn])
__global__ void csr_rowptr_kernel(const int32_t* __restrict__ sorted_keys, int64_t total, int64_t Nn,
                                  int64_t* __restrict__ rowptr, int64_t* __restrict__ nnz_out) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i <= Nn;
       i += (int64_t)gridDim.x * blockDim.x) {
    int64_t lo = 0, hi = total;
    while (lo < hi) {
      const int64_t mid = (lo + hi) >> 1;
      if ((int64_t)sorted_keys[mid] < i) lo = mid + 1; else hi = mid;
    }
    rowptr[i] = lo;
    if (i == Nn && nnz_out) *nnz_out = lo;
  }
}

__global__ void csr_fill_kernel(const int64_t* __restrict__ edge_index, const float* __restrict__ w,
                                int64_t E, const int32_t* __restrict__ sorted_payload, int64_t nnz,
                                const int32_t* __restrict__ loop_eid, int gcn, int32_t* __restrict__ col,
                                float* __restrict__ val) {
  for (int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; p < nnz;
       p += (int64_t)gridDim.x * blockDim.x) {
    const int64_t e = sorted_payload[p];
    if (e < E) {
      col[p] = (int32_t)edge_index[e];
      if (val) val[p] = w ? w[e] : 1.0f;
    } else {
      const int64_t node = e - E;
      col[p] = (int32_t)node;
      const int32_t le = loop_eid[node];
      val[p] = (le >= 0 && w) ? w[le] : 1.0f;
    }
  }
}

// deg[i] = sum of the row's weights in CSR (= edge) order; dis = deg^-1/2 with inf -> 0
__global__ void gcn_degree_kernel(const int64_t* __restrict__ rowptr, const float* __restrict__ val,
                                  int64_t Nn, float* __restrict__ dis) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < Nn;
       i += (int64_t)gridDim.x * blockDim.x) {
    float d = 0.f;
    for (int64_t p = rowptr[i]; p < rowptr[i + 1]; ++p) d = __fadd_rn(d, val[p]);
    float r = __fdiv_rn(1.0f, __fsqrt_rn(d));
    if (isinf(r)) r = 0.f;
    dis[i] = r;
  }
}

__global__ void gcn_scale_kernel(const int64_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                 const float* __restrict__ dis, int64_t Nn, float* __restrict__ val) {
  // one warp per row: val = (dis[src] * w) * dis[dst]
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t i = warp; i < Nn; i += nwarps) {
    const float di = dis[i];
    for (int64_t p = rowptr[i] + lane; p < rowptr[i + 1]; p += 32)
      val[p] = __fmul_rn(__fmul_rn(dis[col[p]], val[p]), di);
  }
}

int key_bits(int64_t Nn) {
  int b = 1;
  while ((1ll << b) <= Nn) ++b;      // keys go up to Nn (sentinel)
  return b;
}

inline size_t al(size_t x) { return (x + 255) & ~size_t(255); }      // workspace arrays start at 256-byte offsets

struct CsrWorkspace {
  size_t keys_in, keys_out, pay_in, pay_out, loop_eid, dis, cub, total;
};

CsrWorkspace csr_layout(int64_t Nn, int64_t E, int mode) {
  const int64_t total = E + (mode == GNNPN_CSR_GCN_NORM ? Nn : 0);
  CsrWorkspace w{};
  size_t off = 0;
  w.keys_in = off;  off += al(total * 4);
  w.keys_out = off; off += al(total * 4);
  w.pay_in = off;   off += al(total * 4);
  w.pay_out = off;  off += al(total * 4);
  w.loop_eid = off; off += al((Nn + 1) * 4);
  w.dis = off;      off += al((Nn + 1) * 4);
  size_t cub_bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, cub_bytes, (const int32_t*)nullptr, (int32_t*)nullptr,
                                  (const int32_t*)nullptr, (int32_t*)nullptr, total, 0, key_bits(Nn));
  w.cub = off;      off += al(cub_bytes + 256);
  w.total = off;
  return w;
}

// ------------------------------------------------------------------ aggregation
// GROUP lanes own one destination row; lane g of the group owns float4 columns g, g+GROUP, ...
// Neighbour (col,val) pairs are staged 32 at a time per group through shared memory, gathers are
// issued UNROLL rows ahead, accumulation is strictly sequential in CSR order per feature
// (mul_rn then add_rn: bit-identical to the CPU index_add_ oracle).  Latency is hidden by occupancy (~60 registers, 4 CTAs of
// 8 warps per SM), not by per-thread pipelining: a variant that requested the next round of gathers and the next batch of
// (col, val) pairs ahead of the accumulation needed 104-128 registers and was slower everywhere (uniform F = 32: 0.91 ->
// 0.80 of the HBM peak, in-degree 8: 0.83 -> 0.55).
// --- shared pieces: one group's accumulation over the edge range [beg, end), and the row epilogue
template <int GROUP, int VPL, int UNROLL>
__device__ __forceinline__ void spmm_accumulate(float4 (&acc)[VPL], int64_t beg, int64_t end, const int32_t* __restrict__ col,
                                                const float* __restrict__ val, const float* __restrict__ x, int64_t ldx,
                                                int F4, int32_t* s_col, float* s_val, int gl, unsigned gmask) {
  for (int64_t e0 = beg; e0 < end; e0 += 32) {
    const int cnt = (int)min((int64_t)32, end - e0);
    __syncwarp(gmask);
    for (int i = gl; i < cnt; i += GROUP) {
      s_col[i] = __ldg(col + e0 + i);
      s_val[i] = val ? __ldg(val + e0 + i) : 1.0f;
    }
    __syncwarp(gmask);
    for (int j0 = 0; j0 < cnt; j0 += UNROLL) {
      float4 g[UNROLL][VPL];
      float w[UNROLL];
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {
        const int j = min(j0 + u, cnt - 1);
        w[u] = s_val[j];
        const float4* src = reinterpret_cast<const float4*>(x + (int64_t)s_col[j] * ldx);
#pragma unroll
        for (int v = 0; v < VPL; ++v) {
          const int c4 = gl + v * GROUP;
          g[u][v] = c4 < F4 ? __ldg(src + c4) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {
        if (j0 + u < cnt) {
#pragma unroll
          for (int v = 0; v < VPL; ++v) {
            acc[v].x = __fadd_rn(acc[v].x, __fmul_rn(w[u], g[u][v].x));
            acc[v].y = __fadd_rn(acc[v].y, __fmul_rn(w[u], g[u][v].y));
            acc[v].z = __fadd_rn(acc[v].z, __fmul_rn(w[u], g[u][v].z));
            acc[v].w = __fadd_rn(acc[v].w, __fmul_rn(w[u], g[u][v].w));
          }
        }
      }
    }
  }
}

struct SpmmEpilogue {
  float self_scale; int mean; const float* bias; const float* scale; const float* shift; int act;
};

template <int GROUP, int VPL>
__device__ __forceinline__ void spmm_finish_row(const float4 (&acc)[VPL], int64_t row, int64_t degree,
                                                const float* __restrict__ x, int64_t ldx, float* __restrict__ y,
                                                int64_t ldy, int F4, const SpmmEpilogue& ep, int gl) {
  const float inv_cnt_den = ep.mean ? (float)max((int64_t)1, degree) : 1.0f;
#pragma unroll
  for (int v = 0; v < VPL; ++v) {
    const int c4 = gl + v * GROUP;
    if (c4 >= F4) continue;
    float4 r = acc[v];
    if (ep.self_scale != 0.f) {
      const float4 xi = __ldg(reinterpret_cast<const float4*>(x + row * ldx) + c4);
      r.x = __fadd_rn(r.x, __fmul_rn(ep.self_scale, xi.x));
      r.y = __fadd_rn(r.y, __fmul_rn(ep.self_scale, xi.y));
      r.z = __fadd_rn(r.z, __fmul_rn(ep.self_scale, xi.z));
      r.w = __fadd_rn(r.w, __fmul_rn(ep.self_scale, xi.w));
    }
    if (ep.mean) {
      r.x = __fdiv_rn(r.x, inv_cnt_den); r.y = __fdiv_rn(r.y, inv_cnt_den);
      r.z = __fdiv_rn(r.z, inv_cnt_den); r.w = __fdiv_rn(r.w, inv_cnt_den);
    }
    bias_bn_act<4>(reinterpret_cast<float*>(&r), ep.bias, ep.scale, ep.shift, ep.act, [&](const float* p, float* x) {
      *reinterpret_cast<float4*>(x) = __ldg(reinterpret_cast<const float4*>(p) + c4);
    });
    reinterpret_cast<float4*>(y + row * ldy)[c4] = r;
  }
}

// long_threshold > 0: rows with more edges are left to the split path below (hub rows of a skewed graph)
template <int GROUP, int VPL, int UNROLL>
__global__ void __launch_bounds__(256) spmm_csr_kernel(
    const int64_t* __restrict__ rowptr, const int32_t* __restrict__ col, const float* __restrict__ val,
    const float* __restrict__ x, int64_t ldx, float* __restrict__ y, int64_t ldy, int64_t n_rows, int F4,
    const SpmmEpilogue ep, int64_t long_threshold) {
  constexpr int GROUPS_PER_CTA = 256 / GROUP;
  __shared__ int32_t s_col[GROUPS_PER_CTA][32];
  __shared__ float s_val[GROUPS_PER_CTA][32];

  const int gl = threadIdx.x % GROUP;                 // lane inside the group
  const int grp = threadIdx.x / GROUP;                // group inside the CTA
  const unsigned lane = threadIdx.x & 31;
  const unsigned gmask = GROUP == 32 ? 0xffffffffu : (((1u << GROUP) - 1u) << (lane / GROUP * GROUP));
  const int64_t row = (int64_t)blockIdx.x * GROUPS_PER_CTA + grp;
  if (row >= n_rows) return;
  const int64_t beg = rowptr[row], end = rowptr[row + 1];
  if (long_threshold > 0 && end - beg > long_threshold) return;

  float4 acc[VPL];
#pragma unroll
  for (int v = 0; v < VPL; ++v) acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
  spmm_accumulate<GROUP, VPL, UNROLL>(acc, beg, end, col, val, x, ldx, F4, s_col[grp], s_val[grp], gl, gmask);
  spmm_finish_row<GROUP, VPL>(acc, row, end - beg, x, ldx, y, ldy, F4, ep, gl);
}

// ---- long-row splitting (hub destinations: a service used by 10^5 compositions would otherwise be ONE group's
// sequential walk).  Rows with more than T edges are cut into chunks of Tc = chunk_len(T) consecutive edges; every chunk is summed
// by one group exactly like a short row (sequential in CSR order), the chunk sums are then added in chunk order.
// Deterministic (fixed order, no atomics in the arithmetic); rows of <= T edges stay bit-identical to index_add_ order,
// split rows differ from the strictly sequential sum by re-association only (~1e-7 relative; tests bound it by 1e-5).
// Edges per chunk of a split row of d edges: Tc, raised for hub rows so that no row has more than ~4096 chunks -- the
// combine walks a row's chunk sums in order (8 loads in flight), so a 7.8M-edge hub cut into 256-edge chunks would be a
// serial tail of 3,800 dependent L2 round trips (measured: 3 ms of a 12 ms launch)
constexpr int kMaxChunksPerRow = 4096;
__host__ __device__ inline int64_t chunk_len_row(int64_t d, int64_t Tc) {
  if (d <= Tc * kMaxChunksPerRow) return Tc;
  return ((d + kMaxChunksPerRow - 1) / kMaxChunksPerRow + 31) / 32 * 32;
}

struct LongRowPlan {
  int* counters;          // [0] number of long rows, [1] number of chunks
  int64_t* row;           // [max_long] row id per slot
  int* chunk_base;        // [max_long] first chunk of the slot's row
  int* chunk_slot;        // [max_chunks] slot a chunk belongs to
  float* partial;         // [max_chunks, F]
  int max_long, max_chunks;
};

__global__ void find_long_rows_kernel(const int64_t* __restrict__ rowptr, int64_t n_rows, int64_t T, int64_t Tc,
                                      LongRowPlan p) {
  for (int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; r < n_rows; r += (int64_t)gridDim.x * blockDim.x) {
    const int64_t d = rowptr[r + 1] - rowptr[r];
    if (d <= T) continue;
    const int64_t C = chunk_len_row(d, Tc);
    const int nch = (int)((d + C - 1) / C);
    const int slot = atomicAdd(p.counters, 1);
    const int cb = atomicAdd(p.counters + 1, nch);
    if (slot >= p.max_long || cb + nch > p.max_chunks) continue;        // cannot happen: both bounds follow from nnz / T
    p.row[slot] = r;
    p.chunk_base[slot] = cb;
    for (int i = 0; i < nch; ++i) p.chunk_slot[cb + i] = slot;
  }
}

template <int GROUP, int VPL, int UNROLL>
__global__ void __launch_bounds__(256) spmm_chunk_kernel(
    const int64_t* __restrict__ rowptr, const int32_t* __restrict__ col, const float* __restrict__ val,
    const float* __restrict__ x, int64_t ldx, int F4, int64_t T, const LongRowPlan p) {
  constexpr int GROUPS_PER_CTA = 256 / GROUP;
  __shared__ int32_t s_col[GROUPS_PER_CTA][32];
  __shared__ float s_val[GROUPS_PER_CTA][32];
  const int gl = threadIdx.x % GROUP, grp = threadIdx.x / GROUP;
  const unsigned lane = threadIdx.x & 31;
  const unsigned gmask = GROUP == 32 ? 0xffffffffu : (((1u << GROUP) - 1u) << (lane / GROUP * GROUP));
  const int n_chunks = min(p.counters[1], p.max_chunks);
  for (int c = blockIdx.x * GROUPS_PER_CTA + grp; c < n_chunks; c += gridDim.x * GROUPS_PER_CTA) {
    const int slot = p.chunk_slot[c];
    const int64_t row = p.row[slot];
    const int64_t rb = rowptr[row], re = rowptr[row + 1];
    const int64_t C = chunk_len_row(re - rb, T);
    const int64_t beg = rb + (int64_t)(c - p.chunk_base[slot]) * C;
    const int64_t end = min(beg + C, re);
    float4 acc[VPL];
#pragma unroll
    for (int v = 0; v < VPL; ++v) acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
    spmm_accumulate<GROUP, VPL, UNROLL>(acc, beg, end, col, val, x, ldx, F4, s_col[grp], s_val[grp], gl, gmask);
#pragma unroll
    for (int v = 0; v < VPL; ++v) {
      const int c4 = gl + v * GROUP;
      if (c4 < F4) reinterpret_cast<float4*>(p.partial + (int64_t)c * F4 * 4)[c4] = acc[v];
    }
  }
}

template <int GROUP, int VPL>
__global__ void __launch_bounds__(256) spmm_combine_kernel(
    const int64_t* __restrict__ rowptr, const float* __restrict__ x, int64_t ldx, float* __restrict__ y, int64_t ldy,
    int F4, int64_t T, const SpmmEpilogue ep, const LongRowPlan p) {
  constexpr int GROUPS_PER_CTA = 256 / GROUP;
  const int gl = threadIdx.x % GROUP, grp = threadIdx.x / GROUP;
  const int n_long = min(p.counters[0], p.max_long);
  for (int s = blockIdx.x * GROUPS_PER_CTA + grp; s < n_long; s += gridDim.x * GROUPS_PER_CTA) {
    const int64_t row = p.row[s];
    const int64_t d = rowptr[row + 1] - rowptr[row];
    const int64_t C = chunk_len_row(d, T);
    const int nch = (int)((d + C - 1) / C), cb = p.chunk_base[s];
    float4 acc[VPL];
#pragma unroll
    for (int v = 0; v < VPL; ++v) acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
    // chunk order = edge order; 8 chunk sums are requested together (independent loads) and then added in order, so a
    // hub row of 10^3..10^4 chunks is not a chain of that many dependent L2 round trips
    constexpr int CU = 8 / VPL;            // 8 float4 loads in flight per lane
    for (int i0 = 0; i0 < nch; i0 += CU) {
      float4 q[CU][VPL];
#pragma unroll
      for (int u = 0; u < CU; ++u) {
        const int i = min(i0 + u, nch - 1);
#pragma unroll
        for (int v = 0; v < VPL; ++v) {
          const int c4 = gl + v * GROUP;
          q[u][v] = c4 < F4 ? __ldcs(reinterpret_cast<const float4*>(p.partial + (int64_t)(cb + i) * F4 * 4) + c4)
                            : make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
#pragma unroll
      for (int u = 0; u < CU; ++u) {
        if (i0 + u < nch) {
#pragma unroll
          for (int v = 0; v < VPL; ++v) {
            if (i0 + u == 0) acc[v] = q[u][v];
            else {
              acc[v].x = __fadd_rn(acc[v].x, q[u][v].x); acc[v].y = __fadd_rn(acc[v].y, q[u][v].y);
              acc[v].z = __fadd_rn(acc[v].z, q[u][v].z); acc[v].w = __fadd_rn(acc[v].w, q[u][v].w);
            }
          }
        }
      }
    }
    spmm_finish_row<GROUP, VPL>(acc, row, d, x, ldx, y, ldy, F4, ep, gl);
  }
}

// NodeEncoder (modelML.py:9-29, only table 0 is reachable) + concat of the remaining float columns:
//   out[i, 0:E) = table[(int)x[i,0], :],  out[i, E:E+C-1) = x[i, 1:C),  zero padding up to ld_out
__global__ void embed_concat_kernel(const float* __restrict__ x, int64_t n, int C, const float* __restrict__ table,
                                    int rows, int E, float* __restrict__ out, int64_t ld_out) {
  const int64_t total = n * ld_out;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total;
       e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = e / ld_out;
    const int j = (int)(e % ld_out);
    float v = 0.f;
    if (j < E) {
      int t = (int)x[i * C];
      t = t < 0 ? 0 : (t >= rows ? rows - 1 : t);
      v = table[(int64_t)t * E + j];
    } else if (j < E + C - 1) {
      v = x[i * C + 1 + (j - E)];
    }
    out[e] = v;
  }
}

inline int64_t chunk_len(int64_t T) {                                       // edges per chunk of a split row
  // 256 edges = 8 staging rounds: amortises the chunk's dependent look-ups (slot -> row -> rowptr).  Chunks of 32 made the
  // chunk pass 3x slower per edge than the short-row kernel (scripts/agg_threshold_probe.py)
  return T / 8 < 256 ? 256 : T / 8;
}

template <int GROUP, int VPL, int UNROLL>
int launch_spmm(const int64_t* rowptr, const int32_t* col, const float* val, const float* x, int64_t ldx,
                float* y, int64_t ldy, int64_t n_rows, int F4, const SpmmEpilogue& ep, int64_t T, const LongRowPlan* plan,
                cudaStream_t st) {
  constexpr int GROUPS_PER_CTA = 256 / GROUP;
  const int64_t blocks = ceil_div(n_rows, GROUPS_PER_CTA);
  if (blocks > 0x7fffffffll) return GNNPN_ERANGE;
  int rc;
  if (plan) {
    cudaMemsetAsync(plan->counters, 0, 2 * sizeof(int), st);
    const int64_t fb = ceil_div(n_rows, 256);
    find_long_rows_kernel<<<(unsigned)(fb < 8 * kNumSMs ? fb : 8 * kNumSMs), 256, 0, st>>>(rowptr, n_rows, T, chunk_len(T), *plan);
    if ((rc = after_launch())) return rc;
  }
  spmm_csr_kernel<GROUP, VPL, UNROLL><<<(unsigned)blocks, 256, 0, st>>>(rowptr, col, val, x, ldx, y, ldy, n_rows, F4, ep,
                                                                       plan ? T : 0);
  if ((rc = after_launch()) || !plan) return rc;
  // persistent grids: they read the chunk / row counts on the device and return at once when there is no long row.  The
  // chunk grid is exactly one resident wave (the static stride gives every CTA the same share: CTAs that only start when
  // others finish -- 8 per SM were launched where 5-6 fit -- ran a second, mostly empty pass: 0.59 -> 0.8 of the HBM peak)
  static const int chunk_ctas_per_sm = [] {
    int nb = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, spmm_chunk_kernel<GROUP, VPL, UNROLL>, 256, 0) != cudaSuccess || nb < 1) {
      cudaGetLastError();
      nb = 4;
    }
    return nb;
  }();
  spmm_chunk_kernel<GROUP, VPL, UNROLL><<<chunk_ctas_per_sm * kNumSMs, 256, 0, st>>>(rowptr, col, val, x, ldx, F4, chunk_len(T), *plan);
  if ((rc = after_launch())) return rc;
  spmm_combine_kernel<GROUP, VPL><<<kNumSMs, 256, 0, st>>>(rowptr, x, ldx, y, ldy, F4, chunk_len(T), ep, *plan);
  return after_launch();
}

template <int G, int V, int U>
struct SpmmShape { static constexpr int GROUP = G, VPL = V, UNROLL = U; };

// The lane-group table: calls fn with the SpmmShape whose kernels aggregate F4 float4 columns (32 / GROUP rows per warp)
template <class Fn>
auto with_spmm_shape(int F4, Fn&& fn) {
  if (F4 <= 8) return fn(SpmmShape<8, 1, 8>{});
  if (F4 <= 16) return fn(SpmmShape<16, 1, 8>{});
  if (F4 <= 32) return fn(SpmmShape<32, 1, 8>{});
  if (F4 <= 64) return fn(SpmmShape<32, 2, 4>{});
  if (F4 <= 128) return fn(SpmmShape<32, 4, 2>{});
  return fn(SpmmShape<32, 8, 1>{});
}

// The long-row threshold a call runs with (0: no split): `requested` when it is >= 0, else the library's choice.
// - Below 2^22 edges nothing is split: there the split path's three extra (tiny) launches cost more than a hub row.
// - Where the lane group is narrower than a warp, 4 or 2 rows share a warp and a 10^3-edge row idles its warp mates, so
//   rows of more than 256 edges are split (in-degree-Zipf sweep, F = 32: 0.53 -> 0.59 of the HBM peak, F = 64: 0.68 ->
//   0.72).
// - Otherwise rows of more than 2048 edges are split.  The QWS co-usage graph's largest row has 1,378 edges: never split,
//   bit-identical to index_add_.
int64_t resolve_long_row_threshold(int64_t nnz, int F, int64_t requested) {
  if (requested >= 0) return requested;
  if (nnz < (int64_t(1) << 22)) return 0;
  return with_spmm_shape(F / 4, [](auto s) -> int64_t { return decltype(s)::GROUP < 32 ? 256 : 2048; });
}

// Workspace of the long-row plan of nnz edges, F columns and threshold T: the LongRowPlan arrays and their capacities
struct LongRowLayout {
  int64_t max_long, max_chunks;
  size_t counters, row, chunk_base, chunk_slot, partial, total;
};

LongRowLayout long_row_layout(int64_t nnz, int F, int64_t T) {
  LongRowLayout w{};
  w.max_long = nnz / (T + 1) + 1;                           // a long row has at least T + 1 edges
  w.max_chunks = nnz / chunk_len(T) + w.max_long + 1;       // sum of ceil(d / Tc) over the long rows
  size_t off = 0;
  w.counters = off;   off += al(2 * sizeof(int));
  w.row = off;        off += al(w.max_long * sizeof(int64_t));
  w.chunk_base = off; off += al(w.max_long * sizeof(int));
  w.chunk_slot = off; off += al(w.max_chunks * sizeof(int));
  w.partial = off;    off += al(w.max_chunks * F * sizeof(float));     // read and written as float4
  w.total = off;
  return w;
}

}  // namespace
}  // namespace gnnpn

using namespace gnnpn;

extern "C" {

int gnnpn_csr_build_workspace_bytes(int64_t n_nodes, int64_t n_edges, int mode, size_t* bytes) {
  GNNPN_REQUIRE(bytes, GNNPN_ENULL);
  GNNPN_REQUIRE(n_nodes >= 0 && n_edges >= 0 && (mode == GNNPN_CSR_PLAIN || mode == GNNPN_CSR_GCN_NORM),
                GNNPN_ESHAPE);
  GNNPN_REQUIRE(n_nodes < 0x7fffffffll && n_edges + n_nodes < 0x7fffffffll, GNNPN_ERANGE);
  *bytes = csr_layout(n_nodes, n_edges, mode).total;
  return GNNPN_OK;
}

int gnnpn_csr_build(const int64_t* edge_index, const float* edge_weight, int64_t E, int64_t Nn, int mode,
                    int64_t* rowptr, int32_t* col, float* val, int64_t* nnz_out, void* workspace,
                    size_t workspace_bytes, void* stream) {
  GNNPN_REQUIRE(rowptr && col && workspace && (edge_index || E == 0), GNNPN_ENULL);
  GNNPN_REQUIRE(Nn >= 0 && E >= 0 && (mode == GNNPN_CSR_PLAIN || mode == GNNPN_CSR_GCN_NORM), GNNPN_ESHAPE);
  GNNPN_REQUIRE(Nn < 0x7fffffffll && E + Nn < 0x7fffffffll, GNNPN_ERANGE);
  const int gcn = mode == GNNPN_CSR_GCN_NORM;
  GNNPN_REQUIRE(!gcn || val, GNNPN_ENULL);
  GNNPN_REQUIRE(!edge_weight || val, GNNPN_ENULL);
  const CsrWorkspace w = csr_layout(Nn, E, mode);
  GNNPN_REQUIRE(workspace_bytes >= w.total, GNNPN_EWORKSPACE);
  cudaStream_t st = (cudaStream_t)stream;
  char* ws = (char*)workspace;
  int32_t* keys_in = (int32_t*)(ws + w.keys_in);
  int32_t* keys_out = (int32_t*)(ws + w.keys_out);
  int32_t* pay_in = (int32_t*)(ws + w.pay_in);
  int32_t* pay_out = (int32_t*)(ws + w.pay_out);
  int32_t* loop_eid = (int32_t*)(ws + w.loop_eid);
  float* dis = (float*)(ws + w.dis);
  const int64_t total = E + (gcn ? Nn : 0);
  const int grid = kNumSMs * 8;
  int rc;
  if (gcn) {
    fill_i32_kernel<<<grid, 256, 0, st>>>(loop_eid, Nn, -1);
    if ((rc = after_launch())) return rc;
  }
  if (total > 0) {
    csr_keys_kernel<<<grid, 256, 0, st>>>(edge_index, E, Nn, gcn, keys_in, pay_in, loop_eid);
    if ((rc = after_launch())) return rc;
    size_t cub_bytes = workspace_bytes - w.cub;
    cudaError_t ce = cub::DeviceRadixSort::SortPairs(ws + w.cub, cub_bytes, keys_in, keys_out, pay_in, pay_out,
                                                     total, 0, key_bits(Nn), st);
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    if (ce != cudaSuccess) return (int)ce;
  }
  csr_rowptr_kernel<<<grid, 256, 0, st>>>(keys_out, total, Nn, rowptr, nnz_out);
  if ((rc = after_launch())) return rc;
  if (total > 0) {
    // entries with the sentinel key sort last and are simply not covered by rowptr[Nn]
    csr_fill_kernel<<<grid, 256, 0, st>>>(edge_index, edge_weight, E, pay_out, total, loop_eid, gcn, col, val);
    if ((rc = after_launch())) return rc;
  }
  if (gcn && Nn > 0) {
    gcn_degree_kernel<<<grid, 256, 0, st>>>(rowptr, val, Nn, dis);
    if ((rc = after_launch())) return rc;
    gcn_scale_kernel<<<grid, 256, 0, st>>>(rowptr, col, dis, Nn, val);
    if ((rc = after_launch())) return rc;
  }
  return GNNPN_OK;
}

int gnnpn_embed_concat_f32(const float* x, int64_t n, int n_cols, const float* table, int table_rows,
                           int embed_dim, float* out, int64_t ld_out, void* stream) {
  GNNPN_REQUIRE(x && table && out, GNNPN_ENULL);
  GNNPN_REQUIRE(n >= 0 && n_cols >= 1 && table_rows >= 1 && embed_dim >= 1 && ld_out >= embed_dim + n_cols - 1,
                GNNPN_ESHAPE);
  if (n == 0) return GNNPN_OK;
  embed_concat_kernel<<<kNumSMs * 4, 256, 0, (cudaStream_t)stream>>>(x, n, n_cols, table, table_rows, embed_dim,
                                                                     out, ld_out);
  return after_launch();
}

size_t gnnpn_spmm_csr_workspace_bytes(int64_t nnz, int F, int64_t long_row_threshold) {
  if (nnz < 0 || F < 4 || (long_row_threshold > 0 && long_row_threshold < 32)) return 0;
  const int64_t T = resolve_long_row_threshold(nnz, F, long_row_threshold);
  return T ? long_row_layout(nnz, F, T).total : 0;
}

int gnnpn_spmm_csr_f32(const int64_t* rowptr, const int32_t* col, const float* val, const float* x, int64_t ldx,
                       float* y, int64_t ldy, int64_t n_rows, int64_t nnz, int F, float self_scale, int mean,
                       const float* bias, const float* scale, const float* shift, int act, int64_t long_row_threshold,
                       void* workspace, size_t workspace_bytes, void* stream) {
  GNNPN_REQUIRE(rowptr && (col || n_rows == 0) && x && y, GNNPN_ENULL);
  GNNPN_REQUIRE(F >= 4 && F % 4 == 0 && F <= 1024 && ldx % 4 == 0 && ldy % 4 == 0 && ldx >= F && ldy >= F && nnz >= 0 &&
                    (long_row_threshold <= 0 || long_row_threshold >= 32),
                GNNPN_ESHAPE);
  GNNPN_REQUIRE((scale == nullptr) == (shift == nullptr), GNNPN_ENULL);
  GNNPN_REQUIRE(aligned16(x) && aligned16(y) && aligned16(bias) && aligned16(scale) && aligned16(shift), GNNPN_EALIGN);
  const int64_t T = resolve_long_row_threshold(nnz, F, long_row_threshold);
  LongRowPlan plan{};
  if (T) {
    GNNPN_REQUIRE(workspace, GNNPN_ENULL);
    GNNPN_REQUIRE(nnz < (1ll << 31) * (int64_t)32, GNNPN_ERANGE);
    const LongRowLayout w = long_row_layout(nnz, F, T);
    GNNPN_REQUIRE(workspace_bytes >= w.total, GNNPN_EWORKSPACE);
    GNNPN_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255u) == 0, GNNPN_EALIGN);
    uint8_t* ws = static_cast<uint8_t*>(workspace);
    plan.counters = reinterpret_cast<int*>(ws + w.counters);
    plan.row = reinterpret_cast<int64_t*>(ws + w.row);
    plan.chunk_base = reinterpret_cast<int*>(ws + w.chunk_base);
    plan.chunk_slot = reinterpret_cast<int*>(ws + w.chunk_slot);
    plan.partial = reinterpret_cast<float*>(ws + w.partial);
    plan.max_long = (int)w.max_long;
    plan.max_chunks = (int)w.max_chunks;
  }
  if (n_rows == 0) return GNNPN_OK;
  const SpmmEpilogue ep{self_scale, mean, bias, scale, shift, act};
  return with_spmm_shape(F / 4, [&](auto s) {
    using S = decltype(s);
    return launch_spmm<S::GROUP, S::VPL, S::UNROLL>(rowptr, col, val, x, ldx, y, ldy, n_rows, F / 4, ep, T,
                                                    T ? &plan : nullptr, (cudaStream_t)stream);
  });
}

}  // extern "C"
