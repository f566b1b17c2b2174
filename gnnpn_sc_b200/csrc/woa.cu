// ESWOA fitness (src/baselines/WOA.py:87-105, `ESWOA.calc`) for a whole batch of whale positions in one launch.
//
// The reference evaluates one composition at a time in numpy float64 (popSize x MAX_Iter x instances calls):
//   conValues[i] = np.cumprod(q_{.,2+i})[-1]                  sequential float64 products, i in {0,1}
//   violate      = #{ i : conValues[i] < lo_i  or  conValues[i] > hi_i }
//   serviceNum   = #{ k : q_{k,0} > 0 }
//   objFunc      = (np.sum(q_{.,0}) / serviceNum + 1 - np.min(q_{.,1})) / 2
//   fitness      = violate + objFunc                          (WOA.py:59,78,119,151)
// One thread = one position; every float64 operation is issued in numpy's order (np.sum's 8-accumulator pairwise
// scheme included) so fitness values -- and therefore every comparison `bestFitness > fitness` of the search -- are
// bit-identical to the reference's.
#include <climits>

#include "common.cuh"

namespace gnnpn {
namespace {

// The fitness (violate + objFunc) of one composition of K <= KMAX picks, b the (lo, hi) pair of each product; violate
// and objFunc also go to viol_out and obj_out when given.  Pick k is row pos[k] of qos (kRow), or entry pos[k] of the
// task's list of size[k] rows from row base[k], a negative pos[k] counting from its end as in Python (kLocal).
// MEAN_ALL: `ML2PN.calc` (src/ML2PN.py:6-12): `np.average(qos[0])` over all K picks instead of sum / #{q0 > 0}, and
// 1.0 added to the objective once per violated constraint, in constraint order, instead of `violate + objFunc` in one
// add (with both violated, (obj + 1) + 1 and obj + 2 can round apart).
enum class WoaPick { kRow, kLocal };
template <int KMAX, bool MEAN_ALL, WoaPick PICK>
__device__ __forceinline__ double woa_fitness(const double* __restrict__ qos, const int32_t* pos, const int32_t* base,
                                              const int32_t* size, int K, const double* b, int* viol_out = nullptr,
                                              double* obj_out = nullptr) {
  double q0s[KMAX];
  double prod[2] = {1.0, 1.0};
  double min_q1 = INFINITY;
  int used = 0;
  for (int k = 0; k < K; ++k) {
    int r = pos[k];
    if constexpr (PICK == WoaPick::kLocal) {
      int v = r % size[k];
      if (v < 0) v += size[k];
      r = base[k] + v;
    }
    const double* row = qos + (int64_t)r * 4;
    q0s[k] = row[0];
    used += row[0] > 0.0;
    min_q1 = fmin(min_q1, row[1]);
    prod[0] = k == 0 ? row[2] : __dmul_rn(prod[0], row[2]);
    prod[1] = k == 0 ? row[3] : __dmul_rn(prod[1], row[3]);
  }
  int viol = 0;
  for (int i = 0; i < 2; ++i) viol += (prod[i] < b[2 * i] || prod[i] > b[2 * i + 1]) ? 1 : 0;
  double obj = __ddiv_rn(numpy_sum<KMAX>(q0s, K), (double)(MEAN_ALL ? K : used));
  obj = __dadd_rn(obj, 1.0);
  obj = __dsub_rn(obj, min_q1);
  obj = __ddiv_rn(obj, 2.0);
  if (viol_out) *viol_out = viol;
  if (obj_out) *obj_out = obj;
  if constexpr (MEAN_ALL) {
    double score = obj;
    for (int i = 0; i < 2; ++i)
      if (prod[i] < b[2 * i] || prod[i] > b[2 * i + 1]) score = __dadd_rn(score, 1.0);
    return score;
  }
  return __dadd_rn((double)viol, obj);
}

constexpr int kMaxTasksWoa = 512;     // picks per composition in woa_fitness_kernel
template <bool MEAN_ALL>
__global__ void woa_fitness_kernel(const double* __restrict__ qos, const int32_t* __restrict__ idx, int64_t idx_ld,
                                   const int32_t* __restrict__ klen, const double* __restrict__ bounds, int64_t P,
                                   int Kmax, int32_t* __restrict__ viol_out, double* __restrict__ obj_out,
                                   double* __restrict__ fit_out) {
  const int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (p >= P) return;
  const int K = klen ? klen[p] : Kmax;
  const double fit = woa_fitness<kMaxTasksWoa, MEAN_ALL, WoaPick::kRow>(
      qos, idx + p * idx_ld, nullptr, nullptr, K, bounds + p * 4, viol_out ? viol_out + p : nullptr,
      obj_out ? obj_out + p : nullptr);
  if (fit_out) fit_out[p] = fit;
}


// ------------------------------------------------------------------------------------------------------------------
// Device-resident ESWOA search (WOA.py:107-162): one CTA per composition instance, one thread per whale, all MAX_Iter
// iterations in one launch.  Same sequential semantics as the reference's loop (and as gnnpn_sc_b200/WOA.py's host
// engine): global phase = in-place mutations, best-so-far replayed in whale order; local phase = moves computed
// speculatively against the current best, committed up to the first improvement, the rest recomputed; `bestPops`
// aliasing kept (best_ref).  Random numbers are counter-based (Philox4x32-10, key = instance seed, counter =
// (slot, whale, phase, iteration)), so the host engine reproduces the run draw for draw with the same generator.
__device__ __forceinline__ void philox_round(uint32_t (&c)[4], uint32_t (&k)[2]) {
  const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
  const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
  const uint32_t n0 = hi1 ^ c[1] ^ k[0], n2 = hi0 ^ c[3] ^ k[1];
  c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
  k[0] += 0x9E3779B9u; k[1] += 0xBB67AE85u;
}
__device__ __forceinline__ double philox_uniform(uint64_t seed, uint32_t slot, uint32_t whale, uint32_t phase, uint32_t t) {
  uint32_t c[4] = {slot, whale, phase, t};
  uint32_t k[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
#pragma unroll
  for (int r = 0; r < 10; ++r) philox_round(c, k);
  return __dmul_rn(__dadd_rn(__dmul_rn((double)(c[0] >> 5), 67108864.0), (double)(c[1] >> 6)), 1.0 / 9007199254740992.0);
}
// one of n choices drawn with u = philox_uniform(...): floor(u * n) (host mirror: PhiloxRng.randint, .choice and .block)
__device__ __forceinline__ int philox_index(double u, int n) { return (int)__dmul_rn(u, (double)n); }

constexpr int kWoaMaxK = 128;       // tasks per instance in the device search
constexpr int kWoaThreads = 128;    // whales per instance (popSize <= 128)

struct WoaSearchArgs {
  const double* qos;        // [T, 4]
  const int32_t* base;      // [I, Kmax] first row of every task's candidate list
  const int32_t* size;      // [I, Kmax]
  const int32_t* klen;      // [I]
  const double* bounds;     // [I, 4]
  int32_t* pops;            // [I, P, Kmax] in/out
  double* best_fit;         // [I] in/out
  int32_t* best_ref;        // [I] in/out: whale whose row IS the best position, or -1
  int32_t* best_vec;        // [I, Kmax] in/out
  const uint64_t* seeds;    // [I]
  double* traj;             // [I, iters] best fitness after every iteration
  int P, Kmax, iters;
};

// one thread's best-so-far scan in whale order (`if bestFitness > fitness`, WOA.py:78-81,119-122); 1 if the best moved
__device__ __forceinline__ int scan_best(const double* fit, int P, double& best, int& ref) {
  int changed = 0;
  for (int w = 0; w < P; ++w)
    if (best > fit[w]) { best = fit[w]; ref = w; changed = 1; }
  return changed;
}

__global__ void __launch_bounds__(kWoaThreads) woa_search_kernel(const WoaSearchArgs a) {
  extern __shared__ double sm_d[];
  const int I = blockIdx.x, i = threadIdx.x;
  const int P = a.P, KM = a.Kmax, K = a.klen[I];
  double* fit = sm_d;                        // [P]
  int32_t* pos = reinterpret_cast<int32_t*>(sm_d + P);   // [P][KM]
  int32_t* newp = pos + P * KM;              // [P][KM] speculative moves
  int32_t* bestv = newp + P * KM;            // [KM]
  int32_t* sz = bestv + KM;
  int32_t* bs = sz + KM;
  int32_t* flag = bs + KM;                   // [P] has_move
  __shared__ double s_best;
  __shared__ int s_ref, s_nxt, s_star, s_skip;
  const uint64_t seed = a.seeds[I];
  const double* bnd = a.bounds + (int64_t)I * 4;
  for (int e = i; e < P * KM; e += blockDim.x) pos[e] = a.pops[(int64_t)I * P * KM + e];
  for (int e = i; e < KM; e += blockDim.x) {
    bestv[e] = a.best_vec[(int64_t)I * KM + e];
    sz[e] = e < K ? a.size[(int64_t)I * KM + e] : 1;
    bs[e] = e < K ? a.base[(int64_t)I * KM + e] : 0;
  }
  if (i == 0) { s_best = a.best_fit[I]; s_ref = a.best_ref[I]; }
  __syncthreads();
  const bool whale = i < P;
  for (int t = 0; t < a.iters; ++t) {
    // ---- global phase (WOA.py:110-122)
    const double prob = __dmul_rn(0.2, __dsub_rn(1.0, __ddiv_rn((double)t, (double)a.iters)));
    double f = INFINITY;
    if (whale && philox_uniform(seed, 0, i, 0, t) < prob) {
      const int rand = philox_index(philox_uniform(seed, 1, i, 0, t), K);
      const int randi = philox_index(philox_uniform(seed, 2, i, 0, t), sz[rand]);
      pos[i * KM + rand] = randi;
      if (s_ref == i) bestv[rand] = randi;                 // the best IS this whale's row: it moves with it
      f = woa_fitness<kWoaMaxK, false, WoaPick::kLocal>(a.qos, pos + i * KM, bs, sz, K, bnd);
    }
    if (whale) fit[i] = f;
    __syncthreads();
    if (i == 0) {
      int ref = s_ref; double best = s_best;
      const int changed = scan_best(fit, P, best, ref);
      s_best = best; s_ref = ref; s_star = changed;
      s_skip = 0.2 > philox_uniform(seed, 0, 0, 1, t);        // exploration skip (WOA.py:124-128)
    }
    __syncthreads();
    if (s_star) {
      for (int e = i; e < K; e += blockDim.x) bestv[e] = pos[s_ref * KM + e];
      __syncthreads();
    }
    if (!s_skip) {
      // ---- local phase (WOA.py:130-155)
      double A = 0, C = 0, e1 = 0, e2 = 0, pp = 1.0;
      if (whale) {
        const double aa = __dsub_rn(2.0, __ddiv_rn(__dmul_rn(2.0, (double)t), (double)a.iters));
        const double r = philox_uniform(seed, 0, i, 2, t), l = philox_uniform(seed, 1, i, 2, t);
        pp = philox_uniform(seed, 2, i, 2, t);
        A = __dsub_rn(__dmul_rn(__dmul_rn(2.0, aa), r), aa);
        C = __dmul_rn(2.0, r);
        e1 = exp(l);
        e2 = cos(__dmul_rn(__dmul_rn(2.0, 3.141592653589793), l));
      }
      const int mode = !whale ? 0 : (pp < 0.5 ? (fabs(A) < 1.0 ? 1 : 0) : 2);
      if (i == 0) s_nxt = 0;
      __syncthreads();
      while (true) {
        const int nxt = s_nxt;
        f = INFINITY;
        if (whale && i >= nxt) {
          flag[i] = mode != 0;
          if (mode) {
            for (int k = 0; k < K; ++k) {
              const double b = (double)bestv[k], x = (double)pos[i * KM + k];
              double v;
              if (mode == 1) v = __dsub_rn(b, __dmul_rn(A, __dsub_rn(__dmul_rn(C, b), x)));
              else v = __dadd_rn(__dmul_rn(__dmul_rn(__dsub_rn(x, b), e1), e2), b);
              int q = (int)rint(v);
              if (abs(q) >= sz[k]) { q %= sz[k]; if (q < 0) q += sz[k]; }
              newp[i * KM + k] = q;
            }
            f = woa_fitness<kWoaMaxK, false, WoaPick::kLocal>(a.qos, newp + i * KM, bs, sz, K, bnd);
          }
          fit[i] = f;
        }
        __syncthreads();
        if (i == 0) {
          int star = P;
          for (int w = nxt; w < P; ++w)
            if (flag[w] && s_best > fit[w]) { star = w; break; }
          s_star = star;
        }
        __syncthreads();
        const int star = s_star;
        const int old_ref = s_ref;
        __syncthreads();
        if (whale && i >= nxt && i <= star && flag[i]) {
          for (int k = 0; k < K; ++k) pos[i * KM + k] = newp[i * KM + k];
          if (old_ref == i && i != star) s_ref = -1;        // pops[i] was rebound: the old list stays the best (WOA.py:150)
        }
        __syncthreads();
        if (star < P) {
          for (int e = i; e < K; e += blockDim.x) bestv[e] = pos[star * KM + e];
          if (i == 0) { s_best = fit[star]; s_ref = star; s_nxt = star + 1; }
        }
        __syncthreads();
        if (star >= P || star + 1 >= P) break;
      }
    }
    if (i == 0) a.traj[(int64_t)I * a.iters + t] = s_best;
    __syncthreads();
  }
  for (int e = i; e < P * KM; e += blockDim.x) a.pops[(int64_t)I * P * KM + e] = pos[e];
  for (int e = i; e < KM; e += blockDim.x) a.best_vec[(int64_t)I * KM + e] = bestv[e];
  if (i == 0) { a.best_fit[I] = s_best; a.best_ref[I] = s_ref; }
}


// ------------------------------------------------------------------------------------------------------------------
// What the host does before the search starts (gnnpn_sc_b200/WOA.py: loadDataOther + _add_s, the seed preparation of
// WOA.start, _Instance.__init__ and _Engine._init_population, whose draws, fitness and best-so-far scan are
// philox_index, woa_fitness and scan_best as in the search), one CTA per instance, for gnnpn_woa_search_f64.
struct WoaPrepareArgs {
  const double* svc_raw;     // [S, 4] JSON values
  const double* svc_round;   // [S, 4] the same rounded to 5 decimals (Python `round`)
  const int32_t* cat_ptr;    // [K + 1]
  const int32_t* req_cat;    // [I, K] requested category per task, request-node order
  const int32_t* n_req;      // [I]
  const double* local;       // [I, K, 4] lo_cost, hi_cost, lo_q, hi_q per category
  const double* global;      // [I, 4]
  const float* seed_rows;    // [I, K, 4] PNHigh's pick per category
  const int32_t* seed_ids;   // [I, K]
  const uint64_t* seeds;     // [I]
  double* qos;               // [I * cap, 4]
  int32_t* ids;              // [I * cap]
  int32_t *base, *size, *klen, *list_cat, *pops, *best_ref, *best_vec, *flags;
  double* best_fit;
  double reduct;
  int64_t cap;
  int K, P;
};

// rows of the candidate table: every instance holds one slot of (category size + 1) rows per category, so a task's list
// and its seed append never need a scan to be placed
__host__ __device__ inline int64_t woa_prepare_rows(int64_t n_instances, int64_t n_services, int K) {
  return n_instances * (n_services + K);
}

// the six rounded rows the reference patches by hand (WOA.py:38-45): row -> (column, replacement)
__constant__ double kPatchRow[6][4] = {{0.05314, 0.55528, 0.94008, 0.95495}, {0.03922, 0.56097, 0.94131, 0.92804},
                                       {0.17292, 0.5995, 0.92651, 0.92459},  {0.33474, 0.55123, 0.90018, 0.97161},
                                       {0.73066, 0.40995, 0.90016, 0.92941}, {0.16904, 0.60902, 0.93639, 0.97272}};
__constant__ int kPatchCol[6] = {1, 1, 2, 3, 3, 2};
__constant__ double kPatchVal[6] = {0.55527, 0.56096, 0.92652, 0.9716, 0.92942, 0.9364};

constexpr uint32_t kFrontSentinel = 0x3FFFFFFFu;   // the front's first entry (1, 0, 1, 1), not a service
constexpr uint32_t kFrontProtected = 0x40000000u;  // the entry's rounded row is in sSet

__device__ __forceinline__ bool rows_equal(const double* a, const double* b) {
  return a[0] == b[0] && a[1] == b[1] && a[2] == b[2] && a[3] == b[3];
}

__global__ void __launch_bounds__(kWoaThreads) woa_prepare_kernel(const WoaPrepareArgs a) {
  const int I = blockIdx.x, tid = threadIdx.x, K = a.K, P = a.P;
  __shared__ double s_sset[kWoaMaxK][4];     // seed rows rounded (sSet)
  __shared__ double s_seed[kWoaMaxK][4];     // the same with the patches: the solution rows
  __shared__ int s_seed_id[kWoaMaxK];
  __shared__ int s_len[kWoaMaxK], s_off[kWoaMaxK], s_cat[kWoaMaxK];     // per task
  __shared__ int s_base[kWoaMaxK], s_size0[kWoaMaxK], s_size[kWoaMaxK], s_lcat[kWoaMaxK], s_match[kWoaMaxK], s_own[kWoaMaxK];
  __shared__ double s_fit[kWoaThreads];
  __shared__ int s_flag, s_ref;
  const int64_t row0 = (int64_t)I * a.cap;

  // ---- seed solution (WOA.start, WOA.py:591-594): PNHigh's picks in category order without the neutral rows
  bool keep = false;
  double raw[4];
  if (tid < K) {
    const float* r = a.seed_rows + ((int64_t)I * K + tid) * 4;
    for (int q = 0; q < 4; ++q) raw[q] = (double)r[q];
    // WOA.start's `sum(r) != 3`.  Python 3.12's sum is compensated (Neumaier), this one sequential; for four float32
    // values in [0, 1] every partial sum is exact, so the two agree, unless a nonzero value is below 2^-28
    keep = __dadd_rn(__dadd_rn(__dadd_rn(raw[0], raw[1]), raw[2]), raw[3]) != 3.0;
  }
  if (tid == 0) s_flag = 0;
  s_match[tid] = INT_MAX;
  s_len[tid] = 0;
  s_cat[tid] = keep;                             // borrowed until the task loop: which seed rows are kept
  const int ns = __syncthreads_count(keep);
  const bool seeded = ns > 0;
  if (keep) {
    int l = 0;                                   // position among the kept rows
    for (int k = 0; k < tid; ++k) l += s_cat[k];
    // float32 values times 1e5 are exact in double, so rint + divide is Python's round(x, 5)
    double rr[4];
    for (int q = 0; q < 4; ++q) rr[q] = __ddiv_rn(rint(__dmul_rn(raw[q], 1e5)), 1e5);
    for (int q = 0; q < 4; ++q) s_sset[l][q] = s_seed[l][q] = rr[q];
    for (int p = 0; p < 6; ++p)
      if (rows_equal(rr, kPatchRow[p])) s_seed[l][kPatchCol[p]] = kPatchVal[p];
    s_seed_id[l] = a.seed_ids[(int64_t)I * K + tid];
  }
  __syncthreads();

  // ---- candidate list of every requested task (loadDataOther + _add_s, WOA.py:484-555): one thread per task
  const int nreq = min(a.n_req[I], K);
  if (a.n_req[I] > K) atomicOr(&s_flag, 8);
  if (tid < nreq) {
    const int cat = a.req_cat[(int64_t)I * K + tid];
    bool ok = cat >= 0 && cat < K;
    for (int j = 0; ok && j < tid; ++j) ok = a.req_cat[(int64_t)I * K + j] != cat;
    if (!ok) atomicOr(&s_flag, 8);
    int len = 0;
    if (ok) {
      const int c0 = a.cat_ptr[cat], c1 = a.cat_ptr[cat + 1];
      const int off = c0 + cat;                   // the category's slot: its size + 1 rows (one seed append)
      s_off[tid] = off;
      s_cat[tid] = cat;
      const double* lb = a.local + ((int64_t)I * K + cat) * 4;
      const double lo_c = lb[0], hi_c = lb[1], lo_q = lb[2], hi_q = lb[3];
      int32_t* out = a.ids + row0 + off;
      // the running front lives in the slot's rows until they are written (it has at most size + 1 entries)
      uint32_t* front = reinterpret_cast<uint32_t*>(a.qos + (row0 + off) * 4);
      const double red = a.reduct;
      auto in_sset = [&](const double* r) {
        for (int l = 0; l < ns; ++l)
          if (rows_equal(r, s_sset[l])) return true;
        return false;
      };
      int nf = 0;
      if (red != 0.0) {
        const double sent[4] = {1.0, 0.0, 1.0, 1.0};
        front[nf++] = kFrontSentinel | (in_sset(sent) ? kFrontProtected : 0u);
      }
      for (int s = c0; s < c1; ++s) {
        const double* f = a.svc_raw + (int64_t)s * 4;
        const double q0 = f[0], q1 = f[1], cost = f[2], quality = f[3];
        if (!(lo_c <= cost && cost <= hi_c && lo_q <= quality && quality <= hi_q)) continue;
        if (red == 0.0) { out[len++] = s; continue; }
        const uint32_t prot = seeded && in_sset(a.svc_round + (int64_t)s * 4) ? kFrontProtected : 0u;
        bool replaced = false;
        for (int x = 0; x < nf; ++x) {
          const uint32_t e = front[x];
          if (e & kFrontProtected) continue;
          const uint32_t eid = e & kFrontSentinel;
          const double e0 = eid == kFrontSentinel ? 1.0 : a.svc_raw[(int64_t)eid * 4];
          const double e1 = eid == kFrontSentinel ? 0.0 : a.svc_raw[(int64_t)eid * 4 + 1];
          if (q0 < e0 && q1 > e1 && e1 < red) {
            front[x] = (uint32_t)s | prot;
            if (len == 0) out[len++] = s;
            else if (x < len) out[x] = s;
            else atomicOr(&s_flag, 2);              // the reference's out[cat][x] = row raises IndexError here
            replaced = true;
            break;
          }
          if ((q0 > e0 && q1 < e1) || (q1 > red && red > q0)) break;
        }
        if (!replaced && (prot || (q1 > red && red > q0))) {
          front[nf++] = (uint32_t)s | prot;
          out[len++] = s;
        }
      }
    }
    s_len[tid] = len;
  }
  __syncthreads();

  // ---- drop the empty lists; the positions after them shift
  const bool nonempty = tid < nreq && s_len[tid] > 0;
  const int kl = __syncthreads_count(nonempty);
  if (nonempty) {
    int l = 0;
    for (int j = 0; j < tid; ++j) l += s_len[j] > 0;
    s_base[l] = (int)(row0 + s_off[tid]);
    s_size0[l] = s_len[tid];
    s_lcat[l] = s_cat[tid];
  }
  if (tid == 0) {
    if (kl == 0) atomicOr(&s_flag, 4);
    // the host path needs one seed row per list: seed row l is looked up in list l (WOA.py:214-220, IndexError past
    // the last list), and the seed position is evaluated against every list (WOA.py:140,263, ValueError when shorter)
    if (ns > kl) atomicOr(&s_flag, 1);
    else if (seeded && ns < kl) atomicOr(&s_flag, 16);
  }
  __syncthreads();

  // ---- candidate rows, rounded when seeded (WOA.py:174-182); first exact match of seed row l in list l
  for (int l = 0; l < kl; ++l) {
    const int n0 = s_size0[l], b = s_base[l];
    for (int r = tid; r < n0; r += blockDim.x) {
      const int s = a.ids[b + r];
      const double* src = (seeded ? a.svc_round : a.svc_raw) + (int64_t)s * 4;
      double row[4] = {src[0], src[1], src[2], src[3]};
      double* dst = a.qos + (int64_t)(b + r) * 4;
      for (int q = 0; q < 4; ++q) dst[q] = row[q];
      if (l < ns && rows_equal(row, s_seed[l])) atomicMin(&s_match[l], r);
    }
  }
  __syncthreads();
  if (tid < kl) {
    int n = s_size0[tid];
    if (tid < ns) {
      if (s_match[tid] == INT_MAX) {                    // an unknown row is appended to its list
        double* dst = a.qos + (int64_t)(s_base[tid] + n) * 4;
        for (int q = 0; q < 4; ++q) dst[q] = s_seed[tid][q];
        a.ids[s_base[tid] + n] = s_seed_id[tid];
        s_own[tid] = n++;
      } else {
        s_own[tid] = s_match[tid];
      }
    }
    s_size[tid] = n;
  }
  if (tid < K) {
    const int64_t o = (int64_t)I * K + tid;
    a.base[o] = tid < kl ? s_base[tid] : 0;
    a.size[o] = tid < kl ? s_size[tid] : 1;
    a.list_cat[o] = tid < kl ? s_lcat[tid] : -1;
  }
  if (tid == 0) a.klen[I] = kl;
  __syncthreads();

  // ---- initial population (WOA.py:50-53, drawn with the sizes before the appends) and its fitness (WOA.py:56-85)
  const uint64_t seed = a.seeds[I];
  const double* bnd = a.global + (int64_t)I * 4;
  if (tid < P) {
    int32_t* row = a.pops + ((int64_t)I * P + tid) * K;
    for (int k = 0; k < K; ++k)
      row[k] = k < kl ? philox_index(philox_uniform(seed, k, tid, 3, 0), s_size0[k]) : 0;
    s_fit[tid] = kl > 0 ? woa_fitness<kWoaMaxK, false, WoaPick::kLocal>(a.qos, row, s_base, s_size, kl, bnd) : INFINITY;
  }
  __syncthreads();
  if (tid == 0) {
    double best = 3.0;
    int ref = -1;
    if (seeded && ns == kl) best = woa_fitness<kWoaMaxK, false, WoaPick::kLocal>(a.qos, s_own, s_base, s_size, kl, bnd);
    scan_best(s_fit, P, best, ref);
    s_ref = ref;
    a.best_fit[I] = best;
    a.best_ref[I] = ref;
    a.flags[I] = s_flag;
  }
  __syncthreads();
  if (tid < K) {
    const int ref = s_ref;
    int v = 0;
    if (tid < kl) v = ref >= 0 ? a.pops[((int64_t)I * P + ref) * K + tid] : (seeded && ns == kl ? s_own[tid] : 0);
    a.best_vec[(int64_t)I * K + tid] = v;
  }
}

}  // namespace
}  // namespace gnnpn

using namespace gnnpn;

extern "C" int gnnpn_woa_fitness_f64(const double* qos, int64_t n_services, const int32_t* idx, int64_t idx_ld,
                                     const int32_t* klen, const double* bounds, int64_t P, int Kmax,
                                     int32_t* viol_out, double* obj_out, double* fit_out, void* stream) {
  GNNPN_REQUIRE(qos && idx && bounds, GNNPN_ENULL);
  GNNPN_REQUIRE(Kmax >= 1 && Kmax <= kMaxTasksWoa && idx_ld >= Kmax && n_services >= 1 && P >= 0, GNNPN_ESHAPE);
  if (P == 0) return GNNPN_OK;
  woa_fitness_kernel<false><<<(unsigned)ceil_div(P, 64), 64, 0, (cudaStream_t)stream>>>(qos, idx, idx_ld, klen, bounds, P,
                                                                                       Kmax, viol_out, obj_out, fit_out);
  return after_launch();
}

extern "C" int gnnpn_ml2pn_score_f64(const double* qos, int64_t n_rows, const int32_t* idx, int64_t idx_ld,
                                     const int32_t* klen, const double* bounds, int64_t P, int Kmax,
                                     int32_t* viol_out, double* obj_out, double* score_out, void* stream) {
  GNNPN_REQUIRE(qos && idx && bounds, GNNPN_ENULL);
  GNNPN_REQUIRE(Kmax >= 1 && Kmax <= kMaxTasksWoa && idx_ld >= Kmax && n_rows >= 1 && P >= 0, GNNPN_ESHAPE);
  if (P == 0) return GNNPN_OK;
  woa_fitness_kernel<true><<<(unsigned)ceil_div(P, 64), 64, 0, (cudaStream_t)stream>>>(qos, idx, idx_ld, klen, bounds, P,
                                                                                      Kmax, viol_out, obj_out, score_out);
  return after_launch();
}

extern "C" int gnnpn_woa_search_f64(const double* qos, int64_t n_services, const int32_t* base, const int32_t* size,
                                    const int32_t* klen, const double* bounds, int32_t* pops, double* best_fit,
                                    int32_t* best_ref, int32_t* best_vec, const uint64_t* seeds, double* traj,
                                    int64_t n_instances, int popSize, int Kmax, int iters, void* stream) {
  GNNPN_REQUIRE(qos && base && size && klen && bounds && pops && best_fit && best_ref && best_vec && seeds && traj, GNNPN_ENULL);
  GNNPN_REQUIRE(popSize >= 1 && popSize <= kWoaThreads && Kmax >= 1 && Kmax <= kWoaMaxK && iters >= 0 && n_services >= 1 &&
                    n_instances >= 0, GNNPN_ESHAPE);
  if (n_instances == 0 || iters == 0) return GNNPN_OK;
  WoaSearchArgs a{qos, base, size, klen, bounds, pops, best_fit, best_ref, best_vec, seeds, traj, popSize, Kmax, iters};
  const size_t smem = (size_t)popSize * 8 + (size_t)(2 * popSize * Kmax + 3 * Kmax + popSize) * 4;
  static size_t configured = 0;
  if (smem > 48 * 1024 && smem > configured) {
    cudaError_t e = cudaFuncSetAttribute(woa_search_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    configured = smem;
  }
  woa_search_kernel<<<(unsigned)n_instances, kWoaThreads, smem, (cudaStream_t)stream>>>(a);
  return after_launch();
}

extern "C" int gnnpn_woa_prepare_f64(const double* svc_raw, const double* svc_round, const int32_t* cat_ptr,
                                     int64_t n_services, int K, const int32_t* req_cat, const int32_t* n_req,
                                     const double* local_bounds, const double* global_bounds, const float* seed_rows,
                                     const int32_t* seed_ids, const uint64_t* seeds, int64_t n_instances, int popSize,
                                     double reduct, double* qos, int32_t* ids, int32_t* base, int32_t* size,
                                     int32_t* klen, int32_t* list_cat, int32_t* pops, double* best_fit,
                                     int32_t* best_ref, int32_t* best_vec, int32_t* flags, void* stream) {
  GNNPN_REQUIRE(svc_raw && svc_round && cat_ptr && req_cat && n_req && local_bounds && global_bounds && seed_rows &&
                    seed_ids && seeds && qos && ids && base && size && klen && list_cat && pops && best_fit && best_ref &&
                    best_vec && flags, GNNPN_ENULL);
  GNNPN_REQUIRE(popSize >= 1 && popSize <= kWoaThreads && K >= 1 && K <= kWoaMaxK && n_services >= 1 &&
                    n_services < (int64_t)kFrontSentinel && n_instances >= 0, GNNPN_ESHAPE);
  const int64_t cap = woa_prepare_rows(1, n_services, K);
  GNNPN_REQUIRE(n_instances * cap <= (int64_t)INT32_MAX, GNNPN_ESHAPE);      // `base` is an int32 row index
  if (n_instances == 0) return GNNPN_OK;
  WoaPrepareArgs a{svc_raw, svc_round, cat_ptr, req_cat, n_req, local_bounds, global_bounds, seed_rows, seed_ids, seeds,
                   qos, ids, base, size, klen, list_cat, pops, best_ref, best_vec, flags, best_fit, reduct, cap, K,
                   popSize};
  woa_prepare_kernel<<<(unsigned)n_instances, kWoaThreads, 0, (cudaStream_t)stream>>>(a);
  return after_launch();
}

extern "C" int64_t gnnpn_woa_prepare_rows(int64_t n_instances, int64_t n_services, int K) {
  return woa_prepare_rows(n_instances, n_services, K);
}
