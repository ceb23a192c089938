// lns.cu -- (c2) LP-guided large-neighbourhood search over placements c[F][N], one WARP per search chain.
//
// Stands in for SCIP's branch and bound inside pywraplp.Solver.Solve() (reference core/solvers/solver.py:37)
// on the step-1 models whose objective has a delay term (NeptuneStep1CPUMinDelay / ...MinDelayAndUtilization,
// neptune_step1.py:63-77) when every function needs the same memory, so that the memory row of a node
// (constraints_step1.py:18-23) is a slot count  sum_f c[f,j] <= floor(M_j / m).
//
// State of a chain: a placement c and node prices lam[j] >= 0 on the CPU rows (constraints_step1.py:57-65).
// For fixed prices every source (f,i) goes to the open pod of f with the smallest PRICED delay
// d[i,j] + lam[j] r[f,j]; the priced cost  g(c, lam) = sum w min_j(d + lam r) - lam.K  is a lower bound of the
// routing LP of c and equals it at the best prices (LP duality for fixed c), so
//   * the prices are kept at the coordinate-wise maximiser for the current placement (dual ascent: the price of
//     an overloaded node is raised to the threshold at which enough flows leave, exactly the fractional
//     knapsack of route_cap.cuh, but only its dual side -- no flow is split here), and
//   * the placement moves are EXACT re-optimisations of all pods of k nodes at once: with the pods outside
//     the k nodes fixed, the priced cost separates over functions, cost_f(T) for the 2^k subsets T of the k
//     nodes is a min-reduction, and the slot limits couple the functions only through the k slot counters,
//     so a dynamic programme over functions with (slots+1)^k states finds the best of ~10^7 joint
//     reassignments (k = 3, F = 10) in a few thousand instructions.
// The DP is run on perturbed costs (noise proportional to an annealed temperature) and its result is always
// accepted; a chain records the best placement it visits (by g, only when no node is overloaded at the
// current prices).  The caller prices the chains' records exactly (route_lp.cu) and returns the best.
// Chains start from randomised roundings of the LP relaxation's c-bar (pdhg_mf.cu) or from seed placements.
// No atomics on floating point, fixed evaluation orders, counter-based random numbers: runs are
// bit-reproducible for a given rng seed.
#include "common.cuh"

namespace neptune {

struct LnsArgs {
  int B, N, F, kind, chains, rounds, k, smax, wpb, S, maxslots;
  double alpha, noise_coef;
  uint64_t rng;
  const double *d, *w, *r, *m, *Mj, *Kj, *maxd;
  const double* guide;     // [B][F][N] c-bar of the relaxation, or null
  const double* lam0;      // [B][N] CPU-row duals of the relaxation (delay units), or null
  const uint8_t* seeds;    // [B][S][F][N] or null
  uint8_t* out_c;          // [B][2*chains][F][N]: per chain one record by the upper bound, one by the lower bound
  double* out_g;           // [B][2*chains] [0,chains): whole-flow objective of the record (upper bound of its true objective);
                           //               [chains,2*chains): priced objective (lower bound); +inf: none
  double* out_lb;          // [B][2*chains] the other end of each record's bracket; may be null
  int32_t* out_round;      // [B][2*chains] round of the record
  uint16_t* out_asg;       // [B][2*chains][F][N] (k_lns_global) each source's pod when the record was taken
};

constexpr double kLnsBig = 1e9;                 // priced delay of "no pod"
constexpr double kFxScale = 1073741824.0;       // 2^30: CPU loads are accumulated in fixed point (integer adds commute)
constexpr int kLnsMaxK = 4;
// chains per block: two blocks per SM, either 8 warps at 128 registers or 12 warps at 80 registers.  A chain-round is
// 3-10 % slower at 80 registers, so 8 is used while all blocks are resident at once (2 * 148); beyond that the 24
// resident warps per SM of the 12-warp build win (the kernel is latency-bound: 30 % issue-active at 16 warps per SM).
constexpr int kLnsWarps = 8, kLnsWarpsWide = 12;

__device__ __forceinline__ uint64_t lns_mix(uint64_t z) {        // splitmix64 finaliser
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
__device__ __forceinline__ double lns_u01(uint64_t h) { return (double)(h >> 11) * (1.0 / 9007199254740992.0); }
__device__ __forceinline__ uint64_t lns_next(uint64_t& s) { s ^= s >> 12; s ^= s << 25; s ^= s >> 27; return s * 2685821657736338717ull; }

// ---- where a chain's state lives ------------------------------------------------------------------------------
// k_lns keeps it in shared memory (N <= 128, F*N <= 4096: pod ids fit a byte, list entries 16 bits); k_lns_global keeps
// it in a workspace slab per chain and reads the instance from global memory (N <= 65534).  Both run lns_chain.cuh: the
// same decisions in the same orders, only the index widths and the memory differ, so on any input both take the records
// of k_lns bit for bit.
struct LnsShared {
  using pod_t = uint8_t;          // node of a source's nearest pod, entries of a function's pod list
  using idx_t = unsigned short;   // entries of the scan and exception lists (indices into F*N)
  using dix_t = int;              // index into the N*N delay matrix
  static constexpr int kNone = 255;
  static constexpr bool kGlobal = false;
};
struct LnsGlobal {
  using pod_t = uint16_t;
  using idx_t = uint32_t;
  using dix_t = int64_t;
  static constexpr int kNone = 0xFFFF;
  static constexpr bool kGlobal = true;
};

// block (k_lns only): dT[N][N] (delay, transposed: the hot loops fix a destination j and run the lanes over sources i),
//        w[F][N], r[F][N], K[N], slots[N]
// chain: lam[N] | loadfx[N] | bestv[F*N] | scratch (costT | dp  /  th  /  exception list) | ints | pod ids | bytes
__host__ __device__ inline size_t lns_block_shared(int N, int F) {
  return ((size_t)N * N + 2 * (size_t)F * N + (size_t)N) * 8 + (size_t)N * 4 + 64;
}
template <class St>
__host__ __device__ inline size_t lns_scratch_bytes(int N, int F, int k, int smax, int maxslots) {
  const size_t fn = (size_t)F * N, nT = (size_t)1 << k, tn = (size_t)(maxslots < F ? maxslots : F) * N;
  const size_t li = sizeof(typename St::idx_t);
  size_t dp = (size_t)F * nT * 8 + (size_t)smax * 8;          // costT, dp (updated in place, one function at a time)
  size_t th = tn * 4 + tn * li;                               // thresholds (float) + their scan list of one node's sources
  if (th < fn * li) th = fn * li;                             // exception list
  return ((dp > th ? dp : th) + 15) & ~(size_t)15;
}
template <class St>
__host__ __device__ inline size_t lns_chain_bytes(int N, int F, int k, int smax, int maxslots) {
  const size_t fn = (size_t)F * N, lp = sizeof(typename St::pod_t);
  size_t b = 0;
  b += (size_t)N * 8;               // lam
  b += (size_t)N * 8;               // loadfx
  b += (fn * 4 + 15) & ~(size_t)15; // bestv (float: it ranks candidates, the records are priced exactly afterwards)
  b += lns_scratch_bytes<St>(N, F, k, smax, maxslots);
  b += ((size_t)F + 33 + (size_t)F) * 4;   // npods, misc (J, rad, mul, incT, number of states), fl
  b += fn * lp;                     // asg
  b += (fn + lp - 1) / lp * lp;     // c (padded: podlist stays aligned)
  b += fn * lp;                     // podlist
  b += (size_t)F * smax;            // choice
  b += (size_t)smax + 2 * (size_t)F + 16;  // supp table, oldT, newT
  return (b + 15) & ~(size_t)15;
}

// instance scalars from k_lns's three lane-strided sums (after warp_sum): noise scale, utilisation weight in delay
// units, delay weight
__device__ __forceinline__ void lns_scalars(const LnsArgs& a, int N, int fn, double sw, double sd, double wm, double* out) {
  double a_d = 1.0, a_u = 0.0;
  if (a.kind == NEPTUNE_KIND_MIN_DELAY_UTIL) { a_u = a.alpha / (double)N; a_d = (sw != 0.0 && wm != 0.0) ? (1.0 - a.alpha) / wm : 0.0; }
  const double dmean = N > 1 ? sd / ((double)N * (N - 1)) : 1.0;
  out[0] = a.noise_coef * (sw / fn) * dmean;
  out[1] = a_d > 0.0 ? a_u / a_d : 0.0;
  out[2] = a_d;
}

// reduce NT per-lane accumulators over the warp: afterwards lane L holds the warp total of accumulator
// t(L) = the top log2(NT) bits of L's 5-bit index read as a number (NT = 8: L >> 2; NT = 16: L >> 1)
template <int NT>
__device__ __forceinline__ double lns_multi_reduce(double (&acc)[NT], int lane) {
  int off = 16;
#pragma unroll
  for (int n = NT; n > 1; n >>= 1, off >>= 1) {
    const bool hi = (lane & off) != 0;
#pragma unroll
    for (int t = 0; t < n / 2; ++t) {
      const double keep = hi ? acc[t + n / 2] : acc[t];
      const double send = hi ? acc[t] : acc[t + n / 2];
      acc[t] = keep + __shfl_xor_sync(0xffffffffu, send, off);
    }
  }
  double v = acc[0];
  for (; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
  return v;
}

template <int KK, int WPB>
__global__ void __launch_bounds__(WPB * 32, 2) k_lns(LnsArgs a) {
  constexpr int NT = 1 << KK;
  const int N = a.N, F = a.F, b = blockIdx.y, lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int chain = blockIdx.x * a.wpb + wid;
  const int fn = F * N, smax = a.smax;
  extern __shared__ __align__(16) unsigned char smem[];
  double* s_dT = (double*)smem;
  double* s_w = s_dT + (size_t)N * N;
  double* s_r = s_w + fn;
  double* s_K = s_r + fn;
  int* s_slots = (int*)(s_K + N);
  __shared__ double s_scal[4];          // noise0, u (utilisation weight in delay units), a_d
  {
    const double* d = a.d + (int64_t)b * N * N;
    const double* w = a.w + (int64_t)b * fn;
    const double* r = a.r + (int64_t)b * fn;
    for (int q = threadIdx.x; q < N * N; q += blockDim.x) { const int i = q / N, j = q - i * N; s_dT[j * N + i] = d[q]; }
    for (int q = threadIdx.x; q < fn; q += blockDim.x) { s_w[q] = w[q]; s_r[q] = r[q]; }
    const double m0 = a.m[(int64_t)b * F];
    for (int j = threadIdx.x; j < N; j += blockDim.x) {
      s_K[j] = a.Kj[(int64_t)b * N + j];
      int sl = m0 > 0.0 ? (int)floor(a.Mj[(int64_t)b * N + j] / m0 + 1e-9) : F;
      s_slots[j] = sl > a.maxslots ? a.maxslots : (sl < 0 ? 0 : sl);
    }
  }
  __syncthreads();
  if (threadIdx.x < 32) {
    // instance scalars: mean workload, mean off-diagonal delay (noise scale), objective weights
    double sw = 0.0, sd = 0.0, wm = 0.0;
    for (int q = lane; q < fn; q += 32) sw += s_w[q];
    for (int q = lane; q < N * N; q += 32) sd += s_dT[q];
    for (int fi = lane; fi < fn; fi += 32) {
      const int f = fi / N, i = fi - f * N;
      const double md = a.maxd ? a.maxd[(int64_t)b * F + f] : INFINITY;
      double best = -INFINITY;
      for (int j = 0; j < N; ++j) { const double v = s_dT[j * N + i]; if (v <= md && v > best) best = v; }
      wm += s_w[fi] * best;
    }
    sw = warp_sum(sw); sd = warp_sum(sd); wm = warp_sum(wm);
    if (lane == 0) {                    // (the formula of lns_scalars, kept inline: k_lns compiles as before)
      double a_d = 1.0, a_u = 0.0;
      if (a.kind == NEPTUNE_KIND_MIN_DELAY_UTIL) { a_u = a.alpha / (double)N; a_d = (sw != 0.0 && wm != 0.0) ? (1.0 - a.alpha) / wm : 0.0; }
      const double dmean = N > 1 ? sd / ((double)N * (N - 1)) : 1.0;
      s_scal[0] = a.noise_coef * (sw / fn) * dmean;
      s_scal[1] = a_d > 0.0 ? a_u / a_d : 0.0;
      s_scal[2] = a_d;
    }
  }
  __syncthreads();
  if (chain >= a.chains) return;                 // (no block-wide barrier below this line)
  // chains anneal from different start temperatures (x0.6, 0.9, 1.2, 1.5 by chain index): no single temperature
  // suits every instance, and a mixed population finds the optimum of more of them than any uniform one
  const double noise0 = s_scal[0] * (0.6 + 0.3 * (double)(chain & 3)), u = s_scal[1], a_d = s_scal[2];
  unsigned char* wp = smem + ((lns_block_shared(N, F) + 15) & ~(size_t)15) + (size_t)wid * lns_chain_bytes<LnsShared>(N, F, KK, smax, a.maxslots);
  using St = LnsShared;
  using pod_t = St::pod_t;
  using idx_t = St::idx_t;
  using dix_t = St::dix_t;
  constexpr int kNone = St::kNone;
  double* dT = s_dT; double* w = s_w; double* r = s_r; double* K = s_K; int* slots = s_slots;
#include "lns_chain.cuh"
}
// ---- k_lns_global: the chain body with its state in a workspace slab (instances too large for shared memory) ------
// Workspace, per instance: the transposed delay matrix, the largest delay of every source within maxd (kind 2), the
// slot counts and the three scalars; then one slab of lns_chain_bytes<LnsGlobal> per chain.
struct LnsGlobalLayout {
  size_t dT, far, slots, scal, state, state_bytes, total;
};
static inline size_t lns_align256(size_t v) { return (v + 255) & ~(size_t)255; }
static inline LnsGlobalLayout lns_global_layout(int B, int N, int F, int chains, int k, int maxslots) {
  LnsGlobalLayout L{};
  const size_t nn = (size_t)N * N, fn = (size_t)F * N;
  int smax = 1; for (int q = 0; q < k; ++q) smax *= 4;
  L.dT = 0;
  L.far = L.dT + lns_align256((size_t)B * nn * 8);
  L.slots = L.far + lns_align256((size_t)B * fn * 8);
  L.scal = L.slots + lns_align256((size_t)B * N * 4);
  L.state = L.scal + lns_align256((size_t)B * 4 * 8);
  L.state_bytes = lns_align256(lns_chain_bytes<LnsGlobal>(N, F, k, smax, maxslots));
  L.total = L.state + (size_t)B * chains * L.state_bytes;
  return L;
}

// transposed delays (dT[j][i] = d[i][j]) and slot counts of every instance; grid (x, B)
__global__ void k_lns_global_stage(LnsArgs a, double* dT_all, int* slots_all) {
  const int N = a.N, F = a.F, b = blockIdx.y;
  const int64_t nn = (int64_t)N * N;
  const double* d = a.d + (int64_t)b * nn;
  double* dT = dT_all + (int64_t)b * nn;
  for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < nn; q += (int64_t)gridDim.x * blockDim.x) {
    const int64_t j = q / N, i = q - j * N;
    dT[q] = d[i * N + j];
  }
  const double m0 = a.m[(int64_t)b * F];
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < N; j += gridDim.x * blockDim.x) {
    int sl = m0 > 0.0 ? (int)floor(a.Mj[(int64_t)b * N + j] / m0 + 1e-9) : F;
    slots_all[(int64_t)b * N + j] = sl > a.maxslots ? a.maxslots : (sl < 0 ? 0 : sl);
  }
}

// largest delay of every source (f,i) within maxd[f]: k_lns's loop over j, one thread per source; grid (x, B)
__global__ void k_lns_global_far(LnsArgs a, const double* dT_all, double* far_all) {
  const int N = a.N, F = a.F, b = blockIdx.y, fn = F * N;
  const double* dT = dT_all + (int64_t)b * N * N;
  for (int fi = blockIdx.x * blockDim.x + threadIdx.x; fi < fn; fi += gridDim.x * blockDim.x) {
    const int f = fi / N, i = fi - f * N;
    const double md = a.maxd ? a.maxd[(int64_t)b * F + f] : INFINITY;
    double best = -INFINITY;
    for (int j = 0; j < N; ++j) { const double v = dT[(int64_t)j * N + i]; if (v <= md && v > best) best = v; }
    far_all[(int64_t)b * fn + fi] = best;
  }
}

// the instance scalars of k_lns, one warp per instance: the same lane-strided sums in the same order, so bit-identical
__global__ void k_lns_global_scalars(LnsArgs a, const double* dT_all, const double* far_all, double* scal) {
  const int N = a.N, F = a.F, b = blockIdx.x, lane = threadIdx.x, fn = F * N;
  const int64_t nn = (int64_t)N * N;
  const double* w = a.w + (int64_t)b * fn;
  const double* dT = dT_all + (int64_t)b * nn;
  double sw = 0.0, sd = 0.0, wm = 0.0;
  for (int q = lane; q < fn; q += 32) sw += w[q];
  for (int64_t q = lane; q < nn; q += 32) sd += dT[q];
  if (far_all) for (int fi = lane; fi < fn; fi += 32) wm += w[fi] * far_all[(int64_t)b * fn + fi];   // kind 2 only
  sw = warp_sum(sw); sd = warp_sum(sd); wm = warp_sum(wm);
  if (lane == 0) lns_scalars(a, N, fn, sw, sd, wm, scal + 4 * (int64_t)b);
}

template <int KK>
__global__ void __launch_bounds__(kLnsWarps * 32, 2) k_lns_global(LnsArgs a, const double* dT_all, const int* slots_all,
                                                                  const double* scal, unsigned char* state, int64_t state_bytes) {
  const int N = a.N, F = a.F, b = blockIdx.y, lane = threadIdx.x & 31;
  const int chain = blockIdx.x * kLnsWarps + (threadIdx.x >> 5);
  if (chain >= a.chains) return;
  const int fn = F * N, smax = a.smax;
  const double* sc = scal + 4 * (int64_t)b;
  const double noise0 = sc[0] * (0.6 + 0.3 * (double)(chain & 3)), u = sc[1], a_d = sc[2];
  const double* dT = dT_all + (int64_t)b * N * N;
  const double* w = a.w + (int64_t)b * fn;
  const double* r = a.r + (int64_t)b * fn;
  const double* K = a.Kj + (int64_t)b * N;
  const int* slots = slots_all + (int64_t)b * N;
  unsigned char* wp = state + ((int64_t)b * a.chains + chain) * state_bytes;
  using St = LnsGlobal;
  using pod_t = St::pod_t;
  using idx_t = St::idx_t;
  using dix_t = St::dix_t;
  constexpr int NT = 1 << KK, kNone = St::kNone;
#include "lns_chain.cuh"
}

}  // namespace neptune

using namespace neptune;

static int g_lns_block_mode = 0;      // 0: by the number of blocks, 1: always 8 chains per block, 2: always 12
extern "C" int neptune_lns_block_mode(int mode) {
  if (mode < 0 || mode > 2) return NEPTUNE_E_ARG;
  g_lns_block_mode = mode;
  return 0;
}

extern "C" int neptune_lns_search(int B, int N, int F, int kind, double alpha, int chains, int rounds, int k,
                                  double noise_coef, uint64_t rng_seed, const double* d, const double* w,
                                  const double* r, const double* m, const double* Mj, const double* Kj,
                                  const double* maxd, const double* guide, const double* lam0, int S,
                                  const uint8_t* seeds, int max_slots, uint8_t* out_c, double* out_g, double* out_lb,
                                  int32_t* out_round, void* stream) {
  if (B <= 0 || N <= 0 || F <= 0 || chains <= 0 || rounds < 0 || k < 2 || k > kLnsMaxK || !d || !w || !r || !m || !Mj ||
      !Kj || !out_c || !out_g || !out_round)
    return NEPTUNE_E_ARG;
  if (kind != NEPTUNE_KIND_MIN_DELAY && kind != NEPTUNE_KIND_MIN_DELAY_UTIL) return NEPTUNE_E_ARG;
  if (seeds && S <= 0) return NEPTUNE_E_ARG;
  if (N > 128 || (int64_t)F * N > 4096) return NEPTUNE_E_SIZE;       // the chain state lives in shared memory
  LnsArgs a{};
  a.B = B; a.N = N; a.F = F; a.kind = kind; a.chains = chains; a.rounds = rounds; a.k = k; a.S = seeds ? S : 0;
  a.alpha = alpha; a.noise_coef = noise_coef; a.rng = rng_seed ? rng_seed : 0x1234567ull;
  a.d = d; a.w = w; a.r = r; a.m = m; a.Mj = Mj; a.Kj = Kj; a.maxd = maxd; a.guide = guide; a.lam0 = lam0; a.seeds = seeds;
  a.out_c = out_c; a.out_g = out_g; a.out_lb = out_lb; a.out_round = out_round;
  // states of the slot counters: (slots+1)^k for the common 3-slot nodes, capped by shared memory
  int smax = 1; for (int q = 0; q < k; ++q) smax *= 4;
  const size_t blk = (lns_block_shared(N, F) + 15) & ~(size_t)15;
  a.maxslots = (max_slots > 0 && max_slots < F) ? max_slots : F;       // bound on floor(Mj / m) the caller vouches for (sizes the scratch)
  const size_t per = lns_chain_bytes<LnsShared>(N, F, k, smax, a.maxslots);
  const int wide_mode = g_lns_block_mode;
  const size_t budget = 112 * 1024;                                     // two blocks per SM (228 KB, 1 KB reserved per block)
  int wpb = kLnsWarps;
  const int64_t blocks8 = (int64_t)B * ((chains + kLnsWarps - 1) / kLnsWarps);
  const bool wide = blocks8 > 2 * kNumSMs && blk + kLnsWarpsWide * per <= budget && !(wide_mode & 1);
  if (wide || (wide_mode & 2)) wpb = kLnsWarpsWide;
  const int cap = wpb;
  while (wpb > 1 && blk + wpb * per > budget) --wpb;
  if (blk + wpb * per > 200 * 1024) return NEPTUNE_E_SIZE;
  if (wpb > chains) wpb = chains;
  a.smax = smax; a.wpb = wpb;
  const size_t sm = blk + wpb * per;
  const dim3 grid((chains + wpb - 1) / wpb, B);
#define NEPTUNE_LNS_LAUNCH(KK_, W_)                                                                                   \
  do {                                                                                                                \
    NEPTUNE_CUDA_OK(cudaFuncSetAttribute(k_lns<KK_, W_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));     \
    k_lns<KK_, W_><<<grid, wpb * 32, sm, (cudaStream_t)stream>>>(a);                                                  \
  } while (0)
  if (cap == kLnsWarpsWide) {
    if (k == 3) NEPTUNE_LNS_LAUNCH(3, kLnsWarpsWide); else if (k == 4) NEPTUNE_LNS_LAUNCH(4, kLnsWarpsWide); else NEPTUNE_LNS_LAUNCH(2, kLnsWarpsWide);
  } else {
    if (k == 3) NEPTUNE_LNS_LAUNCH(3, kLnsWarps); else if (k == 4) NEPTUNE_LNS_LAUNCH(4, kLnsWarps); else NEPTUNE_LNS_LAUNCH(2, kLnsWarps);
  }
#undef NEPTUNE_LNS_LAUNCH
  NEPTUNE_COUNT(1);
  NEPTUNE_LAUNCH_OK();
  return 0;
}

// size rule of neptune_lns_search_global: one warp per chain, every index as wide as LnsGlobal's
static int lns_global_check(int B, int N, int F, int chains, int k) {
  if (B <= 0 || N <= 0 || F <= 0 || chains <= 0 || k < 2 || k > kLnsMaxK) return NEPTUNE_E_ARG;
  if (N > 0xFFFE || (int64_t)F * N > 0x7FFFFFFF || B > 65535) return NEPTUNE_E_SIZE;
  return 0;
}

extern "C" int neptune_lns_search_global_workspace_bytes(int B, int N, int F, int chains, int k, int max_slots, int64_t* bytes) {
  const int rc = lns_global_check(B, N, F, chains, k);
  if (rc) return rc;
  if (!bytes) return NEPTUNE_E_ARG;
  *bytes = (int64_t)lns_global_layout(B, N, F, chains, k, (max_slots > 0 && max_slots < F) ? max_slots : F).total;
  return 0;
}

extern "C" int neptune_lns_search_global(int B, int N, int F, int kind, double alpha, int chains, int rounds, int k,
                                         double noise_coef, uint64_t rng_seed, const double* d, const double* w,
                                         const double* r, const double* m, const double* Mj, const double* Kj,
                                         const double* maxd, const double* guide, const double* lam0, int S,
                                         const uint8_t* seeds, int max_slots, uint8_t* out_c, double* out_g, double* out_lb,
                                         int32_t* out_round, uint16_t* out_asg, void* workspace, int64_t workspace_bytes,
                                         void* stream) {
  const int rc = lns_global_check(B, N, F, chains, k);
  if (rc) return rc;
  if (rounds < 0 || !d || !w || !r || !m || !Mj || !Kj || !out_c || !out_g || !out_round || !out_asg || !workspace)
    return NEPTUNE_E_ARG;
  if (kind != NEPTUNE_KIND_MIN_DELAY && kind != NEPTUNE_KIND_MIN_DELAY_UTIL) return NEPTUNE_E_ARG;
  if (seeds && S <= 0) return NEPTUNE_E_ARG;
  LnsArgs a{};
  a.B = B; a.N = N; a.F = F; a.kind = kind; a.chains = chains; a.rounds = rounds; a.k = k; a.S = seeds ? S : 0;
  a.alpha = alpha; a.noise_coef = noise_coef; a.rng = rng_seed ? rng_seed : 0x1234567ull;
  a.d = d; a.w = w; a.r = r; a.m = m; a.Mj = Mj; a.Kj = Kj; a.maxd = maxd; a.guide = guide; a.lam0 = lam0; a.seeds = seeds;
  a.out_c = out_c; a.out_g = out_g; a.out_lb = out_lb; a.out_round = out_round; a.out_asg = out_asg;
  int smax = 1; for (int q = 0; q < k; ++q) smax *= 4;
  a.maxslots = (max_slots > 0 && max_slots < F) ? max_slots : F;
  a.smax = smax; a.wpb = kLnsWarps;
  const LnsGlobalLayout L = lns_global_layout(B, N, F, chains, k, a.maxslots);
  if (workspace_bytes < (int64_t)L.total) return NEPTUNE_E_NOMEM;
  unsigned char* ws = (unsigned char*)workspace;
  double* dT = (double*)(ws + L.dT);
  double* far = kind == NEPTUNE_KIND_MIN_DELAY_UTIL ? (double*)(ws + L.far) : nullptr;
  int* slots = (int*)(ws + L.slots);
  double* scal = (double*)(ws + L.scal);
  const cudaStream_t st = (cudaStream_t)stream;
  const int64_t nn = (int64_t)N * N;
  const int sx = (int)((nn + 255) / 256 < 1024 ? (nn + 255) / 256 : 1024);
  k_lns_global_stage<<<dim3(sx, B), 256, 0, st>>>(a, dT, slots);
  if (far) {
    const int fx = (int)(((int64_t)F * N + 255) / 256 < 4096 ? ((int64_t)F * N + 255) / 256 : 4096);
    k_lns_global_far<<<dim3(fx, B), 256, 0, st>>>(a, dT, far);
  }
  k_lns_global_scalars<<<B, 32, 0, st>>>(a, dT, far, scal);
  const dim3 grid((chains + kLnsWarps - 1) / kLnsWarps, B);
  unsigned char* state = ws + L.state;
  const int64_t sb = (int64_t)L.state_bytes;
  if (k == 3) k_lns_global<3><<<grid, kLnsWarps * 32, 0, st>>>(a, dT, slots, scal, state, sb);
  else if (k == 4) k_lns_global<4><<<grid, kLnsWarps * 32, 0, st>>>(a, dT, slots, scal, state, sb);
  else k_lns_global<2><<<grid, kLnsWarps * 32, 0, st>>>(a, dT, slots, scal, state, sb);
  NEPTUNE_COUNT(far ? 4 : 3);
  NEPTUNE_LAUNCH_OK();
  return 0;
}
