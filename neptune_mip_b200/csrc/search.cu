// search.cu -- (c2) batched rounding + local search over placements c[F][N].
//
// Stands in for SCIP's primal side (branch and bound + heuristics inside pywraplp.Solver.Solve(),
// reference core/solvers/solver.py:37): once x is eliminated by the nearest-open-pod routing rule
// (efttc_step1.py:196-212) step 1 is a capacitated facility-location problem in c alone, and the
// classical add / drop / swap / replace neighbourhood with exact delta evaluation applies.
//
// One thread block = one search chain; grid = (chains, instances).  Every chain starts from a seed
// placement (EFTTC output, a PDHG rounding, ...), optionally perturbed, and runs best-improvement
// sweeps: each warp evaluates whole moves (exact change of delay, active nodes and CPU overload via a
// per-warp delta-load array in shared memory), a block argmin picks the move, the touched functions
// are re-routed.  At a local optimum the chain keeps its best and kicks itself (iterated local search).
// Thousands of candidate moves are checked per sweep and chain; feasibility of the winner is
// re-verified by the exact checkers (neptune_check_solution) in the caller.
#include "common.cuh"
#include "route_cap.cuh"

namespace neptune {

struct LsArgs {
  int N, F, kind, chains, sweeps, S;
  double alpha, budget;
  uint64_t rng;
  const double *d, *w, *r, *m, *Mj, *Kj, *maxd, *cost, *old;
  const uint8_t* seeds;
  const double* guide;
  int use_smem;              // small instances: d, dT, w, r and the nearest/second-nearest tables live in shared memory
  int step2_mode;            // 0: step-1 objective; 1 "delete" / 2 "create": minimise disruption (step 2)
  const double* bound;       // [B] step 2: the step-1 objective of the placement must stay <= bound[b]
  // workspace
  double* dT;          // [B][N][N]
  double* inst_scal;   // [B][4]: wmax, mu, a_d, a_u
  char* chain_ws;      // [B][chains] blocks
  int64_t chain_stride;
  double* chain_cost;  // [B][chains]
};

struct Chain {
  uint8_t *c, *best_c;
  double *b1, *b2, *load, *mem;
  int *a1, *a2, *cntf, *cntn, *pods;
  // capacity-aware routing scratch (route_cap.cuh)
  double *th, *rho, *cload, *lam;
  int *ch, *sec, *alt;
};

__device__ __forceinline__ int64_t chain_bytes(int N, int F) {
  int64_t fn = (int64_t)F * N;
  int64_t b = 2 * fn + 2 * fn * 8 + 2 * fn * 4 + 2 * (int64_t)N * 8 + (int64_t)F * 4 + (int64_t)N * 4 + fn * 4 + 64;
  b += 2 * fn * 8 + 3 * fn * 4 + 2 * (int64_t)N * 8 + 64;
  return (b + 255) & ~(int64_t)255;
}
static inline int64_t chain_bytes_h(int N, int F) {
  int64_t fn = (int64_t)F * N;
  int64_t b = 2 * fn + 2 * fn * 8 + 2 * fn * 4 + 2 * (int64_t)N * 8 + (int64_t)F * 4 + (int64_t)N * 4 + fn * 4 + 64;
  b += 2 * fn * 8 + 3 * fn * 4 + 2 * (int64_t)N * 8 + 64;
  return (b + 255) & ~(int64_t)255;
}

__device__ __forceinline__ Chain carve(char* p, int N, int F) {
  Chain k;
  const int64_t fn = (int64_t)F * N;
  k.b1 = (double*)p; p += fn * 8;
  k.b2 = (double*)p; p += fn * 8;
  k.th = (double*)p; p += fn * 8;
  k.rho = (double*)p; p += fn * 8;
  k.cload = (double*)p; p += (int64_t)N * 8;
  k.lam = (double*)p; p += (int64_t)N * 8;
  k.load = (double*)p; p += (int64_t)N * 8;
  k.mem = (double*)p; p += (int64_t)N * 8;
  k.a1 = (int*)p; p += fn * 4;
  k.a2 = (int*)p; p += fn * 4;
  k.pods = (int*)p; p += fn * 4;
  k.ch = (int*)p; p += fn * 4;
  k.sec = (int*)p; p += fn * 4;
  k.alt = (int*)p; p += fn * 4;
  k.cntf = (int*)p; p += (int64_t)F * 4;
  k.cntn = (int*)p; p += (int64_t)N * 4;
  k.c = (uint8_t*)p; p += fn;
  k.best_c = (uint8_t*)p;
  return k;
}

constexpr double kBigDelay = 1e8;     // delay charged to a source whose function has no pod yet
constexpr double kCoverage = 1e13;    // cost of a function without any pod (dominates everything else)

__device__ __forceinline__ uint64_t rng_next(uint64_t& s) {   // xorshift64*
  s ^= s >> 12; s ^= s << 25; s ^= s >> 27;
  return s * 2685821657736338717ull;
}

// nearest / second nearest open pod of f for every source (block-wide, threads over i)
__device__ void route_f(const LsArgs& a, const Chain& k, const double* d, int f) {
  const int N = a.N;
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    const double* di = d + (int64_t)i * N;
    double v1 = kBigDelay, v2 = kBigDelay; int j1 = -1, j2 = -1;   // finite: deltas stay finite
    for (int j = 0; j < N; ++j) {
      if (!k.c[(int64_t)f * N + j]) continue;
      const double v = di[j];
      if (v < v1) { v2 = v1; j2 = j1; v1 = v; j1 = j; }
      else if (v < v2) { v2 = v; j2 = j; }
    }
    k.b1[(int64_t)f * N + i] = v1; k.a1[(int64_t)f * N + i] = j1;
    k.b2[(int64_t)f * N + i] = v2; k.a2[(int64_t)f * N + i] = j2;
  }
}

// per-node aggregates from scratch (deterministic): pods, memory (f ascending), CPU load
__device__ void node_state(const LsArgs& a, const Chain& k, const double* w, const double* r, const double* m) {
  const int N = a.N, F = a.F;
  for (int j = threadIdx.x; j < N; j += blockDim.x) {
    double mem = 0.0, load = 0.0; int cnt = 0;
    for (int f = 0; f < F; ++f) {
      if (!k.c[(int64_t)f * N + j]) continue;
      mem += m[f]; ++cnt;
      const double rfj = r[(int64_t)f * N + j];
      const int* a1 = k.a1 + (int64_t)f * N;
      const double* wf = w + (int64_t)f * N;
      double s = 0.0;
      for (int i = 0; i < N; ++i) if (a1[i] == j) s += wf[i];
      load += s * rfj;
    }
    k.mem[j] = mem; k.load[j] = load; k.cntn[j] = cnt;
  }
  for (int f = threadIdx.x; f < F; f += blockDim.x) {
    int cnt = 0;
    for (int j = 0; j < N; ++j) cnt += k.c[(int64_t)f * N + j];
    k.cntf[f] = cnt;
  }
}

struct Cost { double delay, util, over, uncov, flips, pods, memover; };

// whole-block exact cost of the current state (after route_f for all f and node_state)
__device__ Cost full_cost(const LsArgs& a, const Chain& k, const double* w, const double* Kj, double* red) {
  const int N = a.N, F = a.F;
  double dl = 0.0, ut = 0.0, ov = 0.0, uc = 0.0, fl = 0.0, pd = 0.0;
  for (int f = threadIdx.x; f < F; f += blockDim.x) if (k.cntf[f] == 0) uc += 1.0;
  if (a.step2_mode) {
    const double* old = a.old + (int64_t)blockIdx.y * F * N;
    for (int q = threadIdx.x; q < F * N; q += blockDim.x) {
      const bool on = k.c[q] != 0, was = old[q] > 0.0;
      if (on != was) fl += 1.0;
      if (on) pd += 1.0;
    }
  }
  for (int fi = threadIdx.x; fi < F * N; fi += blockDim.x) {
    const double wv = w[fi];
    if (wv != 0.0) dl += wv * k.b1[fi];
  }
  double mo = 0.0;
  const double* Mj = a.Mj + (int64_t)blockIdx.y * N;
  for (int j = threadIdx.x; j < N; j += blockDim.x) {
    if (k.cntn[j]) ut += 1.0;
    const double ex = k.load[j] - Kj[j];
    if (ex > 1e-9) ov += ex;
    if (k.mem[j] > Mj[j]) mo += k.mem[j] - Mj[j];       // only a seed can bring this in; moves never add to it
  }
  Cost c;
  c.delay = block_sum(dl, red); __syncthreads();
  c.util = block_sum(ut, red); __syncthreads();
  c.over = block_sum(ov, red); __syncthreads();
  c.uncov = block_sum(uc, red); __syncthreads();
  c.flips = block_sum(fl, red); __syncthreads();
  c.pods = block_sum(pd, red); __syncthreads();
  c.memover = block_sum(mo, red); __syncthreads();
  __shared__ Cost bc;
  if (threadIdx.x == 0) bc = c;
  __syncthreads();
  return bc;
}

// One elementary change of function f (remove pod j_out and/or add pod j_in), evaluated by one warp:
// returns the delay change (valid in every lane) and accumulates CPU-load changes into delta[].
// Load deltas are accumulated in fixed point (2^-30 cores): integer adds commute, so the sum does not depend on
// the order in which the lanes' atomics land and a run is bit-reproducible.
constexpr double kFxLoad = 1073741824.0;
__device__ __forceinline__ void fx_add(unsigned long long* p, double v) {
  atomicAdd(p, (unsigned long long)(long long)llrint(fmax(fmin(v, 4e9), -4e9) * kFxLoad));
}
__device__ double eval_change(const LsArgs& a, const Chain& k, const double* w, const double* r,
                              const double* dT, int f, int j_out, int j_in, unsigned long long* delta) {
  const int N = a.N, lane = threadIdx.x & 31;
  const double* b1 = k.b1 + (int64_t)f * N; const double* b2 = k.b2 + (int64_t)f * N;
  const int* a1 = k.a1 + (int64_t)f * N; const int* a2 = k.a2 + (int64_t)f * N;
  const double* wf = w + (int64_t)f * N; const double* rf = r + (int64_t)f * N;
  const double* din = j_in >= 0 ? dT + (int64_t)j_in * N : nullptr;
  double dd = 0.0;
  for (int i = lane; i < N; i += 32) {
    const int oa = a1[i];
    const double ob = b1[i];
    int na = oa; double nb = ob;
    if (oa == j_out) { na = a2[i]; nb = b2[i]; }
    if (din) { const double v = din[i]; if (v < nb) { nb = v; na = j_in; } }
    if (na != oa) {
      const double wv = wf[i];
      if (wv != 0.0) {
        dd += wv * (nb - ob);
        if (oa >= 0) fx_add(delta + oa, -wv * rf[oa]);
        if (na >= 0) fx_add(delta + na, wv * rf[na]);
      }
    }
  }
  return warp_sum(dd);
}

// penalty change for the accumulated load deltas; clears delta[] again.  One warp.
__device__ double eval_overload_delta(const LsArgs& a, const Chain& k, const double* Kj, unsigned long long* delta) {
  const int N = a.N, lane = threadIdx.x & 31;
  __syncwarp();
  double dv = 0.0;
  for (int j = lane; j < N; j += 32) {
    const unsigned long long raw = delta[j];
    if (raw != 0ull) {
      const double dl = (double)(long long)raw * (1.0 / kFxLoad);
      const double o0 = fmax(k.load[j] - Kj[j], 0.0), o1 = fmax(k.load[j] + dl - Kj[j], 0.0);
      dv += (o1 > 1e-9 ? o1 : 0.0) - (o0 > 1e-9 ? o0 : 0.0);
      delta[j] = 0ull;
    }
  }
  __syncwarp();
  return warp_sum(dv);
}

enum { MV_NONE = 0, MV_ADD, MV_DROP, MV_SWAP, MV_REPLACE, MV_EXCH, MV_NODE };
// ADD(f, j) | DROP(f, j) | SWAP(f, j -> t) | REPLACE(node j: f -> t) | EXCH((f, j) <-> pod t = g*N + j2)
// | NODE(every pod of node j moves to the empty node t; f = number of functions, step 2 only)
struct Move { int type, f, j, t; };
constexpr int kMaxTabu = 12;
constexpr int kSwapWindow = 96;                // swap targets examined per pod and sweep when N is larger
constexpr int kSubsample = 4;                  // sampled sweeps look at 1/kSubsample of the moves
constexpr int kMaxBatch = 8;                  // disjoint proposals applied together in one sweep
constexpr int64_t kMaxExchange = 1 << 12;     // exchange proposals examined per sweep (sampled beyond that)
constexpr double kUnrepairable = 1e11;        // state whose overload cannot be routed away

__device__ inline void apply_move(const Chain& k, int N, const Move& m, bool undo) {
  const uint8_t on = undo ? 0 : 1, off = undo ? 1 : 0;
  if (m.type == MV_ADD) k.c[(int64_t)m.f * N + m.j] = on;
  else if (m.type == MV_DROP) k.c[(int64_t)m.f * N + m.j] = off;
  else if (m.type == MV_SWAP) { k.c[(int64_t)m.f * N + m.j] = off; k.c[(int64_t)m.f * N + m.t] = on; }
  else if (m.type == MV_REPLACE) { k.c[(int64_t)m.f * N + m.j] = off; k.c[(int64_t)m.t * N + m.j] = on; }
  else if (m.type == MV_EXCH) {
    const int g = m.t / N, j2 = m.t - g * N;
    k.c[(int64_t)m.f * N + m.j] = off; k.c[(int64_t)m.f * N + j2] = on;
    k.c[(int64_t)g * N + j2] = off; k.c[(int64_t)g * N + m.j] = on;
  } else if (m.type == MV_NODE) {
    const int from = undo ? m.t : m.j, to = undo ? m.j : m.t;      // `to` is empty before the move
    for (int f = 0; f < m.f; ++f)
      if (k.c[(int64_t)f * N + from]) { k.c[(int64_t)f * N + from] = 0; k.c[(int64_t)f * N + to] = 1; }
  }
}

__global__ void __launch_bounds__(256) k_ls_prepare(LsArgs a) {
  // per instance: dT, wmax, penalty weight, objective weights
  const int b = blockIdx.x, N = a.N, F = a.F;
  const double* d = a.d + (int64_t)b * N * N;
  double* dT = a.dT + (int64_t)b * N * N;
  for (int k = threadIdx.x; k < N * N; k += blockDim.x) { const int i = k / N, j = k - i * N; dT[(int64_t)j * N + i] = d[k]; }
  __shared__ double red[32];
  const double* w = a.w + (int64_t)b * F * N;
  const double* r = a.r + (int64_t)b * F * N;
  double wm = 0.0, tw = 0.0, dmax = 0.0, rmin = INFINITY, dsum = 0.0, rsum = 0.0, rcnt = 0.0;
  for (int k = threadIdx.x; k < N * N; k += blockDim.x) dsum += d[k];
  for (int fi = threadIdx.x; fi < F * N; fi += blockDim.x) if (r[fi] > 0.0) { rsum += r[fi]; rcnt += 1.0; }
  dsum = block_sum(dsum, red); __syncthreads();
  rsum = block_sum(rsum, red); __syncthreads();
  rcnt = block_sum(rcnt, red); __syncthreads();
  for (int fi = threadIdx.x; fi < F * N; fi += blockDim.x) {
    const int f = fi / N, i = fi - f * N;
    const double md = a.maxd ? a.maxd[(int64_t)b * F + f] : INFINITY;
    double best = -INFINITY;
    for (int j = 0; j < N; ++j) { const double v = d[(int64_t)i * N + j]; if (v <= md && v > best) best = v; dmax = fmax(dmax, v); }
    wm += w[fi] * best; tw += w[fi];
    if (r[fi] > 0.0) rmin = fmin(rmin, r[fi]);
  }
  wm = block_sum(wm, red); __syncthreads();
  tw = block_sum(tw, red); __syncthreads();
  for (int o = 16; o > 0; o >>= 1) { dmax = fmax(dmax, __shfl_xor_sync(0xffffffffu, dmax, o)); rmin = fmin(rmin, __shfl_xor_sync(0xffffffffu, rmin, o)); }
  __shared__ double smx[8], smn[8];
  if ((threadIdx.x & 31) == 0) { smx[threadIdx.x >> 5] = dmax; smn[threadIdx.x >> 5] = rmin; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int q = 1; q < (blockDim.x >> 5); ++q) { dmax = fmax(dmax, smx[q]); rmin = fmin(rmin, smn[q]); }
    double* s = a.inst_scal + (int64_t)b * 4;
    double a_d, a_u;
    if (a.kind == NEPTUNE_KIND_MIN_DELAY) { a_d = 1.0; a_u = 0.0; }
    else if (a.kind == NEPTUNE_KIND_MIN_UTIL) { a_d = 0.0; a_u = 1.0; }
    else { a_u = a.alpha / (double)N; a_d = (tw != 0.0 && wm != 0.0) ? (1.0 - a.alpha) / wm : 0.0; }
    // mu_big: one unit of CPU overload costs more than any reroute that could remove it (used while a
    // state is not routable at all); mu: proposal weight ~ typical repair cost per core (dmean / rmean / 10)
    double mu_big = (isfinite(rmin) ? 4.0 * (dmax + 1.0) / rmin : 1.0) * (a_d > 0.0 ? a_d : 1.0);
    mu_big = fmax(mu_big, 100.0 * a_u);
    const double dmean = dsum / fmax(1.0, (double)N * (double)(N - 1)), rmean = rcnt > 0.0 ? rsum / rcnt : 1.0;
    double mu = a_d > 0.0 ? 0.1 * a_d * dmean / fmax(rmean, 1e-9) : 0.01 * a_u;
    s[0] = mu_big; s[1] = mu; s[2] = a_d; s[3] = a_u;
  }
}

// THREADS = 256 (3 blocks per SM) for small instances, 768 (one block per SM, 24 warps evaluating moves)
// when a sweep has 10^5+ moves (N > 128)
template <int THREADS>
__global__ void __launch_bounds__(THREADS, THREADS == 256 ? 3 : 1) k_local_search(LsArgs a) {
  const int chain = blockIdx.x, b = blockIdx.y, N = a.N, F = a.F;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, nw = blockDim.x >> 5;
  const double* d = a.d + (int64_t)b * N * N;
  const double* dT = a.dT + (int64_t)b * N * N;
  const double* w = a.w + (int64_t)b * F * N;
  const double* r = a.r + (int64_t)b * F * N;
  const double* m = a.m + (int64_t)b * F;
  const double* Mj = a.Mj + (int64_t)b * N;
  const double* Kj = a.Kj + (int64_t)b * N;
  const double* scal = a.inst_scal + (int64_t)b * 4;
  const double mu = scal[1], a_d = scal[2], a_u = scal[3];
  Chain k = carve(a.chain_ws + ((int64_t)b * a.chains + chain) * a.chain_stride, N, F);
  extern __shared__ double dyn[];
  unsigned long long* delta = reinterpret_cast<unsigned long long*>(dyn) + (int64_t)wid * N;   // per-warp load deltas (fixed point)
  if (a.use_smem) {
    // every move evaluation walks d^T, w, r and the nearest / second-nearest tables of one function: at
    // 50x10 all of it (~60 KB) fits next to three resident blocks per SM, so these reads become
    // shared-memory reads instead of L2 round trips
    double* p = dyn + (int64_t)nw * N;
    double* s_d = p; p += (int64_t)N * N;
    double* s_dT = p; p += (int64_t)N * N;
    double* s_w = p; p += (int64_t)F * N;
    double* s_r = p; p += (int64_t)F * N;
    double* s_b1 = p; p += (int64_t)F * N;
    double* s_b2 = p; p += (int64_t)F * N;
    double* s_load = p; p += N; double* s_mem = p; p += N; double* s_K = p; p += N; double* s_M = p; p += N;
    double* s_m = p; p += F;
    int* s_a1 = reinterpret_cast<int*>(p);
    int* s_a2 = s_a1 + (int64_t)F * N;
    int* s_pods = s_a2 + (int64_t)F * N;
    int* s_cntf = s_pods + (int64_t)F * N;
    int* s_cntn = s_cntf + F;
    uint8_t* s_c = reinterpret_cast<uint8_t*>(s_cntn + N);
    for (int q = tid; q < N * N; q += blockDim.x) { s_d[q] = d[q]; s_dT[q] = dT[q]; }
    for (int q = tid; q < F * N; q += blockDim.x) { s_w[q] = w[q]; s_r[q] = r[q]; }
    for (int q = tid; q < N; q += blockDim.x) { s_K[q] = Kj[q]; s_M[q] = Mj[q]; }
    for (int q = tid; q < F; q += blockDim.x) s_m[q] = m[q];
    d = s_d; dT = s_dT; w = s_w; r = s_r; Kj = s_K; Mj = s_M; m = s_m;
    k.b1 = s_b1; k.b2 = s_b2; k.a1 = s_a1; k.a2 = s_a2;
    k.load = s_load; k.mem = s_mem; k.pods = s_pods; k.cntf = s_cntf; k.cntn = s_cntn; k.c = s_c;
  }
  __shared__ double red[32];
  __shared__ double capsh[32];
  __shared__ double wbest[THREADS / 32];
  __shared__ Move wmove[THREADS / 32];
  __shared__ Move mv;
  __shared__ Move batch[kMaxBatch];
  __shared__ int n_batch;
  __shared__ int scan_sh[THREADS];
  __shared__ int n_pods, n_tabu;
  __shared__ uint64_t s_rand[2];
  __shared__ Move tabu_list[kMaxTabu];
  __shared__ double best_total;
  uint64_t rs = a.rng ^ (0x9E3779B97F4A7C15ull * (uint64_t)(chain + 1)) ^ (0xD1B54A32D192ED03ull * (uint64_t)(b + 1));
  rng_next(rs);

  // ---- start placement: a seed, or a rounding of the LP guide ----------------------------------------
  const int seed_id = chain % a.S;
  const uint8_t* seed = a.seeds + ((int64_t)b * a.S + seed_id) * F * N;
  for (int q = tid; q < F * N; q += blockDim.x) k.c[q] = seed[q];
  for (int q = tid; q < nw * N; q += blockDim.x) reinterpret_cast<unsigned long long*>(dyn)[q] = 0ull;
  __syncthreads();
  if (a.guide && chain >= a.S && (chain / a.S) % 2 == 1 && tid == 0) {
    // threshold rounding of c-bar, then memory repair (drop the weakest pods) and coverage repair
    const double* g = a.guide + (int64_t)b * F * N;
    const double thr = 0.15 + 0.1 * (double)((chain / a.S / 2) % 7);
    for (int q = 0; q < F * N; ++q) k.c[q] = g[q] >= thr;
    for (int j = 0; j < N; ++j) {
      while (true) {
        double mem = 0.0; int worst = -1; double wv = INFINITY;
        for (int f = 0; f < F; ++f) if (k.c[(int64_t)f * N + j]) { mem += m[f]; if (g[(int64_t)f * N + j] < wv) { wv = g[(int64_t)f * N + j]; worst = f; } }
        if (mem <= Mj[j] || worst < 0) break;
        k.c[(int64_t)worst * N + j] = 0;
      }
    }
    for (int f = 0; f < F; ++f) {
      int any = 0; for (int j = 0; j < N; ++j) any |= k.c[(int64_t)f * N + j];
      if (!any) {
        int bj = -1; double bv = -1.0;
        for (int j = 0; j < N; ++j) {
          double mem = 0.0; for (int f2 = 0; f2 < F; ++f2) if (k.c[(int64_t)f2 * N + j]) mem += m[f2];
          if (mem + m[f] <= Mj[j] && g[(int64_t)f * N + j] > bv) { bv = g[(int64_t)f * N + j]; bj = j; }
        }
        if (bj >= 0) k.c[(int64_t)f * N + bj] = 1;
      }
    }
  }
  __syncthreads();

  auto rebuild = [&]() {
    for (int f = 0; f < F; ++f) route_f(a, k, d, f);
    __syncthreads();
    node_state(a, k, w, r, m);
    __syncthreads();
  };
  // step 2 (reference neptune_step2.py / constraints_step2.py / objectives.py:55-63), closed form for a
  // fixed placement: W*|c xor old| - (W+1)*(sum_old - sum_c) in "delete" mode (needs sum_c <= sum_old),
  // W*|c xor old| - (W-1)*(sum_c - sum_old) in "create" mode (needs sum_c >= sum_old); the step-1
  // objective must stay below bound = soften_step1_sol * step-1 score.
  const int mode2 = a.step2_mode;
  const double Wd = (double)F * (double)N;
  double sold = 0.0;
  if (mode2) { const double* old = a.old + (int64_t)b * F * N; for (int q = 0; q < F * N; ++q) sold += old[q] > 0.0; }
  const double bound2 = mode2 ? a.bound[b] : 0.0;
  const double pen_unit = 4.0 * Wd * Wd + 1.0;      // larger than any feasible step-2 objective value
  auto disruption = [&](double flips, double pods) -> double {
    const double delta = sold - pods;
    if (mode2 == 1) return Wd * flips + (delta >= 0.0 ? -(Wd + 1.0) * delta : pen_unit * (-delta));
    return Wd * flips + (delta <= 0.0 ? (Wd - 1.0) * delta : pen_unit * delta);
  };
  auto objective = [&](double delay, double util, double over, double uncov, double flips, double pods, double mu_) {
    const double o1 = a_d * delay + a_u * util;
    if (!mode2) return o1 + mu_ * over + kCoverage * uncov;
    const double ex = o1 - bound2 * (1.0 + 1e-12);
    return disruption(flips, pods) + (ex > 0.0 ? 10.0 * pen_unit * (1.0 + ex / fmax(fabs(bound2), 1e-9)) : 0.0) +
           mu_ * over + kCoverage * uncov;
  };
  auto total_of = [&](const Cost& c) { return objective(c.delay, c.util, c.over, c.uncov, c.flips, c.pods, mu) + kCoverage * c.memover; };

  // random kick: `n` random swap / replace changes that keep memory feasible (thread 0)
  auto kick = [&](int n) {
    if (tid == 0) {
      for (int t = 0; t < n; ++t) {
        const int f = (int)(rng_next(rs) % (uint64_t)F);
        int pods[64]; int np = 0;
        for (int j = 0; j < N && np < 64; ++j) if (k.c[(int64_t)f * N + j]) pods[np++] = j;
        const int jn = (int)(rng_next(rs) % (uint64_t)N);
        if (k.c[(int64_t)f * N + jn]) continue;
        double mem = 0.0; for (int f2 = 0; f2 < F; ++f2) if (k.c[(int64_t)f2 * N + jn]) mem += m[f2];
        if (mem + m[f] > Mj[jn]) {
          // replace a random function on jn by f, if that function has another pod
          int cand[64]; int nc = 0;
          for (int f2 = 0; f2 < F && nc < 64; ++f2) if (k.c[(int64_t)f2 * N + jn]) cand[nc++] = f2;
          if (!nc) continue;
          const int f2 = cand[rng_next(rs) % (uint64_t)nc];
          int cnt2 = 0; for (int j = 0; j < N; ++j) cnt2 += k.c[(int64_t)f2 * N + j];
          if (cnt2 < 2 || mem - m[f2] + m[f] > Mj[jn]) continue;
          k.c[(int64_t)f2 * N + jn] = 0;
        }
        k.c[(int64_t)f * N + jn] = 1;
        if (np > 1 && (rng_next(rs) & 1)) k.c[(int64_t)f * N + pods[rng_next(rs) % (uint64_t)np]] = 0;
      }
    }
    __syncthreads();
  };

  if (chain >= a.S && !(a.guide && (chain / a.S) % 2 == 1)) kick(1 + (chain / a.S) % 6);
  rebuild();
  Cost cur = full_cost(a, k, w, Kj, red);
  double cur_total = total_of(cur);
  if (tid == 0) best_total = INFINITY;
  __syncthreads();
  const double mu_big = scal[0];
  // true cost of the current state (block-uniform; all threads must call)
  auto true_total = [&](const Cost& c) -> double {
    if (c.uncov > 0.0 || c.memover > 0.0)
      return objective(c.delay, c.util, c.over, c.uncov, c.flips, c.pods, mu_big) + kCoverage * c.memover;
    if (c.over <= 0.0) return objective(c.delay, c.util, 0.0, 0.0, c.flips, c.pods, 0.0);
    CapRoute q{N, F, d, w, r, Kj, k.c, k.ch, k.sec, k.th, k.rho, k.alt, k.cload, k.lam};
    const CapResult cr = cap_route(q, 48, red, capsh);
    if (cr.feasible) return objective(cr.cost, c.util, 0.0, 0.0, c.flips, c.pods, 0.0);
    return objective(c.delay, c.util, c.over, 0.0, c.flips, c.pods, mu_big) + (mode2 ? 1000.0 * pen_unit : kUnrepairable);
  };
  double cur_true = true_total(cur);
  auto save_best = [&]() {
    // a chain's best must be usable: memory ok by construction, every function placed, CPU rows routable
    if (cur_true < (mode2 ? pen_unit : kUnrepairable) && cur_true < best_total) {
      __syncthreads();
      for (int q = tid; q < F * N; q += blockDim.x) k.best_c[q] = k.c[q];
      if (tid == 0) best_total = cur_true;
    }
    __syncthreads();
  };
  save_best();

  // Moves are PROPOSED by their penalised delta (overload priced at mu, an estimate of the repair cost per
  // core) and ACCEPTED on the true cost of the new state: nearest routing if no node overloads, else the
  // capacity-aware routing of route_cap.cuh.  A rejected proposal is undone and kept tabu until the state
  // changes or the chain is kicked.
  int stall = 0;
  bool stage2 = false;
  bool sampled = true;       // examine a random quarter of the neighbourhood while that still finds improvements
  n_tabu = 0;
  for (int sweep = 0; sweep < a.sweeps; ++sweep) {
    // ---- pod list -------------------------------------------------------------------------------------
    if (tid == 0) { n_pods = 0; s_rand[0] = rng_next(rs); s_rand[1] = rng_next(rs); }   // only thread 0 owns the RNG
    __syncthreads();
    {
      // ordered compaction (ascending q): every thread counts a contiguous chunk, an exclusive scan of the counts
      // over the block gives its write offset -- the pod list does not depend on thread timing
      const int chunk = (F * N + (int)blockDim.x - 1) / (int)blockDim.x;
      const int q0 = tid * chunk, q1 = min(F * N, q0 + chunk);
      int cnt = 0;
      for (int q = q0; q < q1; ++q) cnt += k.c[q] != 0;
      scan_sh[tid] = cnt;
      __syncthreads();
      for (int o = 1; o < (int)blockDim.x; o <<= 1) {
        const int v = tid >= o ? scan_sh[tid - o] : 0;
        __syncthreads();
        scan_sh[tid] += v;
        __syncthreads();
      }
      int at = scan_sh[tid] - cnt;
      for (int q = q0; q < q1; ++q) if (k.c[q]) k.pods[at++] = q;
      if (tid == (int)blockDim.x - 1) n_pods = scan_sh[tid];
    }
    __syncthreads();
    const int P = n_pods;
    // swap targets: all nodes for small N, a window of kSwapWindow nodes (rotating with the sweep) beyond
    const int swin = N <= kSwapWindow ? N : kSwapWindow;
    const int swoff = N <= kSwapWindow ? 0 : (int)(s_rand[1] % (uint64_t)N);
    const int64_t n_add = (int64_t)F * N, n_drop = P, n_swap = (int64_t)P * swin, n_rep = (int64_t)P * F;
    const int64_t pp = (int64_t)P * P;
    const int64_t n_exch = pp < kMaxExchange ? pp : kMaxExchange;
    const int64_t ex_off = (int64_t)(s_rand[0] % (uint64_t)(pp > 0 ? pp : 1));        // block-uniform
    const int64_t ex_stride = pp > kMaxExchange ? (int64_t)(2 * (s_rand[1] % 4096) + 1) : 1;
    // two-stage neighbourhood: the (quadratic) exchange moves are only examined once the basic
    // add / drop / swap / replace neighbourhood has no improving proposal left
    const int64_t n_node = mode2 ? (int64_t)N * N : 0;          // whole-node relocation (step 2 only)
    const int64_t total = n_add + n_drop + n_swap + n_rep + n_node + (stage2 ? n_exch : 0);
    double my_best = -1e-9 * (1.0 + fabs(cur_total));      // only strictly improving proposals
    Move my_mv{MV_NONE, 0, 0, 0};
    const int ntb = n_tabu;
    const int sub = sampled ? kSubsample : 1;
    const int64_t q_first = (int64_t)wid + (int64_t)nw * (int64_t)(sampled ? (s_rand[1] >> 20) % kSubsample : 0);
    for (int64_t q = q_first; q < total; q += (int64_t)nw * sub) {
      Move cand; bool ok = false; double dutil = 0.0, dcov = 0.0, dflip = 0.0, dpods = 0.0, dmem = 0.0;
      auto relief = [&](int j_, double dm) { return fmax(k.mem[j_] + dm - Mj[j_], 0.0) - fmax(k.mem[j_] - Mj[j_], 0.0); };
      if (q < n_add) {
        const int f = (int)(q / N), j = (int)(q - (int64_t)f * N);
        ok = !k.c[q] && k.mem[j] + m[f] <= Mj[j];
        cand = Move{MV_ADD, f, j, -1};
        if (ok && k.cntn[j] == 0) dutil = 1.0;
        if (ok && k.cntf[f] == 0) dcov = -1.0;
      } else if (q < n_add + n_drop) {
        const int pq = k.pods[q - n_add], f = pq / N, j = pq - f * N;
        ok = k.cntf[f] >= 2;
        cand = Move{MV_DROP, f, j, -1};
        if (ok && k.cntn[j] == 1) dutil = -1.0;
        if (ok) dmem = relief(j, -m[f]);
      } else if (q < n_add + n_drop + n_swap) {
        const int64_t t = q - n_add - n_drop;
        const int pq = k.pods[t / swin], f = pq / N, j = pq - f * N, jn = (int)((swoff + t % swin) % N);
        ok = !k.c[(int64_t)f * N + jn] && k.mem[jn] + m[f] <= Mj[jn];
        cand = Move{MV_SWAP, f, j, jn};
        if (ok) dutil = (k.cntn[jn] == 0 ? 1.0 : 0.0) - (k.cntn[j] == 1 ? 1.0 : 0.0);
        if (ok) dmem = relief(j, -m[f]);
      } else if (q < n_add + n_drop + n_swap + n_rep) {
        const int64_t t = q - n_add - n_drop - n_swap;
        const int pq = k.pods[t / F], f = pq / N, j = pq - f * N, fn = (int)(t % F);
        ok = fn != f && !k.c[(int64_t)fn * N + j] && k.cntf[f] >= 2 && k.mem[j] - m[f] + m[fn] <= Mj[j];
        cand = Move{MV_REPLACE, f, j, fn};
        if (ok && k.cntf[fn] == 0) dcov = -1.0;
      } else if (q < n_add + n_drop + n_swap + n_rep + n_node) {
        const int64_t t = q - n_add - n_drop - n_swap - n_rep;
        const int j = (int)(t / N), j2 = (int)(t - (int64_t)j * N);
        ok = j != j2 && k.cntn[j] > 0 && k.cntn[j2] == 0 && k.mem[j] <= Mj[j2];
        cand = Move{MV_NODE, F, j, j2};
      } else {
        // exchange: pods (f, j) and (g, j2) trade nodes -> (f, j2), (g, j); pod counts stay as they are
        const int64_t t = (ex_off + (q - n_add - n_drop - n_swap - n_rep - n_node) * ex_stride) % pp;
        const int p1 = (int)(t / P), p2 = (int)(t - (int64_t)p1 * P);
        if (p1 < p2) {
          const int q1 = k.pods[p1], q2 = k.pods[p2];
          const int f = q1 / N, j = q1 - f * N, g = q2 / N, j2 = q2 - g * N;
          ok = f != g && j != j2 && !k.c[(int64_t)f * N + j2] && !k.c[(int64_t)g * N + j] &&
               k.mem[j] - m[f] + m[g] <= Mj[j] && k.mem[j2] - m[g] + m[f] <= Mj[j2];
          cand = Move{MV_EXCH, f, j, q2};
        }
      }
      if (!ok) continue;
      bool tabu = false;
      for (int t = 0; t < ntb; ++t)
        tabu = tabu || (tabu_list[t].type == cand.type && tabu_list[t].f == cand.f && tabu_list[t].j == cand.j &&
                        tabu_list[t].t == cand.t);
      if (tabu) continue;
      double dd = 0.0;
      if (cand.type == MV_ADD) dd = eval_change(a, k, w, r, dT, cand.f, -1, cand.j, delta);
      else if (cand.type == MV_DROP) dd = eval_change(a, k, w, r, dT, cand.f, cand.j, -1, delta);
      else if (cand.type == MV_SWAP) dd = eval_change(a, k, w, r, dT, cand.f, cand.j, cand.t, delta);
      else if (cand.type == MV_REPLACE) { dd = eval_change(a, k, w, r, dT, cand.f, cand.j, -1, delta);
                                          dd += eval_change(a, k, w, r, dT, cand.t, -1, cand.j, delta); }
      else if (cand.type == MV_NODE) {
        for (int f = 0; f < F; ++f)
          if (k.c[(int64_t)f * N + cand.j]) dd += eval_change(a, k, w, r, dT, f, cand.j, cand.t, delta);
      }
      else { const int g = cand.t / N, j2 = cand.t - g * N;
             dd = eval_change(a, k, w, r, dT, cand.f, cand.j, j2, delta);
             dd += eval_change(a, k, w, r, dT, g, j2, cand.j, delta); }
      const double dov = eval_overload_delta(a, k, Kj, delta);
      double dt;
      if (!mode2) dt = a_d * dd + a_u * dutil + mu * dov + kCoverage * (dcov + dmem);
      else {
        const double* old = a.old + (int64_t)b * F * N;
        auto on = [&](int f_, int j_) { dflip += old[(int64_t)f_ * N + j_] > 0.0 ? -1.0 : 1.0; dpods += 1.0; };
        auto off = [&](int f_, int j_) { dflip += old[(int64_t)f_ * N + j_] > 0.0 ? 1.0 : -1.0; dpods -= 1.0; };
        if (cand.type == MV_ADD) on(cand.f, cand.j);
        else if (cand.type == MV_DROP) off(cand.f, cand.j);
        else if (cand.type == MV_SWAP) { off(cand.f, cand.j); on(cand.f, cand.t); }
        else if (cand.type == MV_REPLACE) { off(cand.f, cand.j); on(cand.t, cand.j); }
        else if (cand.type == MV_NODE) {
          for (int f = 0; f < F; ++f) if (k.c[(int64_t)f * N + cand.j]) { off(f, cand.j); on(f, cand.t); }
        }
        else { const int g = cand.t / N, j2 = cand.t - g * N; off(cand.f, cand.j); on(cand.f, j2); off(g, j2); on(g, cand.j); }
        dt = objective(cur.delay + dd, cur.util + dutil, cur.over + dov, cur.uncov + dcov, cur.flips + dflip,
                       cur.pods + dpods, mu) + kCoverage * (cur.memover + dmem) - cur_total;
      }
      if (dt < my_best) { my_best = dt; my_mv = cand; }
    }
    if (lane == 0) { wbest[wid] = my_best; wmove[wid] = my_mv; }
    __syncthreads();
    if (tid == 0) {
      // the warps' best proposals, best first; keep those that touch pairwise disjoint functions and nodes
      // (their delay changes are then independent and their memory checks stay valid together)
      int order[THREADS / 32];
      for (int q = 0; q < nw; ++q) order[q] = q;
      for (int q = 1; q < nw; ++q) { const int v = order[q]; int p2 = q - 1; while (p2 >= 0 && wbest[order[p2]] > wbest[v]) { order[p2 + 1] = order[p2]; --p2; } order[p2 + 1] = v; }
      int nb = 0;
      int uf[16], un[16], nuf = 0, nun = 0;
      for (int q = 0; q < nw && nb < kMaxBatch; ++q) {
        const Move c = wmove[order[q]];
        if (c.type == MV_NONE) continue;
        if (c.type == MV_NODE) { if (nb == 0) batch[nb++] = c; else continue; break; }
        int fs[2] = {c.f, -1}, ns[2] = {c.j, -1};
        if (c.type == MV_SWAP) ns[1] = c.t;
        else if (c.type == MV_REPLACE) fs[1] = c.t;
        else if (c.type == MV_EXCH) { fs[1] = c.t / N; ns[1] = c.t - (c.t / N) * N; }
        bool clash = false;
        for (int z = 0; z < 2; ++z) {
          for (int y2 = 0; y2 < nuf; ++y2) clash = clash || (fs[z] >= 0 && uf[y2] == fs[z]);
          for (int y2 = 0; y2 < nun; ++y2) clash = clash || (ns[z] >= 0 && un[y2] == ns[z]);
        }
        if (clash) continue;
        for (int z = 0; z < 2; ++z) { if (fs[z] >= 0) uf[nuf++] = fs[z]; if (ns[z] >= 0) un[nun++] = ns[z]; }
        batch[nb++] = c;
      }
      n_batch = nb;
      mv = nb ? batch[0] : Move{MV_NONE, 0, 0, 0};
    }
    __syncthreads();
    if (mv.type != MV_NONE) {
      // ---- apply (the whole disjoint batch first, the single best proposal if that does not pay), re-route
      // the touched functions, refresh node state, price the new state exactly --------------------------
      auto second_f = [&](const Move& m_) { return m_.type == MV_REPLACE ? m_.t : (m_.type == MV_EXCH ? m_.t / N : -1); };
      auto apply_n = [&](int cnt, bool undo) {
        if (tid == 0) for (int z = 0; z < cnt; ++z) apply_move(k, N, batch[z], undo);
        __syncthreads();
        for (int z = 0; z < cnt; ++z) {
          if (batch[z].type == MV_NODE) {
            for (int f = 0; f < F; ++f)
              if (k.c[(int64_t)f * N + batch[z].j] || k.c[(int64_t)f * N + batch[z].t]) route_f(a, k, d, f);
            continue;
          }
          route_f(a, k, d, batch[z].f);
          const int f2 = second_f(batch[z]);
          if (f2 >= 0) route_f(a, k, d, f2);
        }
        __syncthreads();
        node_state(a, k, w, r, m);
        __syncthreads();
      };
      bool accepted = false;
      for (int attempt = (n_batch > 1 ? 0 : 1); attempt < 2 && !accepted; ++attempt) {
        const int cnt = attempt == 0 ? n_batch : 1;
        apply_n(cnt, false);
        const Cost nc = full_cost(a, k, w, Kj, red);
        const double nt = true_total(nc);
        if (nt < cur_true - 1e-9 * (1.0 + fabs(cur_true))) {
          cur = nc; cur_total = total_of(nc); cur_true = nt;
          accepted = true;
        } else {
          apply_n(cnt, true);
        }
      }
      if (accepted) {
        stall = 0; stage2 = false; sampled = true;
        if (tid == 0) n_tabu = 0;
        __syncthreads();
      } else {
        if (tid == 0 && n_tabu < kMaxTabu) tabu_list[n_tabu++] = batch[0];
        __syncthreads();
        if (n_tabu < kMaxTabu) continue;            // try the next-best proposal
        mv.type = MV_NONE;                          // too many rejections: treat as a local optimum
      }
    }
    if (mv.type == MV_NONE && sampled) { sampled = false; continue; }        // nothing in the sample: look at everything
    if (mv.type == MV_NONE && !stage2) { stage2 = true; if (tid == 0) n_tabu = 0; __syncthreads(); continue; }
    if (mv.type == MV_NONE) {
      stage2 = false; sampled = true;
      // ---- local optimum: keep the best, restart from it with a kick -----------------------------------
      save_best();
      if (best_total < INFINITY) {
        for (int q = tid; q < F * N; q += blockDim.x) k.c[q] = k.best_c[q];
        __syncthreads();
      }
      ++stall;
      kick(2 + (int)(s_rand[0] % 4) + (stall > 8 ? 4 : 0));
      rebuild();
      cur = full_cost(a, k, w, Kj, red);
      cur_total = total_of(cur);
      cur_true = true_total(cur);
      if (tid == 0) n_tabu = 0;
      __syncthreads();
    }
  }
  save_best();
  if (tid == 0) a.chain_cost[(int64_t)b * a.chains + chain] = best_total;
}

// pick the best chain per instance and publish its placement / objective
__global__ void __launch_bounds__(256) k_ls_pick(LsArgs a, uint8_t* __restrict__ best_c, double* __restrict__ best_obj,
                                                 int32_t* __restrict__ best_flags) {
  const int b = blockIdx.x, N = a.N, F = a.F;
  __shared__ int pick;
  if (threadIdx.x == 0) {
    int bi = -1; double bv = INFINITY;
    for (int q = 0; q < a.chains; ++q) { const double v = a.chain_cost[(int64_t)b * a.chains + q]; if (v < bv) { bv = v; bi = q; } }
    pick = bi;
    best_obj[b] = bv;
    best_flags[b] = bi >= 0 ? NEPTUNE_OK_ALL : 0;
  }
  __syncthreads();
  const int src = pick >= 0 ? pick : 0;
  Chain k = carve(a.chain_ws + ((int64_t)b * a.chains + src) * a.chain_stride, N, F);
  const uint8_t* from = pick >= 0 ? k.best_c : a.seeds + (int64_t)b * a.S * F * N;   // no feasible chain: first seed
  for (int q = threadIdx.x; q < F * N; q += blockDim.x) best_c[(int64_t)b * F * N + q] = from[q];
}

}  // namespace neptune

using namespace neptune;

extern "C" int neptune_local_search_workspace_bytes(int B, int N, int F, int chains, int64_t* bytes) {
  if (B <= 0 || N <= 0 || F <= 0 || chains <= 0 || !bytes) return NEPTUNE_E_ARG;
  int64_t t = (int64_t)B * N * N * 8 + 256;
  t += (int64_t)B * 4 * 8 + 256;
  t += (int64_t)B * chains * chain_bytes_h(N, F);
  t += (int64_t)B * chains * 8 + 256;
  *bytes = t;
  return 0;
}

// one row of N doubles per warp in shared memory; the only part of it that grows with N without bound
static inline int ls_threads(int N) { return N > 128 ? 768 : 256; }
static inline size_t ls_row_bytes(int N) { return (size_t)(ls_threads(N) / 32) * N * 8; }
constexpr size_t kLsMaxSmem = 200 * 1024;

static int local_search_impl(int step2_mode, const double* bound, int B, int N, int F, int kind, double alpha, int chains, int sweeps,
                                    uint64_t rng_seed, int S, const double* d, const double* w, const double* r,
                                    const double* m, const double* Mj, const double* Kj, const double* maxd,
                                    const double* cost, double budget, const double* old, const uint8_t* seeds,
                                    const double* guide, uint8_t* best_c, double* best_obj, int32_t* best_flags,
                                    void* workspace, int64_t workspace_bytes, void* stream) {
  if (B <= 0 || N <= 0 || F <= 0 || kind < 0 || kind > 2 || chains <= 0 || sweeps < 0 || S <= 0)
    return NEPTUNE_E_ARG;
  if (!d || !w || !r || !m || !Mj || !Kj || !seeds || !best_c || !best_obj || !best_flags || !workspace)
    return NEPTUNE_E_ARG;
  if (step2_mode && (!bound || !old)) return NEPTUNE_E_ARG;
  int64_t need = 0;
  neptune_local_search_workspace_bytes(B, N, F, chains, &need);
  if (workspace_bytes < need) return NEPTUNE_E_NOMEM;
  cudaStream_t s = (cudaStream_t)stream;
  LsArgs a{};
  a.N = N; a.F = F; a.kind = kind; a.chains = chains; a.sweeps = sweeps; a.S = S;
  a.alpha = alpha; a.budget = budget; a.rng = rng_seed ? rng_seed : 0x1234567ull;
  a.d = d; a.w = w; a.r = r; a.m = m; a.Mj = Mj; a.Kj = Kj; a.maxd = maxd; a.cost = cost; a.old = old;
  a.seeds = seeds; a.guide = guide; a.step2_mode = step2_mode; a.bound = bound;
  char* p = (char*)workspace;
  a.dT = (double*)p; p += (((int64_t)B * N * N * 8 + 255) & ~(int64_t)255);
  a.inst_scal = (double*)p; p += 256 * (((int64_t)B * 32 + 255) / 256);
  a.chain_cost = (double*)p; p += (((int64_t)B * chains * 8 + 255) & ~(int64_t)255);
  a.chain_ws = p;
  a.chain_stride = chain_bytes_h(N, F);
  if ((p - (char*)workspace) + (int64_t)B * chains * a.chain_stride > workspace_bytes) return NEPTUNE_E_NOMEM;
  const int threads = ls_threads(N);
  size_t sm = ls_row_bytes(N);
  const size_t tables = (size_t)2 * N * N * 8 + (size_t)4 * F * N * 8 + (size_t)3 * F * N * 4 + (size_t)(4 * N + F) * 8 +
                        (size_t)(F + N) * 4 + (size_t)F * N + 64;
  a.use_smem = (threads == 256 && sm + tables <= 72 * 1024) ? 1 : 0;      // 3 blocks per SM must still fit
  if (a.use_smem) sm += tables;
  if (sm > kLsMaxSmem) return NEPTUNE_E_SIZE;
  if (threads == 256)
    NEPTUNE_CUDA_OK(cudaFuncSetAttribute(k_local_search<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
  else
    NEPTUNE_CUDA_OK(cudaFuncSetAttribute(k_local_search<768>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
  { k_ls_prepare<<<B, 256, 0, s>>>(a); NEPTUNE_COUNT(1); }
  if (threads == 256) { k_local_search<256><<<dim3(chains, B), 256, sm, s>>>(a); NEPTUNE_COUNT(1); }
  else { k_local_search<768><<<dim3(chains, B), 768, sm, s>>>(a); NEPTUNE_COUNT(1); }
  { k_ls_pick<<<B, 256, 0, s>>>(a, best_c, best_obj, best_flags); NEPTUNE_COUNT(1); }
  NEPTUNE_LAUNCH_OK();
  return 0;
}

extern "C" int neptune_local_search(int B, int N, int F, int kind, double alpha, int chains, int sweeps,
                                    uint64_t rng_seed, int S, const double* d, const double* w, const double* r,
                                    const double* m, const double* Mj, const double* Kj, const double* maxd,
                                    const double* cost, double budget, const double* old, const uint8_t* seeds,
                                    const double* guide, uint8_t* best_c, double* best_obj, int32_t* best_flags,
                                    void* workspace, int64_t workspace_bytes, void* stream) {
  return local_search_impl(0, nullptr, B, N, F, kind, alpha, chains, sweeps, rng_seed, S, d, w, r, m, Mj, Kj, maxd,
                           cost, budget, old, seeds, guide, best_c, best_obj, best_flags, workspace, workspace_bytes,
                           stream);
}

extern "C" int neptune_disruption_search(int B, int N, int F, int kind, double alpha, int mode, const double* bound,
                                         int chains, int sweeps, uint64_t rng_seed, int S, const double* d,
                                         const double* w, const double* r, const double* m, const double* Mj,
                                         const double* Kj, const double* maxd, const double* cost, double budget,
                                         const double* old, const uint8_t* seeds, uint8_t* best_c, double* best_obj,
                                         int32_t* best_flags, void* workspace, int64_t workspace_bytes, void* stream) {
  if (mode != 1 && mode != 2) return NEPTUNE_E_ARG;
  return local_search_impl(mode, bound, B, N, F, kind, alpha, chains, sweeps, rng_seed, S, d, w, r, m, Mj, Kj, maxd,
                           cost, budget, old, seeds, nullptr, best_c, best_obj, best_flags, workspace,
                           workspace_bytes, stream);
}

extern "C" int neptune_local_search_fits(int N, int F, int32_t* fits) {
  if (N <= 0 || F <= 0 || !fits) return NEPTUNE_E_ARG;
  *fits = ls_row_bytes(N) <= kLsMaxSmem ? 1 : 0;
  return 0;
}
