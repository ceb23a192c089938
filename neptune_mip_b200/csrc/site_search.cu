// site_search.cu -- best-improvement pod-exchange search over placements c[B][F][N] for the min-delay objective under
// nearest-pod routing, at the sizes the shared-memory searches do not reach (BASELINE config 4: 2000 x 200).
//
//   obj(c) = sum_f sum_i w[f,i] * d1[f,i],   d1 = delay from source i to the nearest open pod of f
//   memory rows sum_f m[f] c[f,j] <= Mj (the real m: several memory sizes work), every function keeps a pod.
//
// Per (instance, function, source) the search keeps the nearest and second-nearest open pod (a1/d1, a2/d2; lowest node
// among equal delays); per node the free memory.  One round:
//   k_ss_tables  : only for the functions changed in the last round ("dirty"):
//                  G[f][j] = sum_i w max(0, d1 - d[i,j])     (gain of adding pod (f, j); k_site_gain's order and rounding)
//                  L[f][j] = sum_{i: a1 = j} w (d2 - d1)     (loss of removing open pod (f, j); +inf with one pod)
//   k_ss_node    : per node j the best of  add (f, j)  and  exchange f_out -> f_in on j          (O(F * pods on j))
//   k_ss_func    : per function f the best relocation j_out -> j_in, j_in among the 4 nodes with the largest G[f][.]
//                  that have memory for f; delta evaluated exactly in O(N) per pair
//   k_ss_resolve : per instance, proposals with delta < -1e-12 (1 + obj) sorted by (delta, nodes before functions,
//                  index); one warp walks them and accepts a proposal when none of its functions and nodes has been
//                  touched in this round.  The objective separates by function and memory by node, so moves on disjoint
//                  functions and nodes are independent: obj after the round = obj before + the accepted deltas.
//   k_ss_memfree, k_ss_pods, k_ss_nearest, k_ss_objf : state of the changed functions and nodes.
// Sums run over ascending i with separate multiply and add (no FMA), no floating-point atomics: a run is
// bit-reproducible and equal to its numpy statement (tests/site_search_reference.py).
#include "common.cuh"

namespace neptune {

constexpr int kSsThreads = 256;
constexpr int kSsFuncThreads = 128;
constexpr int kSsResolveThreads = 512;
constexpr int kSsChunk = 512;           // sources staged per shared-memory chunk
constexpr int kSsCand = 4;              // relocation targets per function
constexpr double kSsMemTol = 1e-9;      // the greedy's memory tolerance (site.cu)

struct SsState {
  int N, F;
  const double *d, *w, *m, *Mj;
  uint8_t* c;                           // [B][F][N], updated in place
  int *a1, *a2, *plist, *npods;         // plist[b][f][0, npods): pods of f in ascending node order
  double *d1, *d2, *G, *L, *memfree, *objf;
  uint8_t* dirty;                       // [B][F]
  double* prop_d;                       // [B][N + F]: nodes first, then functions
  int *prop_x, *prop_y;                 // node: (f_in, f_out or -1); function: (j_out, j_in)
  double* cd;                           // [B][N + F] compacted proposals below the threshold
  int *ci, *sorted;
  int32_t* info;                        // [B][4]
  int* flags;                           // [0] moves accepted (all instances), [1] a function without a pod
};

__device__ __forceinline__ void ss_ordered_compact_begin(int* s_base) {
  if (threadIdx.x == 0) *s_base = 0;
  __syncthreads();
}

// one step of a block-wide ordered compaction: threads whose `on` is set append `val` in thread order
__device__ __forceinline__ void ss_ordered_append(bool on, int* s_wcnt, int* s_base, int* out, int val) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const unsigned bal = __ballot_sync(0xffffffffu, on);
  if (lane == 0) s_wcnt[wid] = __popc(bal);
  __syncthreads();
  int off = *s_base;
  for (int q = 0; q < wid; ++q) off += s_wcnt[q];
  if (on) out[off + __popc(bal & ((1u << lane) - 1u))] = val;
  __syncthreads();
  if (threadIdx.x == 0) { int t = 0; for (int q = 0; q < nw; ++q) t += s_wcnt[q]; *s_base += t; }
  __syncthreads();
}

__global__ void __launch_bounds__(kSsThreads) k_ss_pods(SsState s) {
  const int b = blockIdx.y, f = blockIdx.x, N = s.N;
  const int64_t bf = (int64_t)b * s.F + f;
  if (!s.dirty[bf]) return;
  __shared__ int s_wcnt[32], s_base;
  const uint8_t* __restrict__ c = s.c + bf * N;
  int* out = s.plist + bf * N;
  ss_ordered_compact_begin(&s_base);
  for (int j0 = 0; j0 < N; j0 += blockDim.x) {
    const int j = j0 + threadIdx.x;
    ss_ordered_append(j < N && c[j] != 0, s_wcnt, &s_base, out, j);
  }
  if (threadIdx.x == 0) {
    s.npods[bf] = s_base;
    if (s_base == 0) atomicExch(s.flags + 1, 1);
  }
}

__global__ void __launch_bounds__(kSsThreads) k_ss_nearest(SsState s) {
  const int b = blockIdx.z, f = blockIdx.y, i = blockIdx.x * blockDim.x + threadIdx.x, N = s.N;
  const int64_t bf = (int64_t)b * s.F + f;
  if (!s.dirty[bf] || i >= N) return;
  const int* __restrict__ pods = s.plist + bf * N;
  const double* __restrict__ di = s.d + (int64_t)b * N * N + (int64_t)i * N;
  const int n = s.npods[bf];
  double v1 = INFINITY, v2 = INFINITY;
  int a1 = -1, a2 = -1;
  for (int q = 0; q < n; ++q) {                  // ascending nodes: the first of equal delays wins
    const int j = pods[q];
    const double v = di[j];
    if (v < v1) { v2 = v1; a2 = a1; v1 = v; a1 = j; }
    else if (v < v2) { v2 = v; a2 = j; }
  }
  const int64_t o = bf * N + i;
  s.a1[o] = a1; s.d1[o] = v1; s.a2[o] = a2; s.d2[o] = v2;
}

__global__ void k_ss_objf(SsState s) {
  const int b = blockIdx.y, f = blockIdx.x * blockDim.x + threadIdx.x, N = s.N;
  if (f >= s.F) return;
  const int64_t bf = (int64_t)b * s.F + f;
  if (!s.dirty[bf]) return;
  const double* __restrict__ w = s.w + bf * N;
  const double* __restrict__ d1 = s.d1 + bf * N;
  double acc = 0.0;
  for (int i = 0; i < N; ++i) acc = __dadd_rn(acc, __dmul_rn(w[i], d1[i]));
  s.objf[bf] = acc;
}

__device__ __forceinline__ double ss_objective(const SsState& s, int b) {
  double o = 0.0;
  for (int f = 0; f < s.F; ++f) o = __dadd_rn(o, s.objf[(int64_t)b * s.F + f]);
  return o;
}

__global__ void k_ss_obj(SsState s, double* __restrict__ obj_out, int slot) {
  if (threadIdx.x == 0) obj_out[(int64_t)blockIdx.x * 2 + slot] = ss_objective(s, blockIdx.x);
}

__global__ void __launch_bounds__(kSsThreads) k_ss_memfree(SsState s) {
  const int b = blockIdx.y, j = blockIdx.x * blockDim.x + threadIdx.x, N = s.N;
  if (j >= N) return;
  double mf = s.Mj[(int64_t)b * N + j];
  for (int f = 0; f < s.F; ++f)
    if (s.c[((int64_t)b * s.F + f) * N + j]) mf -= s.m[(int64_t)b * s.F + f];
  s.memfree[(int64_t)b * N + j] = mf;
}

__global__ void __launch_bounds__(kSsThreads) k_ss_tables(SsState s) {
  const int b = blockIdx.z, f = blockIdx.y, j = blockIdx.x * blockDim.x + threadIdx.x, N = s.N;
  const int64_t bf = (int64_t)b * s.F + f;
  if (!s.dirty[bf]) return;
  const double* __restrict__ d = s.d + (int64_t)b * N * N;
  const double* __restrict__ w = s.w + bf * N;
  const double* __restrict__ d1 = s.d1 + bf * N;
  const double* __restrict__ d2 = s.d2 + bf * N;
  const int* __restrict__ a1 = s.a1 + bf * N;
  __shared__ double s_w[kSsChunk], s_d1[kSsChunk], s_d2[kSsChunk];
  __shared__ int s_a1[kSsChunk];
  double g = 0.0, l = 0.0;
  for (int i0 = 0; i0 < N; i0 += kSsChunk) {
    const int n = min(kSsChunk, N - i0);
    __syncthreads();
    for (int t = threadIdx.x; t < n; t += blockDim.x) {
      s_w[t] = w[i0 + t]; s_d1[t] = d1[i0 + t]; s_d2[t] = d2[i0 + t]; s_a1[t] = a1[i0 + t];
    }
    __syncthreads();
    if (j < N) {
      const double* __restrict__ dj = d + (int64_t)i0 * N + j;
#pragma unroll 4
      for (int t = 0; t < n; ++t) {
        const double wv = s_w[t];
        if (wv == 0.0) continue;                               // adds +0: skipping it changes no bit
        g = __dadd_rn(g, __dmul_rn(wv, fmax(s_d1[t] - dj[(int64_t)t * N], 0.0)));
        if (s_a1[t] == j) l = __dadd_rn(l, __dmul_rn(wv, __dsub_rn(s_d2[t], s_d1[t])));
      }
    }
  }
  if (j < N) {
    s.G[bf * N + j] = g;
    s.L[bf * N + j] = s.npods[bf] > 1 ? l : INFINITY;
  }
}

// one thread per node: add (f, j) or exchange f_out -> f_in on j; add first, then f_out ascending, f ascending inside,
// a later candidate must be strictly better
__global__ void __launch_bounds__(128) k_ss_node(SsState s) {
  const int b = blockIdx.y, j = blockIdx.x * blockDim.x + threadIdx.x, N = s.N, F = s.F;
  if (j >= N) return;
  const uint8_t* __restrict__ c = s.c + (int64_t)b * F * N + j;
  const double* __restrict__ G = s.G + (int64_t)b * F * N + j;
  const double* __restrict__ L = s.L + (int64_t)b * F * N + j;
  const double* __restrict__ m = s.m + (int64_t)b * F;
  const double mf = s.memfree[(int64_t)b * N + j];
  double best = INFINITY;
  int bi = -1, bo = -1;
  for (int f = 0; f < F; ++f) {
    if (c[(int64_t)f * N] || !(m[f] <= mf + kSsMemTol)) continue;
    const double v = -G[(int64_t)f * N];
    if (v < best) { best = v; bi = f; bo = -1; }
  }
  for (int fo = 0; fo < F; ++fo) {
    if (!c[(int64_t)fo * N]) continue;
    const double lo = L[(int64_t)fo * N];
    if (lo == INFINITY) continue;                                // fo's only pod: no candidate can be finite
    const double cap = mf + m[fo] + kSsMemTol;
    for (int f = 0; f < F; ++f) {
      if (c[(int64_t)f * N] || !(m[f] <= cap)) continue;
      const double v = __dsub_rn(lo, G[(int64_t)f * N]);
      if (v < best) { best = v; bi = f; bo = fo; }
    }
  }
  const int64_t o = (int64_t)b * (N + F) + j;
  s.prop_d[o] = best; s.prop_x[o] = bi; s.prop_y[o] = bo;
}

// (value, index) pairs: larger value first, lower index among equals; index < 0 = nothing
__device__ __forceinline__ bool ss_better_max(double v, int j, double bv, int bj) {
  if (j < 0) return false;
  return bj < 0 || v > bv || (v == bv && j < bj);
}

// one block per function: relocation j_out -> j_in
__global__ void __launch_bounds__(kSsFuncThreads) k_ss_func(SsState s) {
  const int b = blockIdx.y, f = blockIdx.x, N = s.N, F = s.F;
  const int64_t bf = (int64_t)b * F + f;
  const uint8_t* __restrict__ c = s.c + bf * N;
  const double* __restrict__ G = s.G + bf * N;
  const double* __restrict__ memfree = s.memfree + (int64_t)b * N;
  const double mff = s.m[bf];
  __shared__ int s_cand[kSsCand], s_nc;
  __shared__ double s_v[kSsFuncThreads];
  __shared__ int s_j[kSsFuncThreads];
  __shared__ double s_w[kSsChunk], s_d1[kSsChunk], s_d2[kSsChunk];
  __shared__ int s_a1[kSsChunk];
  const int tid = threadIdx.x;
  if (tid == 0) s_nc = 0;
  __syncthreads();
  // targets: the kSsCand nodes with the largest gain that have memory for f (lowest node among equal gains)
  for (int k = 0; k < kSsCand; ++k) {
    double bv = 0.0; int bj = -1;
    for (int j = tid; j < N; j += blockDim.x) {
      if (c[j] || !(mff <= memfree[j] + kSsMemTol)) continue;
      bool taken = false;
      for (int q = 0; q < k; ++q) taken |= s_cand[q] == j;
      if (!taken && ss_better_max(G[j], j, bv, bj)) { bv = G[j]; bj = j; }
    }
    s_v[tid] = bv; s_j[tid] = bj;
    __syncthreads();
    for (int o = blockDim.x / 2; o > 0; o >>= 1) {
      if (tid < o && ss_better_max(s_v[tid + o], s_j[tid + o], s_v[tid], s_j[tid])) { s_v[tid] = s_v[tid + o]; s_j[tid] = s_j[tid + o]; }
      __syncthreads();
    }
    const int pick = s_j[0];
    __syncthreads();
    if (pick < 0) break;                                         // block-uniform
    if (tid == 0) { s_cand[k] = pick; s_nc = k + 1; }
    __syncthreads();
  }
  if (tid == 0) {                                                // enumeration order: ascending node
    for (int a = 1; a < s_nc; ++a)
      for (int q = a; q > 0 && s_cand[q - 1] > s_cand[q]; --q) { const int t = s_cand[q]; s_cand[q] = s_cand[q - 1]; s_cand[q - 1] = t; }
  }
  __syncthreads();
  const int nc = s_nc, np = s.npods[bf], P = nc * np;
  const int* __restrict__ pods = s.plist + bf * N;
  const double* __restrict__ d = s.d + (int64_t)b * N * N;
  const double* __restrict__ w = s.w + bf * N;
  const double* __restrict__ d1 = s.d1 + bf * N;
  const double* __restrict__ d2 = s.d2 + bf * N;
  const int* __restrict__ a1 = s.a1 + bf * N;
  double best = INFINITY;
  int bp = -1;
  // pair p = q * nc + k: j_out = pods[q] (ascending), j_in = s_cand[k] (ascending)
  for (int p0 = 0; p0 < P; p0 += blockDim.x) {
    const int p = p0 + tid;
    const bool act = p < P;
    const int jo = act ? pods[p / nc] : -1, ji = act ? s_cand[p % nc] : 0;
    double acc = 0.0;
    for (int i0 = 0; i0 < N; i0 += kSsChunk) {
      const int n = min(kSsChunk, N - i0);
      __syncthreads();
      for (int t = tid; t < n; t += blockDim.x) {
        s_w[t] = w[i0 + t]; s_d1[t] = d1[i0 + t]; s_d2[t] = d2[i0 + t]; s_a1[t] = a1[i0 + t];
      }
      __syncthreads();
      if (act) {
        const double* __restrict__ dji = d + (int64_t)i0 * N + ji;
#pragma unroll 4
        for (int t = 0; t < n; ++t) {
          const double wv = s_w[t];
          if (wv == 0.0) continue;                               // adds a signed zero: skipping it changes no bit
          const double dwo = s_a1[t] == jo ? s_d2[t] : s_d1[t];
          acc = __dadd_rn(acc, __dmul_rn(wv, __dsub_rn(fmin(dwo, dji[(int64_t)t * N]), s_d1[t])));
        }
      }
    }
    if (act && acc < best) { best = acc; bp = p; }
  }
  // smallest delta, lowest pair among equals
  s_v[tid] = best; s_j[tid] = bp;
  __syncthreads();
  for (int o = blockDim.x / 2; o > 0; o >>= 1) {
    if (tid < o) {
      const double v2 = s_v[tid + o]; const int p2 = s_j[tid + o];
      if (p2 >= 0 && (s_j[tid] < 0 || v2 < s_v[tid] || (v2 == s_v[tid] && p2 < s_j[tid]))) { s_v[tid] = v2; s_j[tid] = p2; }
    }
    __syncthreads();
  }
  if (tid == 0) {
    const int64_t o = (int64_t)b * (N + F) + N + f;
    const int p = s_j[0];
    s.prop_d[o] = p >= 0 ? s_v[0] : INFINITY;
    s.prop_x[o] = p >= 0 ? pods[p / nc] : -1;
    s.prop_y[o] = p >= 0 ? s_cand[p % nc] : -1;
  }
}

// one block per instance
__global__ void __launch_bounds__(kSsResolveThreads) k_ss_resolve(SsState s) {
  const int b = blockIdx.x, N = s.N, F = s.F, P = N + F, tid = threadIdx.x;
  extern __shared__ uint8_t s_touch[];                           // [0, F) functions, [F, F + N) nodes
  __shared__ int s_wcnt[32], s_base;
  __shared__ double s_thr;
  const double* __restrict__ pd = s.prop_d + (int64_t)b * P;
  const int* __restrict__ px = s.prop_x + (int64_t)b * P;
  const int* __restrict__ py = s.prop_y + (int64_t)b * P;
  double* cd = s.cd + (int64_t)b * P;
  int* ci = s.ci + (int64_t)b * P;
  int* sorted = s.sorted + (int64_t)b * P;
  if (tid == 0) s_thr = __dmul_rn(-1e-12, __dadd_rn(1.0, ss_objective(s, b)));
  for (int k = tid; k < F + N; k += blockDim.x) s_touch[k] = 0;
  for (int f = tid; f < F; f += blockDim.x) s.dirty[(int64_t)b * F + f] = 0;
  ss_ordered_compact_begin(&s_base);                             // (syncs: s_thr visible)
  const double thr = s_thr;
  for (int p0 = 0; p0 < P; p0 += blockDim.x) {
    const int p = p0 + tid;
    ss_ordered_append(p < P && pd[p] < thr, s_wcnt, &s_base, ci, p);
  }
  const int V = s_base;
  for (int k = tid; k < V; k += blockDim.x) cd[k] = pd[ci[k]];
  __syncthreads();
  for (int k = tid; k < V; k += blockDim.x) {                    // rank by (delta, index)
    const double v = cd[k];
    const int idx = ci[k];
    int r = 0;
    for (int q = 0; q < V; ++q) { const double u = cd[q]; r += (u < v || (u == v && ci[q] < idx)) ? 1 : 0; }
    sorted[r] = idx;
  }
  __syncthreads();
  if (tid >= 32) return;
  const int lane = tid;
  int n_add = 0, n_exc = 0, n_rel = 0;
  uint8_t* c = s.c + (int64_t)b * F * N;
  uint8_t* dirty = s.dirty + (int64_t)b * F;
  uint8_t* tf = s_touch;
  uint8_t* tn = s_touch + F;
  for (int k0 = 0; k0 < V; k0 += 32) {
    const int k = k0 + lane;
    const int p = k < V ? sorted[k] : 0;
    const int x = k < V ? px[p] : 0, y = k < V ? py[p] : 0;
    const int cnt = min(32, V - k0);
    for (int t = 0; t < cnt; ++t) {                              // warp-uniform walk in sorted order
      const int pt = __shfl_sync(0xffffffffu, p, t), xt = __shfl_sync(0xffffffffu, x, t), yt = __shfl_sync(0xffffffffu, y, t);
      if (pt < N) {                                              // node pt: f_in = xt, f_out = yt (-1: add)
        if (tn[pt] || tf[xt] || (yt >= 0 && tf[yt])) continue;
        __syncwarp();
        if (lane == 0) {
          c[(int64_t)xt * N + pt] = 1; dirty[xt] = 1; tn[pt] = 1; tf[xt] = 1;
          if (yt >= 0) { c[(int64_t)yt * N + pt] = 0; dirty[yt] = 1; tf[yt] = 1; }
        }
        if (yt >= 0) ++n_exc; else ++n_add;
      } else {                                                   // function pt - N: j_out = xt, j_in = yt
        const int f = pt - N;
        if (tf[f] || tn[xt] || tn[yt]) continue;
        __syncwarp();
        if (lane == 0) {
          c[(int64_t)f * N + xt] = 0; c[(int64_t)f * N + yt] = 1; dirty[f] = 1; tf[f] = 1; tn[xt] = 1; tn[yt] = 1;
        }
        ++n_rel;
      }
      __syncwarp();
    }
  }
  if (lane == 0) {
    const int acc = n_add + n_exc + n_rel;
    if (acc) {
      int32_t* info = s.info + (int64_t)b * 4;
      info[0] += 1; info[1] += n_add; info[2] += n_exc; info[3] += n_rel;
      atomicAdd(s.flags, acc);
    }
  }
}

static inline int64_t ss_align(int64_t v) { return (v + 255) & ~(int64_t)255; }

}  // namespace neptune

using namespace neptune;

extern "C" int neptune_site_search_workspace_bytes(int B, int N, int F, int64_t* bytes) {
  if (B <= 0 || N <= 0 || F <= 0 || !bytes) return NEPTUNE_E_ARG;
  const int64_t fn = (int64_t)B * F * N, bp = (int64_t)B * (N + F);
  *bytes = 3 * ss_align(fn * 4) + 4 * ss_align(fn * 8) + ss_align((int64_t)B * N * 8) + ss_align((int64_t)B * F * 8) +
           ss_align((int64_t)B * F * 4) + ss_align((int64_t)B * F) + 2 * ss_align(bp * 8) + 4 * ss_align(bp * 4) + 256;
  return 0;
}

extern "C" int neptune_site_search(int B, int N, int F, const double* d, const double* w, const double* m,
                                   const double* Mj, const uint8_t* c_in, uint8_t* c_out, int max_rounds,
                                   int32_t* info_out, double* obj_out, void* workspace, int64_t workspace_bytes,
                                   void* stream) {
  if (B <= 0 || N <= 0 || F <= 0 || !d || !w || !m || !Mj || !c_in || !c_out || !info_out || !obj_out || !workspace ||
      max_rounds < 0)
    return NEPTUNE_E_ARG;
  int64_t need = 0;
  neptune_site_search_workspace_bytes(B, N, F, &need);
  if (workspace_bytes < need) return NEPTUNE_E_NOMEM;
  if (F > 65535 || B > 65535) return NEPTUNE_E_SIZE;
  const size_t touch = (size_t)N + F;
  if (touch > 200 * 1024) return NEPTUNE_E_SIZE;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t fn = (int64_t)B * F * N, bp = (int64_t)B * (N + F);
  char* p = (char*)workspace;
  SsState s{};
  s.N = N; s.F = F; s.d = d; s.w = w; s.m = m; s.Mj = Mj; s.c = c_out; s.info = info_out;
  s.a1 = (int*)p; p += ss_align(fn * 4);
  s.a2 = (int*)p; p += ss_align(fn * 4);
  s.plist = (int*)p; p += ss_align(fn * 4);
  s.d1 = (double*)p; p += ss_align(fn * 8);
  s.d2 = (double*)p; p += ss_align(fn * 8);
  s.G = (double*)p; p += ss_align(fn * 8);
  s.L = (double*)p; p += ss_align(fn * 8);
  s.memfree = (double*)p; p += ss_align((int64_t)B * N * 8);
  s.objf = (double*)p; p += ss_align((int64_t)B * F * 8);
  s.npods = (int*)p; p += ss_align((int64_t)B * F * 4);
  s.dirty = (uint8_t*)p; p += ss_align((int64_t)B * F);
  s.prop_d = (double*)p; p += ss_align(bp * 8);
  s.cd = (double*)p; p += ss_align(bp * 8);
  s.prop_x = (int*)p; p += ss_align(bp * 4);
  s.prop_y = (int*)p; p += ss_align(bp * 4);
  s.ci = (int*)p; p += ss_align(bp * 4);
  s.sorted = (int*)p; p += ss_align(bp * 4);
  s.flags = (int*)p;
  if (touch > 48 * 1024)
    NEPTUNE_CUDA_OK(cudaFuncSetAttribute(k_ss_resolve, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)touch));
  if (c_out != c_in) NEPTUNE_CUDA_OK(cudaMemcpyAsync(c_out, c_in, (size_t)fn, cudaMemcpyDeviceToDevice, st));
  NEPTUNE_CUDA_OK(cudaMemsetAsync(info_out, 0, (size_t)B * 4 * sizeof(int32_t), st));
  NEPTUNE_CUDA_OK(cudaMemsetAsync(s.flags, 0, 2 * sizeof(int), st));
  NEPTUNE_CUDA_OK(cudaMemsetAsync(s.dirty, 1, (size_t)B * F, st));
  const dim3 gfn((N + kSsThreads - 1) / kSsThreads, F, B), gn((N + kSsThreads - 1) / kSsThreads, B);
  auto refresh = [&]() {                                         // state of the dirty functions
    { k_ss_pods<<<dim3(F, B), kSsThreads, 0, st>>>(s); NEPTUNE_COUNT(1); }
    { k_ss_nearest<<<gfn, kSsThreads, 0, st>>>(s); NEPTUNE_COUNT(1); }
    { k_ss_objf<<<dim3((F + 127) / 128, B), 128, 0, st>>>(s); NEPTUNE_COUNT(1); }
  };
  { k_ss_memfree<<<gn, kSsThreads, 0, st>>>(s); NEPTUNE_COUNT(1); }
  refresh();
  int h[2] = {0, 0};
  NEPTUNE_CUDA_OK(cudaMemcpyAsync(h, s.flags, 2 * sizeof(int), cudaMemcpyDeviceToHost, st));
  NEPTUNE_CUDA_OK(cudaStreamSynchronize(st));
  if (h[1]) return NEPTUNE_E_ARG;                                // a function without a pod: no objective to search
  { k_ss_obj<<<B, 32, 0, st>>>(s, obj_out, 0); NEPTUNE_COUNT(1); }
  // the host looks at the number of accepted moves every `look` rounds (one 4-byte copy): the search ends when a round
  // accepts nothing (the extra rounds of an instance that has stopped change nothing)
  const int look = 4;
  int h_prev = 0;
  for (int rnd = 0; rnd < max_rounds; ++rnd) {
    { k_ss_tables<<<gfn, kSsThreads, 0, st>>>(s); NEPTUNE_COUNT(1); }
    { k_ss_node<<<dim3((N + 127) / 128, B), 128, 0, st>>>(s); NEPTUNE_COUNT(1); }
    { k_ss_func<<<dim3(F, B), kSsFuncThreads, 0, st>>>(s); NEPTUNE_COUNT(1); }
    { k_ss_resolve<<<B, kSsResolveThreads, touch, st>>>(s); NEPTUNE_COUNT(1); }
    { k_ss_memfree<<<gn, kSsThreads, 0, st>>>(s); NEPTUNE_COUNT(1); }
    refresh();
    if ((rnd + 1) % look == 0 || rnd + 1 == max_rounds) {
      int moves = 0;
      NEPTUNE_CUDA_OK(cudaMemcpyAsync(&moves, s.flags, 4, cudaMemcpyDeviceToHost, st));
      NEPTUNE_CUDA_OK(cudaStreamSynchronize(st));
      if (moves == h_prev) break;                                // nothing accepted in the last `look` rounds
      h_prev = moves;
    }
  }
  { k_ss_obj<<<B, 32, 0, st>>>(s, obj_out, 1); NEPTUNE_COUNT(1); }
  NEPTUNE_LAUNCH_OK();
  return 0;
}
