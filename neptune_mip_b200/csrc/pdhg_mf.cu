// pdhg_mf.cu -- (b) MATRIX-FREE restarted, averaged, diagonally preconditioned PDHG for the LP relaxation
// of the strengthened min-delay placement model (same LP as assemble.cu builds with
// NEPTUNE_FLAG_STRENGTHEN, same algorithm and control logic as pdhg.cu with ruiz_iters = 0).
//
// Replaces the LP work inside pywraplp.Solver.Solve() (reference core/solvers/solver.py:37) for the model
// of neptune/utils/constraints_step1.py:5-65 + objectives.py:4-11.  Every coefficient of that model is a
// closed formula of (w, r, m, d), so nothing of the CSR matrix is read: one PDHG iteration is ONE streaming
// pass over the x-shaped arrays plus O(F*N) work on the small vectors.
//
//   columns  x[f,i,j] in [0,1]  (canonical f*N*N + i*N + j),  c[f,j] in [0,1]
//   rows     C1b (f,j): sum_i x - c >= -eps      y1      C3 (f,i): sum_j x = 1              y3
//            C2  (j)  : sum_f m c <= Mj          y2      C4 (j)  : sum_{f,i} w r x <= Kj     y4
//            S (f,i,j): x - c <= 0               yS      (C1a is a free row in the strengthened model: y = 0)
//   g_x = d*w + y1[f,j] + y3[f,i] + w[f,i] r[f,j] y4[j] + yS[f,i,j]       g_c = -y1 + m[f] y2[j] - sum_i yS
//   Pock-Chambolle (alpha = 1) step sizes generated on the fly:  T_x = 1/(3 + w r),  T_c = 1/(1 + m[f] + N),
//   S_1b = 1/(N+1), S_2 = 1/sum m, S_3 = 1/N, S_4[j] = 1/sum_{f,i} w r, S_S = 1/2.
//
// k_mf_iter (the dominant kernel): per element  x+ = clip(x - tau T_x g_x, 0, 1), xbar = 2x+ - x,
//   yS+ = max(yS + sigma/2 (xbar - cbar[f,j]), 0), running sums; per tile the partial column sums of xbar,
//   w*xbar and yS+ and the row sums of xbar go to small buffers (no atomics, fixed summation order).
// k_mf_small: the F*N-sized updates -- duals y1/y3/y4 from the partial sums (POST), then the c columns of the
//   next iteration (PREC) and the C2 dual (Y2).
// Algorithmic bytes per iteration and instance: X*(8 x + 8 yS + 8 xsum + 8 ysum read, the same written)
//   = 64*X, + 112*F*N (small vectors) + 8*N*N (d, re-read per function from L1/L2)  [X = F*N*N]; the CSR solver
//   moves 16*nnz + 88*cols + 72*rows ~ 260*X for the same iteration.
//
// Three iteration passes, all parity-tested against the numpy statement: tests/test_pdhg_mf_gpu.py up to 70 x 3 and
// 50 x 10; tests/test_pdhg_mf_wide_gpu.py at the branches only wide shapes take, each case pinned to its branch by
// neptune_pdhg_mf_geometry -- k_mf_iter<4, U> / k_mf_eval<4> (65 x 8, 99 x 5, 129 x 40), the C4 dual in 16 slices
// (K4 = F * rt from 65 to 800, the C3 bench instance included), k_mf_small on many blocks with the C2 dual in its own
// launch (F * N > 4096: 130 x 33, 129 x 40, C3, the node-column models), the bulk-copy pass with 64 and 80 functions,
// 17 column tiles (1026 x 2) -- and the restarted solve, decision by decision, against mf_reference.solve_ctl:
//   k_mf_iter_bulk<RED, FUSE> (pdhg_mf_bulk.cuh; even N <= 64, the default for even N in 34..64, i.e. C2): the streams
//     staged through shared memory by the bulk-copy engine (cp.async.bulk + mbarrier), running sums by
//     cp.reduce.async.bulk add.f64, the small-vector update inside the same launch -- 0.75-0.79 of the measured HBM peak
//     where the register passes reach 0.52-0.56 (profiles/r02c_pdhg_bulk.md);
//   k_mf_iter2<KP, U> (even N in 33..64: a lane owns pairs of adjacent columns, 16-byte accesses, cheap reciprocal) and
//   k_mf_iter<K, U> (every other shape: lanes own K strided columns, 8-byte accesses); U rows of a warp are in flight.
// Round 2 measured five further register / staging variants on B200 (bulk-copy staging of 8 KB tiles, strided 16-byte,
// cp.async ring, fused small vectors, pointer bumping: profiles/r02_pdhg_variants.md) -- none beat the two register passes
// and they were removed; what did was taking EVERY consumer input out of global memory and the small-vector kernel out of
// the iteration (pdhg_mf_bulk.cuh).  NEPTUNE_MF_PASS = pair | bulk | bulkred overrides the default pass (measurements).
#include "common.cuh"
#include "pdhg_ctl.cuh"
#include <stdlib.h>
#include <string.h>

namespace neptune {

constexpr int kGeoSeg = 1024;          // column segment used when balancing the row-tile height

struct MfGeo {
  int N, F, K, JT, ct, RT, rt, tiles_inst;
  int cti;                       // column segments of the iteration kernel in use (layout of P3i)
  int with_n;                    // node columns n[j] and rows C5a / C5b / C6 present (min-utilisation, combined objective)
  int64_t X, C, cols, rows, r2, r3, r4, r5, r6, rs;
};

static MfGeo make_geo(int N, int F, int B, int kind = NEPTUNE_KIND_MIN_DELAY) {
  MfGeo G;
  G.N = N; G.F = F;
  G.K = N <= 32 ? 1 : ((N & 1) == 0 || N <= 64 ? 2 : 4);        // columns per lane (even N: one pair of adjacent columns, 16-byte accesses)
  G.JT = 32 * G.K; G.ct = (N + G.JT - 1) / G.JT;
  // row-tile height: the tallest of 64/32/16/8 whose tiles fill the resident blocks evenly (>= 88 % busy in the
  // last round); the partial column sums cost 24 bytes per column and row tile, so taller is cheaper
  G.RT = N <= 64 ? N : 64;
  if (N > 64) {
    const int64_t slots = 2 * kNumSMs;
    int best = 64; double best_eff = 0.0;
    for (int rt_h = 64; rt_h >= 8; rt_h >>= 1) {
      const int64_t units = (int64_t)B * F * ((N + rt_h - 1) / rt_h) * ((N + kGeoSeg - 1) / kGeoSeg);
      const double eff = (double)units / (double)(((units + slots - 1) / slots) * slots);
      if (eff > best_eff + 1e-9) { best_eff = eff; best = rt_h; }
      if (eff >= 0.88) { best = rt_h; break; }
    }
    G.RT = best;
  }
  G.rt = (N + G.RT - 1) / G.RT;
  G.tiles_inst = F * G.rt * G.ct;
  G.cti = G.ct;
  Layout L(N, F, kind, NEPTUNE_FLAG_STRENGTHEN);
  G.with_n = L.with_n;
  G.X = L.X; G.C = L.C; G.cols = L.cols; G.rows = L.rows;
  G.r2 = L.r2; G.r3 = L.r3; G.r4 = L.r4; G.r5 = L.r5; G.r6 = L.r6; G.rs = L.rs;
  return G;
}

// d is the delay matrix AS IT ENTERS THE OBJECTIVE: the caller scales it for the combined objective ((1 - alpha) / the
// largest workload-weighted delay, objectives.py:36-52) and passes zeros for min-utilisation; nothing else reads it.
// cost / budget / objn (objective coefficient of every n[j]) are read only when the model has node columns.
struct MfIn { const double *d, *w, *r, *m, *Mj, *Kj; const double* cost; double budget, objn; const double* bigm; };

constexpr double kMfBigM = 1e6;        // constraints_step1.py:1
// the big M of row C5a for node j: the reference's 10^6, or the caller's (valid) bound on the pods node j can hold
__device__ __forceinline__ double mf_bigm(const MfIn& in, int64_t bj) { return in.bigm ? in.bigm[bj] : kMfBigM; }

struct MfSt {
  double *x, *y, *xsum, *ysum;   // canonical vectors [B][cols] / [B][rows]
  double *cbar;                  // [B][C]        2c+ - c of the running iteration
  double *P1, *P4, *PS;          // [B][F][rt][N] partial column sums (xbar, r*w*xbar, yS+) per row tile
  double *P3;                    // [B][C][ct]    partial row sums per column tile (KKT evaluation pass)
  double *P3i;                   // [B][C][cti]   ... of xbar, written by the iteration pass
  double *S4;                    // [B][N]        1 / sum_{f,i} |w r|
  double *S2;                    // [B]           1 / sum_f |m|
  double *wsum;                  // [B][F]        sum_i |w[f,i]|
  double *scal;                  // [B][tiles_inst][4] per-tile scalars of the KKT evaluation / setup
};

constexpr int kMfThreads = 256;
constexpr int kMfWarps = kMfThreads / 32;

struct Tile { int b, f, it, jt; };
__device__ __forceinline__ Tile decode_tile(const MfGeo& G, int64_t tile) {
  Tile t;
  t.b = (int)(tile / G.tiles_inst);
  int k = (int)(tile - (int64_t)t.b * G.tiles_inst);
  t.jt = k % G.ct; k /= G.ct;
  t.it = k % G.rt; t.f = k / G.rt;
  return t;
}

// cross-warp sum of per-lane column accumulators; thread c < 32*K then owns column c of the tile
template <int K>
__device__ __forceinline__ double column_total(double (*sm)[32 * K], int c) {
  double s = 0.0;
#pragma unroll
  for (int w = 0; w < kMfWarps; ++w) s += sm[w][c];
  return s;
}

// ---------------------------------------------------------------------------------------------------
// the iteration pass
// ---------------------------------------------------------------------------------------------------
// U rows of a warp are in flight together (independent dependency chains; U*K elements per lane)
template <int K, int U>
__global__ void __launch_bounds__(kMfThreads, (K * U >= 4 ? 2 : 3))
k_mf_iter(MfGeo G, MfIn in, MfSt st, const Ctl* __restrict__ ctl, int B) {
  __shared__ double sm[3][kMfWarps][32 * K];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int N = G.N;
  const int64_t NN = (int64_t)N * N;
  const int64_t total = (int64_t)B * G.tiles_inst;
  for (int64_t tile = blockIdx.x; tile < total; tile += gridDim.x) {
    const Tile t = decode_tile(G, tile);
    const int b = t.b, f = t.f;
    if (ctl[b].converged) continue;
    const double tau = ctl[b].tau, shalf = 0.5 * ctl[b].sigma;
    const double* __restrict__ d = in.d + (int64_t)b * NN;
    const double* __restrict__ w = in.w + ((int64_t)b * G.F + f) * N;
    const double* __restrict__ r = in.r + ((int64_t)b * G.F + f) * N;
    const double* __restrict__ y = st.y + (int64_t)b * G.rows;
    const double* __restrict__ y3 = y + G.r3 + (int64_t)f * N;
    double* __restrict__ xp = st.x + (int64_t)b * G.cols + (int64_t)f * NN;
    double* __restrict__ xsp = st.xsum + (int64_t)b * G.cols + (int64_t)f * NN;
    double* __restrict__ sp = st.y + (int64_t)b * G.rows + G.rs + (int64_t)f * NN;
    double* __restrict__ ssp = st.ysum + (int64_t)b * G.rows + G.rs + (int64_t)f * NN;
    const double* __restrict__ cbar = st.cbar + (int64_t)b * G.C + (int64_t)f * N;
    double* __restrict__ P3 = st.P3i + ((int64_t)b * G.C + (int64_t)f * N) * G.cti + t.jt;

    int jj[K]; bool vj[K];
    double y1j[K], rj[K], rr4[K], cb[K];
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const int j = t.jt * G.JT + k * 32 + lane;
      vj[k] = j < N; jj[k] = vj[k] ? j : 0;
      y1j[k] = y[2 * ((int64_t)f * N + jj[k]) + 1];
      rj[k] = __ldg(r + jj[k]);
      rr4[k] = rj[k] * y[G.r4 + jj[k]];
      cb[k] = cbar[jj[k]];
    }
    double a1[K], a4[K], aS[K];
#pragma unroll
    for (int k = 0; k < K; ++k) { a1[k] = 0.0; a4[k] = 0.0; aS[k] = 0.0; }

    const int i0 = t.it * G.RT, i1 = min(N, i0 + G.RT);
    for (int ib = i0 + warp; ib < i1; ib += U * kMfWarps) {
      double xv[U][K], sv[U][K], xs[U][K], ss[U][K], dv[U][K], wfi[U], y3i[U];
      int ro[U]; bool ok[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int i = ib + u * kMfWarps;
        ok[u] = i < i1;
        const int ir = ok[u] ? i : ib;
        ro[u] = ir * N;
        wfi[u] = __ldg(w + ir); y3i[u] = y3[ir];
#pragma unroll
        for (int k = 0; k < K; ++k) {
          const int o = ro[u] + jj[k];
          xv[u][k] = xp[o]; sv[u][k] = sp[o]; xs[u][k] = xsp[o]; ss[u][k] = ssp[o];
          dv[u][k] = __ldg(d + o);
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        double rsum = 0.0;
#pragma unroll
        for (int k = 0; k < K; ++k) {
          if (ok[u] && vj[k]) {
            const int o = ro[u] + jj[k];
            const double wr = fabs(wfi[u] * rj[k]);
            const double g = __dmul_rn(dv[u][k], wfi[u]) + y1j[k] + y3i[u] + wfi[u] * rr4[k] + sv[u][k];
            double xn = xv[u][k] - tau * g / (3.0 + wr);
            xn = fmin(fmax(xn, 0.0), 1.0);
            const double xb = 2.0 * xn - xv[u][k];
            const double sn = fmax(sv[u][k] + shalf * (xb - cb[k]), 0.0);
            xp[o] = xn; sp[o] = sn;
            xsp[o] = xs[u][k] + xn; ssp[o] = ss[u][k] + sn;
            a1[k] += xb; a4[k] += wfi[u] * xb; aS[k] += sn; rsum += xb;
          }
        }
        rsum = warp_sum(rsum);
        if (lane == 0 && ok[u]) P3[(int64_t)(ib + u * kMfWarps) * G.cti] = rsum;
      }
    }
#pragma unroll
    for (int k = 0; k < K; ++k) {
      sm[0][warp][k * 32 + lane] = a1[k]; sm[1][warp][k * 32 + lane] = a4[k]; sm[2][warp][k * 32 + lane] = aS[k];
    }
    __syncthreads();
    for (int c = threadIdx.x; c < 32 * K; c += kMfThreads) {
      const int j = t.jt * G.JT + c;
      if (j < N) {
        const int64_t o = (((int64_t)b * G.F + f) * G.rt + t.it) * N + j;
        st.P1[o] = column_total<K>(sm[0], c);
        st.P4[o] = __ldg(r + j) * column_total<K>(sm[1], c);
        st.PS[o] = column_total<K>(sm[2], c);
      }
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------------
// the iteration pass, pair version (even N > 32): a lane owns KP pairs of ADJACENT columns, so every stream moves
// in 16-byte accesses; one unsigned element offset per row (the five streams share it, the bases are uniform);
// 1/(3 + w r) by a float reciprocal + two Newton steps in double (7 instructions instead of the ~30 of an IEEE
// division; relative error < 1e-15, deterministic); U rows of a warp in flight.  Same tiles, same partial-sum
// buffers and the same summation order per column as k_mf_iter<2*KP, U>, so the rest of the solver is shared.
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ double mf_rcp(double a) {
  float rf;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rf) : "f"(__double2float_rn(a)));
  double r = (double)rf;
  double e = fma(-a, r, 1.0); r = fma(r, e, r);
  e = fma(-a, r, 1.0); r = fma(r, e, r);
  return r;
}

template <int KP, int U>
__global__ void __launch_bounds__(kMfThreads, (KP * U >= 2 ? 2 : 3))
k_mf_iter2(MfGeo G, MfIn in, MfSt st, const Ctl* __restrict__ ctl, int B) {
  constexpr int K = 2 * KP;
  __shared__ double sm[3][kMfWarps][32 * K];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int N = G.N;
  const int64_t NN = (int64_t)N * N;
  const int64_t total = (int64_t)B * G.tiles_inst;
  for (int64_t tile = blockIdx.x; tile < total; tile += gridDim.x) {
    const Tile t = decode_tile(G, tile);
    const int b = t.b, f = t.f;
    if (ctl[b].converged) continue;
    const double tau = ctl[b].tau, shalf = 0.5 * ctl[b].sigma;
    const double* __restrict__ d = in.d + (int64_t)b * NN;
    const double* __restrict__ w = in.w + ((int64_t)b * G.F + f) * N;
    const double* __restrict__ r = in.r + ((int64_t)b * G.F + f) * N;
    const double* __restrict__ y = st.y + (int64_t)b * G.rows;
    const double* __restrict__ y3 = y + G.r3 + (int64_t)f * N;
    double* __restrict__ xp = st.x + (int64_t)b * G.cols + (int64_t)f * NN;
    double* __restrict__ xsp = st.xsum + (int64_t)b * G.cols + (int64_t)f * NN;
    double* __restrict__ sp = st.y + (int64_t)b * G.rows + G.rs + (int64_t)f * NN;
    double* __restrict__ ssp = st.ysum + (int64_t)b * G.rows + G.rs + (int64_t)f * NN;
    const double* __restrict__ cbar = st.cbar + (int64_t)b * G.C + (int64_t)f * N;
    double* __restrict__ P3 = st.P3i + ((int64_t)b * G.C + (int64_t)f * N) * G.cti + t.jt;

    // columns of this lane: pair k covers columns jc[k], jc[k] + 1 (both valid or both invalid: N is even)
    unsigned jc[KP]; bool vj[KP];
    double y1j[K], rj[K], rr4[K], cb[K];
#pragma unroll
    for (int k = 0; k < KP; ++k) {
      const int j = t.jt * G.JT + k * 64 + 2 * lane;
      vj[k] = j < N; jc[k] = vj[k] ? (unsigned)j : 0u;
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const unsigned je = jc[k] + e;
        y1j[2 * k + e] = y[2 * ((int64_t)f * N + je) + 1];
        rj[2 * k + e] = __ldg(r + je);
        rr4[2 * k + e] = rj[2 * k + e] * y[G.r4 + je];
        cb[2 * k + e] = cbar[je];
      }
    }
    double a1[K], a4[K], aS[K];
#pragma unroll
    for (int k = 0; k < K; ++k) { a1[k] = 0.0; a4[k] = 0.0; aS[k] = 0.0; }

    const int i0 = t.it * G.RT, i1 = min(N, i0 + G.RT);
    for (int ib = i0 + warp; ib < i1; ib += U * kMfWarps) {
      double2 xv[U][KP], sv[U][KP], xs[U][KP], ss[U][KP], dv[U][KP];
      double wfi[U], y3i[U];
      unsigned ro[U]; bool ok[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int i = ib + u * kMfWarps;
        ok[u] = i < i1;
        const unsigned ir = ok[u] ? (unsigned)i : (unsigned)ib;
        ro[u] = ir * (unsigned)N;
        wfi[u] = __ldg(w + ir); y3i[u] = y3[ir];
#pragma unroll
        for (int k = 0; k < KP; ++k) {
          const unsigned o = ro[u] + jc[k];
          xv[u][k] = __ldcs(reinterpret_cast<const double2*>(xp + o));
          sv[u][k] = __ldcs(reinterpret_cast<const double2*>(sp + o));
          xs[u][k] = __ldcs(reinterpret_cast<const double2*>(xsp + o));
          ss[u][k] = __ldcs(reinterpret_cast<const double2*>(ssp + o));
          dv[u][k] = __ldg(reinterpret_cast<const double2*>(d + o));
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        double rsum = 0.0;
        const double ty = y3i[u];
#pragma unroll
        for (int k = 0; k < KP; ++k) {
          if (ok[u] && vj[k]) {
            const unsigned o = ro[u] + jc[k];
            double xn[2], sn[2];
#pragma unroll
            for (int e = 0; e < 2; ++e) {
              const int q = 2 * k + e;
              const double xo = e ? xv[u][k].y : xv[u][k].x, so = e ? sv[u][k].y : sv[u][k].x;
              const double de = e ? dv[u][k].y : dv[u][k].x;
              const double wr = fabs(wfi[u] * rj[q]);
              const double g = __dmul_rn(de, wfi[u]) + y1j[q] + ty + wfi[u] * rr4[q] + so;
              double x1 = xo - tau * g * mf_rcp(3.0 + wr);
              x1 = fmin(fmax(x1, 0.0), 1.0);
              const double xb = 2.0 * x1 - xo;
              const double s1 = fmax(so + shalf * (xb - cb[q]), 0.0);
              xn[e] = x1; sn[e] = s1;
              a1[q] += xb; a4[q] += wfi[u] * xb; aS[q] += s1; rsum += xb;
            }
            __stcs(reinterpret_cast<double2*>(xp + o), make_double2(xn[0], xn[1]));
            __stcs(reinterpret_cast<double2*>(sp + o), make_double2(sn[0], sn[1]));
            __stcs(reinterpret_cast<double2*>(xsp + o), make_double2(xs[u][k].x + xn[0], xs[u][k].y + xn[1]));
            __stcs(reinterpret_cast<double2*>(ssp + o), make_double2(ss[u][k].x + sn[0], ss[u][k].y + sn[1]));
          }
        }
        rsum = warp_sum(rsum);
        if (lane == 0 && ok[u]) P3[(int64_t)(ib + u * kMfWarps) * G.cti] = rsum;
      }
    }
    // column c of the tile lives in lane (c % 64) / 2, slot 2 * (c / 64) + (c & 1)
#pragma unroll
    for (int k = 0; k < KP; ++k) {
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int c = k * 64 + 2 * lane + e;
        sm[0][warp][c] = a1[2 * k + e]; sm[1][warp][c] = a4[2 * k + e]; sm[2][warp][c] = aS[2 * k + e];
      }
    }
    __syncthreads();
    for (int c = threadIdx.x; c < 32 * K; c += kMfThreads) {
      const int j = t.jt * G.JT + c;
      if (j < N) {
        const int64_t o = (((int64_t)b * G.F + f) * G.rt + t.it) * N + j;
        st.P1[o] = column_total<K>(sm[0], c);
        st.P4[o] = __ldg(r + j) * column_total<K>(sm[1], c);
        st.PS[o] = column_total<K>(sm[2], c);
      }
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------------
// KKT pieces of a candidate (which = 0: current iterate, 1: running average): the same partial sums from a
// read-only pass, plus per tile {obj.x, sum min(rc_x, 0), sum max(x - c, 0)^2}.  mode 1: only the column
// sums of yS (refreshes PS after a restart / at the start).
// ---------------------------------------------------------------------------------------------------
template <int K>
__global__ void __launch_bounds__(kMfThreads, (K == 4 ? 2 : 3))
k_mf_eval(MfGeo G, MfIn in, MfSt st, const Ctl* __restrict__ ctl, int B, int which, int only_ps) {
  __shared__ double sm[3][kMfWarps][32 * K];
  __shared__ double red[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int N = G.N;
  const int64_t NN = (int64_t)N * N;
  const int64_t total = (int64_t)B * G.tiles_inst;
  for (int64_t tile = blockIdx.x; tile < total; tile += gridDim.x) {
    const Tile t = decode_tile(G, tile);
    const int b = t.b, f = t.f;
    if (ctl[b].converged) continue;
    const double sc = which ? 1.0 / (double)max(ctl[b].avg_count, 1) : 1.0;
    const double* __restrict__ d = in.d + (int64_t)b * NN;
    const double* __restrict__ w = in.w + ((int64_t)b * G.F + f) * N;
    const double* __restrict__ r = in.r + ((int64_t)b * G.F + f) * N;
    const double* __restrict__ xvec = (which ? st.xsum : st.x) + (int64_t)b * G.cols;
    const double* __restrict__ yvec = (which ? st.ysum : st.y) + (int64_t)b * G.rows;
    const double* __restrict__ xp = xvec + (int64_t)f * NN;
    const double* __restrict__ sp = yvec + G.rs + (int64_t)f * NN;

    int jj[K]; bool vj[K];
    double y1j[K], rj[K], rr4[K], cc[K];
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const int j = t.jt * G.JT + k * 32 + lane;
      vj[k] = j < N; jj[k] = vj[k] ? j : 0;
      y1j[k] = yvec[2 * ((int64_t)f * N + jj[k]) + 1] * sc;
      rj[k] = __ldg(r + jj[k]);
      rr4[k] = rj[k] * yvec[G.r4 + jj[k]] * sc;
      cc[k] = xvec[G.X + (int64_t)f * N + jj[k]] * sc;
    }
    double a1[K], a4[K], aS[K];
#pragma unroll
    for (int k = 0; k < K; ++k) { a1[k] = 0.0; a4[k] = 0.0; aS[k] = 0.0; }
    double pobj = 0.0, rcneg = 0.0, ps2 = 0.0;

    const int i0 = t.it * G.RT, i1 = min(N, i0 + G.RT);
    for (int i = i0 + warp; i < i1; i += kMfWarps) {
      const int64_t ro = (int64_t)i * N;
      if (only_ps) {
#pragma unroll
        for (int k = 0; k < K; ++k) if (vj[k]) aS[k] += sp[ro + jj[k]] * sc;
        continue;
      }
      const double wfi = __ldg(w + i), y3i = yvec[G.r3 + (int64_t)f * N + i] * sc;
      double rsum = 0.0;
#pragma unroll
      for (int k = 0; k < K; ++k) {
        if (vj[k]) {
          const double xv = xp[ro + jj[k]] * sc, sv = sp[ro + jj[k]] * sc;
          const double o = __dmul_rn(__ldg(d + ro + jj[k]), wfi);
          const double rc = o + y1j[k] + y3i + wfi * rr4[k] + sv;
          pobj += o * xv;
          rcneg += fmin(rc, 0.0);
          const double viol = fmax(xv - cc[k], 0.0);
          ps2 += viol * viol;
          a1[k] += xv; a4[k] += wfi * xv; aS[k] += sv; rsum += xv;
        }
      }
      rsum = warp_sum(rsum);
      if (lane == 0) st.P3[((int64_t)b * G.C + (int64_t)f * N + i) * G.ct + t.jt] = rsum;
    }
#pragma unroll
    for (int k = 0; k < K; ++k) {
      sm[0][warp][k * 32 + lane] = a1[k]; sm[1][warp][k * 32 + lane] = a4[k]; sm[2][warp][k * 32 + lane] = aS[k];
    }
    __syncthreads();
    for (int c = threadIdx.x; c < 32 * K; c += kMfThreads) {
      const int j = t.jt * G.JT + c;
      if (j < N) {
        const int64_t o = (((int64_t)b * G.F + f) * G.rt + t.it) * N + j;
        if (!only_ps) {
          st.P1[o] = column_total<K>(sm[0], c);
          st.P4[o] = __ldg(r + j) * column_total<K>(sm[1], c);
        }
        st.PS[o] = column_total<K>(sm[2], c);
      }
    }
    if (!only_ps) {
      const double s0 = block_sum(pobj, red), s1 = block_sum(rcneg, red), s2 = block_sum(ps2, red);
      if (threadIdx.x == 0) {
        double* q = st.scal + tile * 4;
        q[0] = s0; q[1] = s1; q[2] = s2; q[3] = 0.0;
      }
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------------
// the small vectors
// ---------------------------------------------------------------------------------------------------
enum { PH_POST = 1, PH_PREC = 2, PH_Y2 = 4 };

// sum of n values p[0], p[stride], p[2*stride], ... in index order, eight loads in flight at a time
__device__ __forceinline__ double strided_sum(const double* __restrict__ p, int n, int64_t stride) {
  double a = 0.0;
  for (int k0 = 0; k0 < n; k0 += 8) {
    double v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) v[u] = (k0 + u < n) ? p[(int64_t)(k0 + u) * stride] : 0.0;
#pragma unroll
    for (int u = 0; u < 8; ++u) a += v[u];
  }
  return a;
}

__global__ void __launch_bounds__(512)
k_mf_small(MfGeo G, MfIn in, MfSt st, const Ctl* __restrict__ ctl, int mask, const int* __restrict__ skip_post,
           int fused) {
  const int b = blockIdx.y;
  if (ctl[b].converged) return;
  if (skip_post && *skip_post) mask &= ~PH_POST;
  const int N = G.N, F = G.F, rt = G.rt, ct = G.cti;
  const int C = (int)G.C;
  const int tid = blockIdx.x * blockDim.x + threadIdx.x, nth = gridDim.x * blockDim.x;
  const double tau = ctl[b].tau, sigma = ctl[b].sigma;
  double* __restrict__ y = st.y + (int64_t)b * G.rows;
  double* __restrict__ ys = st.ysum + (int64_t)b * G.rows;
  double* __restrict__ c = st.x + (int64_t)b * G.cols + G.X;
  double* __restrict__ cs = st.xsum + (int64_t)b * G.cols + G.X;
  double* __restrict__ cbar = st.cbar + (int64_t)b * C;
  const double* __restrict__ P1 = st.P1 + (int64_t)b * F * rt * N;
  const double* __restrict__ P4 = st.P4 + (int64_t)b * F * rt * N;
  const double* __restrict__ PS = st.PS + (int64_t)b * F * rt * N;
  const double* __restrict__ P3 = st.P3i + (int64_t)b * C * ct;
  const double* __restrict__ m = in.m + (int64_t)b * F;
  const bool post = mask & PH_POST, prec = mask & PH_PREC;

  // C4 dual: every load of a thread is issued before the first use (the sums are latency-bound); long sums
  // (large instances: F * rt partials per column) are cut into 16 slices per column and combined in order
  if (post) {
    const double* __restrict__ Kj = in.Kj + (int64_t)b * N;
    const int K4 = F * rt;
    if (K4 <= 64) {
      for (int j = tid; j < N; j += nth) {
        const double a = strided_sum(P4 + j, K4, N);              // P4 already carries r[f,j]
        const double s = sigma * st.S4[(int64_t)b * N + j];
        const double v = y[G.r4 + j] + s * a;
        const double yn = v - s * fmin(v / s, Kj[j]);             // C4: (-inf, Kj]
        y[G.r4 + j] = yn; ys[G.r4 + j] += yn;
      }
    } else {
      __shared__ double slice[512];
      const int cpb = blockDim.x / 16;
      const int jl = threadIdx.x % cpb, sl = threadIdx.x / cpb;
      const int L = (K4 + 15) / 16;
      for (int jb = blockIdx.x; jb * cpb < N; jb += gridDim.x) {
        const int j = jb * cpb + jl;
        const int k0 = sl * L, n = min(L, K4 - k0);
        slice[sl * cpb + jl] = (j < N && n > 0) ? strided_sum(P4 + (int64_t)k0 * N + j, n, N) : 0.0;
        __syncthreads();
        if (sl == 0 && j < N) {
          double a = 0.0;
#pragma unroll
          for (int q = 0; q < 16; ++q) a += slice[q * cpb + jl];
          const double s = sigma * st.S4[(int64_t)b * N + j];
          const double v = y[G.r4 + j] + s * a;
          const double yn = v - s * fmin(v / s, Kj[j]);
          y[G.r4 + j] = yn; ys[G.r4 + j] += yn;
        }
        __syncthreads();
      }
    }
  }
  if (post || prec) {
    const double s1 = sigma / (double)(N + 1), s3 = sigma / (double)N;
    for (int q = tid; q < C; q += nth) {
      const int f = q / N, j = q - f * N;
      const int64_t po = (int64_t)f * rt * N + j;
      double y1 = y[2 * q + 1];
      if (post) {
        const double a1 = strided_sum(P1 + po, rt, N) - cbar[q];
        const double a3 = strided_sum(P3 + (int64_t)q * ct, ct, 1);
        const double y3 = y[G.r3 + q], ys1 = ys[2 * q + 1], ys3 = ys[G.r3 + q];
        const double v1 = y1 + s1 * a1;
        y1 = v1 - s1 * fmax(v1 / s1, -kEps);                      // C1b: [-eps, +inf)
        y[2 * q + 1] = y1; ys[2 * q + 1] = ys1 + y1;
        const double y3n = y3 + s3 * a3 - s3;                     // C3: [1, 1]
        y[G.r3 + q] = y3n; ys[G.r3 + q] = ys3 + y3n;
      }
      if (prec) {
        const double sS = strided_sum(PS + po, rt, N);
        const double mf = m[f];
        double gc = -y1 + mf * y[G.r2 + j] - sS;
        if (G.with_n) gc += y[G.r5 + 2 * j] + y[G.r5 + 2 * j + 1];      // C5a, C5b carry every c[., j]
        const double co = c[q];
        double cn = co - tau * gc / ((G.with_n ? 3.0 : 1.0) + mf + (double)N);
        cn = fmin(fmax(cn, 0.0), 1.0);
        cbar[q] = 2.0 * cn - co;
        c[q] = cn; cs[q] += cn;
      }
    }
  }
  if (mask & PH_Y2) {
    if (fused) __syncthreads();
    const double* __restrict__ Mj = in.Mj + (int64_t)b * N;
    const double s = sigma * st.S2[b];
    for (int j = tid; j < N; j += nth) {
      double a = 0.0;
      for (int f0 = 0; f0 < F; f0 += 8) {
        double v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) v[u] = (f0 + u < F) ? m[f0 + u] * cbar[(int64_t)(f0 + u) * N + j] : 0.0;
#pragma unroll
        for (int u = 0; u < 8; ++u) a += v[u];
      }
      const double vv = y[G.r2 + j] + s * a;
      const double yn = vv - s * fmin(vv / s, Mj[j]);             // C2: (-inf, Mj]
      y[G.r2 + j] = yn; ys[G.r2 + j] += yn;
      if (G.with_n) {
        // node column n[j] from the duals of the previous iteration, then the three rows that see only (c, n)
        double a5 = 0.0;
        for (int f0 = 0; f0 < F; f0 += 8) {
          double v[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) v[u] = (f0 + u < F) ? cbar[(int64_t)(f0 + u) * N + j] : 0.0;
#pragma unroll
          for (int u = 0; u < 8; ++u) a5 += v[u];
        }
        double* __restrict__ nv = st.x + (int64_t)b * G.cols + G.X + C;
        double* __restrict__ ns = st.xsum + (int64_t)b * G.cols + G.X + C;
        const double cj = in.cost[(int64_t)b * N + j], Mb = mf_bigm(in, (int64_t)b * N + j);
        const double y5a = y[G.r5 + 2 * j], y5b = y[G.r5 + 2 * j + 1], y6 = y[G.r6 + j];
        const double gn = in.objn - Mb * y5a - y5b + cj * y6;
        const double no = nv[j];
        double nn = no - tau * gn / (Mb + 1.0 + fabs(cj));
        nn = fmin(fmax(nn, 0.0), 1.0);
        const double nbar = 2.0 * nn - no;
        nv[j] = nn; ns[j] += nn;
        double sr = sigma / ((double)F + Mb);
        double v5 = y5a + sr * (a5 - Mb * nbar);
        v5 = v5 - sr * fmin(v5 / sr, 0.0);                          // C5a: (-inf, 0]
        y[G.r5 + 2 * j] = v5; ys[G.r5 + 2 * j] += v5;
        sr = sigma / ((double)F + 1.0);
        v5 = y5b + sr * (a5 - nbar);
        v5 = v5 - sr * fmax(v5 / sr, -kEps);                        // C5b: [-eps, +inf)
        y[G.r5 + 2 * j + 1] = v5; ys[G.r5 + 2 * j + 1] += v5;
        sr = cj != 0.0 ? sigma / fabs(cj) : sigma;
        v5 = y6 + sr * (cj * nbar);
        v5 = v5 - sr * fmin(v5 / sr, in.budget);                    // C6: (-inf, budget]
        y[G.r6 + j] = v5; ys[G.r6 + j] += v5;
      }
    }
  }
}

}  // namespace neptune
#include "pdhg_mf_bulk.cuh"      // k_mf_iter_bulk<RED, FUSE>: the iteration pass with the streams staged by the bulk-copy engine
namespace neptune {

// rows / c-columns part of the KKT evaluation from the partial sums of k_mf_eval; one block per instance,
// fixed summation order.  Writes ctl[b].acc[ACC_CUR / ACC_AVG + {PRES2, DRES2, POBJ, DOBJ}].
__global__ void __launch_bounds__(256)
k_mf_eval_small(MfGeo G, MfIn in, MfSt st, Ctl* __restrict__ ctl, int which) {
  const int b = blockIdx.x;
  if (ctl[b].converged) return;
  __shared__ double red[32];
  const int N = G.N, F = G.F, rt = G.rt, ct = G.ct;
  const int64_t C = G.C;
  const double sc = which ? 1.0 / (double)max(ctl[b].avg_count, 1) : 1.0;
  const double* __restrict__ xvec = (which ? st.xsum : st.x) + (int64_t)b * G.cols;
  const double* __restrict__ yv = (which ? st.ysum : st.y) + (int64_t)b * G.rows;
  const double* __restrict__ cv = xvec + G.X;
  const double* __restrict__ P1 = st.P1 + (int64_t)b * F * rt * N;
  const double* __restrict__ P4 = st.P4 + (int64_t)b * F * rt * N;
  const double* __restrict__ PS = st.PS + (int64_t)b * F * rt * N;
  const double* __restrict__ P3 = st.P3 + (int64_t)b * C * ct;
  const double* __restrict__ m = in.m + (int64_t)b * F;
  const double* __restrict__ Mj = in.Mj + (int64_t)b * N;
  const double* __restrict__ Kj = in.Kj + (int64_t)b * N;
  double pres2 = 0.0, dres2 = 0.0, pobj = 0.0, dobj = 0.0;
  for (int64_t q = threadIdx.x; q < C; q += blockDim.x) {
    const int f = (int)(q / N), j = (int)(q - (int64_t)f * N);
    const double y1 = yv[2 * q + 1] * sc, cq = cv[q] * sc;
    double a = strided_sum(P1 + (int64_t)f * rt * N + j, rt, N);
    const double sS = strided_sum(PS + (int64_t)f * rt * N + j, rt, N);
    double viol = fmin(a - cq + kEps, 0.0);
    pres2 += viol * viol;
    if (y1 > 0.0) dres2 += y1 * y1; else dobj += kEps * y1;
    a = strided_sum(P3 + q * ct, ct, 1);
    viol = a - 1.0;
    pres2 += viol * viol;
    dobj -= yv[G.r3 + q] * sc;
    double rcc = -y1 + m[f] * yv[G.r2 + j] * sc - sS;
    if (G.with_n) rcc += (yv[G.r5 + 2 * j] + yv[G.r5 + 2 * j + 1]) * sc;
    dobj += fmin(rcc, 0.0);                                       // c in [0, 1]
  }
  for (int64_t j = threadIdx.x; j < N; j += blockDim.x) {
    double a2 = 0.0;
    for (int f = 0; f < F; ++f) a2 += m[f] * cv[(int64_t)f * N + j] * sc;
    const double a4 = strided_sum(P4 + j, F * rt, N);
    double viol = fmax(a2 - Mj[j], 0.0);
    pres2 += viol * viol;
    viol = fmax(a4 - Kj[j], 0.0);
    pres2 += viol * viol;
    const double y2 = yv[G.r2 + j] * sc, y4 = yv[G.r4 + j] * sc;
    if (y2 > 0.0) dobj -= Mj[j] * y2; else dres2 += y2 * y2;
    if (y4 > 0.0) dobj -= Kj[j] * y4; else dres2 += y4 * y4;
    if (G.with_n) {
      double a5 = 0.0;
      for (int f = 0; f < F; ++f) a5 += cv[(int64_t)f * N + j] * sc;
      const double nj = xvec[G.X + C + j] * sc, cj = in.cost[(int64_t)b * N + j], Mb = mf_bigm(in, (int64_t)b * N + j);
      const double y5a = yv[G.r5 + 2 * j] * sc, y5b = yv[G.r5 + 2 * j + 1] * sc, y6 = yv[G.r6 + j] * sc;
      viol = fmax(a5 - Mb * nj, 0.0); pres2 += viol * viol;
      viol = fmin(a5 - nj + kEps, 0.0); pres2 += viol * viol;
      viol = fmax(cj * nj - in.budget, 0.0); pres2 += viol * viol;
      if (y5a < 0.0) dres2 += y5a * y5a;                           // hi = 0: nothing for the dual objective
      if (y5b > 0.0) dres2 += y5b * y5b; else dobj += kEps * y5b;
      if (y6 > 0.0) dobj -= in.budget * y6; else dres2 += y6 * y6;
      const double rcn = in.objn - Mb * y5a - y5b + cj * y6;
      dobj += fmin(rcn, 0.0);                                     // n in [0, 1]
      pobj += in.objn * nj;
    }
  }
  const double* __restrict__ sq = st.scal + (int64_t)b * G.tiles_inst * 4;
  for (int t = threadIdx.x; t < G.tiles_inst; t += blockDim.x) {
    pobj += sq[t * 4 + 0]; dobj += sq[t * 4 + 1]; pres2 += sq[t * 4 + 2];
  }
  const double s0 = block_sum(pres2, red), s1 = block_sum(dres2, red), s2 = block_sum(pobj, red),
               s3 = block_sum(dobj, red);
  if (threadIdx.x == 0) {
    double* acc = ctl[b].acc + (which ? ACC_AVG : ACC_CUR);
    acc[PRES2] = s0; acc[DRES2] = s1; acc[POBJ] = s2; acc[DOBJ] = s3;
  }
}

// ---------------------------------------------------------------------------------------------------
// setup: step-size vectors S4, S2, the norms behind omega0 and the tolerances (same definitions as k_norms
// of pdhg.cu), multipliers of the free C1a rows zeroed.
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_mf_wsum(int N, int64_t n_rows, const double* __restrict__ w,
                                                 double* __restrict__ wsum) {
  const int lane = threadIdx.x & 31;
  const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;     // warp per (instance, function)
  if (row >= n_rows) return;
  double s = 0.0;
  for (int i = lane; i < N; i += 32) s += fabs(w[row * N + i]);
  s = warp_sum(s);
  if (lane == 0) wsum[row] = s;
}

__global__ void __launch_bounds__(256) k_mf_setup(MfGeo G, MfIn in, MfSt st, int nblk) {
  const int b = blockIdx.y;
  __shared__ double red[32];
  const int N = G.N, F = G.F;
  const int64_t NN = (int64_t)N * N;
  const double* __restrict__ d = in.d + (int64_t)b * NN;
  const double* __restrict__ w = in.w + (int64_t)b * F * N;
  const double* __restrict__ r = in.r + (int64_t)b * F * N;
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, nth = (int64_t)gridDim.x * blockDim.x;
  for (int64_t j = tid; j < N; j += nth) {                       // sum_{f,i} |w[f,i] r[f,j]| = sum_f |r[f,j]| * sum_i |w[f,i]|
    double s = 0.0;
    for (int f = 0; f < F; ++f) s += fabs(r[(int64_t)f * N + j]) * st.wsum[(int64_t)b * F + f];
    st.S4[(int64_t)b * N + j] = s > 0.0 ? 1.0 / s : 1.0;
  }
  if (tid == 0) {
    double s = 0.0;
    for (int f = 0; f < F; ++f) s += fabs(in.m[(int64_t)b * F + f]);
    st.S2[b] = s > 0.0 ? 1.0 / s : 1.0;
  }
  double* __restrict__ y = st.y + (int64_t)b * G.rows;
  for (int64_t q = tid; q < G.C; q += nth) y[2 * q] = 0.0;
  double nc2 = 0.0, ncs2 = 0.0;
  for (int64_t q = tid; q < G.X; q += nth) {
    const int f = (int)(q / NN);
    const int64_t rem = q - (int64_t)f * NN;
    const int i = (int)(rem / N), j = (int)(rem - (int64_t)i * N);
    const double wfi = w[(int64_t)f * N + i];
    const double o = __dmul_rn(d[rem], wfi);
    nc2 += o * o;
    ncs2 += o * o / (3.0 + fabs(wfi * r[(int64_t)f * N + j]));
  }
  const double s0 = block_sum(nc2, red), s1 = block_sum(ncs2, red);
  if (threadIdx.x == 0) {
    double* q = st.scal + ((int64_t)b * G.tiles_inst + blockIdx.x) * 4;
    q[0] = s0; q[1] = s1;
  }
  (void)nblk;
}

__global__ void k_mf_setup_norms(MfGeo G, MfIn in, MfSt st, Ctl* __restrict__ ctl, int B, int nblk) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const int N = G.N;
  const double C = (double)G.C;
  double nc2 = 0.0, ncs2 = 0.0;
  for (int k = 0; k < nblk; ++k) {
    nc2 += st.scal[((int64_t)b * G.tiles_inst + k) * 4 + 0];
    ncs2 += st.scal[((int64_t)b * G.tiles_inst + k) * 4 + 1];
  }
  double m2 = 0.0, k2 = 0.0, k2s = 0.0;
  for (int j = 0; j < N; ++j) {
    const double mj = in.Mj[(int64_t)b * N + j], kj = in.Kj[(int64_t)b * N + j];
    if (isfinite(mj)) m2 += mj * mj;
    if (isfinite(kj)) { k2 += kj * kj; k2s += kj * kj * st.S4[(int64_t)b * N + j]; }
  }
  double nb2n = 0.0, nbs2n = 0.0, nc2n = 0.0, ncs2n = 0.0;
  if (G.with_n) {
    const double bud2 = isfinite(in.budget) ? in.budget * in.budget : 0.0;
    nb2n = kEps * kEps * N + bud2 * N;
    nbs2n = kEps * kEps * N / ((double)G.F + 1.0);
    nc2n = in.objn * in.objn * N;
    for (int j = 0; j < N; ++j) {
      const double cj = fabs(in.cost[(int64_t)b * N + j]);
      nbs2n += bud2 * (cj != 0.0 ? 1.0 / cj : 1.0);
      ncs2n += in.objn * in.objn / (mf_bigm(in, (int64_t)b * N + j) + 1.0 + cj);
    }
  }
  double* acc = ctl[b].acc;
  acc[ACC_NB2] = kEps * kEps * C + m2 + C + k2 + nb2n;
  acc[ACC_NC2] = nc2 + nc2n;
  acc[ACC_NBS2] = kEps * kEps * C / (double)(N + 1) + m2 * st.S2[b] + C / (double)N + k2s + nbs2n;
  acc[ACC_NCS2] = ncs2 + ncs2n;
}

// ---------------------------------------------------------------------------------------------------
// restart: x, y <- running average (action 1) or keep (2); sums reset; movement since the last restart
// point in the preconditioned norms (per-block partials, summed in order by k_mf_restart_norms).
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_mf_apply_restart(MfGeo G, MfIn in, MfSt st, double* __restrict__ xres, double* __restrict__ yres,
                   const Ctl* __restrict__ ctl, double* __restrict__ part) {
  const int b = blockIdx.y;
  double* out = part + ((int64_t)b * gridDim.x + blockIdx.x) * 2;
  const int action = ctl[b].action;
  if (action == 0) { if (threadIdx.x == 0) { out[0] = 0.0; out[1] = 0.0; } return; }
  __shared__ double red[32];
  const int N = G.N, F = G.F;
  const int64_t NN = (int64_t)N * N;
  const double inv = 1.0 / (double)max(ctl[b].avg_count, 1);
  const double* __restrict__ w = in.w + (int64_t)b * F * N;
  const double* __restrict__ r = in.r + (int64_t)b * F * N;
  const double* __restrict__ m = in.m + (int64_t)b * F;
  double dx2 = 0.0, dy2 = 0.0;
  const int64_t n = G.cols + G.rows;
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) {
    if (k < G.cols) {
      double diag;
      if (k < G.X) {
        const int f = (int)(k / NN);
        const int64_t rem = k - (int64_t)f * NN;
        const int i = (int)(rem / N), j = (int)(rem - (int64_t)i * N);
        diag = 1.0 / (3.0 + fabs(w[(int64_t)f * N + i] * r[(int64_t)f * N + j]));
      } else if (k < G.X + G.C) {
        const int f = (int)((k - G.X) / N);
        diag = 1.0 / ((G.with_n ? 3.0 : 1.0) + fabs(m[f]) + (double)N);
      } else {
        diag = 1.0 / (mf_bigm(in, (int64_t)b * N + (k - G.X - G.C)) + 1.0 + fabs(in.cost[(int64_t)b * N + (k - G.X - G.C)]));
      }
      const int64_t q = (int64_t)b * G.cols + k;
      const double nv = (action == 1) ? st.xsum[q] * inv : st.x[q];
      const double dl = nv - xres[q];
      dx2 += dl * dl / diag;
      st.x[q] = nv; xres[q] = nv; st.xsum[q] = 0.0;
    } else {
      const int64_t row = k - G.cols;
      double diag;
      if (row < G.r2) diag = (row & 1) ? 1.0 / (double)(N + 1) : 1.0;
      else if (row < G.r3) diag = st.S2[b];
      else if (row < G.r4) diag = 1.0 / (double)N;
      else if (row < G.r5) diag = st.S4[(int64_t)b * N + (row - G.r4)];
      else if (row < G.r6) diag = ((row - G.r5) & 1) ? 1.0 / ((double)F + 1.0) : 1.0 / ((double)F + mf_bigm(in, (int64_t)b * N + ((row - G.r5) >> 1)));
      else if (row < G.rs) { const double cj = fabs(in.cost[(int64_t)b * N + (row - G.r6)]); diag = cj != 0.0 ? 1.0 / cj : 1.0; }
      else diag = 0.5;
      const int64_t q = (int64_t)b * G.rows + row;
      const double nv = (action == 1) ? st.ysum[q] * inv : st.y[q];
      const double dl = nv - yres[q];
      dy2 += dl * dl / diag;
      st.y[q] = nv; yres[q] = nv; st.ysum[q] = 0.0;
    }
  }
  const double s0 = block_sum(dx2, red), s1 = block_sum(dy2, red);
  if (threadIdx.x == 0) { out[0] = s0; out[1] = s1; }
}

__global__ void k_mf_restart_norms(int B, int nblk, const double* __restrict__ part, Ctl* __restrict__ ctl) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  double dx2 = 0.0, dy2 = 0.0;
  for (int k = 0; k < nblk; ++k) { dx2 += part[((int64_t)b * nblk + k) * 2]; dy2 += part[((int64_t)b * nblk + k) * 2 + 1]; }
  ctl[b].acc[ACC_DX2] = dx2; ctl[b].acc[ACC_DY2] = dy2;
}

// the instances still iterating, in increasing order: out[0] = count, out[1..] = indices (one warp, ordered compaction)
__global__ void k_mf_live(int B, const Ctl* __restrict__ ctl, int* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  int count = 0;
  for (int base = 0; base < B; base += 32) {
    const int b = base + lane;
    const bool on = b < B && !ctl[b].converged;
    const unsigned mask = __ballot_sync(0xffffffffu, on);
    if (on) out[1 + count + __popc(mask & ((1u << lane) - 1u))] = b;
    count += __popc(mask);
  }
  if (lane == 0) out[0] = count;
}

static inline size_t mf_align(size_t v) { return (v + 255) & ~(size_t)255; }
constexpr int kMfRestartBlocks = 64;       // blocks per instance of k_mf_apply_restart / k_mf_setup (upper bound)

struct MfWs {
  size_t xsum, xres, ysum, yres, cbar, P1, P4, PS, P3, P3i, S4, S2, wsum, scal, part, ctl, flag, cnt, q0, q1, aP1, aP4, aPS, aP3i, total;
};

static MfWs mf_layout(int B, const MfGeo& G) {
  MfWs W; size_t t = 0;
  auto take = [&](size_t bytes) { size_t o = t; t += mf_align(bytes); return o; };
  const size_t cb = (size_t)B * G.cols * 8, rb = (size_t)B * G.rows * 8;
  const size_t pb = (size_t)B * G.F * G.rt * G.N * 8;
  W.xsum = take(cb); W.xres = take(cb); W.ysum = take(rb); W.yres = take(rb);
  W.cbar = take((size_t)B * G.C * 8);
  W.P1 = take(pb); W.P4 = take(pb); W.PS = take(pb);
  W.P3 = take((size_t)B * G.C * G.ct * 8);
  W.P3i = take((size_t)B * G.C * G.ct * 8);     // cti <= ct (TMA column segments are wider)
  W.S4 = take((size_t)B * G.N * 8); W.S2 = take((size_t)B * 8); W.wsum = take((size_t)B * G.F * 8);
  const size_t per_inst = (size_t)(G.tiles_inst > kMfRestartBlocks ? G.tiles_inst : kMfRestartBlocks);
  W.scal = take((size_t)B * per_inst * 4 * 8);
  W.part = take((size_t)B * kMfRestartBlocks * 2 * 8);
  W.ctl = take((size_t)B * sizeof(Ctl));
  W.flag = take(256);
  W.cnt = take(((size_t)B + 1) * 2 * sizeof(int));     // live list of the bulk pass: count + indices
  // the two small-state buffers the fused launches of a chunk alternate between: y rows [0, rs) | c | cbar per instance
  W.q0 = take((size_t)B * (G.rs + 2 * G.C) * 8); W.q1 = take((size_t)B * (G.rs + 2 * G.C) * 8);
  // ... and the second set of partial sums (a fused launch reads the set the launch before wrote, writes the other)
  W.aP1 = take(pb); W.aP4 = take(pb); W.aPS = take(pb); W.aP3i = take((size_t)B * G.C * G.ct * 8);
  W.total = t + 256;
  return W;
}

template <class Kern> static int mf_grid(Kern kern) {
  int occ = 0;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kMfThreads, 0);
  if (occ < 1) occ = 1;
  return kNumSMs * occ;
}

struct MfPlan {
  int B; MfGeo G; MfIn in; MfSt st; Ctl* ctl; cudaStream_t s;
  int grid_iter, grid_eval, small_blocks, fused;
  int rows_in_flight;            // U of k_mf_iter<K, U> / k_mf_iter2<KP, U>
  int pair;                      // k_mf_iter2 (pairs of adjacent columns, 16-byte accesses) instead of k_mf_iter
  int bulk;                      // k_mf_iter_bulk (streams staged through shared memory by the bulk-copy engine): 1 = four
                                 // streams per stage, 2 = running sums by bulk reduction (two streams per stage)
  BulkCfg bcfg;
  int allow_fuse;                // the caller runs whole chunks (mf_solve_impl): the small-vector update may run inside the pass
  int fuse;                      // ... and does: no k_mf_small launch between the passes of a chunk
  double* q[2];                  // the two small-state buffers of the fused launches
  const int* live;               // [1 + B] count and indices of the instances still iterating (bulk pass), or null
  double *aP1, *aP4, *aPS, *aP3i; // the second set of partial sums (launch k writes set k & 1; set 1 = st.P1, st.P4, st.PS, st.P3i)
  int diag;                      // tools only: bit 2 = time the small-vector kernel alone
};

static void mf_launch_iter(const MfPlan& P) {
  if (P.diag & 4) return;          // tools: time the small-vector kernel alone
  const int64_t total = (int64_t)P.B * P.G.tiles_inst;
  const int g = (int)(total < P.grid_iter ? total : P.grid_iter);
  if (P.bulk) {
    const int threads = (P.bcfg.nw + 1) * 32;
    if (P.bulk == 2) k_mf_iter_bulk<true, false><<<g, threads, P.bcfg.smem, P.s>>>(P.G, P.in, P.st, P.ctl, P.B, P.bcfg, BulkFuse{}, P.live);
    else k_mf_iter_bulk<false, false><<<g, threads, P.bcfg.smem, P.s>>>(P.G, P.in, P.st, P.ctl, P.B, P.bcfg, BulkFuse{}, P.live);
    NEPTUNE_COUNT(1);
    return;
  }
  if (P.pair) {
    if (P.rows_in_flight == 1) k_mf_iter2<1, 1><<<g, kMfThreads, 0, P.s>>>(P.G, P.in, P.st, P.ctl, P.B);
    else k_mf_iter2<1, 2><<<g, kMfThreads, 0, P.s>>>(P.G, P.in, P.st, P.ctl, P.B);
    NEPTUNE_COUNT(1);
    return;
  }
  switch (P.G.K * 10 + P.rows_in_flight) {
    case 11: k_mf_iter<1, 1><<<g, kMfThreads, 0, P.s>>>(P.G, P.in, P.st, P.ctl, P.B); break;
    case 12: k_mf_iter<1, 2><<<g, kMfThreads, 0, P.s>>>(P.G, P.in, P.st, P.ctl, P.B); break;
    case 14: k_mf_iter<1, 4><<<g, kMfThreads, 0, P.s>>>(P.G, P.in, P.st, P.ctl, P.B); break;
    case 21: k_mf_iter<2, 1><<<g, kMfThreads, 0, P.s>>>(P.G, P.in, P.st, P.ctl, P.B); break;
    case 22: k_mf_iter<2, 2><<<g, kMfThreads, 0, P.s>>>(P.G, P.in, P.st, P.ctl, P.B); break;
    case 41: k_mf_iter<4, 1><<<g, kMfThreads, 0, P.s>>>(P.G, P.in, P.st, P.ctl, P.B); break;
    default: k_mf_iter<4, 2><<<g, kMfThreads, 0, P.s>>>(P.G, P.in, P.st, P.ctl, P.B); break;
  }
  NEPTUNE_COUNT(1);
}

// launch k of a chunk with the small-vector update inside the pass: reads the small state the launch before wrote (the
// canonical arrays when it is the first of the chunk -- known on the host, or told by the device flag of graph node 0)
static void mf_launch_fused(const MfPlan& P, int k, const int* first_flag, int force_first) {
  const int64_t total = (int64_t)P.B * P.G.tiles_inst;
  const int g = (int)(total < P.grid_iter ? total : P.grid_iter);
  const int threads = (P.bcfg.nw + 1 + kBulkSmallWarps) * 32;
  BulkFuse fz{P.q[(k + 1) & 1], P.q[k & 1], first_flag, force_first, (int64_t)(P.G.rs + 2 * P.G.C),
              nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  if (k & 1) {          // odd launch: reads the second set, writes the canonical one
    fz.rP1 = P.aP1; fz.rP4 = P.aP4; fz.rPS = P.aPS; fz.rP3 = P.aP3i;
    fz.wP1 = P.st.P1; fz.wP4 = P.st.P4; fz.wPS = P.st.PS; fz.wP3 = P.st.P3i;
  } else {
    fz.rP1 = P.st.P1; fz.rP4 = P.st.P4; fz.rPS = P.st.PS; fz.rP3 = P.st.P3i;
    fz.wP1 = P.aP1; fz.wP4 = P.aP4; fz.wPS = P.aPS; fz.wP3 = P.aP3i;
  }
  if (P.bulk == 2) k_mf_iter_bulk<true, true><<<g, threads, P.bcfg.smem, P.s>>>(P.G, P.in, P.st, P.ctl, P.B, P.bcfg, fz, P.live);
  else k_mf_iter_bulk<false, true><<<g, threads, P.bcfg.smem, P.s>>>(P.G, P.in, P.st, P.ctl, P.B, P.bcfg, fz, P.live);
  NEPTUNE_COUNT(1);
}

// the pass a solve takes when `reserved` does not say: NEPTUNE_MF_PASS = pair | bulk | bulkred (measurements), else the
// compiled default
constexpr int kMfDefaultBulk = 2;        // 0: register passes; 1: bulk-copy staging; 2: bulk-copy staging + bulk reduction (measured: 95.6 us / iteration at C2 x 256 against 125 for the pair pass)
static int mf_default_bulk() {
  const char* e = getenv("NEPTUNE_MF_PASS");
  if (!e || !*e) return kMfDefaultBulk;
  if (!strcmp(e, "bulk")) return 1;
  if (!strcmp(e, "bulkred")) return 2;
  if (!strcmp(e, "pair") || !strcmp(e, "register")) return 0;
  return kMfDefaultBulk;
}

// which pass runs and with how many rows in flight; `reserved`: bit 0 forces the 8-byte pass, bits 8..10 override U,
// bit 12 = bulk-copy staging, bit 13 = bulk-copy staging with the running sums by bulk reduction, bit 11 = register
// passes whatever the default, bits 14..18 = consumer warps of the bulk pass (0 = chosen by shape), bits 19..22 = cap on
// its stages (0 = as many as fit)
static void mf_choose_pass(MfPlan& P, int reserved, const void* x, const void* y, const void* d) {
  const MfGeo& G = P.G;
  switch (G.K) {
    case 1: P.grid_eval = mf_grid(k_mf_eval<1>); break;
    case 2: P.grid_eval = mf_grid(k_mf_eval<2>); break;
    default: P.grid_eval = mf_grid(k_mf_eval<4>); break;
  }
  P.bulk = 0; P.fuse = 0;
  {
    int want = (reserved & (1 << 13)) ? 2 : ((reserved & (1 << 12)) ? 1 : 0);
    const bool forced = want != 0;
    if (!forced && !(reserved & ((1 << 11) | 1))) want = (G.N > 32) ? mf_default_bulk() : 0;    // default: the pair pass's shapes
    const uintptr_t al = (uintptr_t)x | (uintptr_t)y | (uintptr_t)d | (uintptr_t)P.st.xsum | (uintptr_t)P.st.ysum |
                         (uintptr_t)P.in.w | (uintptr_t)P.in.r | (uintptr_t)P.st.cbar;
    if (want && !(G.N & 1) && G.N <= 64 && G.rt == 1 && G.ct == 1 && (al & 15) == 0) {
      // bit 23: keep the small-vector update in its own launches (k_mf_small) even where it could run inside the pass
      const int try_fuse = P.allow_fuse && !(reserved & (1 << 23)) && !G.with_n;
      P.bcfg = bulk_config(G.N, want == 2, (reserved >> 14) & 31, (reserved >> 19) & 15, G.F, try_fuse);
      if (!P.bcfg.ok && try_fuse) P.bcfg = bulk_config(G.N, want == 2, (reserved >> 14) & 31, (reserved >> 19) & 15);
      P.bcfg.diag = (reserved >> 4) & 3;
      if (P.bcfg.ok) {
        cudaError_t e;
        if (P.bcfg.fuse)
          e = want == 2 ? cudaFuncSetAttribute(k_mf_iter_bulk<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)P.bcfg.smem)
                        : cudaFuncSetAttribute(k_mf_iter_bulk<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)P.bcfg.smem);
        else
          e = want == 2 ? cudaFuncSetAttribute(k_mf_iter_bulk<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)P.bcfg.smem)
                        : cudaFuncSetAttribute(k_mf_iter_bulk<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)P.bcfg.smem);
        if (e == cudaSuccess) { P.bulk = want; P.fuse = P.bcfg.fuse; P.grid_iter = kNumSMs; P.pair = 0; P.rows_in_flight = 0; return; }
        (void)cudaGetLastError();
      }
    }
  }
  P.rows_in_flight = (reserved >> 8) & 7;
  P.pair = !(reserved & 1) && !(G.N & 1) && G.K == 2 && G.N <= 64 && (((uintptr_t)x | (uintptr_t)y | (uintptr_t)d) & 15) == 0;
  if (P.pair) {
    if (P.rows_in_flight != 1 && P.rows_in_flight != 2) P.rows_in_flight = 2;
    P.grid_iter = P.rows_in_flight == 1 ? mf_grid(k_mf_iter2<1, 1>) : mf_grid(k_mf_iter2<1, 2>);
    return;
  }
  if (P.rows_in_flight != 1 && P.rows_in_flight != 2 && !(P.rows_in_flight == 4 && G.K == 1))
    P.rows_in_flight = G.K == 4 ? 1 : 2;
  switch (G.K * 10 + P.rows_in_flight) {
    case 11: P.grid_iter = mf_grid(k_mf_iter<1, 1>); break;
    case 12: P.grid_iter = mf_grid(k_mf_iter<1, 2>); break;
    case 14: P.grid_iter = mf_grid(k_mf_iter<1, 4>); break;
    case 21: P.grid_iter = mf_grid(k_mf_iter<2, 1>); break;
    case 22: P.grid_iter = mf_grid(k_mf_iter<2, 2>); break;
    case 41: P.grid_iter = mf_grid(k_mf_iter<4, 1>); break;
    default: P.grid_iter = mf_grid(k_mf_iter<4, 2>); break;
  }
}

static void mf_launch_eval(const MfPlan& P, int which, int only_ps) {
  const int64_t total = (int64_t)P.B * P.G.tiles_inst;
  const int g = (int)(total < P.grid_eval ? total : P.grid_eval);
  switch (P.G.K) {
    case 1: k_mf_eval<1><<<g, kMfThreads, 0, P.s>>>(P.G, P.in, P.st, P.ctl, P.B, which, only_ps); break;
    case 2: k_mf_eval<2><<<g, kMfThreads, 0, P.s>>>(P.G, P.in, P.st, P.ctl, P.B, which, only_ps); break;
    default: k_mf_eval<4><<<g, kMfThreads, 0, P.s>>>(P.G, P.in, P.st, P.ctl, P.B, which, only_ps); break;
  }
  NEPTUNE_COUNT(1);
}

// the small updates around one pass: `mask` of PH_*; in the unfused (large instance) case the C2 dual needs
// every cbar of the instance, so it is a launch of its own
static void mf_launch_small(const MfPlan& P, int mask, const int* skip_post) {
  dim3 g(P.small_blocks, P.B);
  if (P.diag & 4) {          // tools (small-vector kernel alone): NEPTUNE_SMALL_MASK restricts the phases that run
    const char* e = getenv("NEPTUNE_SMALL_MASK");
    if (e && *e) mask &= atoi(e);
    if (!mask) return;
  }
  if (P.fused) {
    const int threads = P.G.C >= 512 ? 512 : (P.G.C <= 64 ? 64 : (int)((P.G.C + 31) / 32) * 32);
    k_mf_small<<<g, threads, 0, P.s>>>(P.G, P.in, P.st, P.ctl, mask, skip_post, 1); NEPTUNE_COUNT(1);
  } else {
    if (mask & (PH_POST | PH_PREC)) {
      k_mf_small<<<g, 256, 0, P.s>>>(P.G, P.in, P.st, P.ctl, mask & (PH_POST | PH_PREC), skip_post, 0); NEPTUNE_COUNT(1);
    }
    if (mask & PH_Y2) { k_mf_small<<<g, 256, 0, P.s>>>(P.G, P.in, P.st, P.ctl, PH_Y2, nullptr, 0); NEPTUNE_COUNT(1); }
  }
}

}  // namespace neptune

using namespace neptune;

// host-only: the tile geometry the solver would use (tests, tools).  out[0..7] = {K columns per lane, JT columns per
// tile, ct column tiles, RT rows per tile, rt row tiles, tiles per instance, F*N <= 4096 (single-block small
// kernel), the default bulk-copy pass of a min-delay solve with an even graph replay runs the small-vector update
// inside its launches}; out[8..15] = geometry of the bulk-copy pass (below)
extern "C" int neptune_pdhg_mf_geometry(int B, int N, int F, int32_t* out) {
  if (B <= 0 || N <= 0 || F <= 0 || !out) return NEPTUNE_E_ARG;
  const MfGeo G = make_geo(N, F, B);
  out[0] = G.K; out[1] = G.JT; out[2] = G.ct; out[3] = G.RT; out[4] = G.rt; out[5] = G.tiles_inst;
  out[6] = G.C <= 4096; out[7] = 0;
  for (int k = 8; k < 16; ++k) out[k] = 0;
  // the bulk-copy pass (pdhg_mf_bulk.cuh): out[8..10] = {applicable, stages, consumer warps} with four streams per stage,
  // out[11..13] = the same with the running sums by bulk reduction, out[14] = the pass a default solve takes for this
  // shape (0 register passes, 1 / 2 bulk), out[15] = dynamic shared memory of the reduction version in bytes
  if (G.rt == 1 && G.ct == 1) {
    const BulkCfg c4 = bulk_config(N, 0, 0, 0), c2 = bulk_config(N, 1, 0, 0);
    out[8] = c4.ok; out[9] = c4.stages; out[10] = c4.nw;
    out[11] = c2.ok; out[12] = c2.stages; out[13] = c2.nw; out[15] = (int32_t)c2.smem;
    const int dflt = N > 32 ? mf_default_bulk() : 0;
    out[14] = (dflt == 1 && c4.ok) ? 1 : ((dflt == 2 && c2.ok) ? 2 : 0);
    out[7] = out[14] ? bulk_config(N, out[14] == 2, 0, 0, F, 1).ok : 0;     // as mf_choose_pass: the fused config fits
  }
  return 0;
}

extern "C" int neptune_pdhg_mf_workspace_bytes(int B, int N, int F, int64_t* bytes) {
  if (B <= 0 || N <= 0 || F <= 0 || !bytes) return NEPTUNE_E_ARG;
  // sized for the layout WITH node columns (N more columns, 3N more rows): valid for every kind
  Layout L(N, F, NEPTUNE_KIND_MIN_DELAY_UTIL, NEPTUNE_FLAG_STRENGTHEN);
  if (L.cols >= (int64_t)INT32_MAX || L.rows >= (int64_t)INT32_MAX) return NEPTUNE_E_SIZE;
  const MfGeo G = make_geo(N, F, B, NEPTUNE_KIND_MIN_DELAY_UTIL);
  *bytes = (int64_t)mf_layout(B, G).total;
  return 0;
}

static int mf_solve_impl(int B, int N, int F, int kind, const double* d, const double* w, const double* r,
                         const double* m, const double* Mj, const double* Kj, const double* cost, double budget,
                         double objn, const double* bigm, const neptune_pdhg_params* prm, double* x, double* y,
                         neptune_pdhg_result* result_d, void* workspace, int64_t workspace_bytes, void* stream) {
  if (B <= 0 || N <= 0 || F <= 0) return NEPTUNE_E_ARG;
  if (kind < 0 || kind > 2) return NEPTUNE_E_ARG;
  if (!d || !w || !r || !m || !Mj || !Kj || !prm || !x || !y || !result_d || !workspace) return NEPTUNE_E_ARG;
  if (kind != NEPTUNE_KIND_MIN_DELAY && !cost) return NEPTUNE_E_ARG;
  int64_t need = 0;
  { int rc = neptune_pdhg_mf_workspace_bytes(B, N, F, &need); if (rc) return rc; }
  if (workspace_bytes < need) return NEPTUNE_E_NOMEM;
  if ((int64_t)B * make_geo(N, F, B).tiles_inst >= (int64_t)INT32_MAX) return NEPTUNE_E_SIZE;
  cudaStream_t caller = (cudaStream_t)stream;
  // side stream, events, graph: released on EVERY return path (an error between BeginCapture and EndCapture also
  // ends the capture, so the side stream is never left capturing)
  struct Guard {
    cudaStream_t s = nullptr; cudaEvent_t ev_in = nullptr, ev_out = nullptr;
    cudaGraph_t graph = nullptr; cudaGraphExec_t gexec = nullptr; bool capturing = false;
    ~Guard() {
      if (capturing && s) { cudaGraph_t g = nullptr; cudaStreamEndCapture(s, &g); if (g) cudaGraphDestroy(g); }
      if (gexec) cudaGraphExecDestroy(gexec);
      if (graph) cudaGraphDestroy(graph);
      if (ev_in) cudaEventDestroy(ev_in);
      if (ev_out) cudaEventDestroy(ev_out);
      if (s) cudaStreamDestroy(s);
    }
  } guard;
  cudaStream_t& s = guard.s;
  cudaEvent_t& ev_in = guard.ev_in; cudaEvent_t& ev_out = guard.ev_out;
  NEPTUNE_CUDA_OK(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
  NEPTUNE_CUDA_OK(cudaEventCreateWithFlags(&ev_in, cudaEventDisableTiming));
  NEPTUNE_CUDA_OK(cudaEventCreateWithFlags(&ev_out, cudaEventDisableTiming));
  NEPTUNE_CUDA_OK(cudaEventRecord(ev_in, caller));
  NEPTUNE_CUDA_OK(cudaStreamWaitEvent(s, ev_in, 0));
  const int check_every = prm->check_every > 0 ? prm->check_every : 64;
  const int max_iters = prm->max_iters > 0 ? prm->max_iters : 20000;

  MfPlan P{};
  P.B = B; P.G = make_geo(N, F, B, kind); P.s = s;
  P.in = MfIn{d, w, r, m, Mj, Kj, cost, budget, objn, bigm};
  const MfGeo& G = P.G;
  const MfWs W = mf_layout(B, G);
  char* base = (char*)workspace;
  double* xres = (double*)(base + W.xres); double* yres = (double*)(base + W.yres);
  double* part = (double*)(base + W.part);
  int* d_flag = (int*)(base + W.flag);          // [0] all done, [1] skip-POST flag of the graph's first node
  Ctl* ctl = (Ctl*)(base + W.ctl);
  P.ctl = ctl;
  P.st = MfSt{x, y, (double*)(base + W.xsum), (double*)(base + W.ysum), (double*)(base + W.cbar),
              (double*)(base + W.P1), (double*)(base + W.P4), (double*)(base + W.PS), (double*)(base + W.P3),
              (double*)(base + W.P3i),
              (double*)(base + W.S4), (double*)(base + W.S2), (double*)(base + W.wsum), (double*)(base + W.scal)};
  P.diag = (prm->reserved >> 4) & 7;
  P.q[0] = (double*)(base + W.q0); P.q[1] = (double*)(base + W.q1);
  P.aP1 = (double*)(base + W.aP1); P.aP4 = (double*)(base + W.aP4); P.aPS = (double*)(base + W.aPS); P.aP3i = (double*)(base + W.aP3i);
  // the fused launches of a graph replay alternate between the two small-state buffers: a replay must be an even number
  // of launches
  P.allow_fuse = ((check_every < 32 ? check_every : 32) & 1) == 0;
  mf_choose_pass(P, prm->reserved, x, y, d);
  P.live = P.bulk ? (const int*)(base + W.cnt) : nullptr;
  // small vectors: one block per instance does POST + PREC + Y2 in one launch while F*N is small; larger
  // instances spread over several blocks and take the C2 dual in a second launch
  P.fused = G.C <= 4096;
  P.small_blocks = P.fused ? 1 : (int)((G.C + 255) / 256 < 8 * kNumSMs ? (G.C + 255) / 256 : 8 * kNumSMs);   // one item per thread: the sums are latency-bound

  const size_t cb = (size_t)B * G.cols * 8, rb = (size_t)B * G.rows * 8;
  NEPTUNE_CUDA_OK(cudaMemsetAsync(ctl, 0, (size_t)B * sizeof(Ctl), s));
  NEPTUNE_CUDA_OK(cudaMemsetAsync(d_flag, 0, 8, s));
  const int nblk = G.tiles_inst < kMfRestartBlocks ? G.tiles_inst : kMfRestartBlocks;
  { k_mf_wsum<<<(int)(((int64_t)B * F * 32 + 255) / 256), 256, 0, s>>>(N, (int64_t)B * F, w, P.st.wsum); NEPTUNE_COUNT(1); }
  { k_mf_setup<<<dim3(nblk, B), 256, 0, s>>>(G, P.in, P.st, nblk); NEPTUNE_COUNT(1); }
  { k_mf_setup_norms<<<(B + 127) / 128, 128, 0, s>>>(G, P.in, P.st, ctl, B, nblk); NEPTUNE_COUNT(1); }
  { k_ctl_init<<<(B + 127) / 128, 128, 0, s>>>(B, ctl, 0.99); NEPTUNE_COUNT(1); }
  if (P.bulk) { k_mf_live<<<1, 32, 0, s>>>(B, ctl, (int*)(base + W.cnt)); NEPTUNE_COUNT(1); }
  NEPTUNE_CUDA_OK(cudaMemsetAsync(P.st.xsum, 0, cb, s));
  NEPTUNE_CUDA_OK(cudaMemsetAsync(P.st.ysum, 0, rb, s));
  NEPTUNE_CUDA_OK(cudaMemcpyAsync(xres, x, cb, cudaMemcpyDeviceToDevice, s));
  NEPTUNE_CUDA_OK(cudaMemcpyAsync(yres, y, rb, cudaMemcpyDeviceToDevice, s));
  mf_launch_eval(P, 0, 1);                      // PS <- column sums of the starting yS
  NEPTUNE_LAUNCH_OK();

  // `inner` iterations = {small(POST unless first of the chunk, PREC, Y2); pass} captured once and replayed;
  // the chunk ends with small(POST).  Step sizes, restart flags and convergence live in device memory.
  const int inner = check_every < 32 ? check_every : 32;
  cudaGraph_t& graph = guard.graph;
  cudaGraphExec_t& gexec = guard.gexec;
  int64_t per_graph = 0;
  {
    int64_t c0 = 0, c1 = 0;
    neptune_launch_count(&c0, 0);
    NEPTUNE_CUDA_OK(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
    guard.capturing = true;
    for (int k = 0; k < inner; ++k) {
      if (P.fuse) { mf_launch_fused(P, k, k == 0 ? d_flag + 1 : nullptr, 0); continue; }
      mf_launch_small(P, PH_POST | PH_PREC | PH_Y2, k == 0 ? d_flag + 1 : nullptr);
      mf_launch_iter(P);
    }
    guard.capturing = false;
    NEPTUNE_CUDA_OK(cudaStreamEndCapture(s, &graph));
    NEPTUNE_CUDA_OK(cudaGraphInstantiate(&gexec, graph, 0));
    neptune_launch_count(&c1, 0);
    per_graph = c1 - c0;
    NEPTUNE_COUNT(-per_graph);
  }
  int h_flag = 0;
  for (int it = 0; it < max_iters && !h_flag; it += check_every) {
    const int chunk = check_every < max_iters - it ? check_every : max_iters - it;      // the last chunk stops at max_iters
    int done = 0;
    bool first = true;
    for (; done + inner <= chunk; done += inner) {
      NEPTUNE_CUDA_OK(cudaMemsetAsync(d_flag + 1, first ? 1 : 0, 1, s));     // int 1 / 0 (little endian)
      NEPTUNE_CUDA_OK(cudaGraphLaunch(gexec, s));
      NEPTUNE_COUNT(per_graph);
      first = false;
    }
    for (; done < chunk; ++done) {
      if (P.fuse) { mf_launch_fused(P, done, nullptr, first ? 1 : 0); first = false; continue; }
      mf_launch_small(P, (first ? 0 : PH_POST) | PH_PREC | PH_Y2, nullptr);
      mf_launch_iter(P);
      first = false;
    }
    if (P.fuse) {
      const bool odd = (chunk - 1) & 1;       // the last launch of the chunk wrote set (chunk - 1) & 1
      k_mf_small_from<<<B, 256, 0, s>>>(G, P.in, P.st, ctl, P.q[(chunk - 1) & 1], (int64_t)(G.rs + 2 * G.C),
                                        odd ? P.st.P1 : P.aP1, odd ? P.st.P4 : P.aP4, odd ? P.st.P3i : P.aP3i); NEPTUNE_COUNT(1);
    } else {
      mf_launch_small(P, PH_POST, nullptr);
    }
    { k_ctl_advance<<<(B + 127) / 128, 128, 0, s>>>(B, ctl, chunk); NEPTUNE_COUNT(1); }
    // KKT of the current iterate and of the running average
    for (int wch = 0; wch < 2; ++wch) {
      mf_launch_eval(P, wch, 0);
      { k_mf_eval_small<<<B, 256, 0, s>>>(G, P.in, P.st, ctl, wch); NEPTUNE_COUNT(1); }
    }
    { k_ctl_decide<<<(B + 127) / 128, 128, 0, s>>>(B, ctl, chunk, prm->eps_abs, prm->eps_rel, max_iters,
                                                 result_d); NEPTUNE_COUNT(1); }
    { k_mf_apply_restart<<<dim3(kMfRestartBlocks, B), 256, 0, s>>>(G, P.in, P.st, xres, yres, ctl, part); NEPTUNE_COUNT(1); }
    { k_mf_restart_norms<<<(B + 127) / 128, 128, 0, s>>>(B, kMfRestartBlocks, part, ctl); NEPTUNE_COUNT(1); }
    { k_ctl_after_restart<<<(B + 127) / 128, 128, 0, s>>>(B, ctl); NEPTUNE_COUNT(1); }
    mf_launch_eval(P, 0, 1);                    // PS of the (possibly replaced) yS for the next PREC
    { k_all_done<<<1, 32, 0, s>>>(B, ctl, d_flag); NEPTUNE_COUNT(1); }
    if (P.bulk) { k_mf_live<<<1, 32, 0, s>>>(B, ctl, (int*)(base + W.cnt)); NEPTUNE_COUNT(1); }
    NEPTUNE_CUDA_OK(cudaMemcpyAsync(&h_flag, d_flag, 4, cudaMemcpyDeviceToHost, s));
    NEPTUNE_CUDA_OK(cudaStreamSynchronize(s));
  }
  NEPTUNE_LAUNCH_OK();
  NEPTUNE_CUDA_OK(cudaEventRecord(ev_out, s));
  NEPTUNE_CUDA_OK(cudaStreamWaitEvent(caller, ev_out, 0));
  NEPTUNE_CUDA_OK(cudaStreamSynchronize(s));
  return 0;          // `guard` releases the graph, its exec, the events and the side stream
}

extern "C" int neptune_pdhg_mf_solve(int B, int N, int F, int kind, const double* d, const double* w,
                                     const double* r, const double* m, const double* Mj, const double* Kj,
                                     const neptune_pdhg_params* prm, double* x, double* y,
                                     neptune_pdhg_result* result_d, void* workspace, int64_t workspace_bytes,
                                     void* stream) {
  if (kind != NEPTUNE_KIND_MIN_DELAY) return NEPTUNE_E_ARG;      // node columns: neptune_pdhg_mf_solve_util
  return mf_solve_impl(B, N, F, kind, d, w, r, m, Mj, Kj, nullptr, 0.0, 0.0, nullptr, prm, x, y, result_d, workspace,
                       workspace_bytes, stream);
}

extern "C" int neptune_pdhg_mf_solve_util(int B, int N, int F, int kind, const double* d_obj, const double* w,
                                          const double* r, const double* m, const double* Mj, const double* Kj,
                                          const double* cost, double budget, double obj_n, const double* big_m,
                                          const neptune_pdhg_params* prm, double* x, double* y,
                                          neptune_pdhg_result* result_d, void* workspace, int64_t workspace_bytes,
                                          void* stream) {
  if (kind != NEPTUNE_KIND_MIN_UTIL && kind != NEPTUNE_KIND_MIN_DELAY_UTIL) return NEPTUNE_E_ARG;
  return mf_solve_impl(B, N, F, kind, d_obj, w, r, m, Mj, Kj, cost, budget, obj_n, big_m, prm, x, y, result_d, workspace,
                       workspace_bytes, stream);
}

// ===================================================================================================
// Step-wise building blocks for the function-block-sharded matrix-free PDHG (SURVEY.md section 8(e); one
// process per GPU, neptune_mip_b200/sharded_mf.py owns the loop and the all-reduce).  The numpy statement it
// follows (tests/mf_reference.ShardedMatrixFree) is proven equal to the unsharded iteration on 2 gloo ranks;
// two NCCL ranks on B200 reproduce the single-rank iterates to 3e-17 (tests/test_sharded_gpu.py).
// A rank holds the functions of its block (F = functions of this rank); the 2N multipliers of the coupling
// rows (y2: C2 memory, y4: C4 CPU) are replicated.  Per iteration:
//   neptune_pdhg_mf_local_step : y1, y3 of the pass that just ran (local), c columns of the next iteration
//                                (local), coupling[2N] = [C4 activity of that pass | C2 activity of the new cbar]
//   (caller: all-reduce of coupling over the ranks -- 2N doubles)
//   neptune_pdhg_mf_pass       : y4, y2 from the global activities (replicated), then the iteration pass
//                                (k_mf_iter, unchanged) over the own functions.
// Step sizes are host scalars; S4[N], S2[1] (global Pock-Chambolle row sums) come from the caller.
// ===================================================================================================
namespace neptune {

struct MfStepWs { size_t cbar, P1, P4, PS, P3i, ctl, total; };

static MfStepWs mf_step_layout(int B, const MfGeo& G) {
  MfStepWs W; size_t t = 0;
  auto take = [&](size_t bytes) { size_t o = t; t += mf_align(bytes); return o; };
  const size_t pb = (size_t)B * G.F * G.rt * G.N * 8;
  W.cbar = take((size_t)B * G.C * 8);
  W.P1 = take(pb); W.P4 = take(pb); W.PS = take(pb);
  W.P3i = take((size_t)B * G.C * G.ct * 8);
  W.ctl = take((size_t)B * sizeof(Ctl));
  W.total = t + 256;
  return W;
}

__global__ void k_mf_set_steps(int B, Ctl* ctl, double tau, double sigma) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  ctl[b].tau = tau; ctl[b].sigma = sigma; ctl[b].converged = 0;
}

// local part of the small-vector work of a rank: POST without the C4 dual (have_pass), PREC always
__global__ void __launch_bounds__(256)
k_mf_shard_local(MfGeo G, MfIn in, MfSt st, double tau, double sigma_prev, int have_pass, int do_prec) {
  const int b = blockIdx.y;
  const int N = G.N, rt = G.rt, ct = G.cti;
  const int C = (int)G.C;
  double* __restrict__ y = st.y + (int64_t)b * G.rows;
  double* __restrict__ ys = st.ysum + (int64_t)b * G.rows;
  double* __restrict__ c = st.x + (int64_t)b * G.cols + G.X;
  double* __restrict__ cs = st.xsum + (int64_t)b * G.cols + G.X;
  double* __restrict__ cbar = st.cbar + (int64_t)b * C;
  const double* __restrict__ P1 = st.P1 + (int64_t)b * G.F * rt * N;
  const double* __restrict__ PS = st.PS + (int64_t)b * G.F * rt * N;
  const double* __restrict__ P3 = st.P3i + (int64_t)b * C * ct;
  const double* __restrict__ m = in.m + (int64_t)b * G.F;
  const double s1 = sigma_prev / (double)(N + 1), s3 = sigma_prev / (double)N;
  for (int q = blockIdx.x * blockDim.x + threadIdx.x; q < C; q += gridDim.x * blockDim.x) {
    const int f = q / N, j = q - f * N;
    const int64_t po = (int64_t)f * rt * N + j;
    double y1 = y[2 * q + 1];
    double sS = 0.0;
    if (have_pass) {
      const double a1 = strided_sum(P1 + po, rt, N) - cbar[q];
      const double a3 = strided_sum(P3 + (int64_t)q * ct, ct, 1);
      const double v1 = y1 + s1 * a1;
      y1 = v1 - s1 * fmax(v1 / s1, -kEps);
      y[2 * q + 1] = y1; ys[2 * q + 1] += y1;
      const double y3n = y[G.r3 + q] + s3 * a3 - s3;
      y[G.r3 + q] = y3n; ys[G.r3 + q] += y3n;
      sS = strided_sum(PS + po, rt, N);
    } else {
      sS = strided_sum(PS + po, rt, N);            // PS of the starting yS (filled by neptune_pdhg_mf_column_sums)
    }
    if (!do_prec) continue;                        // end of a chunk: the c columns stay where they are
    const double mf = m[f];
    const double gc = -y1 + mf * y[G.r2 + j] - sS;
    const double co = c[q];
    double cn = co - tau * gc / (1.0 + mf + (double)N);
    cn = fmin(fmax(cn, 0.0), 1.0);
    cbar[q] = 2.0 * cn - co;
    c[q] = cn; cs[q] += cn;
  }
}

// coupling[b][0:N] = C4 activity of the pending pass over the own functions (0 without one),
// coupling[b][N:2N] = C2 activity of the new cbar over the own functions
__global__ void __launch_bounds__(256)
k_mf_shard_coupling(MfGeo G, MfIn in, MfSt st, int have_pass, double* __restrict__ coupling) {
  const int b = blockIdx.y;
  const int N = G.N, F = G.F;
  const double* __restrict__ P4 = st.P4 + (int64_t)b * F * G.rt * N;
  const double* __restrict__ cbar = st.cbar + (int64_t)b * G.C;
  const double* __restrict__ m = in.m + (int64_t)b * F;
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < N; j += gridDim.x * blockDim.x) {
    coupling[(int64_t)b * 2 * N + j] = have_pass ? strided_sum(P4 + j, F * G.rt, N) : 0.0;
    double a = 0.0;
    for (int f0 = 0; f0 < F; f0 += 8) {
      double v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) v[u] = (f0 + u < F) ? m[f0 + u] * cbar[(int64_t)(f0 + u) * N + j] : 0.0;
#pragma unroll
      for (int u = 0; u < 8; ++u) a += v[u];
    }
    coupling[(int64_t)b * 2 * N + N + j] = a;
  }
}

// replicated dual updates from the all-reduced activities: y4 with the step of the pass it belongs to
// (apply_y4), y2 with the current one (apply_y2)
__global__ void __launch_bounds__(256)
k_mf_shard_apply(MfGeo G, MfIn in, MfSt st, double sigma4, double sigma2, int apply_y4, int apply_y2,
                 const double* __restrict__ coupling) {
  const int b = blockIdx.y;
  const int N = G.N;
  double* __restrict__ y = st.y + (int64_t)b * G.rows;
  double* __restrict__ ys = st.ysum + (int64_t)b * G.rows;
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < N; j += gridDim.x * blockDim.x) {
    if (apply_y4) {
      const double s = sigma4 * st.S4[(int64_t)b * N + j];
      const double v = y[G.r4 + j] + s * coupling[(int64_t)b * 2 * N + j];
      const double yn = v - s * fmin(v / s, in.Kj[(int64_t)b * N + j]);
      y[G.r4 + j] = yn; ys[G.r4 + j] += yn;
    }
    if (apply_y2) {
      const double s = sigma2 * st.S2[b];
      const double v = y[G.r2 + j] + s * coupling[(int64_t)b * 2 * N + N + j];
      const double yn = v - s * fmin(v / s, in.Mj[(int64_t)b * N + j]);
      y[G.r2 + j] = yn; ys[G.r2 + j] += yn;
    }
  }
}

static int mf_step_plan(MfPlan& P, int B, int N, int F, const double* d, const double* w, const double* r,
                        const double* m, const double* Mj, const double* Kj, double* x, double* y, double* xsum,
                        double* ysum, const double* S4, const double* S2, void* ws, int64_t ws_bytes, cudaStream_t s) {
  if (B <= 0 || N <= 0 || F <= 0 || !w || !r || !m || !x || !y || !xsum || !ysum || !S4 || !S2 || !ws) return NEPTUNE_E_ARG;
  P = MfPlan{};
  P.B = B; P.G = make_geo(N, F, B); P.s = s;
  const MfStepWs W = mf_step_layout(B, P.G);
  if (ws_bytes < (int64_t)W.total) return NEPTUNE_E_NOMEM;
  char* base = (char*)ws;
  P.in = MfIn{d, w, r, m, Mj, Kj, nullptr, 0.0, 0.0, nullptr};
  P.ctl = (Ctl*)(base + W.ctl);
  P.st = MfSt{x, y, xsum, ysum, (double*)(base + W.cbar), (double*)(base + W.P1), (double*)(base + W.P4),
              (double*)(base + W.PS), nullptr, (double*)(base + W.P3i), const_cast<double*>(S4),
              const_cast<double*>(S2), nullptr, nullptr};
  mf_choose_pass(P, 0, x, y, d);
  P.small_blocks = (int)((P.G.C + 255) / 256 < 4 * kNumSMs ? (P.G.C + 255) / 256 : 4 * kNumSMs);
  return 0;
}

}  // namespace neptune

extern "C" int neptune_pdhg_mf_step_bytes(int B, int N, int F, int64_t* bytes) {
  if (B <= 0 || N <= 0 || F <= 0 || !bytes) return NEPTUNE_E_ARG;
  Layout L(N, F, NEPTUNE_KIND_MIN_DELAY, NEPTUNE_FLAG_STRENGTHEN);
  if (L.cols >= (int64_t)INT32_MAX || L.rows >= (int64_t)INT32_MAX) return NEPTUNE_E_SIZE;
  *bytes = (int64_t)mf_step_layout(B, make_geo(N, F, B)).total;
  return 0;
}

// PS <- column sums of the current yS (call once before the first local step, and after y was replaced)
extern "C" int neptune_pdhg_mf_column_sums(int B, int N, int F, const double* w, const double* r, const double* m,
                                           double* x, double* y, double* xsum, double* ysum, const double* S4,
                                           const double* S2, void* ws, int64_t ws_bytes, void* stream) {
  MfPlan P;
  { int rc = mf_step_plan(P, B, N, F, nullptr, w, r, m, nullptr, nullptr, x, y, xsum, ysum, S4, S2, ws, ws_bytes,
                          (cudaStream_t)stream); if (rc) return rc; }
  { k_mf_set_steps<<<(B + 127) / 128, 128, 0, P.s>>>(B, P.ctl, 0.0, 0.0); NEPTUNE_COUNT(1); }
  mf_launch_eval(P, 0, 1);
  NEPTUNE_LAUNCH_OK();
  return 0;
}

extern "C" int neptune_pdhg_mf_local_step(int B, int N, int F, const double* w, const double* r, const double* m,
                                          double tau, double sigma_prev, int have_pass, int do_prec, double* x, double* y,
                                          double* xsum, double* ysum, const double* S4, const double* S2, void* ws,
                                          int64_t ws_bytes, double* coupling, void* stream) {
  if (!coupling) return NEPTUNE_E_ARG;
  MfPlan P;
  { int rc = mf_step_plan(P, B, N, F, nullptr, w, r, m, nullptr, nullptr, x, y, xsum, ysum, S4, S2, ws, ws_bytes,
                          (cudaStream_t)stream); if (rc) return rc; }
  dim3 g(P.small_blocks, B), gn((N + 255) / 256, B);
  { k_mf_shard_local<<<g, 256, 0, P.s>>>(P.G, P.in, P.st, tau, sigma_prev, have_pass, do_prec); NEPTUNE_COUNT(1); }
  { k_mf_shard_coupling<<<gn, 256, 0, P.s>>>(P.G, P.in, P.st, have_pass, coupling); NEPTUNE_COUNT(1); }
  NEPTUNE_LAUNCH_OK();
  return 0;
}

extern "C" int neptune_pdhg_mf_pass(int B, int N, int F, const double* d, const double* w, const double* r,
                                    const double* m, const double* Mj, const double* Kj, double tau, double sigma,
                                    double sigma_prev, int have_pass, int run_pass, double* x, double* y, double* xsum,
                                    double* ysum, const double* S4, const double* S2, void* ws, int64_t ws_bytes,
                                    const double* coupling_sum, void* stream) {
  if (!d || !Mj || !Kj || !coupling_sum) return NEPTUNE_E_ARG;
  MfPlan P;
  { int rc = mf_step_plan(P, B, N, F, d, w, r, m, Mj, Kj, x, y, xsum, ysum, S4, S2, ws, ws_bytes,
                          (cudaStream_t)stream); if (rc) return rc; }
  dim3 gn((N + 255) / 256, B);
  // run_pass = 0: end of a chunk -- only the pending C4 dual is applied (the C2 half of coupling_sum is ignored)
  { k_mf_shard_apply<<<gn, 256, 0, P.s>>>(P.G, P.in, P.st, sigma_prev, sigma, have_pass, run_pass, coupling_sum); NEPTUNE_COUNT(1); }
  if (run_pass) {
    { k_mf_set_steps<<<(B + 127) / 128, 128, 0, P.s>>>(B, P.ctl, tau, sigma); NEPTUNE_COUNT(1); }
    mf_launch_iter(P);
  }
  NEPTUNE_LAUNCH_OK();
  return 0;
}
