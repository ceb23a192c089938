// pdhg.cu -- (b) restarted, averaged, diagonally preconditioned PDHG for the LP relaxation of the
// placement model:   min obj.x   s.t.  lo <= A x <= hi,  lb <= x <= ub.
//
// Replaces the LP work inside pywraplp.Solver.Solve() (reference core/solvers/solver.py:37).
// Two kernels per iteration, each ONE pass over one copy of the matrix with the vector update fused
// into the SpMV epilogue (so g = A^T y and A x-bar are never materialised):
//   k_cols<PrimalUpdate> : g = A^T y (CSR of A^T, thread per short column / warp per long one);
//                          x+ = clip(x - tau*T*(obj + g)); x-bar = 2x+ - x; xsum += x+
//   k_rows<DualUpdate>   : a = A x-bar (warp per row; block per long row, shuffle + smem reduce);
//                          v = y + sigma*S*a; y+ = v - sigma*S*clip(v/(sigma*S), lo, hi); ysum += y+
// T = dc^2, S = dr^2 are the Ruiz + Pock-Chambolle equilibration written as diagonal step sizes, so
// the assembled (parity-checked) matrix values are never modified.
// Algorithmic bytes per iteration (fp64 values, int32 indices, int64 row pointers), see DESIGN.md:
//   24*nnz + 8*(cols+1) + 8*(rows+1)              matrix, both copies
//   + cols*(8 x + 8 obj + 8 T + 16 lb/ub + 8 x' + 8 xbar + 16 xsum) + 8*rows (y gather)
//   + rows*(8 y + 8 S + 16 lo/hi + 8 y' + 16 ysum) + 8*cols (xbar gather)
//   = 24*nnz + 88*cols + 72*rows.
#include "common.cuh"
#include "pdhg_ctl.cuh"
#include <cub/cub.cuh>

namespace neptune {

constexpr int kLongRow = 2048;      // rows longer than this get a whole block
constexpr int kShortCol = 8;        // columns of A^T up to this length: one thread each
constexpr int kTaskNnz = 1024;      // non-zeros per warp task of the row kernel
constexpr int kShortRow = 8;        // rows of A up to this length (whole 32-row chunk): one thread each
constexpr int kMaxLongList = 1 << 20;

struct Csr {
  const int64_t* ptr; const int32_t* idx; const double* val;   // val is [B][nnz]
  int64_t n_rows, n_cols, nnz;
};

// ---------------------------------------------------------------------------------------------------
// SpMV cores.  `Epi` consumes one (instance, row, dot) at a time in the thread that owns it.
// ---------------------------------------------------------------------------------------------------
// SpMV over a CSR matrix (A or the stored A^T) whose rows are grouped into warp TASKS: up to 32
// consecutive rows holding about kTaskNnz non-zeros (build_tasks).  Two kernels share the task list:
//   k_spmv_short : tasks whose rows all have <= kShortRow entries (the x / c / n columns of A^T, the C6
//                  and S rows of A): ONE THREAD PER ROW.  Neighbouring rows are neighbours in the CSR
//                  arrays, so a warp still reads contiguous memory; 8/16 B and 16/32 B vector loads
//                  for 2- and 4-entry rows; epilogue operands are loaded before the dot product so
//                  that every load of a row is in flight at once.  Lean (full occupancy).
//   k_spmv_tasks : the other tasks: the warp walks the rows two at a time, lanes striding over a row
//                  (coalesced 128 B / 256 B segments of col_idx / val, 4 loads in flight per lane and
//                  row), shuffle reduction; lane k keeps the dot product of row k and the epilogue
//                  (vector update) runs once per task with all lanes, coalesced.
constexpr int32_t kTaskShort = (int32_t)0x80000000;

template <class Epi>
__global__ void __launch_bounds__(256) k_spmv_short(Csr A, const int32_t* __restrict__ tasks,
                                                    const int32_t* __restrict__ n_tasks,
                                                    const double* __restrict__ xv, Epi epi) {
  const int b = blockIdx.y;
  if (epi.skip(b)) return;
  const double* __restrict__ val = A.val + (int64_t)b * A.nnz;
  const double* __restrict__ x = xv + (int64_t)b * A.n_cols;
  const double xs = epi.xscale(b);
  const int lane = threadIdx.x & 31;
  const int warp0 = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  const int nwarps = (int)(((int64_t)gridDim.x * blockDim.x) >> 5);
  const int nt = *n_tasks;
  for (int ch = warp0; ch < nt; ch += nwarps) {
    const int32_t t0 = tasks[ch];
    if (!(t0 & kTaskShort)) continue;
    const int64_t rb = t0 & ~kTaskShort;
    const int64_t te = (ch + 1 < nt) ? (int64_t)(tasks[ch + 1] & ~kTaskShort) : A.n_rows;
    const int64_t myrow = rb + lane;
    if (myrow >= te) continue;
    const int64_t q0 = A.ptr[myrow], q1 = A.ptr[myrow + 1];
    const typename Epi::Pre pre = epi.pre(b, myrow);
    const int mylen = (int)(q1 - q0);
    double acc = 0.0;
    if (mylen == 2 && (q0 & 1) == 0) {
      const int2 c = __ldcs(reinterpret_cast<const int2*>(A.idx + q0));
      const double2 v = __ldcs(reinterpret_cast<const double2*>(val + q0));
      acc = v.x * x[c.x];
      acc += v.y * x[c.y];
    } else if (mylen == 4 && (q0 & 3) == 0) {
      const int4 c = __ldcs(reinterpret_cast<const int4*>(A.idx + q0));
      const double2 v01 = __ldcs(reinterpret_cast<const double2*>(val + q0));
      const double2 v23 = __ldcs(reinterpret_cast<const double2*>(val + q0 + 2));
      acc = v01.x * x[c.x];
      acc += v01.y * x[c.y];
      acc += v23.x * x[c.z];
      acc += v23.y * x[c.w];
    } else {
      for (int64_t p = q0; p < q1; ++p) acc += __ldcs(val + p) * x[__ldcs(A.idx + p)];
    }
    epi.row(b, myrow, acc * xs, pre);
  }
  epi.finalize(b);
}

template <class Epi>
__global__ void __launch_bounds__(256, 3) k_spmv_tasks(Csr A, const int32_t* __restrict__ tasks,
                                                    const int32_t* __restrict__ n_tasks,
                                                    const double* __restrict__ xv, Epi epi) {
  const int b = blockIdx.y;
  if (epi.skip(b)) return;
  const double* __restrict__ val = A.val + (int64_t)b * A.nnz;
  const double* __restrict__ x = xv + (int64_t)b * A.n_cols;
  const double xs = epi.xscale(b);
  const int lane = threadIdx.x & 31;
  const int warp0 = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  const int nwarps = (int)(((int64_t)gridDim.x * blockDim.x) >> 5);
  const int nt = *n_tasks;
  for (int ch = warp0; ch < nt; ch += nwarps) {
    const int32_t t0 = tasks[ch];
    if (t0 & kTaskShort) continue;
    const int64_t rb = t0;
    const int64_t te = (ch + 1 < nt) ? (int64_t)(tasks[ch + 1] & ~kTaskShort) : A.n_rows;
    const int nr = (int)(te - rb);
    const int64_t myrow = rb + lane;
    const bool mine = lane < nr;
    int64_t q0 = 0, q1 = 0;
    if (mine) { q0 = A.ptr[myrow]; q1 = A.ptr[myrow + 1]; }
    const int mylen = (int)(q1 - q0);
    // four rows at a time, 64 entries of each per pass: 8 index + 8 value loads of a lane are in flight
    // together, then the 8 gathers, then four shuffle reductions -- two memory round trips per four rows of
    // up to 64 entries (the C1 / C3 rows at N = 50), instead of one load -> gather chain per 32 entries.
    double myres = 0.0;
    const typename Epi::Pre pre = (mine && mylen <= kLongRow) ? epi.pre(b, myrow) : typename Epi::Pre{};
    const int64_t tbase = __shfl_sync(0xffffffffu, q0, 0);
    const int32_t* __restrict__ tidx = A.idx + tbase;
    const double* __restrict__ tval = val + tbase;
    for (int k = 0; k < nr; k += 4) {
      int p0[4], p1[4];                                 // offsets relative to the first row of the task
      int maxl = 0;
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int kk = (k + u < nr) ? k + u : k;
        p0[u] = (int)(__shfl_sync(0xffffffffu, q0, kk) - tbase);
        p1[u] = (int)(__shfl_sync(0xffffffffu, q1, kk) - tbase);
        if (k + u >= nr || p1[u] - p0[u] > kLongRow) p1[u] = p0[u];      // nothing to do for this slot
        maxl = max(maxl, p1[u] - p0[u]);
      }
      double acc[4] = {0.0, 0.0, 0.0, 0.0};
      for (int off = 0; off < maxl; off += 64) {
        int ci[8]; double vv[8];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int pa = p0[u] + off + lane, pb = pa + 32;
          const bool va = pa < p1[u], vb = pb < p1[u];
          ci[2 * u] = va ? __ldcs(tidx + pa) : 0;       ci[2 * u + 1] = vb ? __ldcs(tidx + pb) : 0;
          vv[2 * u] = va ? __ldcs(tval + pa) : 0.0;     vv[2 * u + 1] = vb ? __ldcs(tval + pb) : 0.0;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          acc[u] += vv[2 * u] * x[ci[2 * u]];
          acc[u] += vv[2 * u + 1] * x[ci[2 * u + 1]];
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const double r_ = warp_sum(acc[u]);
        if (lane == k + u) myres = r_;
      }
    }
    if (mine && mylen <= kLongRow) epi.row(b, myrow, myres * xs, pre);
  }
  epi.finalize(b);
}

// block per long row; long rows are found by a strided scan over the row list (`long_rows`,
// `n_long` written once per solve by k_find_long_rows).
template <class Epi>
__global__ void __launch_bounds__(256) k_spmv_long(Csr A, const double* __restrict__ xv,
                                                   const int32_t* __restrict__ long_rows,
                                                   const int32_t* __restrict__ n_long, Epi epi) {
  const int b = blockIdx.y;
  if (epi.skip(b)) return;
  __shared__ double sm[32];
  const double* __restrict__ val = A.val + (int64_t)b * A.nnz;
  const double* __restrict__ x = xv + (int64_t)b * A.n_cols;
  const double xs = epi.xscale(b);
  const int nl = *n_long;
  for (int k = blockIdx.x; k < nl; k += gridDim.x) {
    const int64_t row = long_rows[k];
    const int64_t p0 = A.ptr[row], p1 = A.ptr[row + 1];
    double acc = 0.0;
    int64_t p = p0 + threadIdx.x;
    for (; p + 3 * 256 < p1; p += 4 * 256) {
      int c0 = __ldcs(A.idx + p), c1 = __ldcs(A.idx + p + 256), c2 = __ldcs(A.idx + p + 512),
          c3 = __ldcs(A.idx + p + 768);
      double v0 = __ldcs(val + p), v1 = __ldcs(val + p + 256), v2 = __ldcs(val + p + 512),
             v3 = __ldcs(val + p + 768);
      acc += v0 * x[c0]; acc += v1 * x[c1]; acc += v2 * x[c2]; acc += v3 * x[c3];
    }
    for (; p < p1; p += 256) acc += __ldcs(val + p) * x[__ldcs(A.idx + p)];
    acc = block_sum(acc, sm);
    if (threadIdx.x == 0) epi.row(b, row, acc * xs, epi.pre(b, row));
  }
  epi.finalize(b);
}

// Warp tasks of the row kernel: consecutive rows whose first non-zero falls into the same bucket of
// kTaskNnz non-zeros form one task (so a task holds about kTaskNnz non-zeros whatever the row lengths;
// a row longer than a bucket is a task of its own).  tasks[t] = first row of task t.  Built once per
// solve by an ordered stream compaction (cub::DeviceSelect) -- the pattern is shared by the batch.
struct TaskStart {
  const int64_t* ptr;
  __device__ bool operator()(const int32_t& r) const {
    // a new task starts where the non-zero bucket changes, and at least every 32 rows
    return (r & 31) == 0 || (ptr[r] / kTaskNnz) != (ptr[r - 1] / kTaskNnz);
  }
};

// mark the tasks whose rows all have <= kShortRow entries (bit 31 of the start row)
__global__ void k_flag_tasks(const int64_t* __restrict__ ptr, int64_t n_rows, int32_t* __restrict__ tasks,
                             const int32_t* __restrict__ n_tasks, int32_t* __restrict__ kinds) {
  const int nt = *n_tasks;
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < nt; t += gridDim.x * blockDim.x) {
    const int64_t rb = tasks[t];          // not yet flagged: neighbours are read unflagged or masked below
    const int64_t re = (t + 1 < nt) ? (int64_t)(tasks[t + 1] & 0x7fffffff) : n_rows;
    bool sh = true;
    for (int64_t r = rb; r < re; ++r) sh = sh && (ptr[r + 1] - ptr[r] <= kShortRow);
    if (sh) { tasks[t] = (int32_t)rb | (int32_t)0x80000000; kinds[0] = 1; } else kinds[1] = 1;
  }
}

static int build_tasks(const int64_t* row_ptr, int64_t rows, int32_t* tasks, int32_t* n_tasks, int32_t* kinds,
                       cudaStream_t s) {
  cub::CountingInputIterator<int32_t> it(0);
  size_t tmp_bytes = 0;
  TaskStart pred{row_ptr};
  NEPTUNE_CUDA_OK(cub::DeviceSelect::If(nullptr, tmp_bytes, it, tasks, n_tasks, (int)rows, pred, s));
  void* tmp = nullptr;
  NEPTUNE_CUDA_OK(cudaMallocAsync(&tmp, tmp_bytes ? tmp_bytes : 8, s));
  NEPTUNE_CUDA_OK(cub::DeviceSelect::If(tmp, tmp_bytes, it, tasks, n_tasks, (int)rows, pred, s));
  NEPTUNE_COUNT(2);
  NEPTUNE_CUDA_OK(cudaFreeAsync(tmp, s));
  { k_flag_tasks<<<kNumSMs * 4, 256, 0, s>>>(row_ptr, rows, tasks, n_tasks, kinds); NEPTUNE_COUNT(1); }
  return 0;
}

__global__ void k_find_long_rows(const int64_t* __restrict__ ptr, int64_t n_rows,
                                 int32_t* __restrict__ long_rows, int32_t* __restrict__ n_long) {
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n_rows;
       r += (int64_t)gridDim.x * blockDim.x)
    if (ptr[r + 1] - ptr[r] > kLongRow) {
      int k = atomicAdd(n_long, 1);
      if (k < kMaxLongList) long_rows[k] = (int32_t)r;
    }
}

// ---------------------------------------------------------------------------------------------------
// Epilogues
// ---------------------------------------------------------------------------------------------------
struct NoPre {};
struct StoreEpi {            // plain SpMV
  typedef NoPre Pre;
  double* out; int64_t n;
  __device__ bool skip(int) const { return false; }
  __device__ double xscale(int) const { return 1.0; }
  __device__ Pre pre(int, int64_t) const { return Pre{}; }
  __device__ void row(int b, int64_t r, double v, const Pre&) const { out[(int64_t)b * n + r] = v; }
  __device__ void finalize(int) const {}
};

struct PrimalUpdate {        // per column, after g = (A^T y)[col]
  const Ctl* ctl; int64_t cols;
  const double *obj, *lb, *ub, *T;
  double *x, *xbar, *xsum;
  __device__ bool skip(int b) const { return ctl[b].converged != 0; }
  __device__ double xscale(int) const { return 1.0; }
  struct Pre { double xo, o, t, l, u, s; };
  __device__ Pre pre(int b, int64_t c) const {
    const int64_t k = (int64_t)b * cols + c;
    return Pre{x[k], obj[k], T[k], lb[k], ub[k], xsum[k]};
  }
  __device__ void row(int b, int64_t c, double g, const Pre& p) const {
    const int64_t k = (int64_t)b * cols + c;
    const double tau = ctl[b].tau;
    double xn = p.xo - tau * p.t * (p.o + g);
    xn = fmin(fmax(xn, p.l), p.u);
    x[k] = xn;
    xbar[k] = 2.0 * xn - p.xo;
    xsum[k] = p.s + xn;
  }
  __device__ void finalize(int) const {}
};

struct DualUpdate {          // per row, after a = (A xbar)[row]
  const Ctl* ctl; int64_t rows;
  const double *lo, *hi, *S;
  double *y, *ysum;
  __device__ bool skip(int b) const { return ctl[b].converged != 0; }
  __device__ double xscale(int) const { return 1.0; }
  struct Pre { double yo, sc, l, h, s; };
  __device__ Pre pre(int b, int64_t r) const {
    const int64_t k = (int64_t)b * rows + r;
    return Pre{y[k], S[k], lo[k], hi[k], ysum[k]};
  }
  __device__ void row(int b, int64_t r, double a, const Pre& p) const {
    const int64_t k = (int64_t)b * rows + r;
    const double s = ctl[b].sigma * p.sc;
    const double v = p.yo + s * a;
    const double z = fmin(fmax(v / s, p.l), p.h);
    // a free row keeps a zero multiplier exactly: v - s*(v/s) leaves rounding noise that the 1e6 coefficients of
    // the freed C1a rows amplify to ~1e-6 relative in the iterates (seen against the matrix-free solver)
    const double yn = (isinf(p.l) && isinf(p.h)) ? 0.0 : v - s * z;
    y[k] = yn;
    ysum[k] = p.s + yn;
  }
  __device__ void finalize(int) const {}
};

// KKT pieces of a candidate (current iterate or running average) -- rows side:
//   primal residual ||Ax - clip(Ax, lo, hi)||^2 and the row part of the dual objective -g*(y).
struct RowsEval {
  Ctl* ctl; int64_t rows; int which;      // which: 0 current (y), 1 average (ysum / count)
  const double *lo, *hi, *yv;
  double pres2, dobj, dres2;
  __device__ bool skip(int b) const { return ctl[b].converged != 0; }
  __device__ double xscale(int b) const { return which ? 1.0 / (double)max(ctl[b].avg_count, 1) : 1.0; }
  typedef NoPre Pre;
  __device__ Pre pre(int, int64_t) const { return Pre{}; }
  __device__ void row(int b, int64_t r, double a, const Pre&) {
    const int64_t k = (int64_t)b * rows + r;
    const double l = lo[k], h = hi[k];
    const double viol = a - fmin(fmax(a, l), h);
    pres2 += viol * viol;
    const double yy = yv[k] * xscale(b);
    if (yy > 0.0) { if (isfinite(h)) dobj -= h * yy; else dres2 += yy * yy; }
    else if (yy < 0.0) { if (isfinite(l)) dobj -= l * yy; else dres2 += yy * yy; }
  }
  __device__ void finalize(int b) {
    __shared__ double sm[32];
    double a = block_sum(pres2, sm), c = block_sum(dobj, sm), e = block_sum(dres2, sm);
    if (threadIdx.x == 0) {
      double* acc = ctl[b].acc + (which ? ACC_AVG : ACC_CUR);
      if (a != 0.0) atomicAdd(acc + PRES2, a);
      if (c != 0.0) atomicAdd(acc + DOBJ, c);
      if (e != 0.0) atomicAdd(acc + DRES2, e);
    }
  }
};

// columns side: primal objective, reduced-cost part of the dual objective, dual residual.
struct ColsEval {
  Ctl* ctl; int64_t cols; int which;
  const double *obj, *lb, *ub, *xv;
  double pobj, dobj, dres2;
  __device__ bool skip(int b) const { return ctl[b].converged != 0; }
  __device__ double xscale(int b) const { return which ? 1.0 / (double)max(ctl[b].avg_count, 1) : 1.0; }
  typedef NoPre Pre;
  __device__ Pre pre(int, int64_t) const { return Pre{}; }
  __device__ void row(int b, int64_t c, double g, const Pre&) {
    const int64_t k = (int64_t)b * cols + c;
    const double o = obj[k];
    pobj += o * xv[k] * xscale(b);
    const double rc = o + g;
    if (rc > 0.0) { const double l = lb[k]; if (isfinite(l)) dobj += l * rc; else dres2 += rc * rc; }
    else if (rc < 0.0) { const double u = ub[k]; if (isfinite(u)) dobj += u * rc; else dres2 += rc * rc; }
  }
  __device__ void finalize(int b) {
    __shared__ double sm[32];
    double a = block_sum(pobj, sm), c = block_sum(dobj, sm), e = block_sum(dres2, sm);
    if (threadIdx.x == 0) {
      double* acc = ctl[b].acc + (which ? ACC_AVG : ACC_CUR);
      if (a != 0.0) atomicAdd(acc + POBJ, a);
      if (c != 0.0) atomicAdd(acc + DOBJ, c);
      if (e != 0.0) atomicAdd(acc + DRES2, e);
    }
  }
};

// ---------------------------------------------------------------------------------------------------
// Equilibration: Ruiz (inf-norm) passes then one Pock-Chambolle (1-norm) pass, as diagonal scalings
// dr, dc applied on the fly.  One thread per column of A^T; row accumulators via atomics.
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_scale_pass(Csr At, int use_sum, const double* __restrict__ dr,
                                                    const double* __restrict__ dc, const double* __restrict__ lo,
                                                    const double* __restrict__ hi, double* __restrict__ colacc,
                                                    double* __restrict__ rowacc) {
  const int b = blockIdx.y;
  const double* __restrict__ val = At.val + (int64_t)b * At.nnz;
  const int64_t rows = At.n_cols, cols = At.n_rows;
  for (int64_t col = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; col < cols;
       col += (int64_t)gridDim.x * blockDim.x) {
    const int64_t p0 = At.ptr[col], p1 = At.ptr[col + 1];
    const double dcj = dc[(int64_t)b * cols + col];
    double acc = 0.0;
    for (int64_t p = p0; p < p1; ++p) {
      const int r = At.idx[p];
      // a free row (-inf, +inf) never gets a multiplier: it must not distort the equilibration
      if (isinf(lo[(int64_t)b * rows + r]) && isinf(hi[(int64_t)b * rows + r])) continue;
      const double mval = fabs(val[p]) * dr[(int64_t)b * rows + r] * dcj;
      if (use_sum) {
        acc += mval;
        if (mval != 0.0) atomicAdd(rowacc + (int64_t)b * rows + r, mval);
      } else {
        acc = fmax(acc, mval);
        atomicMax(reinterpret_cast<unsigned long long*>(rowacc + (int64_t)b * rows + r),
                  (unsigned long long)__double_as_longlong(mval));
      }
    }
    colacc[(int64_t)b * cols + col] = acc;
  }
}

__global__ void k_scale_update(int64_t n, double* __restrict__ dvec, double* __restrict__ acc) {
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n;
       k += (int64_t)gridDim.x * blockDim.x) {
    const double a = acc[k];
    if (a > 0.0) dvec[k] *= rsqrt(a);
    acc[k] = 0.0;
  }
}

__global__ void k_fill(int64_t n, double* __restrict__ v, double a) {
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n;
       k += (int64_t)gridDim.x * blockDim.x) v[k] = a;
}

__global__ void k_square(int64_t n, double* __restrict__ v) {
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n;
       k += (int64_t)gridDim.x * blockDim.x) v[k] = v[k] * v[k];
}

// ||finite bounds||^2 in the scaled space (per instance) for omega0 and the relative tolerances.
__global__ void __launch_bounds__(256) k_norms(int64_t rows, int64_t cols, const double* __restrict__ lo,
                                               const double* __restrict__ hi, const double* __restrict__ obj,
                                               const double* __restrict__ S, const double* __restrict__ T,
                                               Ctl* ctl) {
  const int b = blockIdx.y;
  __shared__ double sm[32];
  double nb = 0.0, nc = 0.0, nbs = 0.0, ncs = 0.0;
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < rows;
       r += (int64_t)gridDim.x * blockDim.x) {
    const double l = lo[(int64_t)b * rows + r], h = hi[(int64_t)b * rows + r];
    double m = 0.0;
    if (isfinite(l)) m = fabs(l);
    if (isfinite(h)) m = fmax(m, fabs(h));
    nb += m * m;
    nbs += m * m * S[(int64_t)b * rows + r];
  }
  for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < cols;
       c += (int64_t)gridDim.x * blockDim.x) {
    const double o = obj[(int64_t)b * cols + c];
    nc += o * o;
    ncs += o * o * T[(int64_t)b * cols + c];
  }
  nb = block_sum(nb, sm);
  nc = block_sum(nc, sm);
  nbs = block_sum(nbs, sm);
  ncs = block_sum(ncs, sm);
  if (threadIdx.x == 0) {
    if (nb != 0.0) atomicAdd(&ctl[b].acc[ACC_NB2], nb);
    if (nc != 0.0) atomicAdd(&ctl[b].acc[ACC_NC2], nc);
    if (nbs != 0.0) atomicAdd(&ctl[b].acc[ACC_NBS2], nbs);
    if (ncs != 0.0) atomicAdd(&ctl[b].acc[ACC_NCS2], ncs);
  }
}

// Apply the decision: x,y <- average (action 1) or keep current (2); reset sums; measure the
// movement since the last restart point (for the primal-weight update).
__global__ void __launch_bounds__(256) k_apply_restart(int64_t n, int is_primal, Ctl* ctl,
                                                       double* __restrict__ v, double* __restrict__ vsum,
                                                       double* __restrict__ vrestart,
                                                       const double* __restrict__ diag) {
  const int b = blockIdx.y;
  const int action = ctl[b].action;
  if (action == 0) return;
  __shared__ double sm[32];
  const double inv = 1.0 / (double)max(ctl[b].avg_count, 1);
  double d2 = 0.0;
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n;
       k += (int64_t)gridDim.x * blockDim.x) {
    const int64_t q = (int64_t)b * n + k;
    double nv = (action == 1) ? vsum[q] * inv : v[q];
    const double dlt = nv - vrestart[q];
    d2 += dlt * dlt / diag[q];                       // scaled-space norm
    v[q] = nv; vrestart[q] = nv; vsum[q] = 0.0;
  }
  d2 = block_sum(d2, sm);
  if (threadIdx.x == 0 && d2 != 0.0) atomicAdd(&ctl[b].acc[is_primal ? ACC_DX2 : ACC_DY2], d2);
}

static inline int grid1(int64_t work, int threads, int per_sm) {
  int64_t g = ceil_div(work, threads);
  int64_t cap = (int64_t)kNumSMs * per_sm;
  if (g > cap) g = cap;
  return (int)(g < 1 ? 1 : g);
}

struct Side {              // one matrix (A or A^T) with its launch schedule
  Csr M;
  int32_t* tasks; int32_t* n_tasks;       // warp tasks (device)
  int32_t* long_rows; int32_t* n_long;    // rows longer than kLongRow (device list)
  int n_long_h;                           // ... and their number on the host (0: that launch is skipped)
  int has_short, has_wide;                // which task kinds exist (a launch without work is skipped)
};

struct Plan {
  int B; int64_t rows, cols, nnz;
  Side A, At;
  cudaStream_t s;
};

template <class Epi>
static void launch_side(const Plan& P, const Side& S, const double* v, Epi epi) {
  dim3 g(grid1(S.M.n_rows, 256, 16), P.B);     // warps stride over the task list
  if (S.has_short) { k_spmv_short<Epi><<<g, 256, 0, P.s>>>(S.M, S.tasks, S.n_tasks, v, epi); NEPTUNE_COUNT(1); }
  if (S.has_wide) { k_spmv_tasks<Epi><<<g, 256, 0, P.s>>>(S.M, S.tasks, S.n_tasks, v, epi); NEPTUNE_COUNT(1); }
  if (S.n_long_h > 0) {
    dim3 gl(S.n_long_h < kNumSMs * 2 ? S.n_long_h : kNumSMs * 2, P.B);
    { k_spmv_long<Epi><<<gl, 256, 0, P.s>>>(S.M, v, S.long_rows, S.n_long, epi); NEPTUNE_COUNT(1); }
  }
}
template <class Epi> static void launch_rows(const Plan& P, const double* xv, Epi epi) { launch_side(P, P.A, xv, epi); }
template <class Epi> static void launch_cols(const Plan& P, const double* yv, Epi epi) { launch_side(P, P.At, yv, epi); }

// pattern analysis of one matrix: warp tasks + long-row list (device scratch carved from `mem`)
static size_t side_scratch_bytes(int64_t n_rows) { return (size_t)(n_rows + 2) * 4 + (size_t)kMaxLongList * 4 + 512; }

static int analyse_side(Side& S, char* mem, cudaStream_t s) {
  S.tasks = (int32_t*)mem; mem += (((size_t)(S.M.n_rows + 2) * 4 + 255) & ~(size_t)255);
  S.long_rows = (int32_t*)mem; mem += (size_t)kMaxLongList * 4;
  S.n_tasks = (int32_t*)mem; S.n_long = S.n_tasks + 1;
  int32_t* kinds = S.n_tasks + 2;
  NEPTUNE_CUDA_OK(cudaMemsetAsync(S.n_tasks, 0, 16, s));
  { int rc = build_tasks(S.M.ptr, S.M.n_rows, S.tasks, S.n_tasks, kinds, s); if (rc) return rc; }
  { k_find_long_rows<<<grid1(S.M.n_rows, 256, 8), 256, 0, s>>>(S.M.ptr, S.M.n_rows, S.long_rows, S.n_long); NEPTUNE_COUNT(1); }
  int h[3] = {0, 0, 0};
  NEPTUNE_CUDA_OK(cudaMemcpyAsync(h, S.n_long, 12, cudaMemcpyDeviceToHost, s));
  NEPTUNE_CUDA_OK(cudaStreamSynchronize(s));
  S.n_long_h = h[0] < kMaxLongList ? h[0] : kMaxLongList;
  S.has_short = h[1]; S.has_wide = h[2];
  return 0;
}

static inline size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

}  // namespace neptune

using namespace neptune;

extern "C" int neptune_pdhg_workspace_bytes(int B, int64_t rows, int64_t cols, int64_t nnz, int64_t* bytes) {
  if (B <= 0 || rows <= 0 || cols <= 0 || !bytes) return NEPTUNE_E_ARG;
  (void)nnz;
  size_t t = 0;
  t += 5 * align256((size_t)B * cols * 8);     // xbar, xsum, xrestart, T(dc), colacc
  t += 4 * align256((size_t)B * rows * 8);     // ysum, yrestart, S(dr), rowacc
  t += align256((size_t)B * sizeof(Ctl));
  t += align256(side_scratch_bytes(rows)) + align256(side_scratch_bytes(cols));
  t += 1024;
  *bytes = (int64_t)t;
  return 0;
}

static int nnz_of(const int64_t* ptr, int64_t n, int64_t* nnz, cudaStream_t s) {
  NEPTUNE_CUDA_OK(cudaMemcpyAsync(nnz, ptr + n, 8, cudaMemcpyDeviceToHost, s));
  NEPTUNE_CUDA_OK(cudaStreamSynchronize(s));
  return 0;
}

extern "C" int neptune_spmv(int B, int64_t rows, int64_t cols, const int64_t* row_ptr, const int32_t* col_idx,
                            const double* val, const double* x, double* out, void* stream) {
  if (B <= 0 || rows <= 0 || cols <= 0 || !row_ptr || !col_idx || !val || !x || !out) return NEPTUNE_E_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  int64_t nnz = 0;
  { int rc = nnz_of(row_ptr, rows, &nnz, s); if (rc) return rc; }
  char* tmp = nullptr;
  NEPTUNE_CUDA_OK(cudaMallocAsync(&tmp, side_scratch_bytes(rows), s));
  Plan P{};
  P.B = B; P.rows = rows; P.cols = cols; P.nnz = nnz; P.s = s;
  P.A.M = Csr{row_ptr, col_idx, val, rows, cols, nnz};
  { int rc = analyse_side(P.A, tmp, s); if (rc) return rc; }
  launch_rows(P, x, StoreEpi{out, rows});
  NEPTUNE_LAUNCH_OK();
  NEPTUNE_CUDA_OK(cudaFreeAsync(tmp, s));
  return 0;
}

extern "C" int neptune_spmv_t(int B, int64_t rows, int64_t cols, const int64_t* rowT_ptr,
                              const int32_t* colT_idx, const double* valT, const double* y, double* out,
                              void* stream) {
  if (B <= 0 || rows <= 0 || cols <= 0 || !rowT_ptr || !colT_idx || !valT || !y || !out) return NEPTUNE_E_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  int64_t nnz = 0;
  { int rc = nnz_of(rowT_ptr, cols, &nnz, s); if (rc) return rc; }
  char* tmp = nullptr;
  NEPTUNE_CUDA_OK(cudaMallocAsync(&tmp, side_scratch_bytes(cols), s));
  Plan P{};
  P.B = B; P.rows = rows; P.cols = cols; P.nnz = nnz; P.s = s;
  P.At.M = Csr{rowT_ptr, colT_idx, valT, cols, rows, nnz};
  { int rc = analyse_side(P.At, tmp, s); if (rc) return rc; }
  launch_cols(P, y, StoreEpi{out, cols});
  NEPTUNE_LAUNCH_OK();
  NEPTUNE_CUDA_OK(cudaFreeAsync(tmp, s));
  return 0;
}

extern "C" int neptune_pdhg_solve(int B, int64_t rows, int64_t cols, int64_t nnz, const int64_t* row_ptr,
                                  const int32_t* col_idx, const double* val, const int64_t* rowT_ptr,
                                  const int32_t* colT_idx, const double* valT, const double* obj,
                                  const double* lo, const double* hi, const double* col_lb,
                                  const double* col_ub, const neptune_pdhg_params* prm, double* x, double* y,
                                  neptune_pdhg_result* result_d, void* workspace, int64_t workspace_bytes,
                                  void* stream) {
  if (B <= 0 || rows <= 0 || cols <= 0 || nnz <= 0) return NEPTUNE_E_ARG;
  if (!row_ptr || !col_idx || !val || !rowT_ptr || !colT_idx || !valT || !obj || !lo || !hi || !col_lb ||
      !col_ub || !prm || !x || !y || !result_d || !workspace)
    return NEPTUNE_E_ARG;
  int64_t need = 0;
  neptune_pdhg_workspace_bytes(B, rows, cols, nnz, &need);
  if (workspace_bytes < need) return NEPTUNE_E_NOMEM;
  // work on an internal stream (the caller's may be the legacy default stream, which cannot be
  // captured into a graph); ordered after / before the caller's stream with events
  cudaStream_t caller = (cudaStream_t)stream;
  cudaStream_t s = nullptr;
  cudaEvent_t ev_in = nullptr, ev_out = nullptr;
  NEPTUNE_CUDA_OK(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
  NEPTUNE_CUDA_OK(cudaEventCreateWithFlags(&ev_in, cudaEventDisableTiming));
  NEPTUNE_CUDA_OK(cudaEventCreateWithFlags(&ev_out, cudaEventDisableTiming));
  NEPTUNE_CUDA_OK(cudaEventRecord(ev_in, caller));
  NEPTUNE_CUDA_OK(cudaStreamWaitEvent(s, ev_in, 0));
  const int check_every = prm->check_every > 0 ? prm->check_every : 64;
  const int max_iters = prm->max_iters > 0 ? prm->max_iters : 20000;

  // carve the workspace
  char* p = (char*)workspace;
  auto take = [&](size_t bytes) { char* q = p; p += align256(bytes); return q; };
  const size_t cb = (size_t)B * cols * 8, rb = (size_t)B * rows * 8;
  double* xbar = (double*)take(cb); double* xsum = (double*)take(cb); double* xres = (double*)take(cb);
  double* T = (double*)take(cb); double* colacc = (double*)take(cb);
  double* ysum = (double*)take(rb); double* yres = (double*)take(rb);
  double* S = (double*)take(rb); double* rowacc = (double*)take(rb);
  Ctl* ctl = (Ctl*)take((size_t)B * sizeof(Ctl));
  char* scrA = take(side_scratch_bytes(rows));
  char* scrT = take(side_scratch_bytes(cols));

  Csr A{row_ptr, col_idx, val, rows, cols, nnz};
  Csr At{rowT_ptr, colT_idx, valT, cols, rows, nnz};

  // one-off analysis of the (batch-shared) pattern: warp tasks and long-row lists of both copies
  Plan P{};
  P.B = B; P.rows = rows; P.cols = cols; P.nnz = nnz; P.s = s;
  P.A.M = A; P.At.M = At;
  { int rc = analyse_side(P.A, scrA, s); if (rc) return rc; }
  { int rc = analyse_side(P.At, scrT, s); if (rc) return rc; }

  // equilibration: dr = S, dc = T hold the scalings, squared at the end
  const int g_c = grid1((int64_t)B * cols, 256, 16), g_r = grid1((int64_t)B * rows, 256, 16);
  { k_fill<<<g_c, 256, 0, s>>>((int64_t)B * cols, T, 1.0); NEPTUNE_COUNT(1); }
  { k_fill<<<g_r, 256, 0, s>>>((int64_t)B * rows, S, 1.0); NEPTUNE_COUNT(1); }
  NEPTUNE_CUDA_OK(cudaMemsetAsync(rowacc, 0, rb, s));
  NEPTUNE_CUDA_OK(cudaMemsetAsync(colacc, 0, cb, s));
  const int ruiz = prm->ruiz_iters >= 0 ? prm->ruiz_iters : 10;
  for (int it = 0; it <= ruiz; ++it) {
    const int use_sum = (it == ruiz);           // last pass: Pock-Chambolle alpha = 1
    dim3 g(grid1(cols, 256, 16), B);
    { k_scale_pass<<<g, 256, 0, s>>>(At, use_sum, S, T, lo, hi, colacc, rowacc); NEPTUNE_COUNT(1); }
    { k_scale_update<<<g_c, 256, 0, s>>>((int64_t)B * cols, T, colacc); NEPTUNE_COUNT(1); }
    { k_scale_update<<<g_r, 256, 0, s>>>((int64_t)B * rows, S, rowacc); NEPTUNE_COUNT(1); }
  }
  { k_square<<<g_c, 256, 0, s>>>((int64_t)B * cols, T); NEPTUNE_COUNT(1); }
  { k_square<<<g_r, 256, 0, s>>>((int64_t)B * rows, S); NEPTUNE_COUNT(1); }

  // control block, norms, initial state
  NEPTUNE_CUDA_OK(cudaMemsetAsync(ctl, 0, (size_t)B * sizeof(Ctl), s));
  {
    dim3 g(grid1(cols > rows ? cols : rows, 256, 4), B);
    { k_norms<<<g, 256, 0, s>>>(rows, cols, lo, hi, obj, S, T, ctl); NEPTUNE_COUNT(1); }
  }
  { k_ctl_init<<<(B + 127) / 128, 128, 0, s>>>(B, ctl, 0.99); NEPTUNE_COUNT(1); }
  NEPTUNE_CUDA_OK(cudaMemsetAsync(xsum, 0, cb, s));
  NEPTUNE_CUDA_OK(cudaMemsetAsync(ysum, 0, rb, s));
  NEPTUNE_CUDA_OK(cudaMemcpyAsync(xres, x, cb, cudaMemcpyDeviceToDevice, s));
  NEPTUNE_CUDA_OK(cudaMemcpyAsync(yres, y, rb, cudaMemcpyDeviceToDevice, s));
  NEPTUNE_LAUNCH_OK();

  int* d_flag = nullptr; int h_flag = 0;
  NEPTUNE_CUDA_OK(cudaMallocAsync(&d_flag, 4, s));

  PrimalUpdate pu{ctl, cols, obj, col_lb, col_ub, T, x, xbar, xsum};
  DualUpdate du{ctl, rows, lo, hi, S, y, ysum};
  // The inner loop is launch-bound for small batches and exposed to host jitter otherwise: `inner`
  // iterations (2-6 launches each) are captured once into a CUDA graph and replayed; step sizes, restart
  // flags and convergence live in device memory (Ctl), so the graph never changes.
  const int inner = check_every < 32 ? check_every : 32;
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t gexec = nullptr;
  int64_t per_graph = 0;
  {
    int64_t c0 = 0, c1 = 0;
    neptune_launch_count(&c0, 0);
    NEPTUNE_CUDA_OK(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
    for (int k = 0; k < inner; ++k) {
      launch_cols(P, y, pu);
      launch_rows(P, xbar, du);
    }
    NEPTUNE_CUDA_OK(cudaStreamEndCapture(s, &graph));
    NEPTUNE_CUDA_OK(cudaGraphInstantiate(&gexec, graph, 0));
    neptune_launch_count(&c1, 0);
    per_graph = c1 - c0;
    NEPTUNE_COUNT(-per_graph);                      // the capture itself ran nothing
  }
  for (int it = 0; it < max_iters && !h_flag; it += check_every) {
    int done = 0;
    for (; done + inner <= check_every; done += inner) {
      NEPTUNE_CUDA_OK(cudaGraphLaunch(gexec, s));
      NEPTUNE_COUNT(per_graph);
    }
    for (; done < check_every; ++done) {
      launch_cols(P, y, pu);
      launch_rows(P, xbar, du);
    }
    { k_ctl_advance<<<(B + 127) / 128, 128, 0, s>>>(B, ctl, check_every); NEPTUNE_COUNT(1); }
    // KKT of the current iterate and of the running average
    for (int w = 0; w < 2; ++w) {
      launch_rows(P, w ? xsum : x, RowsEval{ctl, rows, w, lo, hi, w ? ysum : y, 0.0, 0.0, 0.0});
      launch_cols(P, w ? ysum : y, ColsEval{ctl, cols, w, obj, col_lb, col_ub, w ? xsum : x, 0.0, 0.0, 0.0});
    }
    { k_ctl_decide<<<(B + 127) / 128, 128, 0, s>>>(B, ctl, check_every, prm->eps_abs, prm->eps_rel, max_iters,
                                                 result_d); NEPTUNE_COUNT(1); }
    {
      dim3 gc(grid1(cols, 256, 8), B), gr(grid1(rows, 256, 8), B);
      { k_apply_restart<<<gc, 256, 0, s>>>(cols, 1, ctl, x, xsum, xres, T); NEPTUNE_COUNT(1); }
      { k_apply_restart<<<gr, 256, 0, s>>>(rows, 0, ctl, y, ysum, yres, S); NEPTUNE_COUNT(1); }
    }
    { k_ctl_after_restart<<<(B + 127) / 128, 128, 0, s>>>(B, ctl); NEPTUNE_COUNT(1); }
    { k_all_done<<<1, 32, 0, s>>>(B, ctl, d_flag); NEPTUNE_COUNT(1); }
    NEPTUNE_CUDA_OK(cudaMemcpyAsync(&h_flag, d_flag, 4, cudaMemcpyDeviceToHost, s));
    NEPTUNE_CUDA_OK(cudaStreamSynchronize(s));
  }
  cudaGraphExecDestroy(gexec);
  cudaGraphDestroy(graph);
  NEPTUNE_LAUNCH_OK();
  NEPTUNE_CUDA_OK(cudaFreeAsync(d_flag, s));
  NEPTUNE_CUDA_OK(cudaEventRecord(ev_out, s));
  NEPTUNE_CUDA_OK(cudaStreamWaitEvent(caller, ev_out, 0));
  NEPTUNE_CUDA_OK(cudaStreamSynchronize(s));
  cudaEventDestroy(ev_in); cudaEventDestroy(ev_out);
  cudaStreamDestroy(s);
  return 0;
}
