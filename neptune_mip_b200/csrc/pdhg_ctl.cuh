// pdhg_ctl.cuh -- per-instance control block of the restarted matrix-free PDHG (pdhg_mf.cu; its numpy statement
// is tests/mf_reference.solve_ctl) and the one-thread-per-instance kernels that take the restart / termination
// decisions on the device (PDLP's KKT-error criteria).  Step sizes, restart flags and convergence live in
// device memory so that the iteration kernels can be replayed from a CUDA graph.
#pragma once
#include "common.cuh"

namespace neptune {

enum Acc { PRES2 = 0, DRES2, POBJ, DOBJ, NACC_PER = 4 };
enum { ACC_CUR = 0, ACC_AVG = NACC_PER, ACC_DX2 = 2 * NACC_PER, ACC_DY2, ACC_NB2, ACC_NC2, ACC_NBS2, ACC_NCS2, NACC };

struct Ctl {
  double tau, sigma, eta, omega;
  double kkt_restart, kkt_prev;
  double norm_b, norm_c;
  double acc[NACC];
  double best[6];                   // reported numbers of the chosen iterate
  int iters, since_restart, restarts, converged;
  int action, avg_count, use_avg, pad;
};

static __global__ void k_ctl_init(int B, Ctl* ctl, double eta) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  Ctl& c = ctl[b];
  c.norm_b = sqrt(c.acc[ACC_NB2]);
  c.norm_c = sqrt(c.acc[ACC_NC2]);
  c.eta = eta;
  // PDLP's initial primal weight ||c|| / ||b||, taken in the equilibrated space
  const double nbs = sqrt(c.acc[ACC_NBS2]), ncs = sqrt(c.acc[ACC_NCS2]);
  c.omega = (nbs > 1e-10 && ncs > 1e-10) ? ncs / nbs : 1.0;
  c.tau = c.eta / c.omega;
  c.sigma = c.eta * c.omega;
  c.kkt_restart = INFINITY; c.kkt_prev = INFINITY;
  for (int k = 0; k < NACC; ++k) c.acc[k] = 0.0;
  for (int k = 0; k < 6; ++k) c.best[k] = 0.0;
  c.iters = 0; c.since_restart = 0; c.restarts = 0; c.converged = 0;
  c.action = 0; c.avg_count = 0; c.use_avg = 0;
}

static __global__ void k_ctl_zero(int B, Ctl* ctl) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b < B) for (int k = 0; k < NACC; ++k) ctl[b].acc[k] = 0.0;
}

// Count the iterations of the chunk that just ran.  Launched BEFORE the KKT evaluation passes: they scale the
// running sums by 1 / avg_count, which must already include the chunk (counting it only in k_ctl_decide made
// the averaged candidate look `check_every` times too large at the first check after every restart, so the
// average was almost never the restart point -- found against the numpy statement of the iteration).
static __global__ void k_ctl_advance(int B, Ctl* ctl, int did_iters) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  Ctl& c = ctl[b];
  if (c.converged) return;
  c.iters += did_iters; c.since_restart += did_iters; c.avg_count += did_iters;
}

// Restart / termination decision, one thread per instance (PDLP's KKT-error criteria:
// sufficient decay 0.2, necessary decay 0.8 + no progress, artificial restart at 36 % of the run).
static __global__ void k_ctl_decide(int B, Ctl* ctl, int did_iters, double eps_abs, double eps_rel, int max_iters,
                             neptune_pdhg_result* res) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  Ctl& c = ctl[b];
  if (c.converged) return;
  double kkt[2]; bool ok[2];
  for (int w = 0; w < 2; ++w) {
    const double* a = c.acc + (w ? ACC_AVG : ACC_CUR);
    const double pres = sqrt(a[PRES2]), dres = sqrt(a[DRES2]);
    const double gap = fabs(a[POBJ] - a[DOBJ]);
    kkt[w] = sqrt(c.omega * c.omega * a[PRES2] + a[DRES2] / (c.omega * c.omega) + gap * gap);
    ok[w] = pres <= eps_abs + eps_rel * c.norm_b && dres <= eps_abs + eps_rel * c.norm_c &&
            gap <= eps_abs + eps_rel * (fabs(a[POBJ]) + fabs(a[DOBJ]));
  }
  const int pick = (ok[1] && !ok[0]) ? 1 : ((ok[0] && !ok[1]) ? 0 : (kkt[1] < kkt[0] ? 1 : 0));
  const double* a = c.acc + (pick ? ACC_AVG : ACC_CUR);
  const bool done = ok[0] || ok[1];
  const bool last = done || c.iters >= max_iters;
  // restart logic on the better candidate
  int action = 0;
  const double cand = kkt[pick];
  if (!last) {
    if (cand <= 0.2 * c.kkt_restart) action = 1 + (pick == 0);
    else if (cand <= 0.8 * c.kkt_restart && cand > c.kkt_prev) action = 1 + (pick == 0);
    else if (c.since_restart >= 0.36 * c.iters && c.iters > 0 && c.restarts > 0) action = 1 + (pick == 0);
    else if (c.restarts == 0 && c.since_restart >= 4 * did_iters) action = 1 + (pick == 0);
  }
  c.kkt_prev = cand;
  if (action) { c.kkt_restart = cand; c.restarts += 1; }
  c.action = action;
  if (last) {
    c.converged = done ? 1 : 2;
    c.use_avg = pick;
    c.action = pick ? 1 : 0;       // materialise the average into x, y if it is the better iterate
  }
  neptune_pdhg_result& r = res[b];
  r.primal_obj = a[POBJ]; r.dual_obj = a[DOBJ];
  r.primal_res = sqrt(a[PRES2]); r.dual_res = sqrt(a[DRES2]);
  r.gap = fabs(a[POBJ] - a[DOBJ]);
  r.step = c.eta; r.primal_weight = c.omega;
  r.iters = c.iters; r.restarts = c.restarts; r.converged = done ? 1 : 0; r.pad = 0;
  for (int k = 0; k < NACC; ++k) c.acc[k] = 0.0;
}

static __global__ void k_ctl_after_restart(int B, Ctl* ctl) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  Ctl& c = ctl[b];
  if (c.action == 0) return;
  if (c.converged == 0) {
    const double dx = sqrt(c.acc[ACC_DX2]), dy = sqrt(c.acc[ACC_DY2]);
    if (dx > 1e-10 && dy > 1e-10 && isfinite(dx) && isfinite(dy)) {
      // PDLP's smoothed update, limited to a factor 2 per restart (early restarts see dy >> dx
      // and would otherwise throw the weight off by orders of magnitude)
      const double nw = exp(0.5 * log(dy / dx) + 0.5 * log(c.omega));
      c.omega = fmin(fmax(nw, 0.5 * c.omega), 2.0 * c.omega);
    }
    c.tau = c.eta / c.omega; c.sigma = c.eta * c.omega;
  }
  c.since_restart = 0; c.avg_count = 0; c.action = 0;
  c.acc[ACC_DX2] = 0.0; c.acc[ACC_DY2] = 0.0;
}

// one warp (a single thread walking B control blocks was 136 us at B = 296 once most instances had converged)
static __global__ void k_all_done(int B, const Ctl* ctl, int* flag) {
  const int lane = threadIdx.x & 31;
  int done = 1;
  for (int b = lane; b < B; b += 32) if (!ctl[b].converged) done = 0;
  done = __all_sync(0xffffffffu, done);
  if (lane == 0) *flag = done;
}

}  // namespace neptune
