/* neptune_b200.h -- C ABI of libneptune_b200.so (hand-written sm_100a kernels for NEPTUNE's
 * function/request placement MIP).
 *
 * The reference (Alessandro-Mosconi/neptune-mip) has no FFI of its own: its solve path is Python
 * calling OR-Tools' `pywraplp` (SWIG) variable by variable.  Each entry point below replaces one
 * stage of that path; the reference interface it stands in for is cited as file:line relative to
 * the reference tree.  The reference-facing plugin (Python classes with the reference's names,
 * `neptune_mip_b200/core/solvers`) binds these with ctypes -- see INTEGRATION.md.
 *
 * Conventions
 *   - every function returns int: 0 ok, <0 invalid argument (NEPTUNE_E_*), >0 a cudaError_t.
 *   - `*_d` / unmarked pointers are DEVICE pointers (borrowed, never freed here);
 *     `*_h` pointers are HOST pointers.  `stream` is a cudaStream_t passed as void*.
 *   - matrices are row-major float64 unless noted:  d[N][N]  node_delay_matrix (i -> j),
 *     w[F][N] workload_matrix, r[F][N] core_per_req_matrix, m[F] function_memory_matrix,
 *     Mj[N] node_memory_matrix, Kj[N] node_cores_matrix, old[F][N] old_allocations_matrix,
 *     maxd[F] max_delay_matrix, cost[N] node_costs  (reference `core/utils/data.py:5-26`).
 *   - batched calls take B same-shaped instances: every per-instance array gains a leading
 *     dimension B (dense, no padding).  The CSR *pattern* (row_ptr/col_idx) is identical for
 *     same-shaped instances and is stored once; values are per instance.
 *   - no global state; re-entrant per stream; no host allocation is returned to the caller.
 */
#ifndef NEPTUNE_B200_H
#define NEPTUNE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NEPTUNE_ABI_VERSION 1

/* objective / model kind (reference classes NeptuneStep1CPUMinDelay / ...MinUtilization /
 * ...MinDelayAndUtilization, `core/solvers/neptune/neptune_step1.py:38-77`; same numbering is used
 * for EfttcStep1CPU*, `core/solvers/efttc/efttc_step1.py:344-441`) */
#define NEPTUNE_KIND_MIN_DELAY      0
#define NEPTUNE_KIND_MIN_UTIL       1
#define NEPTUNE_KIND_MIN_DELAY_UTIL 2

/* assembly flags */
#define NEPTUNE_FLAG_STRENGTHEN 1   /* append the valid rows x[i,f,j] - c[f,j] <= 0 (NOT in the reference
                                        matrix; kept after every reference row, see DESIGN.md) */

#define NEPTUNE_E_ARG     (-1)
#define NEPTUNE_E_SIZE    (-2)   /* index does not fit the ABI's integer widths */
#define NEPTUNE_E_NOMEM   (-3)   /* caller-provided workspace too small */

/* feasibility bits of neptune_check_solution / neptune_eval_placements: bit set <=> check passed
 * (reference `core/solvers/efttc/utils/constraints_step1.py`: c<->x :5-18, memory :22-33,
 * handle_all_requests :37-47, CPU :70-80, n<->c :85-95, budget :126-133) */
#define NEPTUNE_OK_C_X      1
#define NEPTUNE_OK_MEMORY   2
#define NEPTUNE_OK_HANDLE   4
#define NEPTUNE_OK_CPU      8
#define NEPTUNE_OK_N_C     16
#define NEPTUNE_OK_BUDGET  32
#define NEPTUNE_OK_ALL     63

int neptune_abi_version(void);

/* ---- (a) model assembly ------------------------------------------------------------------------
 * Replaces the Python model builders: init_x/init_c/init_n (`neptune/utils/variables.py:4-17`),
 * constrain_c_according_to_x / constrain_memory_usage / constrain_handle_all_requests /
 * constrain_CPU_usage / constrain_n_according_to_c / constrain_budget
 * (`neptune/utils/constraints_step1.py:5-103`) and minimize_network_delay /
 * minimize_node_utilization / minimize_node_delay_and_utilization (`neptune/utils/objectives.py:4-52`).
 * Canonical layout: columns x[i,f,j] -> f*N*N+i*N+j, c[f,j] -> F*N*N+f*N+j, n[j] -> F*N*N+F*N+j;
 * rows C1a/C1b interleaved (f,j) | C2 (j) | C3 (f,i) | C4 (j) | C5a/C5b interleaved (j) | C6 (j)
 * [| S (f,i,j) with NEPTUNE_FLAG_STRENGTHEN].  The result is bit-identical to what the reference's
 * own code hands to pywraplp (tests/test_assemble_gpu.py). */
int neptune_model_sizes(int N, int F, int kind, int flags,
                        int64_t* rows, int64_t* cols, int64_t* nnz);

/* Shared CSR pattern of A and of A^T (any pointer may be NULL to skip that output).
 * row_ptr[rows+1], col_idx[nnz], rowT_ptr[cols+1], colT_idx[nnz] (row ids of A, ascending). */
int neptune_assemble_pattern(int N, int F, int kind, int flags,
                             int64_t* row_ptr, int32_t* col_idx,
                             int64_t* rowT_ptr, int32_t* colT_idx, void* stream);

/* Per-instance numbers: val[B][nnz], valT[B][nnz], obj[B][cols], lo/hi[B][rows],
 * col_lb/col_ub[B][cols], col_int[cols] (0/1, shared), wmax[B] (the reference's
 * max_workload_delay, objectives.py:36-44; written for every kind).  NULL skips an output. */
int neptune_assemble_values(int B, int N, int F, int kind, int flags, double alpha,
                            const double* d, const double* w, const double* r, const double* m,
                            const double* Mj, const double* Kj, const double* maxd,
                            const double* cost, double budget,
                            double* val, double* valT, double* obj, double* lo, double* hi,
                            double* col_lb, double* col_ub, uint8_t* col_int, double* wmax,
                            void* stream);

/* ---- (b) PDHG LP relaxation ----------------------------------------------------------------------
 * Replaces the LP work inside `pywraplp.Solver.Solve()` (`core/solvers/solver.py:37`).
 * Diagonally preconditioned, restarted, averaged PDHG on  min obj.x  s.t. lo <= A x <= hi,
 * lb <= x <= ub, for B same-shaped instances at once.  The entry points below never store A: they
 * regenerate its coefficients from the instance arrays. */
typedef struct neptune_pdhg_params {
  int     max_iters;        /* hard cap on PDHG iterations */
  int     check_every;      /* iterations between KKT evaluations / restart decisions */
  int     ruiz_iters;       /* unused; pass 0 */
  int     reserved;         /* 0.  neptune_pdhg_mf_solve reads it as switches for measurements and tests:
                             * bit 0 = force the 8-byte iteration pass, bits 4..6 = tool diagnostics,
                             * bits 8..10 = rows of a warp in flight (0 = default), bit 11 = register passes whatever the
                             * default, bit 12 = bulk-copy (cp.async.bulk) staged pass, bit 13 = the same with the running
                             * sums by bulk reduction (even N <= 64; other shapes ignore both), bits 14..18 = its consumer
                             * warps, bits 19..22 = cap on its stages, bit 23 = keep the small-vector update of the
                             * bulk pass in its own launches */
  double  eps_rel;          /* termination: relative KKT tolerance */
  double  eps_abs;
} neptune_pdhg_params;

typedef struct neptune_pdhg_result {  /* one per instance, written to device memory */
  double primal_obj;        /* obj . x  of the returned iterate */
  double dual_obj;          /* Lagrangian bound of the returned iterate */
  double primal_res;        /* ||Ax - proj_[lo,hi](Ax)||_2  */
  double dual_res;          /* ||obj + A^T y - proj(reduced costs)||_2 */
  double gap;               /* |primal_obj - dual_obj| */
  double step;              /* final eta */
  double primal_weight;     /* final omega */
  int32_t iters;            /* iterations done */
  int32_t restarts;
  int32_t converged;        /* 1 iff tolerances met */
  int32_t pad;
} neptune_pdhg_result;

/* ---- (b, matrix-free) PDHG without the matrix -------------------------------------------------------
 * The LP relaxation of the STRENGTHENED min-delay model (what neptune_assemble_* builds with kind =
 * NEPTUNE_KIND_MIN_DELAY, flags = NEPTUNE_FLAG_STRENGTHEN: rows of `neptune/utils/constraints_step1.py:5-65`
 * with the C1a rows free, plus x[i,f,j] <= c[f,j] and x <= 1; objective `objectives.py:4-11`), solved with
 * Pock-Chambolle diagonal step sizes (1 / sum_i |A_ij| per column times eta / omega, 1 / sum_j |A_ij| per non-free
 * row times eta * omega; eta = 0.99, omega the primal weight) and PDLP's KKT restart criteria (csrc/pdhg_ctl.cuh).
 * Every coefficient is regenerated from d, w, r, m instead of being read from CSR arrays: one streaming pass over
 * x / yS and their running sums per iteration.  x[B][cols], y[B][rows] are the canonical vectors of that model (in/out, warm
 * start; the multipliers of the free C1a rows are returned as 0).  Other kinds return NEPTUNE_E_ARG. */
int neptune_pdhg_mf_workspace_bytes(int B, int N, int F, int64_t* bytes);
/* host-only: tile geometry of the passes for (B, N, F); out[16] (see csrc/pdhg_mf.cu) */
int neptune_pdhg_mf_geometry(int B, int N, int F, int32_t* out);
int neptune_pdhg_mf_solve(int B, int N, int F, int kind,
                          const double* d, const double* w, const double* r, const double* m,
                          const double* Mj, const double* Kj,
                          const neptune_pdhg_params* params_h,
                          double* x, double* y, neptune_pdhg_result* result_d,
                          void* workspace, int64_t workspace_bytes, void* stream);
/* The same solver for the models with node columns n[j] (`NeptuneStep1CPUMinUtilization`,
 * `NeptuneStep1CPUMinDelayAndUtilization`: reference core/solvers/neptune/neptune_step1.py:38-77): columns x, c, n;
 * the rows above plus C5a (sum_f c[f,j] - M n[j] <= 0), C5b (sum_f c[f,j] - n[j] >= -eps) and C6
 * (cost[j] n[j] <= budget) of utils/constraints_step1.py:69-80, 101-103 -- the canonical layout of
 * neptune_assemble(kind, NEPTUNE_FLAG_STRENGTHEN).  The new rows and columns are O(N): they live in the small-vector
 * kernel, the streaming pass is unchanged.  d_obj[B][N][N] is the delay matrix AS IT ENTERS THE OBJECTIVE
 * (objectives.py:24-52): zeros for kind 1, d * (1 - alpha) / (largest workload-weighted delay) for kind 2; obj_n is
 * the coefficient of every n[j] (1, or alpha / N).  big_m[B][N] (or NULL for the reference's 10^6) is the M of row C5a per
 * node: any valid bound on the pods node j can hold keeps the MIP unchanged and tightens the relaxation ("node cut":
 * with floor(Mj / m) the LP bound of the combined objective goes from 5 % to 81-90 % of the MIP optimum on the small
 * goldens).  Workspace: neptune_pdhg_mf_workspace_bytes. */
int neptune_pdhg_mf_solve_util(int B, int N, int F, int kind, const double* d_obj, const double* w,
                               const double* r, const double* m, const double* Mj, const double* Kj,
                               const double* cost, double budget, double obj_n, const double* big_m,
                               const neptune_pdhg_params* prm, double* x, double* y,
                               neptune_pdhg_result* result_d, void* workspace, int64_t workspace_bytes,
                               void* stream);

/* ---- (b, matrix-free, sharded) step-wise building blocks of the matrix-free iteration for the
 * function-block-sharded solver (neptune_mip_b200/sharded_mf.py, one process per GPU; SURVEY.md section 8(e)): a rank
 * owns the functions of its block, the 2N coupling rows (C2 memory, C4 CPU) are replicated, and the caller all-reduces
 * their activities once per iteration; step sizes are host scalars.  The numpy statement they follow is
 * tests/mf_reference.ShardedMatrixFree; on B200 two NCCL ranks reproduce the single-rank iterates to 3e-17
 * (profiles/r02_sharded_mf.md).  F = functions of THIS rank; x / y / xsum / ysum are the canonical vectors of
 * the rank's local model; S4[B][N], S2[B] are the GLOBAL Pock-Chambolle row scalings (caller all-reduces the sums);
 * coupling[B][2N] = [C4 activity of the pending pass | C2 activity of the new cbar] over the own functions.
 *   column_sums : once before the first local step (and after y was replaced): column sums of yS
 *   local_step  : y1, y3 of the pending pass (have_pass), c columns of the next iteration (do_prec), coupling out
 *   (caller: all-reduce of coupling)
 *   pass        : y4 (have_pass, step sigma_prev) and y2 (run_pass, step sigma) from the global activities, then the
 *                 iteration pass over the own functions (run_pass) */
int neptune_pdhg_mf_step_bytes(int B, int N, int F, int64_t* bytes);
int neptune_pdhg_mf_column_sums(int B, int N, int F, const double* w, const double* r, const double* m,
                                double* x, double* y, double* xsum, double* ysum, const double* S4, const double* S2,
                                void* workspace, int64_t workspace_bytes, void* stream);
int neptune_pdhg_mf_local_step(int B, int N, int F, const double* w, const double* r, const double* m,
                               double tau, double sigma_prev, int have_pass, int do_prec,
                               double* x, double* y, double* xsum, double* ysum, const double* S4, const double* S2,
                               void* workspace, int64_t workspace_bytes, double* coupling, void* stream);
int neptune_pdhg_mf_pass(int B, int N, int F, const double* d, const double* w, const double* r, const double* m,
                         const double* Mj, const double* Kj, double tau, double sigma, double sigma_prev,
                         int have_pass, int run_pass, double* x, double* y, double* xsum, double* ysum,
                         const double* S4, const double* S2, void* workspace, int64_t workspace_bytes,
                         const double* coupling_sum, void* stream);

/* ---- (c) exact evaluation, rounding, local search -------------------------------------------------
 * neptune_check_solution: the reference's six checkers and three scorers
 * (`efttc/utils/constraints_step1.py:5-133`, `efttc/utils/objectives.py:23-98`) on dense
 * x[N][F][N] (index [i][f][j]), c[F][N], n[N] for B solutions of B instances, every sum in the
 * reference's order.  flags_out[B] (NEPTUNE_OK_* bits), scores_out[B][3] = {delay, util, combined}. */
int neptune_check_solution(int B, int N, int F, double alpha,
                           const double* d, const double* w, const double* r, const double* m,
                           const double* Mj, const double* Kj, const double* maxd,
                           const double* cost, double budget,
                           const double* x, const double* c, const double* n,
                           int32_t* flags_out, double* scores_out, void* stream);

/* neptune_route_placements: closed-form routing of `change_x_one`
 * (`efttc/efttc_step1.py:196-212`): x[i,f,j] = 1/|B| on the (1e-6-)nearest open pods of f.
 * c[B][F][N] (uint8 0/1) -> x[B][N][F][N], n[B][N] (float64). */
int neptune_route_placements(int B, int N, int F, const double* d, const uint8_t* c,
                             double* x, double* n, void* stream);

/* neptune_route_capacitated: routing of a fixed placement that also honours the CPU rows
 * (`constrain_CPU_usage`, constraints_step1.py:57-65): nearest open pod first, then per overloaded
 * node the flows with the smallest delay increase per freed core are moved (the last one split).
 * Pods left without any request are closed in c_out (C1b, constraints_step1.py:12-15).
 * c[B][F][N] uint8 -> c_out[B][F][N], x[B][N][F][N], n[B][N], obj_out[B] (sum x*d*w), feas_out[B]. */
int neptune_route_capacitated(int B, int N, int F, const double* d, const double* w, const double* r,
                              const double* Kj, const uint8_t* c, uint8_t* c_out, double* x, double* n,
                              double* obj_out, int32_t* feas_out, void* stream);

/* neptune_eval_placements: P candidate placements per instance, never materialising x:
 * c[B][P][F][N] (uint8) -> obj_out[B][P][3] {delay, util, combined}, flags_out[B][P],
 * overload_out[B][P] (sum_j max(0, cpu_load_j - K_j), 0 when the CPU check passes). */
int neptune_eval_placements(int B, int P, int N, int F, double alpha,
                            const double* d, const double* w, const double* r, const double* m,
                            const double* Mj, const double* Kj, const double* maxd,
                            const double* cost, double budget, const uint8_t* c,
                            double* obj_out, int32_t* flags_out, double* overload_out,
                            void* stream);

/* neptune_local_search: per instance, `chains` independent add/drop/swap searches seeded from
 * seeds[B][S][F][N] (uint8; e.g. EFTTC output, PDHG roundings), `sweeps` best-improvement sweeps
 * each.  Returns the best feasible placement per instance: best_c[B][F][N] (uint8),
 * best_obj[B], best_flags[B]. */
int neptune_local_search(int B, int N, int F, int kind, double alpha, int chains, int sweeps,
                         uint64_t rng_seed, int S,
                         const double* d, const double* w, const double* r, const double* m,
                         const double* Mj, const double* Kj, const double* maxd,
                         const double* cost, double budget, const double* old,
                         const uint8_t* seeds, const double* guide /* c-bar [B][F][N] or NULL */,
                         uint8_t* best_c, double* best_obj, int32_t* best_flags,
                         void* workspace, int64_t workspace_bytes, void* stream);
int neptune_local_search_workspace_bytes(int B, int N, int F, int chains, int64_t* bytes);
/* *fits = 1 when neptune_local_search (and neptune_disruption_search) take instances of N nodes and F functions,
 * 0 when they return NEPTUNE_E_SIZE for them (a chain's shared-memory rows exceed 200 KiB: N > 1066).  Host only. */
int neptune_local_search_fits(int N, int F, int32_t* fits);

/* neptune_disruption_search: step 2 "minimise disruption" (reference NeptuneStep2*, neptune_step2.py:5-93,
 * constraints_step2.py:5-89, objectives.py:55-63) as a search over placements with the step-2 objective in
 * closed form: W*|c xor old| - (W+1)*(sum_old - sum_c) for mode 1 ("delete", needs sum_c <= sum_old),
 * W*|c xor old| - (W-1)*(sum_c - sum_old) for mode 2 ("create"), W = F*N, subject to the step-1 rows and
 * to step-1 objective(kind) <= bound[b] (= soften_step1_sol * step-1 score).  Same workspace as
 * neptune_local_search.  best_obj[b] = +inf when no chain found a placement satisfying mode and bound. */
int neptune_disruption_search(int B, int N, int F, int kind, double alpha, int mode, const double* bound,
                              int chains, int sweeps, uint64_t rng_seed, int S,
                              const double* d, const double* w, const double* r, const double* m,
                              const double* Mj, const double* Kj, const double* maxd,
                              const double* cost, double budget, const double* old,
                              const uint8_t* seeds, uint8_t* best_c, double* best_obj, int32_t* best_flags,
                              void* workspace, int64_t workspace_bytes, void* stream);

/* neptune_route_lp: EXACT routing of fixed placements -- the LP the reference's step-1 MIP reduces to once c
 * is fixed (rows constraints_step1.py:47-65, objective objectives.py:4-11), solved per placement by a
 * dense-tableau dual simplex started from the nearest-open-pod routing and restricted to the sources of the
 * nodes whose CPU row binds (csrc/route_lp.cu).  P placements per instance: c[B][P][F][N] (uint8) ->
 * obj_out[B][P] (sum x*d*w of the LP optimum), status_out[B][P] (1 = optimal and every open pod keeps a share
 * >= 1 - eps, 0 = infeasible, 2 = the tableau does not fit `tableau_doubles`: use neptune_route_capacitated),
 * optional c_out[B][P][F][N] (pods nobody uses closed), x[B][P][N][F][N], n[B][P][N], info_out[B][P][2]
 * (pivots, nodes priced).  Workspace from neptune_route_lp_workspace_bytes. */
int neptune_route_lp(int B, int P, int N, int F, const double* d, const double* w, const double* r,
                     const double* Kj, const uint8_t* c, uint8_t* c_out, double* x, double* n,
                     double* obj_out, int32_t* status_out, int32_t* info_out, int64_t tableau_doubles,
                     void* workspace, int64_t workspace_bytes, void* stream);
int neptune_route_lp_workspace_bytes(int B, int P, int N, int F, int64_t tableau_doubles, int64_t* bytes);

/* neptune_lns_search: step-1 search for the models with a delay term (kind 0 and 2) when every function needs
 * the same memory (the memory row is then a slot count per node): `chains` warp-sized chains per instance, each
 * `rounds` exact k-node re-optimisations (dynamic programme over functions with the slot counters as state) on
 * the priced nearest-pod cost, node prices on the CPU rows kept at their coordinate-wise dual optimum, annealed
 * cost perturbation of relative size `noise_coef` (csrc/lns.cu).  Chains start from randomised roundings of
 * guide[B][F][N] (c-bar of the LP relaxation) and lam0[B][N] (its CPU-row duals), and/or from
 * seeds[B][S][F][N]; any of the three may be NULL (no guide: every chain starts from a seed).  Every chain returns
 * two records (2*chains per instance): entries [0, chains) are the chains' best placements by the objective with
 * every source routed WHOLE to its nearest priced pod (feasible, so an upper bound of the placement's true
 * objective), entries [chains, 2*chains) the best by the priced objective (a lower bound; equal to the routing LP
 * where the prices are optimal, i.e. where the optimum splits flows).  out_c[B][2*chains][F][N], out_g[B][2*chains]
 * (the bound the record was chosen by; +inf = none), out_lb[B][2*chains] (optional: the other end of the bracket),
 * out_round[B][2*chains].  Price the records exactly with neptune_route_lp. */
int neptune_lns_search(int B, int N, int F, int kind, double alpha, int chains, int rounds, int k,
                       double noise_coef, uint64_t rng_seed,
                       const double* d, const double* w, const double* r, const double* m,
                       const double* Mj, const double* Kj, const double* maxd,
                       const double* guide, const double* lam0, int S, const uint8_t* seeds,
                       int max_slots /* >= max_j floor(Mj / m), or 0 for F: sizes the shared-memory scratch */,
                       uint8_t* out_c, double* out_g, double* out_lb, int32_t* out_round, void* stream);
/* neptune_lns_search_global: neptune_lns_search with every chain's state in a workspace slab instead of shared memory,
 * for instances the shared-memory kernel refuses (N > 128 or F*N > 4096; BASELINE configs 3 and 4).  Same arguments and
 * the same records bit for bit wherever both run (same random streams, evaluation and summation orders, decisions), at
 * any N <= 65534 with F*N < 2^31; kind 1 is refused (NEPTUNE_E_ARG), larger sizes NEPTUNE_E_SIZE, a workspace smaller
 * than neptune_lns_search_global_workspace_bytes NEPTUNE_E_NOMEM.  It also returns out_asg[B][2*chains][F][N] (uint16):
 * the node of each source's nearest priced pod when the record was taken.  A record is taken only with no node
 * overloaded, so routing every source whole to that pod is a feasible point of the MIP whose delay is the record's
 * upper bound -- a routing for records too large for neptune_route_lp.  The workspace holds each instance's
 * transposed delay matrix (8 N^2 bytes) and about 13 F*N bytes per chain. */
int neptune_lns_search_global(int B, int N, int F, int kind, double alpha, int chains, int rounds, int k,
                              double noise_coef, uint64_t rng_seed,
                              const double* d, const double* w, const double* r, const double* m,
                              const double* Mj, const double* Kj, const double* maxd,
                              const double* guide, const double* lam0, int S, const uint8_t* seeds, int max_slots,
                              uint8_t* out_c, double* out_g, double* out_lb, int32_t* out_round, uint16_t* out_asg,
                              void* workspace, int64_t workspace_bytes, void* stream);
/* workspace of neptune_lns_search_global (host arithmetic, no device needed) */
int neptune_lns_search_global_workspace_bytes(int B, int N, int F, int chains, int k, int max_slots, int64_t* bytes);
/* chains per thread block of neptune_lns_search: 0 (default) = 8 while all blocks are resident at once, 12 (at 80
 * registers) beyond; 1 = always 8; 2 = always 12.  The results do not depend on it (a chain's random stream is a
 * function of its index only); it is a tuning and measurement switch. */
int neptune_lns_block_mode(int mode);

/* ---- (d2) round-robin delay-improvement greedy (csrc/site.cu) ---------------------------------------
 * A placement for instances too large for the one-block-per-instance EFTTC kernel and the shared-memory searches
 * (BASELINE config 4).  The move is EFTTC's `find_best_node_by_delay_improvement`
 * (`core/solvers/efttc/efttc_step1.py:214-288`): gain(f, j) = sum_i w[f,i] max(0, cur[f,i] - d[i,j]); every function
 * proposes its best node in every round, a node accepts in order of gain while its memory lasts (`:290-312`).
 * c_out[B][F][N] uint8, info_out[B][2] = {rounds that placed a pod, pods}.  `unserved_delay` (> every d) is the delay
 * of a source whose function has no pod yet.  CPU capacity is left to neptune_route_capacitated + the checkers. */
int neptune_site_greedy_workspace_bytes(int B, int N, int F, int64_t* bytes);
int neptune_site_greedy(int B, int N, int F, const double* d, const double* w, const double* m, const double* Mj,
                        double unserved_delay, int max_rounds, uint8_t* c_out, int32_t* info_out,
                        void* workspace, int64_t workspace_bytes, void* stream);

/* neptune_site_search: best-improvement pod-exchange search for the min-delay objective under nearest-pod routing,
 * obj = sum_f sum_i w[f,i] * (delay from i to the nearest open pod of f), at any size (csrc/site_search.cu).  Starts
 * from c_in[B][F][N] (uint8; every function with a pod, memory rows sum_f m[f] c[f,j] <= Mj held; e.g.
 * neptune_site_greedy's placement) and keeps both.  Per round every node proposes its best add or exchange (one
 * function leaves, another enters), every function its best relocation of one pod; proposals touching disjoint
 * functions and nodes are accepted in order of improvement.  Stops when a round accepts nothing or after max_rounds.
 * c_out[B][F][N] (may equal c_in), info_out[B][4] = {rounds that accepted a move, adds, exchanges, relocations},
 * obj_out[B][2] = {objective at the start, at the end}.  Deterministic.  NEPTUNE_E_ARG when a function of c_in has
 * no pod.  Workspace from neptune_site_search_workspace_bytes. */
int neptune_site_search_workspace_bytes(int B, int N, int F, int64_t* bytes);
int neptune_site_search(int B, int N, int F, const double* d, const double* w, const double* m, const double* Mj,
                        const uint8_t* c_in, uint8_t* c_out, int max_rounds, int32_t* info_out, double* obj_out,
                        void* workspace, int64_t workspace_bytes, void* stream);

/* neptune_route_two_choice: routing of ONE placement per instance at sizes where the per-instance routers do not
 * finish (C4: 400 000 sources).  Every source sends the share theta[j1] to its nearest pod and the rest to its
 * second-nearest one; theta[j] starts at 1 and is lowered until node j's CPU row holds (`constrain_CPU_usage`,
 * constraints_step1.py:57-65; `constrain_handle_all_requests` :27-33 holds by construction).  Pods that are nobody's
 * nearest are closed.  c[B][F][N] -> c_out, x[B][N][F][N] (may be NULL), n_out[B][N], obj_out[B] (objectives.py:4-11
 * on that x), feas_out[B] (1 = every CPU row holds), *iters_out (host int). */
int neptune_route_two_choice_workspace_bytes(int B, int N, int F, int64_t* bytes);
int neptune_route_two_choice(int B, int N, int F, const double* d, const double* w, const double* r, const double* Kj,
                             const uint8_t* c, uint8_t* c_out, double* x, double* n_out, double* obj_out,
                             int32_t* feas_out, int32_t* iters_out, int max_iters,
                             void* workspace, int64_t workspace_bytes, void* stream);

/* ---- (d) EFTTC greedy -----------------------------------------------------------------------------
 * Replaces `EfttcStepBase.solve()` (`core/solvers/efttc/efttc_step1.py:39-90` and helpers
 * :92-312, score_local :356-439).  One thread block per instance; deterministic, same
 * iteration orders, tie-breaks and tolerances as the reference.
 * c_out[B][F][N] (uint8), n_out[B][N] (uint8), info_out[B][4] = {ttc iterations, pods,
 * reference_would_raise_KeyError (efttc_step1.py:118), stop reason}. */
int neptune_efttc(int B, int N, int F, int kind, double alpha,
                  const double* d, const double* w, const double* r, const double* m,
                  const double* Mj, const double* Kj, const double* old,
                  const double* cost, double budget,
                  uint8_t* c_out, uint8_t* n_out, int32_t* info_out,
                  void* workspace, int64_t workspace_bytes, void* stream);
int neptune_efttc_workspace_bytes(int B, int N, int F, int64_t* bytes);

/* small helper: out[k] = in[k] ? 1.0 : 0.0 (placements travel as uint8, the checkers read float64) */
int neptune_u8_to_f64(int64_t n, const uint8_t* in, double* out, void* stream);

/* number of kernels this library launched since the last reset (host-side counter; bench.py's
 * `gpu_launches`) */
int neptune_launch_count(int64_t* count, int reset);

/* ---- host-buffer convenience (the e2e path of bench.py) -----------------------------------------
 * Same as neptune_efttc + neptune_route_placements + neptune_check_solution but with HOST
 * buffers: copies inputs H2D, runs on `stream`, copies c/n/flags/scores D2H and synchronises. */
int neptune_efttc_host(int B, int N, int F, int kind, double alpha,
                       const double* d_h, const double* w_h, const double* r_h, const double* m_h,
                       const double* Mj_h, const double* Kj_h, const double* old_h,
                       const double* maxd_h, const double* cost_h, double budget,
                       uint8_t* c_out_h, uint8_t* n_out_h, int32_t* info_out_h,
                       int32_t* flags_out_h, double* scores_out_h, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NEPTUNE_B200_H */
