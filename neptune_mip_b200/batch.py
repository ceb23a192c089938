"""Batched solve path: B same-shaped instances through the LP relaxation (matrix-free PDHG, all three objectives)
-> EFTTC -> local search (or, for the min-delay model at sizes the searches with shared-memory chain state do not take,
greedy -> pod-exchange search -> two-choice routing) -> exact check in one go (what bench.py times, and what a sweep like BASELINE.json's config 5 calls)."""
from __future__ import annotations

import os

import dataclasses
from dataclasses import dataclass
from typing import Optional

import numpy as np
import torch

from . import device
from ._lib import FLAG_STRENGTHEN, KINDS, OK_ALL, OK_C_X, OK_CPU, OK_HANDLE, OK_MEMORY, OK_N_C, NeptuneError

# the checks of the min-delay model: it has no budget row (C6), so the budget flag does not make its answer infeasible
MIN_DELAY_FLAGS = OK_HANDLE | OK_MEMORY | OK_CPU | OK_C_X | OK_N_C


@dataclass
class BatchParams:
    kind: str = "min_delay"
    alpha: float = 0.5
    lp_iters: int = 2048          # PDHG iterations on the strengthened relaxation (bound + rounding guide)
    lp_check_every: int = 256
    chains: int = 16              # local-search chains per instance (add/drop/swap search)
    sweeps: int = 200
    rng_seed: int = 1
    search: str = "auto"          # "auto": slot-count LNS (csrc/lns.cu) where it applies, else the add/drop/swap search, and for the
                                  # min-delay model at sizes neither takes (N > 1066) the pod-exchange search; "local": always the
                                  # add/drop/swap search; "site": always the pod-exchange search (min-delay only); "lns": the
                                  # slot-count LNS at every size (kinds 0 and 2, one memory size): beyond shared memory (N > 128 or
                                  # F*N > 4096) with the chain state in global memory, started from the pod-exchange search's placement
    lp_cut: bool = True           # relax with the Chvatal-Gomory rounding of the memory rows (one memory size per instance)
    lns_chains: int = 96          # warp-sized chains per instance
    lns_fill_waves: bool = False  # raise the chain count (at most 1.5x) until the blocks of the search fill whole waves of the GPU
                                  # (measured: NOT free -- 32 x 144 chains take 9.1 s where 32 x 96 take 7.1 s; fill the waves with instances instead)
    lns_rounds: int = 20000       # k-node re-optimisations per chain
    lns_k: int = 3
    lns_noise: float = 0.1
    lns_phases: int = 1           # > 1: population restarts from the best records between phases (lns_rounds is the total)
    lns_cooling: float = 0.6      # temperature factor from one phase to the next
    lns_restart_pool: int = 16    # records a restart phase draws its start placements from
    lns_local_chains: int = -1    # > 0: the add/drop/swap search, restarted from the best records, adds one candidate; -1: 16 chains when F*N <= 256
    lns_k4_chains: int = 0        # > 0: a second population of chains that re-optimise four nodes per round
    lns_final_k4: int = 3000      # > 0: rounds of a final phase that restarts one 4-node chain from every record
    lns_final_noise: float = 0.3  # its temperature, as a fraction of lns_noise
    lns_polish: int = -12         # > 0: iterations of exact steepest descent (every single-pod change priced by the routing LP) from the best
                                  # record; < 0: that many, but only for tiny instances (F*N <= 64); 0: never
    elites: int = 32              # chain records priced exactly (routing LP) per instance


@dataclass
class BatchResult:
    c: torch.Tensor               # uint8 [B,F,N]
    x: torch.Tensor               # float64 [B,N,F,N]
    n: torch.Tensor               # float64 [B,N]
    flags: torch.Tensor           # int32 [B]
    scores: torch.Tensor          # float64 [B,3]
    lp: Optional[np.ndarray]      # PDHG result records (primal/dual objective, residuals, iterations)
    pdhg_ms: float = 0.0          # device time of the PDHG call (CUDA events on the launch stream)
    pdhg_iters: int = 0
    model_dims: tuple = (0, 0, 0)
    pdhg_bytes_per_iter: int = 0  # algorithmic bytes one PDHG iteration of the whole batch moves (DESIGN.md section 3b)
    pdhg_path: str = ""           # "matrix-free" when the LP ran
    search_path: str = ""         # "lns" | "local" | "site"
    lns_round: Optional[torch.Tensor] = None     # [B] round at which the returned placement was recorded by its chain
    lns_ms: float = 0.0
    lns_diag: Optional[dict] = None              # elite_g[B,E] priced objective, elite_val[B,E] exact objective (inf: infeasible)


def solve_batch(inst: device.InstanceBatch, prm: BatchParams, time_pdhg: bool = False) -> BatchResult:
    kind = prm.kind
    lp_res, guide, lam0, pdhg_ms, iters, dims = None, None, None, 0.0, 0, (0, 0, 0)
    bytes_iter, path = 0, ""
    use_lns = prm.search in ("auto", "lns") and device.lns_supported(inst, kind)
    delay_term = KINDS.get(kind, kind) != 2 or bool((objective_weights(inst, kind, prm.alpha)[0] > 0).all())
    if use_lns and not delay_term:
        use_lns = False         # no workload: the combined objective has no delay term (objectives.py:34-35), nothing to price
    lns_global = prm.search == "lns" and not device.lns_supported(inst, kind)
    if lns_global and not (delay_term and device.lns_global_supported(inst, kind)):
        raise ValueError("search='lns' needs a delay term in the objective and one memory size per instance")
    use_site = prm.search == "site" or (prm.search == "auto" and KINDS.get(kind, kind) == 0 and not use_lns
                                        and not device.local_search_fits(inst.N, inst.F))
    if use_site and KINDS.get(kind, kind) != 0:
        raise ValueError("search='site' solves the min-delay model only")
    cut = prm.lp_cut and (use_lns or lns_global or (use_site and device.one_memory_size(inst)))
    inst_lp = device.slot_relaxation(inst) if cut else inst
    if prm.lp_iters > 0:
        N, F, B = inst.N, inst.F, inst.B
        X = F * N * N
        # the relaxation is solved matrix-free (nothing is assembled; every coefficient of the strengthened model is
        # regenerated from d, w, r, m inside the iteration kernels); the models with node columns n[j] add O(N) rows
        # and columns that live in the small-vector kernel (neptune_pdhg_mf_solve_util)
        kk = KINDS.get(kind, kind)
        rows, cols, nnz = device.model_sizes(N, F, kk, FLAG_STRENGTHEN)
        if time_pdhg:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        xs, ys, lp_res = device.pdhg_mf_solve(inst_lp, max_iters=prm.lp_iters, check_every=prm.lp_check_every,
                                              eps_rel=1e-6, eps_abs=1e-9, kind=kk, alpha=prm.alpha, node_cut=prm.lp_cut)
        lam0 = ys[:, 3 * F * N + N:3 * F * N + 2 * N].contiguous()       # duals of the CPU rows C4
        if kk == 2:      # the combined objective scales the delays: prices back in delay units for the search
            a_d = objective_weights(inst, kind, prm.alpha)[0]
            lam0 = lam0 / torch.where(a_d > 0, a_d, torch.ones_like(a_d))[:, None]
        bytes_iter, path = B * (64 * X + 112 * F * N + 8 * N * N), "matrix-free"
        if time_pdhg:
            e1.record()
            e1.synchronize()
            pdhg_ms = e0.elapsed_time(e1)
        dims = (rows, cols, nnz)
        iters = int(lp_res["iters"].max())
        guide = xs[:, X:X + F * N].contiguous()
        del xs, ys
    if use_site:
        best_c, x, n, flags, scores = site_step1(inst, prm.alpha)
        return BatchResult(best_c, x, n, flags, scores, lp_res, pdhg_ms, iters, dims, bytes_iter, path, "site")
    if lns_global:
        # the relaxation guides the chains (roundings of c-bar, CPU-row prices) only where it converged everywhere
        conv = lp_res is not None and bool((lp_res["converged"] != 0).all())
        best_c, x, n, flags, scores, lns_round, lns_ms, lns_diag = lns_global_step1(
            inst, kind, prm, guide if conv else None, lam0 if conv else None, time_it=time_pdhg)
        return BatchResult(best_c, x, n, flags, scores, lp_res, pdhg_ms, iters, dims, bytes_iter, path, "lns",
                           lns_round, lns_ms, lns_diag)
    cache = {}

    def get_seeds():
        """EFTTC placements of the three objectives (one thread block per instance: seconds at 50x10, so the LP-guided
        search only asks for them when it needs a fallback or feeds the add/drop/swap search)"""
        if "s" not in cache:
            cache["s"] = torch.stack([device.efttc(inst, k, prm.alpha)[0] for k in ("min_delay", "min_util", "min_delay_util")],
                                     dim=1).contiguous()
        return cache["s"]

    lns_round, lns_ms, lns_diag = None, 0.0, None
    if use_lns:
        if prm.lns_local_chains < 0:
            prm = dataclasses.replace(prm, lns_local_chains=16 if inst.F * inst.N <= 256 else 0)
        lns_seeds = get_seeds() if (prm.lns_local_chains > 0 or guide is None) else None
        best_c, x, n, flags, scores, lns_round, lns_ms, lns_diag = lns_step1(inst, kind, prm, guide, lam0, lns_seeds, time_it=time_pdhg)
    else:
        seeds = get_seeds()
        fallback = seeds[:, KINDS[kind]]
        best_c, best_obj, _ = device.local_search(inst, kind, seeds, prm.alpha, prm.chains, prm.sweeps,
                                                  prm.rng_seed, guide)
        bad = ~torch.isfinite(best_obj)
        if bool(bad.any()):
            best_c[bad] = fallback[bad]
        # final routing honours the CPU rows (splits flows on binding nodes) and closes pods nobody uses
        best_c, x, n, _, _ = device.route_capacitated(inst, best_c)
        flags, scores = device.check_solution(inst, x, device.u8_to_f64(best_c), n, prm.alpha)
    bad = flags != OK_ALL
    if bool(bad.any()):
        # rare (a pod starved by a split flow that no free source can top up): fall back, per instance, to the
        # first EFTTC seed that passes every check -- a worse objective, never an infeasible answer
        seeds = get_seeds()
        for k in (KINDS[kind], 1, 2, 0):
            cf, xf, nf, _, _ = device.route_capacitated(inst, seeds[:, k].contiguous())
            ff, sf = device.check_solution(inst, xf, device.u8_to_f64(cf), nf, prm.alpha)
            take = bad & (ff == OK_ALL)
            if bool(take.any()):
                best_c[take], x[take], n[take], flags[take], scores[take] = cf[take], xf[take], nf[take], ff[take], sf[take]
                bad = flags != OK_ALL
            if not bool(bad.any()):
                break
    return BatchResult(best_c, x, n, flags, scores, lp_res, pdhg_ms, iters, dims, bytes_iter, path,
                       "lns" if use_lns else "local", lns_round, lns_ms, lns_diag)


def site_step1(inst: device.InstanceBatch, alpha=0.5):
    """Min-delay placement at any size: round-robin greedy -> pod-exchange search -> two-choice routing -> checkers.
    The searched placement is kept where it passes the model's checks (MIN_DELAY_FLAGS) and routes no worse than the
    greedy's; elsewhere the greedy's routed placement stands in.  Neither EFTTC nor the capacity-aware router runs here
    (neither finishes at BASELINE config 4).  Returns (c uint8[B,F,N], x, n, flags, scores)."""
    M = MIN_DELAY_FLAGS
    cg, _ = device.site_greedy(inst)
    cs, _, _ = device.site_search(inst, cg)
    c, x, n, obj, _, _ = device.route_two_choice(inst, cs)
    flags, scores = device.check_solution(inst, x, device.u8_to_f64(c), n, alpha)
    _, _, _, obj_g, _, _ = device.route_two_choice(inst, cg, want_x=False)
    failed = (flags & M) != M
    bad = failed | (obj_g < obj)
    if bool(bad.any()):
        cf, xf, nf, _, _, _ = device.route_two_choice(inst, cg)
        ff, sf = device.check_solution(inst, xf, device.u8_to_f64(cf), nf, alpha)
        take = bad & (((ff & M) == M) | failed)
        if bool(take.any()):
            c[take], x[take], n[take], flags[take], scores[take] = cf[take], xf[take], nf[take], ff[take], sf[take]
        del xf
    return c, x, n, flags, scores


def lns_global_step1(inst: device.InstanceBatch, kind, prm: "BatchParams", guide, lam0, time_it=False):
    """The slot-count search at sizes beyond shared memory (`lns_search_global`).  EFTTC (one block per instance) and the
    capacity-aware router do not finish at BASELINE config 4, so neither runs: chain 0 starts from the pod-exchange
    search's placement (`site_greedy` -> `site_search`), the other chains from it too or, with a guide, from roundings
    of c-bar; records the routing LP cannot price keep the whole-flow routing they were certified with.  The start
    placement routed by `route_two_choice` is one more candidate: the answer is never worse than it.
    Returns what `lns_step1` returns."""
    kk = KINDS.get(kind, kind)
    M, col = (MIN_DELAY_FLAGS, 0) if kk == 0 else (OK_ALL, 2)
    cg, _ = device.site_greedy(inst)
    cs, _, _ = device.site_search(inst, cg)
    del cg
    prm = dataclasses.replace(prm, lns_local_chains=0, lns_polish=0)
    c, x, n, flags, scores, rnd, ms, diag = lns_step1(inst, kind, prm, guide, lam0, cs[:, None].contiguous(), time_it,
                                                      global_state=True)
    c2, x2, n2, _, _, _ = device.route_two_choice(inst, cs)
    f2, s2 = device.check_solution(inst, x2, device.u8_to_f64(c2), n2, prm.alpha)
    ok, ok2 = (flags & M) == M, (f2 & M) == M
    take = ok2 & (~ok | (s2[:, col] < scores[:, col]))
    if bool(take.any()):
        c[take], x[take], n[take], flags[take], scores[take] = c2[take], x2[take], n2[take], f2[take], s2[take]
        rnd[take] = -1
    diag["start_won"] = take
    return c, x, n, flags, scores, rnd, ms, diag


_DEBUG_SYNC = int(os.environ.get("NEPTUNE_DEBUG_SYNC", "0"))


def polish_exact(inst: device.InstanceBatch, kind, alpha, c: torch.Tensor, max_iters: int = 12, depth: int = 2,
                 chunk: int = 4096):
    """Steepest descent with EVERY neighbour priced exactly by the routing LP (`neptune_route_lp` on the whole batch
    of candidates: the "thousands of candidate placements per launch" of the north star).  Neighbourhoods by size,
    the next one only when the smaller ones hold no improvement: all single pod flips (add / drop), all PAIRS of flips
    (moves of a pod, swaps of two functions on a node, two adds, ...), all TRIPLES.  For small instances where most
    CPU rows bind: there the node prices of the search stall below the LP value, its records are loose, and the
    optimum is one or two coupled changes away (a pod swap on a full node plus the re-routing it allows).
    c uint8[B,F,N] -> (improved c, its exact value [B]); memory is a slot count (lns_supported)."""
    B, N, F = inst.B, inst.N, inst.F
    FN = F * N
    dev = c.device
    a_d, a_u = objective_weights(inst, kind, alpha)
    slots = torch.floor(inst.Mj / inst.m[:, :1] + 1e-9).clamp_(max=float(F))                      # [B,N]
    # the tableau of such an instance is small: rows <= N + F*N + pods, a slab of 2^17 doubles per candidate is ample
    slab = 1 << 17 if FN <= 64 else 1 << 19
    ar = torch.arange(FN, device=dev)
    masks = {}

    def flip_masks(size):
        if size not in masks:
            comb = torch.combinations(ar, r=size) if size > 1 else ar[:, None]                    # [M,size]
            mk = torch.zeros((comb.shape[0], FN), dtype=torch.uint8, device=dev)
            mk.scatter_(1, comb, 1)
            masks[size] = mk.reshape(-1, F, N)
        return masks[size]

    depth = int(os.environ.get("NEPTUNE_POLISH_DEPTH", depth))
    zero_ws = bool(os.environ.get("NEPTUNE_RLP_ZERO"))

    def value(cands):
        if _DEBUG_SYNC == 1:
            torch.cuda.synchronize(); print("polish: before route_lp", tuple(cands.shape), flush=True)
        ws = None
        if zero_ws:
            ws = torch.zeros(296 * ((1 << 20) + (slab << 3)), dtype=torch.uint8, device=dev)
        pr = device.route_lp(inst, cands.contiguous(), tableau_doubles=slab, workspace=ws)
        if _DEBUG_SYNC in (1, 2):
            torch.cuda.synchronize(); print("polish: after route_lp", tuple(cands.shape), "status counts", torch.bincount(pr["status"].reshape(-1), minlength=3).tolist(), flush=True)
        v = a_d[:, None] * pr["obj"] + a_u[:, None] * pr["n"].sum(dim=-1)
        return torch.where(pr["status"] == 1, v, torch.full_like(v, float("inf")))

    def best_of(cur, size):
        mk = flip_masks(size)
        best = torch.full((B,), float("inf"), dtype=torch.float64, device=dev)
        pick = cur.clone()
        for lo in range(0, mk.shape[0], chunk):
            cands = cur[:, None] ^ mk[None, lo:lo + chunk]                                        # [B,M,F,N]
            # slot limits and coverage: an invalid candidate is replaced by the current placement (it cannot win)
            bad = (cands.sum(dim=2).to(torch.float64) > slots[:, None, :]).any(dim=2) | (cands.sum(dim=3) == 0).any(dim=2)
            cands = torch.where(bad[:, :, None, None], cur[:, None].expand_as(cands), cands)
            vals = value(cands)
            v, arg = vals.min(dim=1)                                                              # first minimum: deterministic
            take = v < best
            pick = torch.where(take[:, None, None], cands[torch.arange(B, device=dev), arg], pick)
            best = torch.where(take, v, best)
        return best, pick

    cur = c.clone()
    cur_val = value(cur[:, None])[:, 0]
    size, it = 1, 0
    while it < max_iters and size <= depth:
        if size == 3 and B * (FN ** 3) // 6 > 4_000_000:      # bounded work: triples only where they are cheap
            break
        best, pick = best_of(cur, size)
        better = best < cur_val - 1e-9 * (1.0 + cur_val.abs())
        if bool(better.any()):
            cur = torch.where(better[:, None, None], pick, cur)
            cur_val = torch.where(better, best, cur_val)
            size = 1
            it += 1
        else:
            size += 1
    return cur, cur_val


objective_weights = device.objective_weights      # (a_d[B], a_u[B]) of the three objectives


def _route_lp_or_none(inst: device.InstanceBatch, c_u8: torch.Tensor, want_x=False):
    """`route_lp`, or None where the library refuses the size (F*N > 2^24)"""
    try:
        return device.route_lp(inst, c_u8, want_x=want_x)
    except NeptuneError as e:
        if "size does not fit" not in str(e):
            raise
        return None


def fill_waves(B: int, chains: int, chains_per_block: int = 8, resident_blocks: int = 2 * 148, cap: float = 1.5) -> int:
    """Largest chain count with the same number of waves of search blocks (`chains_per_block` chains per block, two
    blocks per SM), at most `cap` times what was asked.  32 instances x 96 chains (384 blocks = 1.3 waves) take as long
    as 48 x 96 (576 blocks = 1.95 waves), so idle block slots exist -- but filling them with more chains of the SAME
    instances also grows the record pricing and the final phase (9.1 s against 7.1 s at 32 x 144): off by default, the
    bench fills the waves with instances (batch 48)."""
    per_inst = -(-chains // chains_per_block)
    waves = -(-(B * per_inst) // resident_blocks)
    fit = (waves * resident_blocks) // B
    return max(chains, min(fit * chains_per_block, int(cap * chains) // chains_per_block * chains_per_block))


def lns_step1(inst: device.InstanceBatch, kind, prm: "BatchParams", guide, lam0, seeds, time_it=False, global_state=False):
    """Slot-count LNS -> exact pricing of the best chain records (routing LP) -> exact routing + checkers of the
    winner.  Returns (c uint8[B,F,N], x, n, flags, scores, round[B], search ms, diagnostics).  `global_state`: the
    chains run in `lns_search_global`, and a record the routing LP does not price (tableau too large, or the size
    refused) is valued and routed by the whole-flow routing its chain certified it with."""
    B, N, F = inst.B, inst.N, inst.F
    if time_it:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    phases = max(1, prm.lns_phases)
    rounds = max(1, prm.lns_rounds // phases)
    main_chains = fill_waves(B, prm.lns_chains) if prm.lns_fill_waves else prm.lns_chains
    pops = []                 # populations: dict(c, g, r, other, chains), records [0, chains) by upper bound, [chains, 2 chains) by lower

    search = device.lns_search_global if global_state else device.lns_search

    def population(chains, n_rounds, k, noise, rng, guide_, seeds_, round_scale=1, round_offset=0):
        out = search(inst, kind, prm.alpha, chains, n_rounds, k, noise, rng, guide_, lam0, seeds_)
        pops.append(dict(c=out[0], g=out[1], r=out[2] * round_scale + round_offset, other=search.last_other_bound,
                         chains=chains, asg=out[3] if global_state else None))

    def records(upper, keys=("c", "g", "r", "other")):
        part = lambda t, p: t[:, :p["chains"]] if upper else t[:, p["chains"]:]          # noqa: E731
        return tuple(torch.cat([part(p[key], p) for p in pops], dim=1) for key in keys)

    for ph in range(phases):
        noise = prm.lns_noise * (prm.lns_cooling ** ph)
        if ph == 0:
            # start from roundings of the relaxation; optionally a second population that re-optimises four nodes at a
            # time (half as many, dearer rounds): it misses other instances than the three-node one does
            population(main_chains, rounds, prm.lns_k, noise, prm.rng_seed, guide, seeds)
            if prm.lns_k4_chains > 0:
                population(prm.lns_k4_chains, max(1, rounds // 2), 4, noise, prm.rng_seed + 104729, guide, seeds, round_scale=2)
        else:
            # population restart ("go with the winners"): every chain restarts from one of the best records so far
            # (drawn half from the records by upper bound, half from those by lower bound)
            halves = []
            for upper in (True, False):
                rc, rg, _, _ = records(upper)
                S = max(1, min(prm.lns_restart_pool // 2, rg.shape[1]))
                _, top = torch.topk(rg, S, dim=1, largest=False)
                halves.append(torch.gather(rc, 1, top[:, :, None, None].expand(B, S, F, N)))
            pool = torch.cat(halves, dim=1).contiguous()
            population(main_chains, rounds, prm.lns_k, noise, prm.rng_seed + 7919 * ph, None, pool, round_offset=ph * rounds)
    if prm.lns_final_k4 > 0:
        # intensification: every record so far is the start of one chain that re-optimises FOUR nodes at a time, almost
        # cold -- moves no three-node step can make
        allc = torch.cat([records(True)[0], records(False)[0]], dim=1).contiguous()
        population(allc.shape[1], prm.lns_final_k4, 4, prm.lns_noise * prm.lns_final_noise, prm.rng_seed + 15485863, None, allc,
                   round_offset=prm.lns_rounds)
    ub_c, ub_g, ub_r, _ = records(True)
    lb_c, lb_g, lb_r, lb_u = records(False)
    # elites: the best records of either kind, half each (a lower and an upper bound do not rank against each other)
    Eh = max(1, min(prm.elites // 2, ub_g.shape[1]))
    _, iu = torch.topk(ub_g, Eh, dim=1, largest=False)
    _, il = torch.topk(lb_g, Eh, dim=1, largest=False)
    out_c = torch.cat([ub_c, lb_c], dim=1)
    out_g = torch.cat([ub_g, lb_g], dim=1)
    out_round = torch.cat([ub_r, lb_r], dim=1)
    idx = torch.cat([iu, il + ub_g.shape[1]], dim=1)
    E = idx.shape[1]
    elite = torch.gather(out_c, 1, idx[:, :, None, None].expand(B, E, F, N)).contiguous()
    if global_state:
        out_a = torch.cat([records(True, ("asg",))[0], records(False, ("asg",))[0]], dim=1)
        elite_asg = torch.gather(out_a, 1, idx[:, :, None, None].expand(B, E, F, N))
        del out_a
        # the whole-flow value of each elite: the bound of the records by upper bound, the other bound of the others
        elite_wf = torch.gather(torch.cat([ub_g, lb_u], dim=1), 1, idx)
    if prm.lns_local_chains > 0:
        # one more candidate from the add/drop/swap search (it prices overload by a penalty instead of node prices and
        # does better where most CPU rows bind); restarted from the best records
        pool = torch.cat([elite[:, :2], elite[:, Eh:Eh + 2]] + ([seeds] if seeds is not None else []), dim=1).contiguous()
        lc, lobj, _ = device.local_search(inst, kind, pool, prm.alpha, prm.lns_local_chains, prm.sweeps, prm.rng_seed, None)
        lc = torch.where(torch.isfinite(lobj)[:, None, None], lc, elite[:, 0])
        elite = torch.cat([elite, lc[:, None]], dim=1).contiguous()
        idx = torch.cat([idx, idx[:, :1]], dim=1)
        E += 1
    pr = _route_lp_or_none(inst, elite) if global_state else device.route_lp(inst, elite)
    a_d, a_u = objective_weights(inst, kind, prm.alpha)
    if pr is None:        # the size is refused: every record keeps its certified whole-flow routing
        st0 = torch.full((B, E), 2, dtype=torch.int32, device=elite.device)
        pr = dict(obj=torch.full((B, E), float("inf"), dtype=torch.float64, device=elite.device), status=st0,
                  n=torch.zeros((B, E, N), dtype=torch.float64, device=elite.device), info=torch.zeros((B, E, 2), dtype=torch.int32, device=elite.device))
    val = a_d[:, None] * pr["obj"] + a_u[:, None] * pr["n"].sum(dim=-1)
    val = torch.where(pr["status"] == 1, val, torch.full_like(val, float("inf")))
    if global_state:
        val = torch.where(pr["status"] == 2, elite_wf, val)
    order = torch.argsort(val, dim=1, stable=True)
    ar = torch.arange(B, device=val.device)
    best_c = x = n = flags = scores = rnd = None
    polished = None
    if prm.lns_polish > 0 or (prm.lns_polish < 0 and F * N <= 64 and B * (F * N) ** 2 <= 400000):
        # tiny instances: exact steepest descent from the best priced record
        start = elite[ar, order[:, 0]].contiguous()
        if _DEBUG_SYNC in (1, 2, 3):
            torch.cuda.synchronize(); print('before polish', flush=True)
        polished, pval = polish_exact(inst, kind, prm.alpha, start, max_iters=abs(prm.lns_polish) if prm.lns_polish else 12)
        if _DEBUG_SYNC:
            torch.cuda.synchronize(); print('polish done', flush=True)
    # the checks an answer must pass: the min-delay model has no budget row, so at sizes where only the global-state
    # search runs its answers need not pass the budget check (the shared-memory path keeps asking for all six)
    M = MIN_DELAY_FLAGS if global_state and KINDS.get(kind, kind) == 0 else OK_ALL

    def certified_routing(pick):
        """(c, x, n, unrouted[B]) of the picked records' whole-flow routings; a chain that never took a record returns its
        current routing, where a source may have no pod (node id >= N): such an instance is marked, not routed"""
        a_ = elite_asg[ar, pick]
        bad = (a_ >= N).flatten(1).any(dim=1)
        return (*device.routing_of_assignment(inst, torch.where(bad[:, None, None], torch.zeros_like(a_), a_)), bad)
    for rank in range(E):
        pick = order[:, rank]
        cand = elite[ar, pick].contiguous() if not (rank == 0 and polished is not None) else polished
        if global_state and bool((pr["status"][ar, pick] == 2).all()):
            fin = None            # no instance would use the exact routing: skip the LP
        else:
            fin = _route_lp_or_none(inst, cand[:, None].contiguous(), want_x=True) if global_state else \
                device.route_lp(inst, cand[:, None].contiguous(), want_x=True)
        unrouted = None           # instances whose certified routing leaves a source without a pod (no record)
        if fin is None:
            cc, cx, cn, unrouted = certified_routing(pick)
        else:
            cx, cc, cn = fin["x"][:, 0].contiguous(), fin["c_out"][:, 0].contiguous(), fin["n"][:, 0].contiguous()
            st = fin["status"][:, 0]
            big = st == 2
            if bool(big.any()) and global_state:      # the routing the record was certified with
                hc, hx, hn, unrouted = certified_routing(pick)
                cc[big], cx[big], cn[big] = hc[big], hx[big], hn[big]
                unrouted = unrouted & big
            elif bool(big.any()):       # tableau larger than the slab: the heuristic capacity-aware routing stands in
                hc, hx, hn, _, _ = device.route_capacitated(inst, cand)
                cc[big], cx[big], cn[big] = hc[big], hx[big], hn[big]
        fl, sc = device.check_solution(inst, cx, device.u8_to_f64(cc), cn, prm.alpha)
        if unrouted is not None:
            fl = torch.where(unrouted, torch.zeros_like(fl), fl)
        if best_c is None:
            best_c, x, n, flags, scores = cc, cx, cn, fl, sc
            rnd = torch.gather(out_round, 1, torch.gather(idx, 1, pick[:, None]))[:, 0]
        else:
            take = ((flags & M) != M) & ((fl & M) == M)
            if bool(take.any()):
                best_c[take], x[take], n[take], flags[take], scores[take] = cc[take], cx[take], cn[take], fl[take], sc[take]
        if bool(((flags & M) == M).all()):
            break
    ms = 0.0
    if time_it:
        e1.record()
        e1.synchronize()
        ms = e0.elapsed_time(e1)
    diag = dict(elite_g=torch.gather(out_g, 1, idx), elite_val=val, n_upper=Eh, lb_other=torch.gather(lb_u, 1, il), elite_c=elite, pivots=pr["info"][..., 0], status=pr["status"],
                fell_back=(flags != OK_ALL))
    return best_c, x, n, flags, scores, rnd, ms, diag
