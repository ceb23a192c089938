#!/usr/bin/env python
"""bench.py -- placement instances/sec on BASELINE.json's config 2 (50 nodes x 10 functions, min-delay).

A step = one pass of the whole hot path over one batch of B synthetic C2 instances per GPU:
matrix-free PDHG on the slot-cut LP relaxation (b; run to convergence: bound, rounding guide, CPU-row prices)
-> EFTTC seeds (d) -> LP-guided slot-count search (c2, csrc/lns.cu) -> exact routing LP of the best chain
records (csrc/route_lp.cu) -> the reference's checkers/scorers (c1).  The search budget is the one at which the
returned placements reach the HiGHS optima of tests/golden/mip_optima.json (`quality`), i.e. `value` is a
throughput at (near) equal quality, not at a shorter budget.  `value` is instances/s with the inputs already in
HBM; `e2e` repeats the measurement from pinned HOST buffers through the batched plugin call, with the H2D copy of
every input and the D2H read of placements, routing, flags and scores inside the timed region.
`--impl reference` times the reference's CPU path (oracle port: the reference's model restated in numpy + HiGHS
standing in for the un-vendored OR-Tools/SCIP wheel) and prints the gap each instance is left with at the cap.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

N_NODES, N_FUNCS = 50, 10
WORKLOAD = "C2: 50 nodes x 10 functions, random symmetric delays, min-delay objective (NeptuneMinDelay step 1)"
L2_BYTES = 126e6


def make_hosts(cfg, batch, seed0):
    from neptune_mip_b200 import synth
    from neptune_mip_b200.core.utils import data_to_solver_input
    from neptune_mip_b200.device import InstanceBatch
    datas = [data_to_solver_input(synth.config_payload(cfg, seed0 + s), 1, with_db=False) for s in range(batch)]
    return InstanceBatch.host_arrays(datas)


def gold_optima(cfg):
    path = os.path.join(ROOT, "tests", "golden", "mip_optima.json")
    if not os.path.exists(path):
        return {}
    return {r["seed"]: r for r in json.load(open(path)) if r["config"] == cfg and r["optimal"]}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe), once per second."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_evt = index, [], threading.Event()

    def run(self):
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
                if out.returncode == 0 and out.stdout.strip():
                    self.rows.append([t.strip() for t in out.stdout.strip().split(",")])
            except Exception:
                pass
            self._stop_evt.wait(1.0)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=3)
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [nm for k, nm in enumerate(names) if any(r[2 + k].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons,
                "samples": len(self.rows), "sampled_on": "rank 0, 1 Hz"}


# ---------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the reference's CPU path (oracle port) on the host cores
# ---------------------------------------------------------------------------------------------------
def _cpu_one(args):
    seed, limit = args
    sys.path.insert(0, ROOT)
    from neptune_mip_b200 import synth
    from neptune_mip_b200.core.utils import data_to_solver_input
    from oracle import mip, model
    t0 = time.time()
    a = model.arrays_from_data(data_to_solver_input(synth.config_payload("C2", seed), 1, with_db=False))
    out = mip.solve_step1(a, "min_delay", time_limit=limit)
    return dict(seed=seed, seconds=time.time() - t0, optimal=bool(out["optimal"]), objective=out["objective"],
                gap=out["gap"])


def cpu_reference(n_instances, limit, procs, seed0=0):
    """Wall time of `n_instances` C2 step-1 MIPs, `procs` worker processes (the reference forks up to 10
    workers, main.py:69), each solve capped at `limit` seconds (an unsolved instance counts as done at
    the cap, which can only flatter the CPU)."""
    from concurrent.futures import ProcessPoolExecutor
    t0 = time.time()
    with ProcessPoolExecutor(procs) as ex:
        recs = list(ex.map(_cpu_one, [(seed0 + s, limit) for s in range(n_instances)]))
    wall = time.time() - t0
    return wall, recs


def cpu_quality(recs):
    """Where the CPU arm stands at its cap, against the proven optima (so the two arms' qualities can be compared)."""
    gold = gold_optima("C2")
    gaps = {r["seed"]: (r["objective"] - gold[r["seed"]]["objective"]) / abs(gold[r["seed"]]["objective"])
            for r in recs if r["seed"] in gold and r["objective"] is not None}
    return {"proven_optimal_inside_cap": int(sum(r["optimal"] for r in recs)), "instances": len(recs),
            "reference_optima_known": len(gaps), "within_1e4": int(sum(g <= 1e-4 for g in gaps.values())),
            "max_rel_gap": float(max(gaps.values())) if gaps else None,
            "rel_gap_at_cap_by_seed": {str(k): float(f"{v:.3g}") for k, v in sorted(gaps.items())},
            "no_incumbent": int(sum(r["objective"] is None for r in recs))}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    procs = max(1, min(cores, 10))
    n_inst = args.ref_instances if args.ref_instances > 0 else max(procs, 4)
    limit = args.ref_limit
    walls = []
    recs = []
    for it in range(args.warmup + args.steps):
        # step 0 takes seeds 0.. (the ones with proven optima in tests/golden, so its quality can be stated)
        wall, r = cpu_reference(n_inst, limit, procs, seed0=0 if it == args.warmup else 1000 * (it + 1))
        if it >= args.warmup:
            walls.append(wall)
        if it == args.warmup:
            recs = r
    ms = 1e3 * sum(walls) / max(len(walls), 1)
    value = n_inst / (ms / 1e3)
    solved = sum(r["optimal"] for r in recs)
    sample = (f"{n_inst} C2 instances per step, {procs} processes, HiGHS (stand-in for SCIP) capped at {limit:.0f} s "
              f"per instance; {solved}/{n_inst} proven optimal inside the cap in the first timed step "
              "(unsolved ones are counted as finished at the cap)")
    gold = gold_optima("C2")
    full = sorted(r["seconds"] for r in gold.values())
    line = {"impl": "reference", "metric": "placement instances/sec", "value": value, "unit": "instances/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "batch_per_step": n_inst, "time_limit_s": limit},
            "cpu_baseline": {"value": value, "unit": "instances/s", "cores": procs, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "instances/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "quality": cpu_quality(recs),
            "seconds_to_proven_optimum": {"median": full[len(full) // 2] if full else None, "max": full[-1] if full else None,
                                          "n": len(full), "source": "tests/golden/mip_optima.json (HiGHS, one process per "
                                          "instance, mip_rel_gap 0, when the fixture was generated in the build container)"}}
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------
def pdhg_roofline(device, host_fn, B, iters, peak, peak_src, in_step=None):
    """Achieved HBM GB/s of the PDHG iteration (C2: k_mf_iter_bulk, the bulk-copy staged pass with the small-vector update
    inside the launch): algorithmic bytes (DESIGN.md section 3b: 64 B per x column + the F*N-sized vectors + d) over the
    CUDA-event time of the solver call."""
    import torch
    X = N_FUNCS * N_NODES * N_NODES
    if in_step is not None:
        ms, it, bytes_iter, note = in_step
    else:
        inst = device.InstanceBatch.from_host(host_fn(B))
        lp = device.slot_relaxation(inst)
        device.pdhg_mf_solve(lp, max_iters=64, check_every=64)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        device.pdhg_mf_solve(lp, max_iters=iters, check_every=iters, eps_rel=1e-12, eps_abs=1e-14)
        e1.record()
        e1.synchronize()
        ms, it = e0.elapsed_time(e1), iters
        bytes_iter = B * (64 * X + 112 * N_FUNCS * N_NODES + 8 * N_NODES * N_NODES)
        note = (f"probe outside the timed steps: the same kernels on {B} C2 instances (working set {B * 32 * X // 1000000} MB "
                f"> L2), {iters} iterations, one solver call timed with CUDA events -- the step's own batch is L2-resident")
    ach = bytes_iter * it / (ms / 1e3) / 1e9
    tpath = os.path.join(ROOT, "profiles", "r02c_pdhg_traffic.json")
    traffic = None
    if os.path.exists(tpath):
        t = json.load(open(tpath))
        traffic = {"dram_bytes_per_iteration": t["per_instance_dram_bytes"] * B, "captured_on": t.get("kernel_build")}
    return {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
            "traffic": traffic["dram_bytes_per_iteration"] if traffic else None, "traffic_source": traffic["captured_on"] if traffic else None,
            "kernel": "PDHG iteration (matrix-free) = k_mf_iter_bulk<RED, FUSE>: one launch per iteration -- x, yS, d and the "
                      "function's vectors staged through shared memory by cp.async.bulk + mbarrier (one producer lane), updated "
                      "in place by the consumer warps, written back by bulk stores, running sums by cp.reduce.async.bulk "
                      "add.f64, the F*N-sized vectors (k_mf_small's arithmetic) updated by two small-vector warps of the same "
                      "launch; tools and tests can still ask for the register passes k_mf_iter2 / k_mf_iter + k_mf_small",
            "bytes_per_iteration": bytes_iter, "iterations_timed": it, "pdhg_ms": ms, "us_per_iteration": 1e3 * ms / it,
            "peak_source": peak_src, "measured": note}


def run_ours(args):
    import ctypes

    import torch
    import torch.distributed as dist

    from neptune_mip_b200 import _lib, device, sharding
    from neptune_mip_b200.batch import BatchParams, solve_batch

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    lib = _lib.load()
    device.lns_block_mode(args.lns_block_mode)

    B = args.batch
    prm = BatchParams(kind="min_delay", lp_iters=args.lp_iters, lp_check_every=256, chains=args.chains, sweeps=args.sweeps,
                      search=args.search, lns_chains=args.lns_chains, lns_rounds=args.lns_rounds, lns_k=args.lns_k,
                      lns_noise=args.lns_noise, lns_phases=args.lns_phases, elites=args.elites, lns_final_k4=args.lns_final_k4)
    # instances are sharded across ranks by seed (weak scaling: B per GPU): rank r owns the contiguous block
    # sharding.shard_range(world*B, r, world) = [r*B, (r+1)*B) -- no data-path collective
    lo, hi = sharding.shard_range(world * B, rank, world)
    host = make_hosts("C2", hi - lo, lo)
    pinned = {k: torch.from_numpy(host[k]).pin_memory() for k in device.InstanceBatch.FIELDS}
    inst = device.InstanceBatch.from_host(host, pinned=pinned)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    cnt = ctypes.c_int64()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        lib.neptune_launch_count(ctypes.byref(cnt), 1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        outs = [fn() for _ in range(steps)]
        e1.record()
        barrier()
        lib.neptune_launch_count(ctypes.byref(cnt), 0)
        ms = e0.elapsed_time(e1)
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), outs, int(cnt.value)

    # ---- device-resident throughput ("value") ---------------------------------------------------------------
    acc = {"pdhg_ms": 0.0, "iters": 0, "bytes": 0, "lns_ms": 0.0, "path": "", "search": ""}

    def step_resident():
        res = solve_batch(inst, prm, time_pdhg=True)
        acc["pdhg_ms"] += res.pdhg_ms
        acc["iters"] += res.pdhg_iters
        acc["bytes"], acc["path"], acc["search"] = res.pdhg_bytes_per_iter, res.pdhg_path, res.search_path
        acc["lns_ms"] += res.lns_ms
        return res

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    for _ in range(args.warmup):
        solve_batch(inst, prm)
    ms_total, outs, launches = timed(step_resident, args.steps, 0)
    clocks = sampler.stop() if sampler else None
    ms_step = ms_total / args.steps
    value = world * B / (ms_step / 1e3)

    # ---- end to end from pinned host buffers through the batched plugin call -------------------------
    d2h = {}

    def step_e2e_pinned():
        ib = device.InstanceBatch(B=B, N=host["N"], F=host["F"], budget=host["budget"],
                                  **{k: pinned[k].to("cuda", non_blocking=True) for k in device.InstanceBatch.FIELDS})
        res = solve_batch(ib, prm)
        out = (res.c.cpu(), res.x.cpu(), res.flags.cpu(), res.scores.cpu())
        d2h["bytes"] = sum(t.numel() * t.element_size() for t in out)
        return out

    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    ms_e2e_total, _, _ = timed(step_e2e_pinned, e2e_steps, 1)
    ms_e2e = ms_e2e_total / e2e_steps
    e2e_value = world * B / (ms_e2e / 1e3)

    # ---- quality of what was computed (parity bar: feasible, objective vs the reference optimum) --------
    last = outs[-1]
    flags = last.flags.cpu().numpy()
    delay = last.scores[:, 0].cpu().numpy()
    quality = {"feasible": int((flags == 63).sum()), "instances": int(B)}
    gold = gold_optima("C2")
    if rank == 0 and gold:
        known = [s for s in sorted(gold) if s < B]
        gaps = {s: (delay[s] - gold[s]["objective"]) / abs(gold[s]["objective"]) for s in known}
        if gaps:
            quality.update(reference_optima_known=len(gaps), max_rel_gap=float(max(gaps.values())),
                           within_1e4=int(sum(g <= 1e-4 for g in gaps.values())),
                           rel_gap_by_seed={str(s): float(f"{g:.3g}") for s, g in gaps.items()})
            if last.lns_round is not None:
                # when the answer was in hand: the LP relaxation of the batch, then the share of the search up to the
                # round at which the chain that produced the returned placement recorded it (rounds have equal length)
                rounds = last.lns_round.cpu().numpy()
                pd_ms, ls_ms = acc["pdhg_ms"] / args.steps, acc["lns_ms"] / args.steps
                total_r = prm.lns_rounds + prm.lns_final_k4
                t14 = {s: pd_ms + ls_ms * min(1.0, (rounds[s] + 1) / max(1, total_r)) for s in known if gaps[s] <= 1e-4}
                if t14:
                    v = sorted(t14.values())
                    quality["time_to_1e4_ms"] = {"median": v[len(v) // 2], "max": v[-1], "reached": len(v), "of": len(known),
                                                 "note": "batch wall time until the returned placement was recorded: LP relaxation + the "
                                                         "search up to that round; null for instances that never get within 1e-4",
                                                 "by_seed": {str(s): (round(t14[s], 1) if s in t14 else None) for s in known}}
            ref_s = sorted(gold[s]["seconds"] for s in known)
            quality["reference_seconds_to_proven_optimum"] = {"median": ref_s[len(ref_s) // 2], "max": ref_s[-1],
                                                              "source": "tests/golden/mip_optima.json: HiGHS, one process per instance, build container"}
    if last.lp is not None:
        lp = last.lp
        # dual objective of the slot-cut relaxation: a lower bound on the MIP optimum up to the remaining dual residual
        quality.update(lp_bound_mean=float(np.mean(lp["dual_obj"])), lp_primal_mean=float(np.mean(lp["primal_obj"])),
                       lp_dual_residual_mean=float(np.mean(lp["dual_res"])), lp_converged=int(lp["converged"].sum()),
                       lp_iterations_max=int(lp["iters"].max()),
                       mean_gap_to_lp_bound=float(np.mean((delay - lp["dual_obj"]) / np.maximum(np.abs(delay), 1e-9))))

    # ---- roofline of the HBM-bound kernel of the path (the PDHG iteration) -----------------------------------
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    X = N_FUNCS * N_NODES * N_NODES
    roof = None
    if acc["iters"] and acc["path"] == "matrix-free":
        if B * 32 * X > L2_BYTES:
            roof = pdhg_roofline(device, None, B, 0, peak, peak_src,
                                 in_step=(acc["pdhg_ms"], acc["iters"], acc["bytes"], "inside the timed steps (CUDA events around the solver call)"))
        elif rank == 0:
            roof = pdhg_roofline(device, lambda b: make_hosts("C2", b, 0), args.probe_batch, 2048, peak, peak_src)
        if roof:
            roof["pdhg_share_of_step"] = acc["pdhg_ms"] / ms_total
            roof["search_share_of_step"] = acc["lns_ms"] / ms_total
            roof["note"] = ("the step is dominated by the search kernel k_lns (shared-memory / issue bound: no HBM or tensor roofline applies, "
                            "profiles/r02_lns_summary.md); the roofline is stated for the HBM-bound kernel of the path")

    line = {"metric": "placement instances/sec", "value": value, "unit": "instances/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "batch_per_gpu": B, "lp_iters_cap": args.lp_iters, "search": acc["search"],
                       "lns_chains": args.lns_chains, "lns_rounds": args.lns_rounds, "lns_k": args.lns_k, "lns_noise": args.lns_noise, "lns_final_k4_rounds": args.lns_final_k4,
                       "elites": args.elites, "lp_path": acc["path"],
                       "l2": ("PDHG working set of the batch (%d MB) exceeds the 126 MB L2" % (B * 32 * X // 1000000)) if B * 32 * X > L2_BYTES else
                             "the step's PDHG working set is L2-resident (the search sets the batch size); the HBM roofline is probed on " + str(args.probe_batch) + " instances, see roofline.measured"},
            "e2e": {"value": e2e_value, "unit": "instances/s", "h2d_bytes_per_step": inst.h2d_bytes(),
                    "d2h_bytes_per_step": d2h.get("bytes", 0), "ms_per_step": ms_e2e, "steps": e2e_steps},
            "gpu_launches": launches, "clocks": clocks, "quality": quality,
            "step_breakdown_ms": {"pdhg": acc["pdhg_ms"] / args.steps, "search_and_pricing": acc["lns_ms"] / args.steps}}
    if roof:
        line["roofline"] = roof

    # ---- the other configs BASELINE.json names, once each (not part of `value`) ------------------------------
    if not args.no_extra:
        extra = {}
        try:
            extra["c5_sweep"] = c5_sweep(args, rank, world, barrier)
        except Exception as e:  # pragma: no cover
            extra["c5_sweep"] = {"error": f"{type(e).__name__}: {e}"}
        if rank == 0:
            try:
                extra["c3_pdhg"] = c3_pdhg(peak)
            except Exception as e:  # pragma: no cover
                extra["c3_pdhg"] = {"error": f"{type(e).__name__}: {e}"}
        if rank == 0 and world == 1:
            try:
                sys.path.insert(0, os.path.join(ROOT, "tools"))
                import c4_placement
                extra["c4_placement"] = c4_placement.record(args.c4_nodes, args.c4_funcs, lp_iters=64)
            except Exception as e:  # pragma: no cover
                extra["c4_placement"] = {"error": f"{type(e).__name__}: {e}"}
        if world > 1:
            try:
                extra["c4_sharded"] = c4_sharded(args, rank, world, peak)
            except Exception as e:  # pragma: no cover
                extra["c4_sharded"] = {"error": f"{type(e).__name__}: {e}"}
        line["sub_records"] = extra

    if rank == 0 and world == 1 and not args.no_cpu:
        procs = max(1, min(os.cpu_count() or 1, 10))
        n_inst = procs
        wall, recs = cpu_reference(n_inst, 15.0, procs)
        line["cpu_baseline"] = {"value": n_inst / wall, "unit": "instances/s", "cores": procs, "kind": "port",
                                "sample": f"{n_inst} C2 instances (seeds 0..{n_inst - 1}), oracle model + HiGHS capped at 15 s each, "
                                          f"{sum(r['optimal'] for r in recs)}/{n_inst} proven optimal inside the cap",
                                "quality_at_cap": cpu_quality(recs)}
    if rank == 0 and args.dump_outputs:
        dump_outputs(last, args.dump_outputs)
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


DUMP_BYTES = 64 << 20


def dump_outputs(res, out_dir):
    """What the last timed step returned to its caller, one float64 `<name>.npy` per array: placement `c`, routing `x`,
    node counts `n`, check `flags`, `scores`, the PDHG records as `lp_<field>` and the search round `lns_round`.  Every
    array has the instance as its first axis; when they would exceed DUMP_BYTES together, a seeded sample of instances is
    kept, and `instances.npy` always lists the instances written."""
    arrays = {"c": res.c, "x": res.x, "n": res.n, "flags": res.flags, "scores": res.scores}
    if res.lp is not None:
        arrays.update({f"lp_{k}": res.lp[k] for k in res.lp.dtype.names if k != "pad"})
    if res.lns_round is not None:
        arrays["lns_round"] = res.lns_round
    arrays = {k: (v.cpu().numpy() if hasattr(v, "cpu") else np.asarray(v)).astype(np.float64) for k, v in arrays.items()}
    B = len(arrays["c"])
    per_instance = sum(v.nbytes for v in arrays.values()) // B
    keep = np.arange(B)
    if per_instance * B > DUMP_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(B, DUMP_BYTES // per_instance, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "instances.npy"), keep.astype(np.float64))
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), v[keep])


def c5_sweep(args, rank, world, barrier):
    """BASELINE config 5: 4096 independent 20x5 instances sharded over the ranks -- EFTTC and the Neptune step-1 path."""
    import torch
    import torch.distributed as dist

    from neptune_mip_b200 import device, sharding
    from neptune_mip_b200.batch import BatchParams, solve_batch
    total = args.c5_instances
    lo, hi = sharding.shard_range(total, rank, world)
    inst = device.InstanceBatch.from_host(make_hosts("C5", hi - lo, lo))

    def timed(fn):
        fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn()
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), out

    ms_e, _ = timed(lambda: device.efttc(inst, "min_delay"))
    prm = BatchParams(kind="min_delay", lp_iters=8192, lp_check_every=256, lns_chains=16, lns_rounds=2000, lns_noise=0.1,
                      elites=8, lns_local_chains=0, lns_final_k4=0)
    ms_n, res = timed(lambda: solve_batch(inst, prm))
    rec = {"workload": f"C5: {total} x (20 nodes x 5 functions), min-delay, sharded over {world} rank(s)",
           "efttc_instances_per_s": total / (ms_e / 1e3), "efttc_ms": ms_e,
           "neptune_instances_per_s": total / (ms_n / 1e3), "neptune_ms": ms_n,
           "neptune_feasible_on_rank0": int((res.flags == 63).sum()), "neptune_instances_on_rank0": hi - lo}
    gold = gold_optima("C5")
    if rank == 0 and gold:
        d = res.scores[:, 0].cpu().numpy()
        gaps = [(d[s] - gold[s]["objective"]) / abs(gold[s]["objective"]) for s in sorted(gold) if s < hi - lo]
        rec.update(reference_optima_known=len(gaps), within_1e4=int(sum(g <= 1e-4 for g in gaps)), max_rel_gap=float(max(gaps)))
    return rec


def c3_pdhg(peak):
    """BASELINE config 3 (500 x 50): the PDHG iteration alone, HBM roofline."""
    import torch

    from neptune_mip_b200 import device, synth
    from neptune_mip_b200.core.utils import data_to_solver_input
    N, F, iters = 500, 50, 2048          # long enough for the solve's set-up and KKT passes (one set per call) to be ~1 % of it
    inst = device.InstanceBatch.from_datas([data_to_solver_input(synth.config_payload("C3", 0), 1, with_db=False)])
    lp = device.slot_relaxation(inst)
    device.pdhg_mf_solve(lp, max_iters=32, check_every=32)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    device.pdhg_mf_solve(lp, max_iters=iters, check_every=iters, eps_rel=1e-12, eps_abs=1e-14)
    e1.record()
    e1.synchronize()
    ms = e0.elapsed_time(e1)
    bytes_iter = 64 * F * N * N + 112 * F * N + 8 * N * N
    ach = bytes_iter * iters / (ms / 1e3) / 1e9
    return {"workload": "C3: 500 nodes x 50 functions, one instance, slot-cut relaxation, matrix-free PDHG", "iterations": iters,
            "us_per_iteration": 1e3 * ms / iters, "bytes_per_iteration": bytes_iter, "achieved_gbs": ach, "frac_of_measured_hbm": ach / peak}


def c4_sharded(args, rank, world, peak):
    """BASELINE config 4 (2000 x 200): function-block-sharded matrix-free PDHG, one all-reduce of 2N doubles per iteration."""
    from neptune_mip_b200 import sharded_mf
    return sharded_mf.bench_record(rank, world, peak, n_nodes=args.c4_nodes, n_funcs=args.c4_funcs, iters=args.c4_iters)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=48,
                    help="instances per GPU per step (48 x 96 chains = 576 search blocks = two full waves of 2 x 148 resident blocks)")
    ap.add_argument("--lp-iters", type=int, default=50000, help="cap on PDHG iterations (the solver stops at 1e-6 relative KKT error)")
    ap.add_argument("--search", default="auto", choices=["auto", "local"])
    ap.add_argument("--lns-chains", type=int, default=96)
    ap.add_argument("--lns-rounds", type=int, default=20000)
    ap.add_argument("--lns-k", type=int, default=3)
    ap.add_argument("--lns-noise", type=float, default=0.1)
    ap.add_argument("--lns-phases", type=int, default=1)
    ap.add_argument("--lns-final-k4", type=int, default=3000, help="rounds of the final phase: one 4-node chain restarted from every record")
    ap.add_argument("--elites", type=int, default=32)
    ap.add_argument("--lns-block-mode", type=int, default=0, choices=[0, 1, 2],
                    help="chains per block of the search kernel: 0 automatic, 1 = 8, 2 = 12 (same results)")
    ap.add_argument("--chains", type=int, default=8, help="add/drop/swap search (--search local)")
    ap.add_argument("--sweeps", type=int, default=400)
    ap.add_argument("--e2e-steps", type=int, default=2, help="steps of the end-to-end leg (at most --steps)")
    ap.add_argument("--probe-batch", type=int, default=296, help="instances of the PDHG roofline probe: two per SM (working set 0.8 MB each, 237 MB > L2); 256 instances measure 4.90 TB/s where 296 measure 5.12")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-extra", action="store_true", help="skip the C5 / C3 / C4 sub-records")
    ap.add_argument("--c5-instances", type=int, default=4096)
    ap.add_argument("--c4-nodes", type=int, default=2000)
    ap.add_argument("--c4-funcs", type=int, default=200)
    ap.add_argument("--c4-iters", type=int, default=64)
    ap.add_argument("--ref-limit", type=float, default=20.0, help="--impl reference: HiGHS cap per instance (s)")
    ap.add_argument("--ref-instances", type=int, default=0, help="--impl reference: instances per step (0 = one per worker)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (rank 0's instances) as DIR/<name>.npy, at most 64 MB")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
