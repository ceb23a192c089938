#!/usr/bin/env python
"""BASELINE config 4 (2000 nodes x 200 functions) on ONE GPU: what the pod-exchange search adds to the greedy placement.

  greedy (k_site_*) -> pod-exchange search (k_ss_*, csrc/site_search.cu) -> two-choice routing (k_tc_*) -> checkers
  -> lower bound of the slot-cut LP relaxation after --lp-iters matrix-free PDHG iterations.

Prints one JSON object: nearest-pod and routed objectives of the greedy and of the searched placement, the search's
rounds and moves by kind, device times of every stage, the LP bound and the gap.  `--c2` instead prints the gaps to the
HiGHS optima of the 15 C2 seeds (tests/golden/mip_optima.json) of greedy + two-choice, of the pod-exchange path and of
the default (slot-count LNS) path.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def gpu_info():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def timed(fn):
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record(); out = fn(); e1.record(); e1.synchronize()
    return e0.elapsed_time(e1), out


def routed(inst, c):
    from neptune_mip_b200 import device
    ms_r, (c2, x, n, obj, feas, iters) = timed(lambda: device.route_two_choice(inst, c))
    ms_c, (flags, scores) = timed(lambda: device.check_solution(inst, x, device.u8_to_f64(c2), n))
    del x
    return dict(objective=float(scores.cpu()[0, 0]), routing_feasible=bool(int(feas.cpu()[0])), routing_iterations=iters,
                flags=int(flags.cpu()[0]), ms_routing=ms_r, ms_checkers=ms_c)


def record(n_nodes=2000, n_funcs=200, lp_iters=512, seed=0):
    import torch
    from neptune_mip_b200 import device, synth
    from neptune_mip_b200.batch import MIN_DELAY_FLAGS
    from neptune_mip_b200.core.utils import data_to_solver_input

    data = data_to_solver_input(synth.random_payload(n_nodes, n_funcs, seed, node_cores=None), 1, with_db=False)
    inst = device.InstanceBatch.from_datas([data])
    device.site_search(inst, device.site_greedy(inst)[0], max_rounds=1)                          # module load
    ms_g, (cg, ginfo) = timed(lambda: device.site_greedy(inst))
    ms_s, (cs, info, obj) = timed(lambda: device.site_search(inst, cg))
    ms_s2, (cs2, info2, obj2) = timed(lambda: device.site_search(inst, cg))
    rg, rs = routed(inst, cg), routed(inst, cs)
    info = info.cpu()[0].tolist()
    rec = {"workload": f"{n_nodes} nodes x {n_funcs} functions, seed {seed}, one instance, one GPU", "gpu": gpu_info(),
           "greedy": {"rounds": int(ginfo.cpu()[0, 0]), "pods": int(cg.sum()), "ms": ms_g,
                      "nearest_pod_objective": float(obj.cpu()[0, 0]), "routed": rg},
           "search": {"rounds_with_moves": info[0], "adds": info[1], "exchanges": info[2], "relocations": info[3],
                      "ms": ms_s, "ms_second_run": ms_s2, "ms_per_round": ms_s / max(info[0], 1),
                      "identical_second_run": bool(torch.equal(cs, cs2) and torch.equal(obj, obj2) and torch.equal(info2.cpu()[0], torch.tensor(info, dtype=torch.int32))),
                      "pods": int(cs.sum()), "nearest_pod_objective": float(obj.cpu()[0, 1]), "routed": rs},
           "note": "ms: CUDA events around each call, one call after a warm-up of both kernels' modules; the search's "
                   "ms_per_round divides by the rounds that moved a pod (the host stops within 4 rounds of the last one)"}
    rec["search"]["nearest_pod_gain"] = 1.0 - rec["search"]["nearest_pod_objective"] / rec["greedy"]["nearest_pod_objective"]
    rec["search"]["routed_gain"] = 1.0 - rs["objective"] / rg["objective"]
    rec["search"]["model_checks_pass"] = (rs["flags"] & MIN_DELAY_FLAGS) == MIN_DELAY_FLAGS
    if lp_iters > 0:
        lp = device.slot_relaxation(inst)
        ms_lp, (_, _, sol) = timed(lambda: device.pdhg_mf_solve(lp, max_iters=lp_iters, check_every=min(lp_iters, 256)))
        bound = float(sol["dual_obj"][0])
        rec["lp"] = {"iterations": int(sol["iters"][0]), "ms": ms_lp, "dual_bound": bound, "primal_obj": float(sol["primal_obj"][0]),
                     "converged": bool(sol["converged"][0]),
                     "gap_greedy": (rg["objective"] - bound) / rg["objective"],
                     "gap_searched": (rs["objective"] - bound) / rs["objective"],
                     "note": "slot-cut relaxation; the dual objective (box terms included) is a lower bound at every iterate"}
    return rec


def c2_record():
    import numpy as np
    from neptune_mip_b200 import device, synth
    from neptune_mip_b200.batch import BatchParams, solve_batch
    from neptune_mip_b200.core.utils import data_to_solver_input
    gold = {r["seed"]: r for r in json.load(open(os.path.join(ROOT, "tests", "golden", "mip_optima.json")))
            if r["config"] == "C2" and r["optimal"]}
    seeds = sorted(gold)
    opt = np.array([gold[s]["objective"] for s in seeds])
    inst = device.InstanceBatch.from_datas([data_to_solver_input(synth.config_payload("C2", s), 1, with_db=False) for s in seeds])
    cg, _ = device.site_greedy(inst)
    cg2, x, n, _, _, _ = device.route_two_choice(inst, cg)
    greedy = device.check_solution(inst, x, device.u8_to_f64(cg2), n)[1][:, 0].cpu().numpy()
    ms_site, site = timed(lambda: solve_batch(inst, BatchParams(search="site", lp_iters=0)))
    ms_lns, lns = timed(lambda: solve_batch(inst, BatchParams()))

    def gaps(v):
        g = (v - opt) / opt
        return {"mean": float(g.mean()), "max": float(g.max()), "per_seed": [float(f"{x:.3e}") for x in g]}
    return {"workload": f"C2 (50 x 10), seeds {seeds} with proven HiGHS optima, one batch, one GPU", "gpu": gpu_info(),
            "greedy_two_choice": gaps(greedy),
            "site_search_two_choice": dict(gaps(site.scores[:, 0].cpu().numpy()), ms=ms_site, path=site.search_path),
            "default_path": dict(gaps(lns.scores[:, 0].cpu().numpy()), ms=ms_lns, path=lns.search_path),
            "note": "gap = (routed objective - optimum) / optimum; ms: whole solve_batch call of the 15-instance batch "
                    "(the pod-exchange row without the LP: lp_iters=0; the default row with its 2048 LP iterations)"}


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--nodes", type=int, default=2000)
    ap.add_argument("--funcs", type=int, default=200)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--lp-iters", type=int, default=512)
    ap.add_argument("--c2", action="store_true", help="the C2 comparison instead of the C4 record")
    a = ap.parse_args()
    print(json.dumps(c2_record() if a.c2 else record(a.nodes, a.funcs, a.lp_iters, a.seed)))
