"""GPU measurement of the slot-count search with its chain state in global memory (`search="lns"` at C3 / C4 sizes).

usage: python tools/lns_global.py [out.json]          (default profiles/r04_lns_global.json)

Records, with the card's name and power limit read in the same run:
  * C3 seeds 0-3 (one batch of four): objective and wall time of search="auto" (the add/drop/swap search at this size)
    against search="lns" at two budgets, next to the slot-cut LP relaxation's dual objective (gap to the bound);
  * C4 seed 0: the site path (greedy -> pod-exchange search -> two-choice routing) against search="lns";
  * time per chain-round: C2 (both kernels, same records), C3 and C4 (global-state kernel)."""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT]

import numpy as np  # noqa: E402
import torch  # noqa: E402

from neptune_mip_b200 import device, synth  # noqa: E402
from neptune_mip_b200.batch import MIN_DELAY_FLAGS, BatchParams, solve_batch  # noqa: E402
from neptune_mip_b200.core.utils import data_to_solver_input  # noqa: E402


def batch(name, seeds):
    return device.InstanceBatch.from_datas([data_to_solver_input(synth.config_payload(name, s), 1, with_db=False) for s in seeds])


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, time.perf_counter() - t0


def solve_record(inst, prm):
    res, sec = timed(lambda: solve_batch(inst, prm))
    flags = res.flags.cpu().numpy()
    return dict(search_path=res.search_path, seconds=sec, objective=res.scores[:, 0].cpu().tolist(),
                min_delay_checks_pass=[bool((f & MIN_DELAY_FLAGS) == MIN_DELAY_FLAGS) for f in flags],
                lp_dual_obj=[float(v) for v in res.lp["dual_obj"]] if res.lp is not None else None,
                lp_converged=[int(v) for v in res.lp["converged"]] if res.lp is not None else None)


def round_time(inst, chains, rounds, shared):
    """kernel wall time of one search call / rounds: every chain of the batch runs concurrently"""
    fn = device.lns_search if shared else device.lns_search_global
    kw = dict(chains=chains, k=3, noise_coef=0.1, rng_seed=1)
    fn(inst, "min_delay", rounds=2, **kw)                  # warm-up (module load, allocations)
    out, sec = timed(lambda: fn(inst, "min_delay", rounds=rounds, **kw))
    return dict(kernel="k_lns" if shared else "k_lns_global", B=inst.B, chains=chains, rounds=rounds, seconds=sec,
                ms_per_round=1e3 * sec / rounds), out


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r04_lns_global.json")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    rep = dict(gpu=dict(device=torch.cuda.get_device_name(0), nvidia_smi=smi))

    # ---- time per chain-round ------------------------------------------------------------------------------------
    c2 = batch("C2", range(32))
    a, ra = round_time(c2, 96, 1000, shared=True)
    b, rb = round_time(c2, 96, 1000, shared=False)
    b["records_equal_k_lns"] = bool(all(torch.equal(u, v) for u, v in zip(ra[:3], rb[:3])))
    del c2
    c3 = batch("C3", range(4))
    c3r, _ = round_time(c3, 64, 200, shared=False)
    c4 = batch("C4", [0])
    c4r, _ = round_time(c4, 64, 20, shared=False)
    rep["chain_round"] = dict(c2_shared=a, c2_global=b, c3_global=c3r, c4_global=c4r)
    torch.cuda.empty_cache()

    # ---- C3 seeds 0-3: add/drop/swap against the slot-count search ------------------------------------------------
    lp = 4096
    budgets = {"small": dict(lns_chains=32, lns_rounds=1000, lns_final_k4=0, elites=8),
               "large": dict(lns_chains=96, lns_rounds=4000, lns_final_k4=500, elites=16)}
    c3rep = dict(instances="C3 (500 x 50) seeds 0-3, one batch", lp_iters=lp,
                 auto=solve_record(c3, BatchParams(search="auto", lp_iters=lp)))
    for name, kw in budgets.items():
        c3rep["lns_" + name] = dict(params=kw, **solve_record(c3, BatchParams(search="lns", lp_iters=lp, **kw)))
    bound = np.array(c3rep["lns_small"]["lp_dual_obj"])
    for key in ("auto", "lns_small", "lns_large"):
        c3rep[key]["gap_to_slot_cut_lp_bound"] = ((np.array(c3rep[key]["objective"]) - bound) / bound).tolist()
    rep["c3"] = c3rep
    torch.cuda.empty_cache()

    # ---- C4 seed 0: site path against the slot-count search -------------------------------------------------------
    c4rep = dict(instances="C4 (2000 x 200) seed 0", lp_iters=256,
                 site=solve_record(c4, BatchParams(search="site", lp_iters=256)))
    torch.cuda.empty_cache()
    kw = dict(lns_chains=64, lns_rounds=300, lns_final_k4=0, elites=4)
    c4rep["lns"] = dict(params=kw, **solve_record(c4, BatchParams(search="lns", lp_iters=256, **kw)))
    bound = np.array(c4rep["lns"]["lp_dual_obj"])
    for key in ("site", "lns"):
        c4rep[key]["gap_to_lp_dual_obj"] = ((np.array(c4rep[key]["objective"]) - bound) / bound).tolist()
    rep["c4"] = c4rep

    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as fh:
        json.dump(rep, fh, indent=1)
    print(json.dumps(rep, indent=1))


if __name__ == "__main__":
    main()
