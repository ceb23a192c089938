"""GPU experiment: the passes of the matrix-free PDHG (neptune_pdhg_mf_solve) against each other -- time per
iteration, achieved GB/s and iterate differences of the register, pair and bulk-copy passes at C2 (batch), C3, the
per-GPU share of C4 and C5; the small-vector kernel alone; plain copy ceilings; iterations to 1e-6 on C2 (the bulk
mode also writes its rows to mf_bulk.json).
    python tools/mf_check.py [--variants] [--small-phases] [--bulk-diag] [--bulk] [--ceiling] [--converge]"""
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

from neptune_mip_b200 import device, synth
from neptune_mip_b200._lib import FLAG_STRENGTHEN
from neptune_mip_b200.core.utils import data_to_solver_input

out = {"equality": [], "converged": [], "timing": []}


def batch_of(N, F, B, cores, seed0=0):
    datas = [data_to_solver_input(synth.random_payload(N, F, seed0 + s, node_cores=cores), 1, with_db=False)
             for s in range(B)]
    return device.InstanceBatch.from_datas(datas)


def synth_batch(N, F, B, seed=0):
    """random instance arrays made on the device (large shapes: no payload round trip)"""
    g = torch.Generator(device="cuda").manual_seed(seed)
    f64 = dict(dtype=torch.float64, device="cuda")
    D = torch.randint(1, 50, (B, N, N), generator=g, device="cuda").to(torch.float64)
    D = torch.floor((D + D.transpose(1, 2)) / 2)
    D.diagonal(dim1=1, dim2=2).zero_()
    W = torch.randint(0, 20, (B, F, N), generator=g, device="cuda").to(torch.float64)
    cores = torch.randint(1, 5, (B, F, N), generator=g, device="cuda").to(torch.float64)
    dest = torch.randint(1, 10, (B, F, N), generator=g, device="cuda").to(torch.float64)
    r = cores / dest
    load = (W.sum(dim=2, keepdim=True) * r).sum(dim=1).mean(dim=1, keepdim=True)     # mean CPU need per node
    Kj = torch.ceil(2.5 * load).expand(B, N).contiguous()
    return device.InstanceBatch(B=B, N=N, F=F, d=D.contiguous(), w=W, r=r, m=torch.full((B, F), 30.0, **f64),
                                Mj=torch.full((B, N), 100.0, **f64), Kj=Kj, old=torch.ones((B, F, N), **f64),
                                maxd=torch.full((B, F), 1000.0, **f64), cost=torch.full((B, N), 5.0, **f64),
                                budget=300.0)


def timed(fn):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    r = fn()
    e1.record()
    e1.synchronize()
    return r, e0.elapsed_time(e1)


def bytes_iter(inst):
    X = inst.F * inst.N * inst.N
    return inst.B * (64 * X + 112 * inst.F * inst.N + 8 * inst.N ** 2)


def variants():
    """the two iteration passes, one and two rows of a warp in flight; the small-vector kernel alone"""
    for name, inst, iters in (("C2 batch 256", synth_batch(50, 10, 256), 512), ("C3 500x50", synth_batch(500, 50, 1), 256),
                              ("C4 share 2000x25", synth_batch(2000, 25, 1), 64), ("C5 4096 x 20x5", synth_batch(20, 5, 4096), 256)):
        ref = None
        for scalar in (True, False):
            for u in (1, 2):
                kw = dict(scalar_kernel=scalar, rows_in_flight=u)
                device.pdhg_mf_solve(inst, max_iters=32, check_every=32, **kw)
                (xu, yu, _), ms = timed(lambda: device.pdhg_mf_solve(inst, max_iters=iters, check_every=iters, eps_rel=1e-12, eps_abs=1e-14, **kw))
                if ref is None:
                    ref = (xu, yu)
                print("VAR", name, "8-byte pass" if scalar else "default pass (pairs where N is even and 33..64)", "rows in flight", u,
                      "us/iter %.1f" % (1e3 * ms / iters), "GB/s %.0f" % (bytes_iter(inst) * iters / ms / 1e6),
                      "max |dx| vs first %.1e" % float((xu - ref[0]).abs().max()), "max |dy| %.1e" % float((yu - ref[1]).abs().max()), flush=True)
        device.pdhg_mf_solve(inst, max_iters=32, check_every=32, _diag=4)
        _, ms = timed(lambda: device.pdhg_mf_solve(inst, max_iters=iters, check_every=iters, eps_rel=1e-12, eps_abs=1e-14, _diag=4))
        print("VAR", name, "small-vector kernel alone us/iter %.1f" % (1e3 * ms / iters), flush=True)


def bulk():
    """the bulk-copy staged pass (csrc/pdhg_mf_bulk.cuh) against the pair pass: time per iteration and iterate difference,
    over consumer-warp counts and stage caps"""
    rows = []
    for name, inst, iters in (("C2 batch 256", synth_batch(50, 10, 256), 512), ("64x10 batch 128", synth_batch(64, 10, 128), 256),
                              ("34x10 batch 512", synth_batch(34, 10, 512), 256), ("C2 batch 48 (L2-resident)", synth_batch(50, 10, 48), 512)):
        kwt = dict(max_iters=iters, check_every=iters, eps_rel=1e-12, eps_abs=1e-14)
        device.pdhg_mf_solve(inst, max_iters=32, check_every=32, register_pass=True)
        (xr, yr, _), ms = timed(lambda: device.pdhg_mf_solve(inst, register_pass=True, **kwt))
        (_, _, _), ms2 = timed(lambda: device.pdhg_mf_solve(inst, register_pass=True, **kwt))
        ms = min(ms, ms2)
        print("BULK", name, "pair pass (registers) us/iter %.1f GB/s %.0f" % (1e3 * ms / iters, bytes_iter(inst) * iters / ms / 1e6), flush=True)
        rows.append({"shape": name, "pass": "pair", "us_per_iter": 1e3 * ms / iters, "gbs": bytes_iter(inst) * iters / ms / 1e6})
        full = name.startswith("C2 batch 256")
        for mode in (2, 1):
            for warps in ((0, 8, 10, 15) if full else (0,)):
                for cap in ((0, 3, 2) if (full and warps == 0) else (0,)):
                    kw = dict(bulk=mode, bulk_warps=warps, bulk_stages=cap)
                    try:
                        device.pdhg_mf_solve(inst, max_iters=32, check_every=32, **kw)
                        (xb, yb, _), ms = timed(lambda: device.pdhg_mf_solve(inst, **kw, **kwt))
                        (_, _, _), ms2 = timed(lambda: device.pdhg_mf_solve(inst, **kw, **kwt))
                    except Exception as e:          # a trap inside the kernel poisons the context: stop here
                        print("BULK", name, kw, "FAILED", repr(e), flush=True)
                        raise
                    ms = min(ms, ms2)
                    dx, dy = float((xb - xr).abs().max()), float((yb - yr).abs().max())
                    print("BULK", name, "bulk mode %d (%s) warps %d stage cap %d" % (mode, "sums by bulk reduction" if mode == 2 else "four streams staged", warps, cap),
                          "us/iter %.1f GB/s %.0f" % (1e3 * ms / iters, bytes_iter(inst) * iters / ms / 1e6), "max |dx| %.1e |dy| %.1e vs pair" % (dx, dy), flush=True)
                    rows.append({"shape": name, "pass": "bulk%d" % mode, "warps": warps, "stage_cap": cap, "us_per_iter": 1e3 * ms / iters,
                                 "gbs": bytes_iter(inst) * iters / ms / 1e6, "max_dx": dx, "max_dy": dy})
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    json.dump(rows, open(os.path.join(ROOT, "gpurun_out", "mf_bulk.json"), "w"), indent=1)


def bulk_diag():
    """where the bulk-copy pass spends its time: arithmetic only (no copies), copy-through (no arithmetic), loads only"""
    inst, iters = synth_batch(50, 10, 256), 512
    kwt = dict(max_iters=iters, check_every=iters, eps_rel=1e-12, eps_abs=1e-14)
    for mode in (1, 2):
        for diag, what in ((0, "full"), (1, "arithmetic only (no copies)"), (2, "copy through (no arithmetic)"), (3, "loads only")):
            for cap in (0, 2):
                for warps in ((0, 8) if diag == 1 else (0,)):
                    for unfused in (False, True):
                        kw = dict(bulk=mode, bulk_stages=cap, bulk_warps=warps, _diag=diag, unfused_small=unfused)
                        device.pdhg_mf_solve(inst, max_iters=32, check_every=32, **kw)
                        _, ms = timed(lambda: device.pdhg_mf_solve(inst, **kw, **kwt))
                        print("BDIAG C2 batch 256 mode %d stage cap %d warps %d %s %s us/iter %.1f" % (mode, cap, warps, "small vectors in their own launch" if unfused else "small vectors inside the pass", what, 1e3 * ms / iters), flush=True)
    device.pdhg_mf_solve(inst, max_iters=32, check_every=32, _diag=4)
    _, ms = timed(lambda: device.pdhg_mf_solve(inst, _diag=4, **kwt))
    print("BDIAG small-vector kernel alone us/iter %.1f" % (1e3 * ms / iters), flush=True)


def small_phases():
    """the small-vector kernel alone, phase by phase (NEPTUNE_SMALL_MASK: 1 POST, 2 PREC, 4 Y2), at C3 and the C4 share"""
    for name, inst, iters in (("C3 500x50", synth_batch(500, 50, 1), 256), ("C4 share 2000x25", synth_batch(2000, 25, 1), 64)):
        for mask in (7, 1, 2, 4, 3):
            os.environ["NEPTUNE_SMALL_MASK"] = str(mask)
            device.pdhg_mf_solve(inst, max_iters=32, check_every=32, _diag=4)
            _, ms = timed(lambda: device.pdhg_mf_solve(inst, max_iters=iters, check_every=iters, eps_rel=1e-12, eps_abs=1e-14, _diag=4))
            print("SMALL", name, "phases mask", mask, "us/iter %.1f" % (1e3 * ms / iters), flush=True)
        os.environ.pop("NEPTUNE_SMALL_MASK", None)
        _, ms = timed(lambda: device.pdhg_mf_solve(inst, max_iters=iters, check_every=iters, eps_rel=1e-12, eps_abs=1e-14))
        print("SMALL", name, "whole iteration us/iter %.1f GB/s %.0f" % (1e3 * ms / iters, bytes_iter(inst) * iters / ms / 1e6), flush=True)


def ceiling():
    """what plain torch kernels reach on this box for copy / read-modify-write streams"""
    n = 1 << 27
    a = torch.empty(n, dtype=torch.float64, device="cuda"); b = torch.empty_like(a)

    def rate(fn, nbytes, reps=10):
        fn(); best = 1e9
        for _ in range(reps):
            _, ms = timed(fn); best = min(best, ms)
        return nbytes / best / 1e6
    print("CEIL copy 1 GiB f64 (read + write) GB/s %.0f" % rate(lambda: b.copy_(a), 16 * n), flush=True)
    m = 256 * 25000
    xs = [torch.zeros(m, dtype=torch.float64, device="cuda") for _ in range(4)]
    print("CEIL a.add_(b) on 51 MB streams (2 reads + 1 write) GB/s %.0f" % rate(lambda: (xs[0].add_(xs[1]), xs[2].add_(xs[3])), 2 * 24 * m), flush=True)


def converge():
    """iterations to 1e-6 on the slot-cut relaxation of C2 (what the solve path runs)"""
    from neptune_mip_b200.core.utils import data_to_solver_input as d2s
    inst = device.InstanceBatch.from_datas([d2s(synth.config_payload("C2", s), 1, with_db=False) for s in range(16)])
    for cut in (False, True):
        lp = device.slot_relaxation(inst) if cut else inst
        (_, _, res), ms = timed(lambda: device.pdhg_mf_solve(lp, max_iters=60000, check_every=256, eps_rel=1e-6, eps_abs=1e-9))
        print("CONV C2 seeds 0-15", "slot-cut" if cut else "memory rows", "iters", res["iters"].tolist(), "converged", int(res["converged"].sum()),
              "bound", [round(float(v), 1) for v in res["dual_obj"][:4]], "ms %.0f" % ms, flush=True)


if __name__ == "__main__":
    torch.cuda.set_device(0)
    t0 = time.time()
    if "--variants" in sys.argv:
        variants()
    if "--small-phases" in sys.argv:
        small_phases()
    if "--bulk-diag" in sys.argv:
        bulk_diag()
    if "--bulk" in sys.argv:
        bulk()
    if "--ceiling" in sys.argv:
        ceiling()
    if "--converge" in sys.argv:
        converge()
    print("mf_check done in %.1f s" % (time.time() - t0))
