"""(c2) The slot-count search with its chain state in global memory (`neptune_lns_search_global`, csrc/lns.cu) and the
`search="lns"` solve path built on it.

CPU: the workspace size is the closed form of its layout at C2, C3 and C4; kind 1, N = 65535 and a short workspace are
refused.  GPU: on every case of the shared-memory kernel's golden the records are the golden's bit for bit (so the two
kernels compute the same thing); the same for the combined objective with an LP guide and prices; at C3 the routing each
record was certified with is feasible and its delay is the record's upper bound; runs are reproducible; the solve path
at C3 and C4 passes the min-delay checks between the LP bound and the site placement's objective."""
import ctypes
import hashlib
import json
import os

import numpy as np
import pytest

from helpers import cuda_batch
from neptune_mip_b200 import _lib, synth

HERE = os.path.dirname(os.path.abspath(__file__))


# ---- CPU: size arithmetic and refusals ----------------------------------------------------------------------------

def _a(v, q):
    return (v + q - 1) // q * q


def closed_form_workspace(B, N, F, chains, k, max_slots):
    """per instance: transposed delays, largest delay within maxd per source, slot counts, 4 scalars (each section
    aligned to 256 bytes); per chain: lam, loadfx, bestv, scratch, ints, pod ids (uint16), placement, DP tables"""
    fn, smax = F * N, 4 ** k
    ms = max_slots if 0 < max_slots < F else F
    tn = ms * N
    scratch = _a(max(F * 2 ** k * 8 + smax * 8, max(tn * 4 + tn * 4, fn * 4)), 16)
    chain = 16 * N + _a(4 * fn, 16) + scratch + (2 * F + 33) * 4 + 2 * fn + _a(fn, 2) + 2 * fn + F * smax + smax + 2 * F + 16
    return (_a(B * N * N * 8, 256) + _a(B * fn * 8, 256) + _a(B * N * 4, 256) + _a(B * 32, 256)
            + B * chains * _a(_a(chain, 16), 256))


@pytest.mark.parametrize("B,N,F,chains,k,max_slots", [(32, 50, 10, 96, 3, 3), (2, 500, 50, 16, 3, 3), (1, 2000, 200, 8, 4, 3),
                                                      (1, 2000, 200, 8, 3, 0), (1, 501, 51, 5, 2, 7)])
def test_workspace_bytes_closed_form(B, N, F, chains, k, max_slots):
    lib = _lib.load()
    need = ctypes.c_int64()
    assert lib.neptune_lns_search_global_workspace_bytes(B, N, F, chains, k, max_slots, ctypes.byref(need)) == 0
    assert need.value == closed_form_workspace(B, N, F, chains, k, max_slots)


def test_refusals_without_a_device():
    lib = _lib.load()
    need = ctypes.c_int64()
    assert lib.neptune_lns_search_global_workspace_bytes(1, 65534, 2, 1, 3, 0, ctypes.byref(need)) == 0
    assert lib.neptune_lns_search_global_workspace_bytes(1, 65535, 2, 1, 3, 0, ctypes.byref(need)) == -2
    assert lib.neptune_lns_search_global_workspace_bytes(1, 50, 10, 1, 5, 0, ctypes.byref(need)) == -1
    p = ctypes.c_void_p(16)          # never dereferenced: every refusal happens before a launch

    def call(N, kind, ws_bytes):
        return lib.neptune_lns_search_global(1, N, 10, kind, ctypes.c_double(0.5), 8, 10, 3, ctypes.c_double(0.1),
                                             ctypes.c_uint64(1), p, p, p, p, p, p, None, None, None, 0, None, 0,
                                             p, p, None, p, p, p, ws_bytes, None)
    assert lib.neptune_lns_search_global_workspace_bytes(1, 50, 10, 8, 3, 0, ctypes.byref(need)) == 0
    assert call(50, 1, need.value) == -1                 # min-utilisation: no delay term to price
    assert call(65535, 0, 1 << 40) == -2                 # pod ids are 16 bits, 0xFFFF = none
    assert call(50, 0, need.value - 1) == -3             # workspace too small


# ---- GPU ----------------------------------------------------------------------------------------------------------

def _digest(c, g, lb, rnd):
    return {"out_c_sha256": hashlib.sha256(c.cpu().numpy().tobytes()).hexdigest(),
            "out_g": [float(v).hex() for v in g.cpu().flatten().tolist()],
            "out_lb": [float(v).hex() for v in lb.cpu().flatten().tolist()],
            "out_round": [int(v) for v in rnd.cpu().flatten().tolist()]}


@pytest.mark.gpu
def test_records_equal_the_shared_memory_golden():
    """every case of the shared-memory kernel's golden, through the global-state kernel (block mode does not apply)"""
    from neptune_mip_b200 import device
    from test_lns_records_gpu import CASES, GOLD, _instances
    want = json.load(open(GOLD))
    insts, raw = {}, {}
    for case, (iname, k, chains, rounds, _mode, rng, seeds_from) in CASES.items():
        inst = insts.setdefault(iname, _instances(iname))
        seeds = raw[seeds_from].contiguous() if seeds_from else None
        c, g, rnd, _ = device.lns_search_global(inst, "min_delay", chains=chains, rounds=rounds, k=k, noise_coef=0.1,
                                                rng_seed=rng, seeds_u8=seeds)
        raw[case] = c
        got = _digest(c, g, device.lns_search_global.last_other_bound, rnd)
        for key in ("out_round", "out_g", "out_lb", "out_c_sha256"):
            assert got[key] == want[case][key], (case, key)


@pytest.mark.gpu
def test_combined_objective_equals_the_shared_memory_kernel():
    """kind 2 with an LP guide and CPU-row prices (the golden covers min-delay only): both kernels, same records"""
    import torch
    from neptune_mip_b200 import device
    from neptune_mip_b200.batch import objective_weights
    inst = cuda_batch([synth.config_payload("C2", s) for s in (1, 2)])
    N, F = inst.N, inst.F
    xs, ys, _ = device.pdhg_mf_solve(device.slot_relaxation(inst), max_iters=512, check_every=128, kind=2, alpha=0.5,
                                     node_cut=True)
    guide = xs[:, F * N * N:F * N * N + F * N].contiguous()
    a_d = objective_weights(inst, 2, 0.5)[0]
    lam0 = (ys[:, 3 * F * N + N:3 * F * N + 2 * N] / a_d[:, None]).contiguous()
    kw = dict(alpha=0.5, chains=24, rounds=500, k=3, noise_coef=0.1, rng_seed=5, guide=guide, lam0=lam0)
    c1, g1, r1 = device.lns_search(inst, "min_delay_util", **kw)
    lb1 = device.lns_search.last_other_bound
    c2, g2, r2, _ = device.lns_search_global(inst, "min_delay_util", **kw)
    lb2 = device.lns_search_global.last_other_bound
    assert torch.isfinite(g1).any()
    assert torch.equal(c1, c2) and torch.equal(r1, r2)
    assert torch.equal(g1, g2) and torch.equal(lb1, lb2)


def _c3(seeds=(0, 1)):
    return cuda_batch([synth.config_payload("C3", s) for s in seeds])


@pytest.mark.gpu
def test_certified_routing_at_c3():
    """the routing each record was taken with passes the min-delay checks, its delay is the record's upper bound, and the
    exact routing LP of the placement is no larger"""
    import torch
    from neptune_mip_b200 import device
    from neptune_mip_b200.batch import MIN_DELAY_FLAGS
    inst = _c3()
    chains = 8
    c, g, _, asg = device.lns_search_global(inst, "min_delay", chains=chains, rounds=150, k=3, noise_coef=0.1, rng_seed=3)
    other = device.lns_search_global.last_other_bound
    ub = torch.cat([g[:, :chains], other[:, chains:]], dim=1)       # the whole-flow value of every record
    assert torch.isfinite(g).any()
    pr = device.route_lp(inst, c)
    checked = 0
    for rec in range(2 * chains):
        if not bool(torch.isfinite(g[:, rec]).all()):
            continue
        cc, x, n = device.routing_of_assignment(inst, asg[:, rec].contiguous())
        assert torch.equal(cc & c[:, rec], cc)                       # only pods of the record are used
        flags, scores = device.check_solution(inst, x, device.u8_to_f64(cc), n)
        assert bool(((flags & MIN_DELAY_FLAGS) == MIN_DELAY_FLAGS).all()), (rec, flags)
        delay = scores[:, 0]
        assert torch.allclose(delay, ub[:, rec], rtol=1e-9, atol=0.0), (rec, delay, ub[:, rec])
        ok = pr["status"][:, rec] == 1
        assert bool((pr["obj"][:, rec][ok] <= delay[ok] * (1 + 1e-9)).all())
        checked += 1
    assert checked > 0


@pytest.mark.gpu
def test_reproducible_at_c3():
    import torch
    from neptune_mip_b200 import device
    inst = _c3((2,))
    kw = dict(chains=8, rounds=100, k=3, noise_coef=0.1)
    a = device.lns_search_global(inst, "min_delay", rng_seed=7, **kw)
    b = device.lns_search_global(inst, "min_delay", rng_seed=7, **kw)
    d = device.lns_search_global(inst, "min_delay", rng_seed=8, **kw)
    assert all(torch.equal(u, v) for u, v in zip(a, b))
    assert not torch.equal(a[0], d[0]) or not torch.equal(a[1], d[1])


def _site_objective(inst):
    from neptune_mip_b200 import device
    cg, _ = device.site_greedy(inst)
    cs, _, _ = device.site_search(inst, cg)
    c2, x, n, _, _, _ = device.route_two_choice(inst, cs)
    _, sc = device.check_solution(inst, x, device.u8_to_f64(c2), n)
    return sc[:, 0].cpu().numpy()


def _check_solve(inst, prm):
    from neptune_mip_b200.batch import MIN_DELAY_FLAGS, solve_batch
    res = solve_batch(inst, prm)
    assert res.search_path == "lns"
    flags = res.flags.cpu().numpy()
    assert np.all((flags & MIN_DELAY_FLAGS) == MIN_DELAY_FLAGS), flags
    got = res.scores[:, 0].cpu().numpy()
    assert np.all(got >= res.lp["dual_obj"] * (1 - 1e-9)), (got, res.lp["dual_obj"])
    assert np.all(got <= _site_objective(inst) * (1 + 1e-12)), got
    again = solve_batch(inst, prm)
    assert np.array_equal(again.c.cpu().numpy(), res.c.cpu().numpy())
    return res


@pytest.mark.gpu
def test_solve_path_at_c3():
    from neptune_mip_b200.batch import BatchParams
    _check_solve(_c3(), BatchParams(search="lns", lp_iters=2048, lns_chains=16, lns_rounds=300, lns_final_k4=50, elites=8))


@pytest.mark.gpu
def test_solve_path_at_c4():
    from neptune_mip_b200.batch import BatchParams
    inst = cuda_batch([synth.config_payload("C4", 0)])
    _check_solve(inst, BatchParams(search="lns", lp_iters=256, lns_chains=8, lns_rounds=60, lns_final_k4=0, elites=4))


@pytest.mark.gpu
def test_class_at_c3_returns():
    """the drop-in class with search="lns" at C3 size (budget raised: the adapter's default budget is about the number
    of nodes, not about the search)"""
    from neptune_mip_b200.core.solvers import NeptuneStep1CPUMinDelay
    from neptune_mip_b200.core.utils import data_to_solver_input
    data = data_to_solver_input(synth.config_payload("C3", 0), 1, with_db=False)
    data.node_budget = 1e9
    s = NeptuneStep1CPUMinDelay(search="lns", lp_iters=1024, lns_chains=16, lns_rounds=200, lns_final_k4=0, elites=8,
                                verbose=False)
    s.load_data(data)
    assert s.solve() == True        # noqa: E712
