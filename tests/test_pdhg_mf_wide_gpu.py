"""Matrix-free PDHG (`neptune_pdhg_mf_solve`) at the shapes C3 and C4 run: every branch the solver takes only there --
four strided columns per lane (odd N > 64), the C4 dual summed in 16 slices per column (F * rt > 64 partials), the
small-vector update on many blocks with the C2 dual in its own launch (F * N > 4096), the bulk-copy pass with many
functions, many column tiles -- against the numpy statement of the iteration (tests/mf_reference.py).  Each case reads
the tile geometry the library chooses for its batch and asserts the branch it is meant to cover, so a change of the
geometry heuristics cannot silently move a case off its branch.

Also: the restarted solve against `mf_reference.solve_ctl`, the device's control logic stated in numpy (same
iteration count, restart count and primal weight), and bitwise batch independence on the wide branches."""
import ctypes
import functools

import numpy as np
import pytest

from helpers import arrays_of, cuda_batch, float_payload
from mf_reference import MatrixFree, node_cut_bigm, run_fixed, solve_ctl
from neptune_mip_b200 import synth

pytestmark = pytest.mark.gpu

UNREACHABLE = dict(eps_rel=1e-13, eps_abs=1e-15)


def loaded_payload(N, F, seed, capacity=0.25, function_memory=45):
    """`synth.random_payload` with the CPU capacity of every node cut to `capacity` times the generator's default
    (which is 2.5 x the mean demand per node) and memory for two functions per node: the C4 rows bind within the first
    iterations, and the C2 rows as soon as the c columns grow, so both coupling duals leave zero."""
    auto = synth.random_payload(N, F, seed, node_cores=None)["node_cores"][0]
    return synth.random_payload(N, F, seed, node_cores=max(1, int(round(auto * capacity))), function_memory=function_memory)


def geometry(B, N, F):
    """The branches `neptune_pdhg_mf_geometry` reports for a min-delay solve of B instances of N x F."""
    from neptune_mip_b200 import _lib
    out = (ctypes.c_int32 * 16)()
    assert _lib.load().neptune_pdhg_mf_geometry(B, N, F, out) == 0
    o = list(out)
    return dict(K=o[0], ct=o[2], RT=o[3], rt=o[4], K4=F * o[4], small="one-block" if o[6] else "many-blocks",
                bulk=o[14], bulk_fused=o[7])


def branch(B, N, F):
    """(K, small-vector kernel, C4 dual summation, default pass) of the solve -- what the case ids spell"""
    g = geometry(B, N, F)
    return (g["K"], g["small"], "sliced" if g["K4"] > 64 else "one-pass",
            ("bulk-fused" if g["bulk_fused"] else "bulk") if g["bulk"] else "register")


def _close(got, want, tol):
    return np.abs(got - want).max() <= tol * (1.0 + np.abs(want).max())


def _rows(N, F, y):
    """(y2, y4) of a canonical min-delay y vector"""
    C = F * N
    return y[2 * C:2 * C + N], y[3 * C + N:3 * C + 2 * N]


def _assert_equals_run_fixed(x, y, res, payloads, iters, ref):
    """the candidate after `iters` iterations equals run_fixed's, with the tolerances of tests/test_pdhg_mf_gpu.py;
    the two candidates' KKT errors are not tied, so the pick cannot differ by rounding"""
    for b in range(len(payloads)):
        xr, yr, info = ref[b]
        k0, k1 = info["kkt"]
        assert abs(k0 - k1) > 1e-6 * max(k0, k1), (b, k0, k1)
        assert _close(x[b].cpu().numpy(), xr, 1e-9), b
        assert _close(y[b].cpu().numpy(), yr, 1e-9), b
        assert abs(res[b]["primal_obj"] - info["primal_obj"]) <= 1e-9 * (1 + abs(info["primal_obj"]))
        assert abs(res[b]["dual_obj"] - info["dual_obj"]) <= 1e-9 * (1 + abs(info["dual_obj"]))
        assert abs(res[b]["primal_res"] - info["primal_res"]) <= 1e-9 * (1 + info["primal_res"])
        assert abs(res[b]["primal_weight"] - info["omega"]) <= 1e-12 * info["omega"]
        assert res[b]["iters"] == iters and res[b]["converged"] == 0


# ------------------------------------------------------------------------------------------------------------------
# 1. branch-pinned parity at wide shapes (B = 2)
# ------------------------------------------------------------------------------------------------------------------
# (id, N, F, iterations, payload(seed), expected branch(B = 2), coupling duals the reference must show active).
# Iteration counts: one graph replay of 32 + 1, or two + 6.
def _loaded(N, F, capacity=0.25):
    return lambda s: loaded_payload(N, F, s, capacity)


WIDE = [
    ("65x8", 65, 8, 33, _loaded(65, 8), (4, "one-block", "sliced", "register"), ("y4",)),                 # K4 = 72
    ("99x5", 99, 5, 70, _loaded(99, 5), (4, "one-block", "sliced", "register"), ("y4",)),                 # K4 = 65
    ("64x64", 64, 64, 33, _loaded(64, 64), (2, "one-block", "one-pass", "bulk"), ("y2", "y4")),           # F*N = 4096, K4 = 64
    ("100x40", 100, 40, 70, _loaded(100, 40), (2, "one-block", "sliced", "register"), ("y2", "y4")),      # K4 = 280
    ("130x33", 130, 33, 33, _loaded(130, 33), (2, "many-blocks", "sliced", "register"), ("y2", "y4")),    # ct = 3, K4 = 561
    ("129x40", 129, 40, 33, _loaded(129, 40), (4, "many-blocks", "sliced", "register"), ("y2", "y4")),
    ("50x80", 50, 80, 70, _loaded(50, 80), (2, "one-block", "sliced", "bulk"), ("y2", "y4")),             # fused bulk does not fit
    ("1026x2", 1026, 2, 70, _loaded(1026, 2, 0.05), (2, "one-block", "sliced", "register"), ("y4",)),     # 17 column tiles
    ("99x5-float", 99, 5, 33, lambda s: float_payload(99, 5, 11 + s), (4, "one-block", "sliced", "register"), ()),
]
WIDE_BY_ID = {c[0]: c for c in WIDE}

# the default pass, and the register passes with one and two rows of a warp in flight where the default is the bulk-copy
# pass (even N <= 64); elsewhere the default IS the 8-byte pass (two rows in flight, one for K = 4)
PASSES = {"default": {}, "8-byte-rows1": dict(scalar_kernel=True, rows_in_flight=1),
          "8-byte-rows2": dict(scalar_kernel=True, rows_in_flight=2), "pair-rows1": dict(register_pass=True, rows_in_flight=1),
          "pair-rows2": dict(register_pass=True, rows_in_flight=2)}
WIDE_PARAMS = [(c[0], v) for c in WIDE
               for v in (PASSES if c[5][3] != "register" else ("8-byte-rows1", "8-byte-rows2"))]


def _wide_id(name):
    K, small, c4, dflt = WIDE_BY_ID[name][5]
    return f"{name}-K{K}-small-{small}-c4-{c4}-{dflt}"


@functools.lru_cache(maxsize=None)
def _wide_reference(name):
    _, N, F, iters, make, _, _ = WIDE_BY_ID[name]
    payloads = [make(s) for s in range(2)]
    return payloads, [run_fixed(arrays_of(p), iters) for p in payloads]


@pytest.mark.parametrize("name,variant", WIDE_PARAMS, ids=[f"{_wide_id(n)}-{v}" for n, v in WIDE_PARAMS])
def test_wide_iterates_equal_the_numpy_reference(name, variant):
    """`iters` iterations without a restart, then the better candidate: x, y, objectives, primal residual and primal
    weight equal `run_fixed`'s (1e-9 of the largest entry; the weight to 1e-12)"""
    from neptune_mip_b200 import device
    _, N, F, iters, _, want, active = WIDE_BY_ID[name]
    assert branch(2, N, F) == want
    payloads, ref = _wide_reference(name)
    for b in range(2):                      # the coupling rows the case is meant to exercise do bind
        y2, y4 = _rows(N, F, ref[b][1])
        assert all(np.abs({"y2": y2, "y4": y4}[k]).max() > 1e-3 for k in active), (b, active)
    x, y, res = device.pdhg_mf_solve(cuda_batch(payloads), max_iters=iters, check_every=iters, **UNREACHABLE,
                                     **PASSES[variant])
    _assert_equals_run_fixed(x, y, res, payloads, iters, ref)


def test_c3_bench_workload_equals_the_numpy_reference():
    """the C3 record of bench.py: 500 x 50, one instance, slot-cut relaxation (`device.slot_relaxation`), 33
    iterations; the reference runs on the same slot-relaxed arrays (m = 1, Mj = floor(Mj / m) capped by F)"""
    from neptune_mip_b200 import device
    assert branch(1, 500, 50) == (2, "many-blocks", "sliced", "register")
    g = geometry(1, 500, 50)
    assert (g["ct"], g["rt"], g["K4"]) == (8, 16, 800)
    p = synth.config_payload("C3", 0)
    lp = device.slot_relaxation(cuda_batch([p]))
    a = dict(arrays_of(p))
    a["Mj"] = np.minimum(np.floor(a["Mj"] / a["m"][0] + 1e-9), float(a["F"]))
    a["m"] = np.ones_like(a["m"])
    assert np.array_equal(lp.Mj[0].cpu().numpy(), a["Mj"]) and np.array_equal(lp.m[0].cpu().numpy(), a["m"])
    x, y, res = device.pdhg_mf_solve(lp, max_iters=33, check_every=33, **UNREACHABLE)
    ref = run_fixed(a, 33)
    _assert_equals_run_fixed(x, y, res, [p], 33, [ref])


@pytest.mark.parametrize("node_cut", [False, True], ids=["bigM", "node-cut"])
@pytest.mark.parametrize("kind", ["min_util", "min_delay_util"])
def test_node_variable_models_at_130x33(kind, node_cut):
    """node columns (C5a / C5b / C6 in the small-vector kernel) with the C2 dual and the node rows in their own launch
    (F * N > 4096)"""
    from neptune_mip_b200 import device
    assert branch(2, 130, 33) == (2, "many-blocks", "sliced", "register")
    payloads = [loaded_payload(130, 33, s) for s in range(2)]
    ref = []
    for p in payloads:
        a = arrays_of(p)
        ref.append(run_fixed(a, 33, kind, 0.5, node_cut_bigm(a) if node_cut else None))
    x, y, res = device.pdhg_mf_solve(cuda_batch(payloads), max_iters=33, check_every=33, **UNREACHABLE, kind=kind,
                                     alpha=0.5, node_cut=node_cut)
    _assert_equals_run_fixed(x, y, res, payloads, 33, ref)


# ------------------------------------------------------------------------------------------------------------------
# 2. the restart trajectory
# ------------------------------------------------------------------------------------------------------------------
# (id, N, F, payload, expected branch at B = 1, max_iters, check_every, eps_abs, eps_rel); the converged runs stop on
# the tolerance, the fixed-budget runs on max_iters with at least two restarts behind them
RESTART = [
    ("12x5-K1-converged", 12, 5, lambda: synth.random_payload(12, 5, 1, node_cores=25), (1, "one-block", "one-pass", "register"),
     20000, 64, 1e-9, 1e-6),
    ("50x4-bulk-fused-converged", 50, 4, lambda: synth.random_payload(50, 4, 0, node_cores=25),
     (2, "one-block", "one-pass", "bulk-fused"), 20000, 64, 1e-9, 1e-6),
    ("33x3-K2-odd-converged", 33, 3, lambda: synth.random_payload(33, 3, 0, node_cores=60), (2, "one-block", "one-pass", "register"),
     20000, 64, 1e-9, 1e-6),
    ("65x8-K4-converged", 65, 8, lambda: synth.random_payload(65, 8, 1, node_cores=None), (4, "one-block", "sliced", "register"),
     20000, 64, 1e-9, 1e-5),
    ("130x33-many-blocks-1024", 130, 33, lambda: loaded_payload(130, 33, 0), (2, "many-blocks", "sliced", "register"),
     1024, 64, 1e-15, 1e-13),
    ("129x40-K4-many-blocks-1024", 129, 40, lambda: loaded_payload(129, 40, 0), (4, "many-blocks", "sliced", "register"),
     1024, 64, 1e-15, 1e-13),
]

# x, y after the restarted solve, relative to the largest entry: measured on B200 at 3e-15 .. 1.9e-13 over these six runs
# (the largest after 11 648 iterations and 16 restarts at 65 x 8)
TRAJECTORY_TOL = 1e-11


@pytest.mark.parametrize("case", RESTART, ids=[c[0] for c in RESTART])
def test_restart_trajectory_equals_the_control_logic(case):
    """`neptune_pdhg_mf_solve` with restarts against `mf_reference.solve_ctl` (k_ctl_decide / k_ctl_after_restart in
    numpy): the same number of iterations, of restarts and the same convergence flag; primal weight and objectives to
    1e-9.  Every floating-point decision of the reference is at least 1e-7 relative away from its threshold, so a
    rounding difference cannot take the other branch."""
    from neptune_mip_b200 import device
    name, N, F, make, want, max_iters, check_every, eps_abs, eps_rel = case
    assert branch(1, N, F) == want
    p = make()
    mf = MatrixFree(arrays_of(p))
    info, log = solve_ctl(mf, max_iters, check_every, eps_abs, eps_rel)
    for e in log:
        for label, v, t in e["decisions"]:
            assert not np.isfinite(t) or abs(v - t) > 1e-7 * abs(t), (e["iters"], label, v, t)
    if max_iters == 1024:
        assert info["converged"] == 0 and info["restarts"] >= 2 and info["iters"] == 1024
    else:
        assert info["converged"] == 1
    x, y, res = device.pdhg_mf_solve(cuda_batch([p]), max_iters=max_iters, check_every=check_every, eps_abs=eps_abs,
                                     eps_rel=eps_rel)
    r = res[0]
    assert (int(r["iters"]), int(r["restarts"]), int(r["converged"])) == (info["iters"], info["restarts"], info["converged"])
    assert abs(r["primal_weight"] - info["primal_weight"]) <= 1e-9 * info["primal_weight"]
    for k in ("primal_obj", "dual_obj"):
        assert abs(r[k] - info[k]) <= 1e-9 * (1 + abs(info[k])), k
    xr, yr = mf.pack()
    dx = np.abs(x[0].cpu().numpy() - xr).max() / (1 + np.abs(xr).max())
    dy = np.abs(y[0].cpu().numpy() - yr).max() / (1 + np.abs(yr).max())
    print(f"{name}: iters {info['iters']} restarts {info['restarts']} max|dx| {dx:.2e} max|dy| {dy:.2e} (relative)")
    assert dx <= TRAJECTORY_TOL and dy <= TRAJECTORY_TOL


# ------------------------------------------------------------------------------------------------------------------
# 3. batch independence on the wide branches
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,F,payloads", [
    (65, 8, lambda: [synth.random_payload(65, 8, 0, node_cores=None), loaded_payload(65, 8, 0, 0.5),
                     synth.random_payload(65, 8, 1, node_cores=None)]),
    (130, 33, lambda: [synth.random_payload(130, 33, 0, node_cores=None), loaded_payload(130, 33, 0, 0.5),
                       synth.random_payload(130, 33, 1, node_cores=None)]),
], ids=["65x8-K4", "130x33-many-blocks"])
def test_wide_instances_of_a_batch_converge_independently(N, F, payloads):
    """as test_pdhg_mf_gpu.test_instances_of_a_batch_converge_independently at 8 x 4: every instance of a batch takes
    bitwise the trajectory it takes alone, restarts and convergence included, while the others run on.  The tile
    geometry of N > 64 depends on the batch size (row-tile height); these shapes have the same for 1 and 3 instances,
    so the summation orders agree"""
    from neptune_mip_b200 import device
    ps = payloads()
    assert geometry(len(ps), N, F) == geometry(1, N, F)
    kw = dict(max_iters=20000, check_every=128, eps_rel=1e-4, eps_abs=1e-9)
    x, y, res = device.pdhg_mf_solve(cuda_batch(ps), **kw)
    assert len(set(res["iters"].tolist())) > 1
    for b, p in enumerate(ps):
        xs, ys, rs = device.pdhg_mf_solve(cuda_batch([p]), **kw)
        assert res[b]["converged"] == 1 and res[b]["iters"] == rs[0]["iters"] and res[b]["restarts"] == rs[0]["restarts"]
        assert np.array_equal(x[b].cpu().numpy(), xs[0].cpu().numpy())
        assert np.array_equal(y[b].cpu().numpy(), ys[0].cpu().numpy())
