"""(b) matrix-free PDHG (`neptune_pdhg_mf_solve`): the kernels reproduce the numpy statement of the iteration
(tests/mf_reference.py, proven equal to the CSR iteration on the strengthened oracle matrix in
tests/test_mf_reference.py), that matrix is exactly the one the device assembles in the solver's canonical layout,
and the solver reaches the HiGHS LP optimum."""
import ctypes

import numpy as np
import pytest

from helpers import KIND_NAMES, arrays_of, cuda_batch, float_payload
from mf_reference import MatrixFree, MatrixFreeN, node_cut_bigm, run_fixed, solve, strengthened
from neptune_mip_b200 import synth
from oracle import mip as omip

pytestmark = pytest.mark.gpu

# (name, payload factory, iterations): odd and even N, N <= 32 / <= 64 / > 64 (1, 2, 4 columns per lane; one and
# several row / column tiles), iteration counts that are one graph replay, several, and replay + remainder
CASES = [
    ("C1-3x2", lambda s: synth.test_py_payload(), 64),
    ("8x4", lambda s: synth.random_payload(8, 4, s, node_cores=30), 64),
    ("12x5", lambda s: synth.random_payload(12, 5, s, node_cores=25), 96),
    ("20x5", lambda s: synth.random_payload(20, 5, s, node_cores=100), 40),
    ("33x3", lambda s: synth.random_payload(33, 3, s, node_cores=60), 33),
    ("50x10", lambda s: synth.random_payload(50, 10, s, node_cores=200), 64),
    ("70x3", lambda s: synth.random_payload(70, 3, s, node_cores=60), 64),
    ("7x3-float", lambda s: float_payload(7, 3, 5 + s), 64),
]


def _close(got, want, tol):
    scale = 1.0 + np.abs(want).max()
    return np.abs(got - want).max() <= tol * scale


@pytest.mark.parametrize("name,make,iters", CASES, ids=[c[0] for c in CASES])
@pytest.mark.parametrize("variant", ["default-pass", "8-byte-pass"])
def test_iterates_equal_the_numpy_reference(name, make, iters, variant):
    """After `iters` iterations (no restart inside) the returned candidate -- current iterate or running
    average, whichever has the smaller KKT error -- equals the reference's.  Tolerance 1e-9 relative to the
    largest entry: the kernels only differ from numpy in summation order and FMA contraction."""
    from neptune_mip_b200 import device
    payloads = [make(s) for s in range(2)]
    inst = cuda_batch(payloads)
    x, y, res = device.pdhg_mf_solve(inst, max_iters=iters, check_every=iters, eps_rel=1e-13, eps_abs=1e-15,
                                     scalar_kernel=variant == "8-byte-pass")
    for b, p in enumerate(payloads):
        xr, yr, info = run_fixed(arrays_of(p), iters)
        assert _close(x[b].cpu().numpy(), xr, 1e-9), (name, b)
        assert _close(y[b].cpu().numpy(), yr, 1e-9), (name, b)
        assert abs(res[b]["primal_obj"] - info["primal_obj"]) <= 1e-9 * (1 + abs(info["primal_obj"]))
        assert abs(res[b]["dual_obj"] - info["dual_obj"]) <= 1e-9 * (1 + abs(info["dual_obj"]))
        assert abs(res[b]["primal_res"] - info["primal_res"]) <= 1e-9 * (1 + info["primal_res"])
        assert abs(res[b]["primal_weight"] - info["omega"]) <= 1e-12 * info["omega"]
        assert res[b]["iters"] == iters and res[b]["converged"] == 0
        assert np.all(y[b].cpu().numpy()[0:2 * inst.F * inst.N:2] == 0.0)      # free C1a rows


@pytest.mark.parametrize("shape", [(34, 3), (50, 4), (64, 3), (130, 2), (300, 2)])
def test_pair_pass_equals_the_8_byte_pass(shape):
    """even N in 33..64 runs the pair pass (16-byte accesses, reciprocal by Newton steps) by default: same
    arithmetic as the 8-byte pass up to the last bits of 1/(3 + w r); wider shapes take the 8-byte pass either way;
    one and two rows of a warp in flight"""
    from neptune_mip_b200 import device
    inst = cuda_batch([synth.random_payload(shape[0], shape[1], s, node_cores=60) for s in range(2)])
    kw = dict(max_iters=33, check_every=33, eps_rel=1e-13, eps_abs=1e-15)
    xa, ya, ra = device.pdhg_mf_solve(inst, scalar_kernel=True, **kw)
    for u in (0, 1, 2):
        xb, yb, rb = device.pdhg_mf_solve(inst, rows_in_flight=u, **kw)
        assert _close(xb.cpu().numpy(), xa.cpu().numpy(), 1e-11) and _close(yb.cpu().numpy(), ya.cpu().numpy(), 1e-11)
        assert np.allclose(ra["primal_obj"], rb["primal_obj"], rtol=1e-11)


def _bulk_geometry(N, F, B=2):
    from neptune_mip_b200 import _lib
    out = (ctypes.c_int32 * 16)()
    assert _lib.load().neptune_pdhg_mf_geometry(B, N, F, out) == 0
    return list(out)[8:]


@pytest.mark.parametrize("shape", [(50, 4), (34, 3), (64, 3), (20, 5), (8, 4), (2, 2)])
@pytest.mark.parametrize("mode", [1, 2], ids=["staged-sums", "bulk-reduction"])
@pytest.mark.parametrize("unfused", [False, True], ids=["small-vectors-in-pass", "small-vectors-own-launch"])
def test_bulk_copy_pass_equals_the_register_passes(shape, mode, unfused):
    """even N <= 64: the pass with its streams staged through shared memory by cp.async.bulk (mode 1: x, yS and both
    running sums; mode 2: the running sums added by cp.reduce.async.bulk) does the arithmetic of the pair pass; the
    column sums are taken over another grouping of the rows, so the comparison is 1e-11, not bitwise.  Shapes whose
    stage does not fit twice (N > 50 with four streams) fall back to the register pass -- the geometry says which.
    By default the small-vector update (k_mf_small's arithmetic) runs inside the pass, per block and instance, on two
    alternating small-state buffers; `unfused_small` keeps it in its own launches."""
    from neptune_mip_b200 import device
    ok4, st4, nw4, ok2, st2, nw2, dflt, smem2 = _bulk_geometry(*shape)
    assert ok2 == 1 and ok4 == (0 if shape[0] > 50 else 1)
    inst = cuda_batch([synth.random_payload(shape[0], shape[1], s, node_cores=60) for s in range(3)])
    kw = dict(max_iters=70, check_every=70, eps_rel=1e-13, eps_abs=1e-15)
    xa, ya, ra = device.pdhg_mf_solve(inst, scalar_kernel=True, **kw)
    xb, yb, rb = device.pdhg_mf_solve(inst, bulk=mode, unfused_small=unfused, **kw)
    assert _close(xb.cpu().numpy(), xa.cpu().numpy(), 1e-11) and _close(yb.cpu().numpy(), ya.cpu().numpy(), 1e-11)
    assert np.allclose(ra["primal_obj"], rb["primal_obj"], rtol=1e-11) and np.allclose(ra["dual_obj"], rb["dual_obj"], rtol=1e-9)
    # bit-reproducible: fixed summation orders, one addition per element in the reduction
    xc, yc, rc = device.pdhg_mf_solve(inst, bulk=mode, unfused_small=unfused, **kw)
    assert np.array_equal(xb.cpu().numpy(), xc.cpu().numpy()) and np.array_equal(yb.cpu().numpy(), yc.cpu().numpy())


@pytest.mark.parametrize("mode,warps,stages,unfused", [(1, 0, 0, False), (2, 0, 0, False), (2, 0, 0, True), (2, 8, 2, False), (2, 15, 3, True),
                                                       (2, 5, 4, False), (1, 10, 2, True), (2, 13, 2, False)])
def test_bulk_copy_pass_many_tiles_per_block(mode, warps, stages, unfused):
    """more tiles per block than stages (every stage and both barrier phases are reused many times), every geometry the
    tools can ask for; against the numpy statement of the iteration on two instances and the pair pass on all"""
    from neptune_mip_b200 import device
    B = 96                                                   # 960 slabs over 148 blocks: 6-7 tiles per block
    payloads = [synth.random_payload(50, 10, s, node_cores=200) for s in range(B)]
    inst = cuda_batch(payloads)
    kw = dict(max_iters=70, check_every=70, eps_rel=1e-13, eps_abs=1e-15)      # two graph replays of 32 + a remainder of 6
    xa, ya, ra = device.pdhg_mf_solve(inst, register_pass=True, **kw)
    xb, yb, rb = device.pdhg_mf_solve(inst, bulk=mode, bulk_warps=warps, bulk_stages=stages, unfused_small=unfused, **kw)
    assert _close(xb.cpu().numpy(), xa.cpu().numpy(), 1e-11) and _close(yb.cpu().numpy(), ya.cpu().numpy(), 1e-11)
    for b in (0, B - 1):
        xr, yr, info = run_fixed(arrays_of(payloads[b]), 70)
        assert _close(xb[b].cpu().numpy(), xr, 1e-9) and _close(yb[b].cpu().numpy(), yr, 1e-9)


@pytest.mark.parametrize("mode", [1, 2])
@pytest.mark.parametrize("unfused", [False, True])
def test_bulk_copy_pass_frozen_instances_and_solo_runs(mode, unfused):
    """converged instances go through the barrier protocol without copies: their state stays frozen, the others take
    exactly the trajectory of their solo runs (restarts included)"""
    from neptune_mip_b200 import device
    ps = [synth.random_payload(8, 4, 1, node_cores=200), synth.random_payload(8, 4, 1, node_cores=12),
          synth.random_payload(8, 4, 2, node_cores=30)]
    kw = dict(max_iters=20000, check_every=128, eps_rel=1e-6, eps_abs=1e-9, bulk=mode, unfused_small=unfused)
    x, y, res = device.pdhg_mf_solve(cuda_batch(ps), **kw)
    assert len(set(res["iters"].tolist())) > 1
    for b, p in enumerate(ps):
        xs, ys, rs = device.pdhg_mf_solve(cuda_batch([p]), **kw)
        assert res[b]["converged"] == 1 and res[b]["iters"] == rs[0]["iters"] and res[b]["restarts"] == rs[0]["restarts"]
        assert np.array_equal(x[b].cpu().numpy(), xs[0].cpu().numpy())
        assert np.array_equal(y[b].cpu().numpy(), ys[0].cpu().numpy())


def test_strengthened_assembly_equals_the_reference_statement():
    """the strengthened model the device assembles (`assemble(..., flags=FLAG_STRENGTHEN)`: the model whose canonical
    x / y vectors the matrix-free solver reads and writes) IS the matrix of `mf_reference.strengthened`, on which
    tests/test_mf_reference.py proves the numpy matrix-free iteration equal to the CSR iteration.  Exact equality of
    the pattern, the values, the row and column bounds and the objective, for all three objectives at 20x5 and 8x4,
    three instances in one batch each"""
    from neptune_mip_b200 import device
    from neptune_mip_b200._lib import FLAG_STRENGTHEN
    for (N, F), cores in (((20, 5), 100), ((8, 4), 30)):
        payloads = [synth.random_payload(N, F, s, node_cores=cores) for s in range(3)]
        inst = cuda_batch(payloads)
        for kind in KIND_NAMES:
            mdl = device.assemble(inst, kind, 0.5, flags=FLAG_STRENGTHEN)
            for b, p in enumerate(payloads):
                ref = strengthened(arrays_of(p), kind, 0.5)
                A, case = ref["A"], (N, F, kind, b)
                assert (mdl.rows, mdl.cols, mdl.nnz) == (A.shape[0], A.shape[1], A.nnz), case
                assert np.array_equal(mdl.row_ptr.cpu().numpy(), A.indptr), case
                assert np.array_equal(mdl.col_idx.cpu().numpy(), A.indices), case
                assert np.array_equal(mdl.val[b].cpu().numpy(), A.data), case
                for got, key in ((mdl.lo, "lo"), (mdl.hi, "hi"), (mdl.obj, "obj"), (mdl.col_lb, "lb"), (mdl.col_ub, "ub")):
                    assert np.array_equal(got[b].cpu().numpy(), ref[key]), (key,) + case


@pytest.mark.parametrize("shape,cores", [((12, 5), 25), ((8, 4), 12), ((10, 3), 20)])
def test_reaches_the_highs_lp_optimum(shape, cores):
    """LP value of the strengthened relaxation: |obj - obj_highs| <= 1e-4 * (1 + |obj_highs|) (BASELINE.json's
    1e-4 relative), primal and dual side, with the convergence flag set."""
    from neptune_mip_b200 import device
    p = synth.random_payload(shape[0], shape[1], 1, node_cores=cores)
    lp = omip.solve_model(strengthened(arrays_of(p)), relax=True)
    x, y, res = device.pdhg_mf_solve(cuda_batch([p]), max_iters=30000, check_every=128, eps_rel=1e-6, eps_abs=1e-9)
    assert res[0]["converged"] == 1
    assert abs(res[0]["primal_obj"] - lp["objective"]) <= 1e-4 * (1 + abs(lp["objective"]))
    assert abs(res[0]["dual_obj"] - lp["objective"]) <= 1e-4 * (1 + abs(lp["objective"]))
    xs = x[0].cpu().numpy()
    assert xs.min() >= 0.0 and xs.max() <= 1.0
    # same restart decisions as the numpy statement of the solver (regression guard: with the running average
    # mis-scaled at the KKT checks the device solver needed ~10x the iterations)
    ref = solve(MatrixFree(arrays_of(p)), max_iters=30000, check=128, eps=1e-6)
    assert ref["converged"] and res[0]["iters"] <= 3 * ref["iters"] + 128, (res[0]["iters"], ref["iters"])


def test_instances_of_a_batch_converge_independently():
    """per-instance step sizes, restarts and convergence: every instance of a batch takes exactly the trajectory
    it takes alone (a converged instance is frozen while the others run on)"""
    from neptune_mip_b200 import device
    ps = [synth.random_payload(8, 4, 1, node_cores=200), synth.random_payload(8, 4, 1, node_cores=12),
          synth.random_payload(8, 4, 2, node_cores=30)]
    kw = dict(max_iters=20000, check_every=128, eps_rel=1e-6, eps_abs=1e-9)
    x, y, res = device.pdhg_mf_solve(cuda_batch(ps), **kw)
    assert len(set(res["iters"].tolist())) > 1                       # they do stop at different times
    for b, p in enumerate(ps):
        xs, ys, rs = device.pdhg_mf_solve(cuda_batch([p]), **kw)
        assert res[b]["converged"] == 1 and res[b]["iters"] == rs[0]["iters"] and res[b]["restarts"] == rs[0]["restarts"]
        assert np.array_equal(x[b].cpu().numpy(), xs[0].cpu().numpy())
        assert np.array_equal(y[b].cpu().numpy(), ys[0].cpu().numpy())


UTIL_CASES = [c for c in CASES if c[0] in ("C1-3x2", "8x4", "12x5", "33x3", "50x10", "70x3")]


@pytest.mark.parametrize("name,make,iters", UTIL_CASES, ids=[c[0] for c in UTIL_CASES])
@pytest.mark.parametrize("kind", ["min_util", "min_delay_util"])
def test_node_variable_models_iterates_equal_the_numpy_reference(name, make, iters, kind):
    """`neptune_pdhg_mf_solve_util` (columns x, c, n; rows + C5a / C5b / C6, reference neptune_step1.py:38-77): the
    candidate after `iters` iterations equals the numpy statement, which tests/test_mf_reference.py proves equal to
    the CSR iteration on the oracle's matrix of that model.  1e-9 relative to the largest entry."""
    from neptune_mip_b200 import device
    payloads = [make(s) for s in range(2)]
    inst = cuda_batch(payloads)
    x, y, res = device.pdhg_mf_solve(inst, max_iters=iters, check_every=iters, eps_rel=1e-13, eps_abs=1e-15, kind=kind, alpha=0.5)
    N, F = inst.N, inst.F
    assert x.shape[1] == F * N * N + F * N + N and y.shape[1] == 3 * F * N + 2 * N + 3 * N + F * N * N
    for b, p in enumerate(payloads):
        xr, yr, info = run_fixed(arrays_of(p), iters, kind, 0.5)
        assert _close(x[b].cpu().numpy(), xr, 1e-9), (name, b)
        assert _close(y[b].cpu().numpy(), yr, 1e-9), (name, b)
        assert abs(res[b]["primal_obj"] - info["primal_obj"]) <= 1e-9 * (1 + abs(info["primal_obj"]))
        assert abs(res[b]["dual_obj"] - info["dual_obj"]) <= 1e-9 * (1 + abs(info["dual_obj"]))
        assert abs(res[b]["primal_res"] - info["primal_res"]) <= 1e-9 * (1 + info["primal_res"])
        assert abs(res[b]["primal_weight"] - info["omega"]) <= 1e-12 * info["omega"]
        assert res[b]["iters"] == iters and res[b]["converged"] == 0


@pytest.mark.parametrize("kind", ["min_util", "min_delay_util"])
def test_node_variable_models_reach_the_highs_lp_optimum(kind):
    """LP value of the reference's relaxation with node columns: HiGHS on the oracle's matrix and the matrix-free
    solver agree to 1e-4 relative."""
    from neptune_mip_b200 import device
    p = synth.random_payload(12, 5, 1, node_cores=25)
    lp = omip.solve_model(strengthened(arrays_of(p), kind, 0.5), relax=True)
    inst = cuda_batch([p])
    x, y, res = device.pdhg_mf_solve(inst, max_iters=60000, check_every=128, eps_rel=1e-6, eps_abs=1e-9, kind=kind, alpha=0.5)
    assert res[0]["converged"] == 1
    tol = 1e-4 * (1 + abs(lp["objective"]))
    assert abs(res[0]["primal_obj"] - lp["objective"]) <= tol and abs(res[0]["dual_obj"] - lp["objective"]) <= tol
    n = x[0, -inst.N:].cpu().numpy()
    assert n.min() >= 0.0 and n.max() <= 1.0


@pytest.mark.parametrize("kind", ["min_util", "min_delay_util"])
def test_node_cut_iterates_and_lp_value(kind):
    """per-node M of row C5a (`node_cut=True`): iterates equal the numpy statement with that M, and the converged value is
    the HiGHS optimum of the oracle's matrix with the same coefficient -- far above the vacuous bound of M = 10^6"""
    from neptune_mip_b200 import device
    p = synth.random_payload(12, 5, 1, node_cores=25)
    a = arrays_of(p)
    inst = cuda_batch([p])
    x, y, res = device.pdhg_mf_solve(inst, max_iters=96, check_every=96, eps_rel=1e-13, eps_abs=1e-15, kind=kind, node_cut=True)
    xr, yr, info = run_fixed(a, 96, kind, 0.5, node_cut_bigm(a))
    assert _close(x[0].cpu().numpy(), xr, 1e-9) and _close(y[0].cpu().numpy(), yr, 1e-9)
    lp_cut = omip.solve_model(strengthened(a, kind, 0.5, node_cut_bigm(a)), relax=True)["objective"]
    lp_ref = omip.solve_model(strengthened(a, kind, 0.5), relax=True)["objective"]
    x, y, res = device.pdhg_mf_solve(inst, max_iters=60000, check_every=128, eps_rel=1e-6, eps_abs=1e-9, kind=kind, node_cut=True)
    assert res[0]["converged"] == 1
    tol = 1e-4 * (1 + abs(lp_cut))
    assert abs(res[0]["primal_obj"] - lp_cut) <= tol and abs(res[0]["dual_obj"] - lp_cut) <= tol
    assert res[0]["dual_obj"] > 5 * lp_ref


def test_other_model_kinds_are_refused():
    """`neptune_pdhg_mf_solve` is the min-delay entry point; the n-column models have their own
    (`neptune_pdhg_mf_solve_util`)"""
    import torch
    from neptune_mip_b200 import _lib, device
    lib = _lib.load()
    inst = cuda_batch([synth.random_payload(8, 4, 0, node_cores=30)])
    need = ctypes.c_int64()
    assert lib.neptune_pdhg_mf_workspace_bytes(1, 8, 4, ctypes.byref(need)) == 0 and need.value > 0
    ws = torch.empty(need.value, dtype=torch.uint8, device="cuda")
    rows, cols, _ = device.model_sizes(8, 4, 0, 1)
    x = torch.zeros(cols, dtype=torch.float64, device="cuda")
    y = torch.zeros(rows, dtype=torch.float64, device="cuda")
    res = torch.zeros(128, dtype=torch.uint8, device="cuda")
    prm = _lib.PdhgParams(64, 64, 0, 0, 1e-6, 1e-9)
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    args = [p(inst.d), p(inst.w), p(inst.r), p(inst.m), p(inst.Mj), p(inst.Kj), ctypes.byref(prm), p(x), p(y), p(res), p(ws)]
    for kind in (1, 2):
        assert lib.neptune_pdhg_mf_solve(1, 8, 4, kind, *args, ws.numel(), None) == -1
    assert lib.neptune_pdhg_mf_solve(1, 8, 4, 0, *args, 16, None) == -3          # workspace too small
    assert lib.neptune_pdhg_mf_solve(1, 8, 4, 0, *args, ws.numel(), None) == 0
