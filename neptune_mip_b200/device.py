"""Device-side plumbing: torch tensors for HBM + streams, ctypes calls into libneptune_b200.so.

Everything numeric happens in the CUDA kernels behind the C ABI (`include/neptune_b200.h`); this
module only allocates tensors, passes raw device pointers and checks return codes.  A missing
library or GPU raises -- there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np
import torch

from . import _lib
from ._lib import KINDS, NeptuneError, PdhgParams, check


def _require_cuda():
    if not torch.cuda.is_available():
        raise NeptuneError("neptune_mip_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


@dataclass
class InstanceBatch:
    """B same-shaped placement instances resident in HBM (float64, row-major, leading dim B)."""
    B: int
    N: int
    F: int
    d: torch.Tensor        # [B,N,N]
    w: torch.Tensor        # [B,F,N]
    r: torch.Tensor        # [B,F,N]
    m: torch.Tensor        # [B,F]
    Mj: torch.Tensor       # [B,N]
    Kj: torch.Tensor       # [B,N]
    old: torch.Tensor      # [B,F,N]
    maxd: torch.Tensor     # [B,F]
    cost: torch.Tensor     # [B,N]
    budget: float

    FIELDS = ("d", "w", "r", "m", "Mj", "Kj", "old", "maxd", "cost")

    @staticmethod
    def host_arrays(datas: Sequence) -> dict:
        """Stack the `Data` fields the kernels read into float64 numpy arrays (host)."""
        def stack(attr):
            return np.ascontiguousarray(np.stack([np.asarray(getattr(x, attr), dtype=np.float64) for x in datas]))
        N, F = len(datas[0].nodes), len(datas[0].functions)
        for x in datas:
            if len(x.nodes) != N or len(x.functions) != F:
                raise ValueError("a batch must hold same-shaped instances")
        budgets = {float(x.node_budget) for x in datas}
        if len(budgets) != 1:
            raise ValueError("a batch must share node_budget")
        return dict(N=N, F=F, B=len(datas), budget=budgets.pop(),
                    d=stack("node_delay_matrix").reshape(len(datas), N, N),
                    w=stack("workload_matrix").reshape(len(datas), F, N),
                    r=stack("core_per_req_matrix").reshape(len(datas), F, N),
                    m=stack("function_memory_matrix").reshape(len(datas), F),
                    Mj=stack("node_memory_matrix").reshape(len(datas), N),
                    Kj=stack("node_cores_matrix").reshape(len(datas), N),
                    old=stack("old_allocations_matrix").reshape(len(datas), F, N),
                    maxd=stack("max_delay_matrix").reshape(len(datas), F),
                    cost=stack("node_costs").reshape(len(datas), N))

    @classmethod
    def from_host(cls, h: dict, device="cuda", pinned: Optional[dict] = None) -> "InstanceBatch":
        """H2D copy (from pinned staging buffers when given) on the current stream."""
        _require_cuda()
        kw = {}
        for k in cls.FIELDS:
            src = torch.from_numpy(h[k])
            if pinned is not None:
                pinned[k].copy_(src)
                src = pinned[k]
            kw[k] = src.to(device, non_blocking=True)
        return cls(B=h["B"], N=h["N"], F=h["F"], budget=h["budget"], **kw)

    @classmethod
    def from_datas(cls, datas: Sequence, device="cuda") -> "InstanceBatch":
        return cls.from_host(cls.host_arrays(datas), device)

    def h2d_bytes(self) -> int:
        return sum(getattr(self, k).numel() * 8 for k in self.FIELDS)

    def inst_ptrs(self):
        """(d, w, r, m, Mj, Kj, maxd, cost, budget) in the order the C ABI takes them."""
        return [_ptr(self.d), _ptr(self.w), _ptr(self.r), _ptr(self.m), _ptr(self.Mj), _ptr(self.Kj),
                _ptr(self.maxd), _ptr(self.cost), C.c_double(self.budget)]


@dataclass
class Model:
    """Assembled LP/MIP model of a batch: shared CSR pattern (+ transpose) and per-instance values."""
    B: int
    N: int
    F: int
    kind: int
    flags: int
    rows: int
    cols: int
    nnz: int
    row_ptr: torch.Tensor
    col_idx: torch.Tensor
    rowT_ptr: torch.Tensor
    colT_idx: torch.Tensor
    val: torch.Tensor
    valT: torch.Tensor
    obj: torch.Tensor
    lo: torch.Tensor
    hi: torch.Tensor
    col_lb: torch.Tensor
    col_ub: torch.Tensor
    col_int: torch.Tensor
    wmax: torch.Tensor


def model_sizes(N, F, kind, flags=0):
    lib = _lib.load()
    rows, cols, nnz = C.c_int64(), C.c_int64(), C.c_int64()
    check(lib.neptune_model_sizes(N, F, kind, flags, C.byref(rows), C.byref(cols), C.byref(nnz)),
          "neptune_model_sizes")
    return rows.value, cols.value, nnz.value


def assemble(inst: InstanceBatch, kind, alpha=0.5, flags=0, with_transpose=True) -> Model:
    _require_cuda()
    lib = _lib.load()
    kind = KINDS.get(kind, kind)
    rows, cols, nnz = model_sizes(inst.N, inst.F, kind, flags)
    dev = inst.d.device
    B = inst.B
    f64 = dict(dtype=torch.float64, device=dev)
    row_ptr = torch.empty(rows + 1, dtype=torch.int64, device=dev)
    col_idx = torch.empty(nnz, dtype=torch.int32, device=dev)
    rowT_ptr = torch.empty(cols + 1, dtype=torch.int64, device=dev) if with_transpose else None
    colT_idx = torch.empty(nnz, dtype=torch.int32, device=dev) if with_transpose else None
    val = torch.empty((B, nnz), **f64)
    valT = torch.empty((B, nnz), **f64) if with_transpose else None
    obj = torch.empty((B, cols), **f64)
    lo = torch.empty((B, rows), **f64)
    hi = torch.empty((B, rows), **f64)
    col_lb = torch.empty((B, cols), **f64)
    col_ub = torch.empty((B, cols), **f64)
    col_int = torch.empty(cols, dtype=torch.uint8, device=dev)
    wmax = torch.zeros(B, **f64)
    check(lib.neptune_assemble_pattern(inst.N, inst.F, kind, flags, _ptr(row_ptr), _ptr(col_idx),
                                       _ptr(rowT_ptr), _ptr(colT_idx), _stream()), "neptune_assemble_pattern")
    check(lib.neptune_assemble_values(B, inst.N, inst.F, kind, flags, C.c_double(alpha), *inst.inst_ptrs(),
                                      _ptr(val), _ptr(valT), _ptr(obj), _ptr(lo), _ptr(hi), _ptr(col_lb),
                                      _ptr(col_ub), _ptr(col_int), _ptr(wmax), _stream()),
          "neptune_assemble_values")
    return Model(B, inst.N, inst.F, kind, flags, rows, cols, nnz, row_ptr, col_idx, rowT_ptr, colT_idx,
                 val, valT, obj, lo, hi, col_lb, col_ub, col_int, wmax)


_PDHG_DTYPE = np.dtype([("primal_obj", "f8"), ("dual_obj", "f8"), ("primal_res", "f8"), ("dual_res", "f8"),
                        ("gap", "f8"), ("step", "f8"), ("primal_weight", "f8"), ("iters", "i4"),
                        ("restarts", "i4"), ("converged", "i4"), ("pad", "i4")])


def objective_weights(inst: InstanceBatch, kind, alpha=0.5):
    """(a_d[B], a_u[B]): objective = a_d * (workload-weighted delay) + a_u * (active nodes), reference
    objectives.py:4-52 -- (1, 0) for min-delay, (0, 1) for min-utilisation, ((1 - alpha) / the largest
    workload-weighted delay, alpha / N) for the combined objective."""
    k = KINDS.get(kind, kind)
    one = torch.ones(inst.B, dtype=torch.float64, device=inst.d.device)
    if k == 0:
        return one, 0 * one
    if k == 1:
        return 0 * one, one
    far = torch.where(inst.d[:, None, :, :] <= inst.maxd[:, :, None, None], inst.d[:, None, :, :],
                      torch.full_like(inst.d[:, None, :, :], -float("inf"))).amax(dim=-1)          # [B,F,N]
    wmax = (inst.w * far).sum(dim=(1, 2))
    wsum = inst.w.sum(dim=(1, 2))
    a_d = torch.where((wsum != 0) & (wmax != 0), (1.0 - alpha) / wmax, 0 * one)
    return a_d, one * (alpha / inst.N)


def pdhg_mf_solve(inst: InstanceBatch, max_iters=20000, check_every=64, eps_rel=1e-6, eps_abs=1e-8,
                  x0: Optional[torch.Tensor] = None, y0: Optional[torch.Tensor] = None, workspace=None,
                  scalar_kernel=False, rows_in_flight=0, _diag=0, kind="min_delay", alpha=0.5, node_cut=False,
                  bulk=0, bulk_warps=0, bulk_stages=0, register_pass=False, unfused_small=False):
    """Matrix-free PDHG on the strengthened relaxation (`neptune_pdhg_mf_solve`, and `neptune_pdhg_mf_solve_util`
    for the models with node columns): nothing is assembled, every coefficient is regenerated from the instance
    arrays.  Returns (x[B,cols], y[B,rows], results) in the canonical layout of
    `assemble(inst, kind, flags=FLAG_STRENGTHEN)`.  `node_cut` (models with node columns): the big M of row C5a becomes
    the number of pods node j can hold, floor(Mj / min_f m) capped by F -- valid for the MIP, and the relaxation then says
    something about the node term.  `bulk` (even N <= 64): 1 = the iteration pass with its streams staged through shared
    memory by the bulk-copy engine, 2 = the same with the running sums added by bulk reduction; `register_pass` forces
    the register passes whatever the library's default; `bulk_warps` / `bulk_stages` override the bulk pass's geometry
    (measurements); `unfused_small` keeps the small-vector update of the bulk pass in its own launches."""
    _require_cuda()
    lib = _lib.load()
    from ._lib import FLAG_STRENGTHEN
    k = KINDS.get(kind, kind)
    rows, cols, _ = model_sizes(inst.N, inst.F, k, FLAG_STRENGTHEN)
    dev = inst.d.device
    x = torch.zeros((inst.B, cols), dtype=torch.float64, device=dev) if x0 is None else x0
    y = torch.zeros((inst.B, rows), dtype=torch.float64, device=dev) if y0 is None else y0
    need = C.c_int64()
    check(lib.neptune_pdhg_mf_workspace_bytes(inst.B, inst.N, inst.F, C.byref(need)), "neptune_pdhg_mf_workspace_bytes")
    if workspace is None or workspace.numel() < need.value:
        workspace = torch.empty(need.value, dtype=torch.uint8, device=dev)
    res = torch.zeros(inst.B * _PDHG_DTYPE.itemsize, dtype=torch.uint8, device=dev)
    # reserved (tools and tests): bit 0 = force the 8-byte iteration pass, bits 4..6 = tool diagnostics,
    # bits 8..10 = rows of a warp in flight (0 = default), bit 11 = register passes, bit 12 / 13 = bulk-copy pass
    # (staged sums / sums by bulk reduction), bits 14..18 = its consumer warps, bits 19..22 = cap on its stages,
    # bit 23 = small-vector update in its own launches (not inside the bulk pass)
    reserved = ((1 if scalar_kernel else 0) | (_diag << 4) | (rows_in_flight << 8) | ((1 << 11) if register_pass else 0)
                | ((1 << 12) if bulk == 1 else 0) | ((1 << 13) if bulk == 2 else 0) | ((bulk_warps & 31) << 14)
                | ((bulk_stages & 15) << 19) | ((1 << 23) if unfused_small else 0))
    prm = PdhgParams(max_iters, check_every, 0, reserved, eps_rel, eps_abs)
    if k == 0:
        check(lib.neptune_pdhg_mf_solve(inst.B, inst.N, inst.F, 0, _ptr(inst.d), _ptr(inst.w), _ptr(inst.r),
                                        _ptr(inst.m), _ptr(inst.Mj), _ptr(inst.Kj), C.byref(prm), _ptr(x), _ptr(y),
                                        _ptr(res), _ptr(workspace), workspace.numel(), _stream()),
              "neptune_pdhg_mf_solve")
    else:
        # the delay matrix as it enters the objective (objectives.py:24-52): zeros, or d scaled per instance
        a_d, a_u = objective_weights(inst, k, alpha)
        d_obj = (inst.d * a_d[:, None, None]).contiguous()
        big_m = None
        if node_cut:
            m_min = inst.m.amin(dim=1, keepdim=True)
            big_m = torch.where(m_min > 0, torch.floor(inst.Mj / torch.where(m_min > 0, m_min, torch.ones_like(m_min)) + 1e-9),
                                torch.full_like(inst.Mj, float(inst.F))).clamp_(min=0.0, max=float(inst.F)).contiguous()
        check(lib.neptune_pdhg_mf_solve_util(inst.B, inst.N, inst.F, k, _ptr(d_obj), _ptr(inst.w), _ptr(inst.r),
                                             _ptr(inst.m), _ptr(inst.Mj), _ptr(inst.Kj), _ptr(inst.cost),
                                             C.c_double(float(inst.budget)), C.c_double(float(a_u[0])), _ptr(big_m), C.byref(prm),
                                             _ptr(x), _ptr(y), _ptr(res), _ptr(workspace), workspace.numel(), _stream()),
              "neptune_pdhg_mf_solve_util")
    out = np.frombuffer(res.cpu().numpy().tobytes(), dtype=_PDHG_DTYPE)
    return x, y, out


def check_solution(inst: InstanceBatch, x: torch.Tensor, c: torch.Tensor, n: torch.Tensor, alpha=0.5):
    """The reference's six checkers + three scorers.  x[B,N,F,N], c[B,F,N], n[B,N] float64 on device.
    Returns (flags int32[B], scores float64[B,3]) as device tensors."""
    lib = _lib.load()
    dev = inst.d.device
    flags = torch.empty(inst.B, dtype=torch.int32, device=dev)
    scores = torch.empty((inst.B, 3), dtype=torch.float64, device=dev)
    check(lib.neptune_check_solution(inst.B, inst.N, inst.F, C.c_double(alpha), *inst.inst_ptrs(),
                                     _ptr(x), _ptr(c), _ptr(n), _ptr(flags), _ptr(scores), _stream()),
          "neptune_check_solution")
    return flags, scores


def route_placements(inst: InstanceBatch, c_u8: torch.Tensor):
    """c[B,F,N] uint8 -> (x[B,N,F,N], n[B,N]) float64 by the nearest-open-pod rule."""
    lib = _lib.load()
    dev = inst.d.device
    x = torch.empty((inst.B, inst.N, inst.F, inst.N), dtype=torch.float64, device=dev)
    n = torch.empty((inst.B, inst.N), dtype=torch.float64, device=dev)
    check(lib.neptune_route_placements(inst.B, inst.N, inst.F, _ptr(inst.d), _ptr(c_u8), _ptr(x), _ptr(n),
                                       _stream()), "neptune_route_placements")
    return x, n


def eval_placements(inst: InstanceBatch, c_u8: torch.Tensor, alpha=0.5):
    """c[B,P,F,N] uint8 -> (obj[B,P,3], flags[B,P], overload[B,P])."""
    lib = _lib.load()
    dev = inst.d.device
    P = c_u8.shape[1]
    obj = torch.empty((inst.B, P, 3), dtype=torch.float64, device=dev)
    flags = torch.empty((inst.B, P), dtype=torch.int32, device=dev)
    over = torch.empty((inst.B, P), dtype=torch.float64, device=dev)
    check(lib.neptune_eval_placements(inst.B, P, inst.N, inst.F, C.c_double(alpha), *inst.inst_ptrs(),
                                      _ptr(c_u8), _ptr(obj), _ptr(flags), _ptr(over), _stream()),
          "neptune_eval_placements")
    return obj, flags, over


def efttc(inst: InstanceBatch, kind, alpha=0.5, workspace=None):
    """GPU EFTTC.  Returns (c uint8[B,F,N], n uint8[B,N], info int32[B,4])."""
    lib = _lib.load()
    kind = KINDS.get(kind, kind)
    dev = inst.d.device
    need = C.c_int64()
    check(lib.neptune_efttc_workspace_bytes(inst.B, inst.N, inst.F, C.byref(need)), "neptune_efttc_workspace_bytes")
    if workspace is None or workspace.numel() < need.value:
        workspace = torch.empty(need.value, dtype=torch.uint8, device=dev)
    c = torch.empty((inst.B, inst.F, inst.N), dtype=torch.uint8, device=dev)
    n = torch.empty((inst.B, inst.N), dtype=torch.uint8, device=dev)
    info = torch.empty((inst.B, 4), dtype=torch.int32, device=dev)
    check(lib.neptune_efttc(inst.B, inst.N, inst.F, kind, C.c_double(alpha), _ptr(inst.d), _ptr(inst.w),
                            _ptr(inst.r), _ptr(inst.m), _ptr(inst.Mj), _ptr(inst.Kj), _ptr(inst.old),
                            _ptr(inst.cost), C.c_double(inst.budget), _ptr(c), _ptr(n), _ptr(info),
                            _ptr(workspace), workspace.numel(), _stream()), "neptune_efttc")
    return c, n, info


def site_greedy(inst: InstanceBatch, max_rounds: int = 0):
    """Round-robin delay-improvement greedy (`neptune_site_greedy`): c uint8[B,F,N], info int32[B,2] = (rounds, pods).
    For the sizes the EFTTC block and the shared-memory searches do not reach (C4)."""
    _require_cuda()
    lib = _lib.load()
    dev = inst.d.device
    need = C.c_int64()
    check(lib.neptune_site_greedy_workspace_bytes(inst.B, inst.N, inst.F, C.byref(need)), "neptune_site_greedy_workspace_bytes")
    ws = torch.empty(need.value, dtype=torch.uint8, device=dev)
    c = torch.empty((inst.B, inst.F, inst.N), dtype=torch.uint8, device=dev)
    info = torch.empty((inst.B, 2), dtype=torch.int32, device=dev)
    unserved = 2.0 * float(inst.d.max()) + 1.0
    rounds = max_rounds if max_rounds > 0 else inst.N * inst.F
    check(lib.neptune_site_greedy(inst.B, inst.N, inst.F, _ptr(inst.d), _ptr(inst.w), _ptr(inst.m), _ptr(inst.Mj),
                                  C.c_double(unserved), rounds, _ptr(c), _ptr(info), _ptr(ws), ws.numel(), _stream()),
          "neptune_site_greedy")
    return c, info


def site_search(inst: InstanceBatch, c_u8: torch.Tensor, max_rounds: int = 0):
    """Best-improvement pod-exchange search for the min-delay objective under nearest-pod routing
    (`neptune_site_search`) from c_u8[B,F,N] (every function with a pod, e.g. `site_greedy`'s placement), at any size.
    Returns (c uint8[B,F,N], info int32[B,4] = (rounds, adds, exchanges, relocations),
    obj float64[B,2] = nearest-pod objective at the start and at the end).  max_rounds <= 0: until a round accepts
    nothing (at most N*F rounds)."""
    _require_cuda()
    lib = _lib.load()
    dev = inst.d.device
    assert c_u8.shape == (inst.B, inst.F, inst.N) and c_u8.dtype == torch.uint8 and c_u8.is_contiguous()
    need = C.c_int64()
    check(lib.neptune_site_search_workspace_bytes(inst.B, inst.N, inst.F, C.byref(need)), "neptune_site_search_workspace_bytes")
    ws = torch.empty(need.value, dtype=torch.uint8, device=dev)
    c = torch.empty_like(c_u8)
    info = torch.empty((inst.B, 4), dtype=torch.int32, device=dev)
    obj = torch.empty((inst.B, 2), dtype=torch.float64, device=dev)
    rounds = max_rounds if max_rounds > 0 else inst.N * inst.F
    check(lib.neptune_site_search(inst.B, inst.N, inst.F, _ptr(inst.d), _ptr(inst.w), _ptr(inst.m), _ptr(inst.Mj),
                                  _ptr(c_u8), _ptr(c), rounds, _ptr(info), _ptr(obj), _ptr(ws), ws.numel(), _stream()),
          "neptune_site_search")
    return c, info, obj


def route_two_choice(inst: InstanceBatch, c_u8: torch.Tensor, want_x=True, max_iters=500):
    """Nearest / second-nearest routing with per-node shares lowered until the CPU rows hold (`neptune_route_two_choice`):
    the router for sizes the per-instance ones do not reach.  c_u8[B,F,N] ->
    (c_out uint8[B,F,N], x[B,N,F,N] or None, n[B,N], obj[B], feasible int32[B], iterations)."""
    _require_cuda()
    lib = _lib.load()
    dev = inst.d.device
    assert c_u8.shape == (inst.B, inst.F, inst.N) and c_u8.is_contiguous()
    need = C.c_int64()
    check(lib.neptune_route_two_choice_workspace_bytes(inst.B, inst.N, inst.F, C.byref(need)), "neptune_route_two_choice_workspace_bytes")
    ws = torch.empty(need.value, dtype=torch.uint8, device=dev)
    c_out = torch.empty_like(c_u8)
    x = torch.empty((inst.B, inst.N, inst.F, inst.N), dtype=torch.float64, device=dev) if want_x else None
    n = torch.empty((inst.B, inst.N), dtype=torch.float64, device=dev)
    obj = torch.empty(inst.B, dtype=torch.float64, device=dev)
    feas = torch.empty(inst.B, dtype=torch.int32, device=dev)
    iters = C.c_int32(0)
    check(lib.neptune_route_two_choice(inst.B, inst.N, inst.F, _ptr(inst.d), _ptr(inst.w), _ptr(inst.r), _ptr(inst.Kj),
                                       _ptr(c_u8), _ptr(c_out), _ptr(x), _ptr(n), _ptr(obj), _ptr(feas), C.byref(iters),
                                       max_iters, _ptr(ws), ws.numel(), _stream()), "neptune_route_two_choice")
    return c_out, x, n, obj, feas, int(iters.value)


def u8_to_f64(t: torch.Tensor) -> torch.Tensor:
    lib = _lib.load()
    out = torch.empty(t.shape, dtype=torch.float64, device=t.device)
    check(lib.neptune_u8_to_f64(t.numel(), _ptr(t), _ptr(out), _stream()), "neptune_u8_to_f64")
    return out


def efttc_host(h: dict, kind, alpha=0.5):
    """Host-buffer entry point (`neptune_efttc_host`): numpy in, numpy out, copies inside the call."""
    _require_cuda()
    lib = _lib.load()
    kind = KINDS.get(kind, kind)
    B, N, F = h["B"], h["N"], h["F"]
    c = np.empty((B, F, N), dtype=np.uint8)
    n = np.empty((B, N), dtype=np.uint8)
    info = np.empty((B, 4), dtype=np.int32)
    flags = np.empty(B, dtype=np.int32)
    scores = np.empty((B, 3), dtype=np.float64)
    hp = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    check(lib.neptune_efttc_host(B, N, F, kind, C.c_double(alpha), hp(h["d"]), hp(h["w"]), hp(h["r"]),
                                 hp(h["m"]), hp(h["Mj"]), hp(h["Kj"]), hp(h["old"]), hp(h["maxd"]),
                                 hp(h["cost"]), C.c_double(h["budget"]), hp(c), hp(n), hp(info), hp(flags),
                                 hp(scores), _stream()), "neptune_efttc_host")
    return c, n, info, flags, scores


def local_search(inst: InstanceBatch, kind, seeds_u8: torch.Tensor, alpha=0.5, chains=296, sweeps=400,
                 rng_seed=1, guide: Optional[torch.Tensor] = None, workspace=None):
    """Batched add/drop/swap/replace search.  seeds_u8[B,S,F,N] uint8 -> (best_c uint8[B,F,N],
    best_obj float64[B], best_flags int32[B]); best_obj is +inf where no chain found a feasible placement."""
    lib = _lib.load()
    kind = KINDS.get(kind, kind)
    dev = inst.d.device
    S = seeds_u8.shape[1]
    need = C.c_int64()
    check(lib.neptune_local_search_workspace_bytes(inst.B, inst.N, inst.F, chains, C.byref(need)),
          "neptune_local_search_workspace_bytes")
    if workspace is None or workspace.numel() < need.value:
        workspace = torch.empty(need.value, dtype=torch.uint8, device=dev)
    best_c = torch.empty((inst.B, inst.F, inst.N), dtype=torch.uint8, device=dev)
    best_obj = torch.empty(inst.B, dtype=torch.float64, device=dev)
    best_flags = torch.empty(inst.B, dtype=torch.int32, device=dev)
    check(lib.neptune_local_search(inst.B, inst.N, inst.F, kind, C.c_double(alpha), chains, sweeps,
                                   C.c_uint64(rng_seed), S, *inst.inst_ptrs(), _ptr(inst.old), _ptr(seeds_u8),
                                   _ptr(guide), _ptr(best_c), _ptr(best_obj), _ptr(best_flags),
                                   _ptr(workspace), workspace.numel(), _stream()), "neptune_local_search")
    return best_c, best_obj, best_flags


def route_capacitated(inst: InstanceBatch, c_u8: torch.Tensor):
    """CPU-capacity-aware routing.  Returns (c_out uint8[B,F,N], x[B,N,F,N], n[B,N], obj[B], feasible int32[B])."""
    lib = _lib.load()
    dev = inst.d.device
    c_out = torch.empty_like(c_u8)
    x = torch.empty((inst.B, inst.N, inst.F, inst.N), dtype=torch.float64, device=dev)
    n = torch.empty((inst.B, inst.N), dtype=torch.float64, device=dev)
    obj = torch.empty(inst.B, dtype=torch.float64, device=dev)
    feas = torch.empty(inst.B, dtype=torch.int32, device=dev)
    check(lib.neptune_route_capacitated(inst.B, inst.N, inst.F, _ptr(inst.d), _ptr(inst.w), _ptr(inst.r),
                                        _ptr(inst.Kj), _ptr(c_u8), _ptr(c_out), _ptr(x), _ptr(n), _ptr(obj),
                                        _ptr(feas), _stream()), "neptune_route_capacitated")
    return c_out, x, n, obj, feas


def route_lp(inst: InstanceBatch, c_u8: torch.Tensor, want_x=False, tableau_doubles=1 << 19, workspace=None):
    """Exact routing LP of P fixed placements per instance (`neptune_route_lp`, dual simplex on device).
    c_u8[B,P,F,N] uint8 -> dict(obj[B,P], status int32[B,P] (1 optimal, 0 infeasible, 2 tableau too large),
    c_out uint8[B,P,F,N], n[B,P,N], info int32[B,P,2], x[B,P,N,F,N] when `want_x`)."""
    lib = _lib.load()
    dev = inst.d.device
    assert c_u8.dim() == 4 and c_u8.shape[0] == inst.B and c_u8.is_contiguous()
    P = c_u8.shape[1]
    need = C.c_int64()
    check(lib.neptune_route_lp_workspace_bytes(inst.B, P, inst.N, inst.F, tableau_doubles, C.byref(need)),
          "neptune_route_lp_workspace_bytes")
    if workspace is None or workspace.numel() < need.value:
        workspace = torch.empty(need.value, dtype=torch.uint8, device=dev)
    c_out = torch.empty_like(c_u8)
    x = torch.empty((inst.B, P, inst.N, inst.F, inst.N), dtype=torch.float64, device=dev) if want_x else None
    n = torch.empty((inst.B, P, inst.N), dtype=torch.float64, device=dev)
    obj = torch.empty((inst.B, P), dtype=torch.float64, device=dev)
    status = torch.empty((inst.B, P), dtype=torch.int32, device=dev)
    info = torch.empty((inst.B, P, 2), dtype=torch.int32, device=dev)
    check(lib.neptune_route_lp(inst.B, P, inst.N, inst.F, _ptr(inst.d), _ptr(inst.w), _ptr(inst.r), _ptr(inst.Kj),
                               _ptr(c_u8), _ptr(c_out), _ptr(x), _ptr(n), _ptr(obj), _ptr(status), _ptr(info),
                               tableau_doubles, _ptr(workspace), workspace.numel(), _stream()), "neptune_route_lp")
    return dict(obj=obj, status=status, c_out=c_out, n=n, info=info, x=x)


def one_memory_size(inst: InstanceBatch) -> bool:
    """Every function of an instance needs the same, positive memory: the memory rows are slot counts."""
    return bool((inst.m == inst.m[:, :1]).all()) and bool((inst.m > 0).all())


def lns_supported(inst: InstanceBatch, kind) -> bool:
    """The slot-count search needs a delay term in the objective, one memory size for all functions of an
    instance, and a chain state that fits shared memory."""
    kind = KINDS.get(kind, kind)
    if kind not in (0, 2) or inst.N > 128 or inst.F * inst.N > 4096:
        return False
    return one_memory_size(inst)


def lns_global_supported(inst: InstanceBatch, kind) -> bool:
    """The slot-count search with its chain state in global memory (`lns_search_global`): a delay term, one memory
    size per instance, N <= 65534."""
    kind = KINDS.get(kind, kind)
    return kind in (0, 2) and inst.N <= 65534 and inst.F * inst.N < 2 ** 31 and one_memory_size(inst)


def local_search_fits(N: int, F: int) -> bool:
    """Whether the add/drop/swap search (`local_search`, `disruption_search`) takes N x F instances
    (`neptune_local_search_fits`; host arithmetic, no device needed)."""
    fits = C.c_int32()
    check(_lib.load().neptune_local_search_fits(N, F, C.byref(fits)), "neptune_local_search_fits")
    return bool(fits.value)


def lns_block_mode(mode: int) -> None:
    """Chains per block of `lns_search`: 0 automatic (8, or 12 when the blocks of 8 would not all be resident), 1 = 8,
    2 = 12.  Same results either way."""
    check(_lib.load().neptune_lns_block_mode(int(mode)), "neptune_lns_block_mode")


def lns_search(inst: InstanceBatch, kind, alpha=0.5, chains=32, rounds=4000, k=3, noise_coef=0.06, rng_seed=1,
               guide: Optional[torch.Tensor] = None, lam0: Optional[torch.Tensor] = None,
               seeds_u8: Optional[torch.Tensor] = None):
    """LP-guided k-node re-optimisation search (`neptune_lns_search`).  Returns every chain's record:
    (c uint8[B,2*chains,F,N], g float64[B,2*chains], round int32[B,2*chains]): entries [:chains] are the chains' best
    placements by the whole-flow objective (an upper bound of the true objective), entries [chains:] by the priced
    objective (a lower bound); g is the bound the record was chosen by (+inf: none)."""
    lib = _lib.load()
    kind = KINDS.get(kind, kind)
    dev = inst.d.device
    S = 0 if seeds_u8 is None else seeds_u8.shape[1]
    out_c = torch.empty((inst.B, 2 * chains, inst.F, inst.N), dtype=torch.uint8, device=dev)
    out_g = torch.empty((inst.B, 2 * chains), dtype=torch.float64, device=dev)
    out_round = torch.empty((inst.B, 2 * chains), dtype=torch.int32, device=dev)
    out_lb = torch.empty((inst.B, 2 * chains), dtype=torch.float64, device=dev)
    max_slots = int(torch.floor(inst.Mj / inst.m[:, :1] + 1e-9).max().clamp(min=0, max=inst.F).item())
    check(lib.neptune_lns_search(inst.B, inst.N, inst.F, kind, C.c_double(alpha), chains, rounds, k,
                                 C.c_double(noise_coef), C.c_uint64(rng_seed), _ptr(inst.d), _ptr(inst.w), _ptr(inst.r),
                                 _ptr(inst.m), _ptr(inst.Mj), _ptr(inst.Kj), _ptr(inst.maxd), _ptr(guide), _ptr(lam0),
                                 S, _ptr(seeds_u8), max_slots, _ptr(out_c), _ptr(out_g), _ptr(out_lb), _ptr(out_round), _stream()),
          "neptune_lns_search")
    lns_search.last_other_bound = out_lb          # the other end of each record's bracket (diagnostics)
    return out_c, out_g, out_round


def lns_search_global_workspace_bytes(B: int, N: int, F: int, chains: int, k: int, max_slots: int) -> int:
    """Workspace of `lns_search_global` (`neptune_lns_search_global_workspace_bytes`; host arithmetic, no device needed)."""
    need = C.c_int64()
    check(_lib.load().neptune_lns_search_global_workspace_bytes(B, N, F, chains, k, max_slots, C.byref(need)),
          "neptune_lns_search_global_workspace_bytes")
    return need.value


def lns_search_global(inst: InstanceBatch, kind, alpha=0.5, chains=32, rounds=4000, k=3, noise_coef=0.06, rng_seed=1,
                      guide: Optional[torch.Tensor] = None, lam0: Optional[torch.Tensor] = None,
                      seeds_u8: Optional[torch.Tensor] = None):
    """`lns_search` with every chain's state in global memory (`neptune_lns_search_global`): any N <= 65534, and where
    both run the same records bit for bit.  Returns (c, g, round) as `lns_search` does, plus asg int32[B,2*chains,F,N]:
    the node each source was routed to, whole, when its chain took the record (no node overloaded: a feasible routing
    whose delay is the upper bound of entries [:chains])."""
    lib = _lib.load()
    kind = KINDS.get(kind, kind)
    dev = inst.d.device
    B, N, F = inst.B, inst.N, inst.F
    S = 0 if seeds_u8 is None else seeds_u8.shape[1]
    out_c = torch.empty((B, 2 * chains, F, N), dtype=torch.uint8, device=dev)
    out_g = torch.empty((B, 2 * chains), dtype=torch.float64, device=dev)
    out_round = torch.empty((B, 2 * chains), dtype=torch.int32, device=dev)
    out_lb = torch.empty((B, 2 * chains), dtype=torch.float64, device=dev)
    out_asg = torch.empty((B, 2 * chains, F, N), dtype=torch.int16, device=dev)       # uint16 node ids
    max_slots = int(torch.floor(inst.Mj / inst.m[:, :1] + 1e-9).max().clamp(min=0, max=F).item())
    ws = torch.empty(lns_search_global_workspace_bytes(B, N, F, chains, k, max_slots), dtype=torch.uint8, device=dev)
    check(lib.neptune_lns_search_global(B, N, F, kind, C.c_double(alpha), chains, rounds, k, C.c_double(noise_coef),
                                        C.c_uint64(rng_seed), _ptr(inst.d), _ptr(inst.w), _ptr(inst.r), _ptr(inst.m),
                                        _ptr(inst.Mj), _ptr(inst.Kj), _ptr(inst.maxd), _ptr(guide), _ptr(lam0), S,
                                        _ptr(seeds_u8), max_slots, _ptr(out_c), _ptr(out_g), _ptr(out_lb), _ptr(out_round),
                                        _ptr(out_asg), _ptr(ws), ws.numel(), _stream()), "neptune_lns_search_global")
    del ws
    lns_search_global.last_other_bound = out_lb
    return out_c, out_g, out_round, out_asg.to(torch.int32) & 0xFFFF


def routing_of_assignment(inst: InstanceBatch, asg: torch.Tensor):
    """asg int[B,F,N] (node of every source) -> (c uint8[B,F,N], x[B,N,F,N], n[B,N]): every source routed whole to its
    node, only the pods some source uses open."""
    B, N, F = inst.B, inst.N, inst.F
    if bool((asg >= N).any()) or bool((asg < 0).any()):
        raise ValueError("routing_of_assignment: a source without a node (a chain that took no record)")
    idx = asg.to(torch.int64)
    c = torch.zeros((B, F, N), dtype=torch.uint8, device=asg.device)
    c.scatter_(2, idx, 1)
    x = torch.zeros((B, N, F, N), dtype=torch.float64, device=asg.device)
    x.scatter_(3, idx.permute(0, 2, 1)[..., None], 1.0)
    n = (c.amax(dim=1) > 0).to(torch.float64)
    return c, x, n


def slot_relaxation(inst: InstanceBatch) -> InstanceBatch:
    """The instance whose memory rows are replaced by their Chvatal-Gomory rounding: with one memory size m per
    instance,  sum_f m c[f,j] <= Mj  implies  sum_f c[f,j] <= floor(Mj / m)  for integer c
    (`constraints_step1.py:18-23`).  Valid for the MIP and much tighter for its LP relaxation (50x10: bound
    0.2-1 % below the optimum instead of 14 %).  Only m and Mj differ from `inst`."""
    import dataclasses
    slots = torch.floor(inst.Mj / inst.m[:, :1] + 1e-9).clamp_(max=float(inst.F))
    return dataclasses.replace(inst, m=torch.ones_like(inst.m), Mj=slots)


def disruption_search(inst: InstanceBatch, kind, mode: str, bound: torch.Tensor, seeds_u8: torch.Tensor, alpha=0.5,
                      chains=64, sweeps=300, rng_seed=1, workspace=None):
    """Step-2 search (`neptune_disruption_search`): mode "delete" | "create", bound[B] float64 on device.
    Returns (best_c uint8[B,F,N], best_obj float64[B] = step-2 objective or +inf, flags int32[B])."""
    lib = _lib.load()
    kind = KINDS.get(kind, kind)
    dev = inst.d.device
    S = seeds_u8.shape[1]
    need = C.c_int64()
    check(lib.neptune_local_search_workspace_bytes(inst.B, inst.N, inst.F, chains, C.byref(need)),
          "neptune_local_search_workspace_bytes")
    if workspace is None or workspace.numel() < need.value:
        workspace = torch.empty(need.value, dtype=torch.uint8, device=dev)
    best_c = torch.empty((inst.B, inst.F, inst.N), dtype=torch.uint8, device=dev)
    best_obj = torch.empty(inst.B, dtype=torch.float64, device=dev)
    best_flags = torch.empty(inst.B, dtype=torch.int32, device=dev)
    check(lib.neptune_disruption_search(inst.B, inst.N, inst.F, kind, C.c_double(alpha),
                                        {"delete": 1, "create": 2}[mode], _ptr(bound), chains, sweeps,
                                        C.c_uint64(rng_seed), S, *inst.inst_ptrs(), _ptr(inst.old), _ptr(seeds_u8),
                                        _ptr(best_c), _ptr(best_obj), _ptr(best_flags), _ptr(workspace),
                                        workspace.numel(), _stream()), "neptune_disruption_search")
    return best_c, best_obj, best_flags
