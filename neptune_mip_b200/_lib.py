"""ctypes binding of libneptune_b200.so (the C ABI declared in include/neptune_b200.h).

There is NO CPU fallback: if the library is missing or a call returns a CUDA error this module
raises.  PyTorch is only used by the callers for device memory and streams; no torch type crosses
this boundary (plain pointers and sizes).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libneptune_b200.so")

KIND_MIN_DELAY, KIND_MIN_UTIL, KIND_MIN_DELAY_UTIL = 0, 1, 2
KINDS = {"min_delay": 0, "min_util": 1, "min_delay_util": 2}
FLAG_STRENGTHEN = 1
OK_C_X, OK_MEMORY, OK_HANDLE, OK_CPU, OK_N_C, OK_BUDGET, OK_ALL = 1, 2, 4, 8, 16, 32, 63
FLAG_NAMES = ("c_x", "memory", "handle_all", "cpu", "n_c", "budget")


class PdhgParams(C.Structure):
    _fields_ = [("max_iters", C.c_int), ("check_every", C.c_int), ("ruiz_iters", C.c_int),
                ("reserved", C.c_int), ("eps_rel", C.c_double), ("eps_abs", C.c_double)]


PDHG_RESULT_FIELDS = ("primal_obj", "dual_obj", "primal_res", "dual_res", "gap", "step", "primal_weight")
PDHG_RESULT_BYTES = 7 * 8 + 4 * 4


class NeptuneError(RuntimeError):
    pass


_p, _i, _i64, _d = C.c_void_p, C.c_int, C.c_int64, C.c_double
_INST = [_p] * 8 + [_d]          # d w r m Mj Kj maxd cost budget

_SIGNATURES = {
    "neptune_abi_version": [],
    "neptune_model_sizes": [_i, _i, _i, _i, C.POINTER(_i64), C.POINTER(_i64), C.POINTER(_i64)],
    "neptune_assemble_pattern": [_i, _i, _i, _i, _p, _p, _p, _p, _p],
    "neptune_assemble_values": [_i, _i, _i, _i, _i, _d] + _INST + [_p] * 9 + [_p],
    "neptune_pdhg_mf_workspace_bytes": [_i, _i, _i, C.POINTER(_i64)],
    "neptune_pdhg_mf_geometry": [_i, _i, _i, C.POINTER(C.c_int32)],
    "neptune_pdhg_mf_solve_util": [_i, _i, _i, _i] + [_p] * 7 + [_d, _d, _p] + [C.POINTER(PdhgParams)] + [_p] * 3 + [_p, _i64, _p],
    "neptune_pdhg_mf_solve": [_i, _i, _i, _i] + [_p] * 6 + [C.POINTER(PdhgParams)] + [_p] * 3 + [_p, _i64, _p],
    "neptune_pdhg_mf_step_bytes": [_i, _i, _i, C.POINTER(_i64)],
    "neptune_pdhg_mf_column_sums": [_i, _i, _i] + [_p] * 9 + [_p, _i64, _p],
    "neptune_pdhg_mf_local_step": [_i, _i, _i] + [_p] * 3 + [_d, _d, _i, _i] + [_p] * 6 + [_p, _i64, _p, _p],
    "neptune_pdhg_mf_pass": [_i, _i, _i] + [_p] * 6 + [_d, _d, _d, _i, _i] + [_p] * 6 + [_p, _i64, _p, _p],
    "neptune_check_solution": [_i, _i, _i, _d] + _INST + [_p] * 5 + [_p],
    "neptune_route_placements": [_i, _i, _i, _p, _p, _p, _p, _p],
    "neptune_route_capacitated": [_i, _i, _i] + [_p] * 10 + [_p],
    "neptune_route_lp": [_i, _i, _i, _i] + [_p] * 11 + [_i64, _p, _i64, _p],
    "neptune_route_lp_workspace_bytes": [_i, _i, _i, _i, _i64, C.POINTER(_i64)],
    "neptune_site_greedy_workspace_bytes": [_i, _i, _i, C.POINTER(_i64)],
    "neptune_site_greedy": [_i, _i, _i, _p, _p, _p, _p, _d, _i, _p, _p, _p, _i64, _p],
    "neptune_site_search_workspace_bytes": [_i, _i, _i, C.POINTER(_i64)],
    "neptune_site_search": [_i, _i, _i, _p, _p, _p, _p, _p, _p, _i, _p, _p, _p, _i64, _p],
    "neptune_route_two_choice_workspace_bytes": [_i, _i, _i, C.POINTER(_i64)],
    "neptune_route_two_choice": [_i, _i, _i] + [_p] * 4 + [_p] * 6 + [C.POINTER(C.c_int32), _i, _p, _i64, _p],
    "neptune_lns_block_mode": [_i],
    "neptune_lns_search": [_i, _i, _i, _i, _d, _i, _i, _i, _d, C.c_uint64] + [_p] * 9 + [_i, _p, _i, _p, _p, _p, _p, _p],
    "neptune_lns_search_global": [_i, _i, _i, _i, _d, _i, _i, _i, _d, C.c_uint64] + [_p] * 9 + [_i, _p, _i] + [_p] * 6 + [_i64, _p],
    "neptune_lns_search_global_workspace_bytes": [_i, _i, _i, _i, _i, _i, C.POINTER(_i64)],
    "neptune_eval_placements": [_i, _i, _i, _i, _d] + _INST + [_p] * 4 + [_p],
    "neptune_local_search": [_i, _i, _i, _i, _d, _i, _i, C.c_uint64, _i] + _INST + [_p] * 6 + [_p, _i64, _p],
    "neptune_disruption_search": [_i, _i, _i, _i, _d, _i, _p, _i, _i, C.c_uint64, _i] + _INST + [_p] * 5 + [_p, _i64, _p],
    "neptune_local_search_workspace_bytes": [_i, _i, _i, _i, C.POINTER(_i64)],
    "neptune_local_search_fits": [_i, _i, C.POINTER(C.c_int32)],
    "neptune_efttc": [_i, _i, _i, _i, _d] + [_p] * 8 + [_d] + [_p] * 3 + [_p, _i64, _p],
    "neptune_efttc_workspace_bytes": [_i, _i, _i, C.POINTER(_i64)],
    "neptune_u8_to_f64": [_i64, _p, _p, _p],
    "neptune_launch_count": [C.POINTER(_i64), _i],
    "neptune_efttc_host": [_i, _i, _i, _i, _d] + [_p] * 9 + [_d] + [_p] * 5 + [_p],
}

_lib = None


def declared_symbols():
    """Every function include/neptune_b200.h declares (kept in sync by tests/test_abi.py)."""
    return sorted(_SIGNATURES)


def load():
    """dlopen the in-tree library (built by `__graft_entry__.build()` / csrc/Makefile)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NeptuneError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  neptune_mip_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, argtypes in _SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the .so does not export it
        fn.argtypes = argtypes
        fn.restype = C.c_int
    _lib = lib
    return lib


def check(rc, what):
    if rc == 0:
        return
    if rc < 0:
        names = {-1: "invalid argument", -2: "size does not fit the ABI", -3: "workspace too small"}
        raise NeptuneError(f"{what}: {names.get(rc, rc)}")
    raise NeptuneError(f"{what}: CUDA error {rc}")
