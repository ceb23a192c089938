"""The C-ABI library loads on a CPU-only box and exports every symbol include/neptune_b200.h declares."""
import ctypes
import os
import re

from neptune_mip_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_functions():
    text = open(os.path.join(ROOT, "include", "neptune_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\bint\s+(neptune_\w+)\s*\(", text)))


def test_header_and_binding_agree():
    assert header_functions() == _lib.declared_symbols()


def test_library_exports_every_declared_symbol():
    assert os.path.exists(_lib.LIB_PATH), "build first: python -c 'import __graft_entry__ as g; g.build()'"
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in header_functions():
        assert hasattr(lib, name), name
    assert _lib.load().neptune_abi_version() == 1


def test_model_sizes_without_gpu():
    """Pure host arithmetic of the ABI (no kernel launch): the SURVEY.md section 8 size table."""
    lib = _lib.load()
    r, c, z = ctypes.c_int64(), ctypes.c_int64(), ctypes.c_int64()
    table = {(3, 2): (24, 24, 90), (50, 10): (1600, 25500, 101500), (500, 50): (76000, 12525000, 50075000),
             (2000, 200): (1204000, 800400000, 3201200000), (20, 5): (340, 2100, 8300)}
    for (N, F), want in table.items():
        assert lib.neptune_model_sizes(N, F, 0, 0, ctypes.byref(r), ctypes.byref(c), ctypes.byref(z)) == 0
        assert (r.value, c.value, z.value) == want
    assert lib.neptune_model_sizes(3, 2, 2, 0, ctypes.byref(r), ctypes.byref(c), ctypes.byref(z)) == 0
    assert (r.value, c.value, z.value) == (33, 27, 111)
    assert lib.neptune_model_sizes(0, 2, 0, 0, None, None, None) == -1
    assert lib.neptune_model_sizes(3, 2, 7, 0, None, None, None) == -1
    # 4000 x 400 would need > 2^31 columns: refused, not truncated
    assert lib.neptune_model_sizes(4000, 400, 0, 0, None, None, None) == -2


def test_no_cpu_fallback_without_gpu():
    import pytest
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from neptune_mip_b200 import device, synth
    from neptune_mip_b200.core.utils import data_to_solver_input
    data = data_to_solver_input(synth.test_py_payload(), 1, with_db=False)
    with pytest.raises(_lib.NeptuneError):
        device.InstanceBatch.from_datas([data])


def test_matrix_free_tile_geometry_covers_every_shape():
    """host arithmetic only: the tiles of the matrix-free passes cover N x N exactly once (even N > 32: pairs of
    adjacent columns, two columns per lane; odd wide N: four strided columns), workspaces hold the state"""
    lib = _lib.load()
    out = (ctypes.c_int32 * 16)()
    need = ctypes.c_int64()
    for (B, N, F) in [(1, 3, 2), (256, 50, 10), (4096, 20, 5), (1, 33, 3), (2, 64, 3), (2, 34, 3), (1, 56, 2), (1, 8, 4), (1, 65, 1), (1, 500, 50), (1, 2000, 25),
                      (1, 2000, 200), (3, 1026, 2), (1, 130, 2), (1, 131, 2)]:
        assert lib.neptune_pdhg_mf_geometry(B, N, F, out) == 0
        K, JT, ct, RT, rt, tiles, single = list(out)[:7]
        assert JT == 32 * K and K in (1, 2, 4) and (K == 1) == (N <= 32)
        assert K == (1 if N <= 32 else 2 if (N % 2 == 0 or N <= 64) else 4)
        assert (ct - 1) * JT < N <= ct * JT and (rt - 1) * RT < N <= rt * RT and 1 <= RT <= 64
        assert tiles == F * rt * ct and single == (F * N <= 4096)
        # bulk-copy pass: even N <= 64 only; a stage is 4 (2 with bulk reduction) slabs of N*N doubles, at least two stages
        ok4, st4, nw4, ok2, st2, nw2, dflt, smem2 = list(out)[8:]
        if N % 2 or N > 64:
            assert (ok4, ok2, dflt) == (0, 0, 0)
        else:
            slab = (8 * N * N + 127) // 128 * 128
            vec = ((7 * N + 4) * 8 + 127) // 128 * 128          # a stage: 2 or 4 read-write slabs + the delay matrix + the small vectors
            assert ok2 == 1 and 2 <= st2 <= 8 and 4 <= nw2 <= 15 and smem2 <= 227 * 1024 and smem2 >= st2 * (3 * slab + vec)
            assert (nw2 * ((N + nw2 - 1) // nw2) >= N) and ok4 == (1 if 2 * (5 * slab + vec) + 3 * nw4 * N * 8 + 512 <= 227 * 1024 else 0)
            if ok4:
                assert st4 >= 2 and st4 * (5 * slab + vec) <= 227 * 1024
        assert dflt in (0, 1, 2) and (N > 32 or dflt == 0)
        assert out[7] in (0, 1) and (out[7] == 0 or dflt != 0)        # small-vector update inside the bulk pass
        assert lib.neptune_pdhg_mf_workspace_bytes(B, N, F, ctypes.byref(need)) == 0
        X, C = F * N * N, F * N
        assert need.value >= 8 * B * (2 * (X + C) + 2 * (3 * C + 2 * N + X))        # xsum, xres, ysum, yres at least
    # C2 (50 x 10) runs the small-vector update inside the bulk pass; with 80 functions its two buffers do not fit
    for (N, F, fused) in [(50, 10, 1), (50, 80, 0), (64, 3, 0), (34, 3, 1), (12, 5, 0)]:
        assert lib.neptune_pdhg_mf_geometry(256, N, F, out) == 0 and out[7] == fused, (N, F)
    assert lib.neptune_pdhg_mf_geometry(0, 3, 2, out) == -1
    assert lib.neptune_pdhg_mf_workspace_bytes(1, 4000, 400, ctypes.byref(need)) == -2
