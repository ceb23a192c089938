"""Function-block-sharded matrix-free PDHG: 2 ranks must reproduce the unsharded iterates (one GPU, gloo for the
exchange -- the NCCL path is the same code with `dist.all_reduce` on device tensors)."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_matrix_free_single_rank_equals_the_numpy_iteration():
    """world size 1: the step-wise entry points (local step / pass / flush) reproduce tests/mf_reference.MatrixFree;
    65 x 8 runs four strided columns per lane, 130 x 33 three column tiles and 17 row tiles (561 partial sums per column
    of the C4 activity), both with CPU capacities tight enough that the C4 rows bind"""
    import numpy as np
    from helpers import arrays_of, data_of
    from mf_reference import MatrixFree
    from neptune_mip_b200 import synth
    from neptune_mip_b200.sharded_mf import ShardedMF
    for (N, F, cores, iters) in ((12, 5, 25, 96), (50, 4, 200, 40), (70, 3, 60, 33), (65, 8, 38, 33), (130, 33, 154, 33)):
        p = synth.random_payload(N, F, 1, node_cores=cores)
        lp = ShardedMF(data_of(p))
        ref = MatrixFree(arrays_of(p))
        lp.tau, lp.sigma = ref.eta / ref.omega, ref.eta * ref.omega          # the reference's primal-weighted steps
        lp.iterate(iters)
        for _ in range(iters):
            ref.step()
        xr, yr = ref.pack()
        x, y = lp.x[0].cpu().numpy(), lp.y[0].cpu().numpy()
        assert np.abs(x - xr).max() <= 1e-9 * (1 + np.abs(xr).max()), (N, F)
        assert np.abs(y - yr).max() <= 1e-9 * (1 + np.abs(yr).max()), (N, F)
        want = ref.kkt(ref.state())
        for u, v in zip(lp._kkt(lp.x, lp.y), want):
            assert abs(u - v) <= 1e-9 * (1 + abs(v))


def test_matrix_free_two_ranks_match_single_rank():
    env = dict(os.environ, NEPTUNE_DIST_BACKEND="gloo")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29535", os.path.join(ROOT, "tools", "sharded_run.py"), "mf-parity", "24", "6", "150"]
    out = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert "MF-PARITY world=2" in out.stdout


def test_matrix_free_two_ranks_match_single_rank_uneven_split():
    """33 functions over 2 ranks (17 + 16): the ranks' blocks differ in size, and 130 nodes give three column tiles and
    many row tiles per function; tight CPU capacities make the replicated C4 dual move"""
    env = dict(os.environ, NEPTUNE_DIST_BACKEND="gloo", NEPTUNE_NODE_CORES="154")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29537", os.path.join(ROOT, "tools", "sharded_run.py"), "mf-parity", "130", "33", "70"]
    out = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert "MF-PARITY world=2 N=130 F=33" in out.stdout


def test_matrix_free_sharded_solve_reaches_the_single_gpu_optimum():
    env = dict(os.environ, NEPTUNE_DIST_BACKEND="gloo", NEPTUNE_NODE_CORES="12")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29536", os.path.join(ROOT, "tools", "sharded_run.py"), "mf-solve", "8", "4", "40000"]
    out = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert "MF-SOLVE world=2" in out.stdout
