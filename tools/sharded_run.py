"""torchrun entry: function-block-sharded matrix-free PDHG (neptune_mip_b200/sharded_mf.py) vs the unsharded
iteration (parity), vs the single-GPU solver (solve), and timing.
  python -m torch.distributed.run --nproc-per-node 2 tools/sharded_run.py mf-parity|mf-solve|mf-time N F [iters]"""
import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np, torch, torch.distributed as dist
from neptune_mip_b200 import synth, sharding
from neptune_mip_b200.core.utils import data_to_solver_input
from neptune_mip_b200.sharded_mf import ShardedMF

mode, N, F = sys.argv[1], int(sys.argv[2]), int(sys.argv[3])
if mode not in ("mf-parity", "mf-solve", "mf-time"):
    sys.exit(__doc__)
iters = int(sys.argv[4]) if len(sys.argv) > 4 else 100
backend = os.environ.get("NEPTUNE_DIST_BACKEND", "nccl")
rank, ws, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ.get("LOCAL_RANK", 0))
ngpu = torch.cuda.device_count()
torch.cuda.set_device(local % ngpu)
dist.init_process_group(backend, **({"device_id": torch.device("cuda", local)} if backend == "nccl" else {}))
_nc = os.environ.get("NEPTUNE_NODE_CORES")
data = data_to_solver_input(synth.random_payload(N, F, 1 if _nc else 0, node_cores=int(_nc) if _nc else None), 1, with_db=False)
lp = ShardedMF(data)
if mode == "mf-parity":
    lp.iterate(iters)
    xloc = lp.x[0, : lp.Fg * N * N].reshape(lp.Fg, N * N).contiguous()
    xall = sharding.gather_rows(xloc.cpu(), F) if backend != "nccl" else sharding.gather_rows(xloc, F).cpu()
    ycoup = torch.cat([lp.y[0, lp.r2:lp.r2 + N], lp.y[0, lp.r4:lp.r4 + N]]).cpu()
    kkt = lp._kkt(lp.x, lp.y)                    # collective: every rank calls it
    if rank == 0:
        import neptune_mip_b200.sharded_mf as shm
        shm.world = lambda: (0, 1)               # reference: every function on one rank (no exchange)
        ref = ShardedMF(data)
        ref.iterate(iters)
        xr = ref.x[0, : F * N * N].reshape(F, N * N).cpu()
        yr = torch.cat([ref.y[0, ref.r2:ref.r2 + N], ref.y[0, ref.r4:ref.r4 + N]]).cpu()
        kr = ref._kkt(ref.x, ref.y)
        dx = float((xall - xr).abs().max()); dy = float((ycoup - yr).abs().max())
        print(f"MF-PARITY world={ws} N={N} F={F} iters={iters} max|dx|={dx:.3e} max|dy_coupling|={dy:.3e} "
              f"kkt sharded={kkt} single={kr} exchanged doubles/iter={lp.exchanged_doubles / max(lp.iters, 1):.1f}", flush=True)
        assert dx <= 1e-9 * (1 + float(xr.abs().max())) and dy <= 1e-9 * (1 + float(yr.abs().max()))
        assert all(abs(u - v) <= 1e-9 * (1 + abs(v)) for u, v in zip(kkt, kr))
elif mode == "mf-solve":
    info = lp.solve(max_iters=iters, check_every=128, eps_rel=1e-6)
    if rank == 0:
        from neptune_mip_b200 import device
        _, _, res = device.pdhg_mf_solve(device.InstanceBatch.from_datas([data]), max_iters=iters, check_every=128,
                                         eps_rel=1e-6, eps_abs=1e-9)
        print(f"MF-SOLVE world={ws} N={N} F={F} sharded: {info} | single GPU: primal={res[0]['primal_obj']:.9g} "
              f"dual={res[0]['dual_obj']:.9g} iters={res[0]['iters']} converged={res[0]['converged']}", flush=True)
        tol = 1e-4 * (1 + abs(float(res[0]["primal_obj"])))
        assert info["converged"] and res[0]["converged"] == 1 and abs(info["primal_obj"] - float(res[0]["primal_obj"])) <= tol
else:
    lp.iterate(5)
    torch.cuda.synchronize(); dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); lp.iterate(iters); e1.record(); e1.synchronize()
    ms = sharding.max_over_ranks(e0.elapsed_time(e1), device="cuda")
    by = 64 * lp.X + 112 * lp.Cn + 8 * N * N
    if rank == 0:
        print(f"MF-TIME world={ws} N={N} F={F} (Fg={lp.Fg}) {ms / iters * 1e3:.1f} us/iter  {by * iters / ms / 1e6:.1f} GB/s per GPU  "
              f"exchange {16 * N} B/iter", flush=True)
dist.destroy_process_group()
