"""Function-block-sharded MATRIX-FREE PDHG for one large instance (SURVEY.md section 8(e), BASELINE config 4).
The iteration it drives is stated in numpy by `tests/mf_reference.ShardedMatrixFree`, which a world_size-2 gloo test
proves equal to the unsharded iteration; on B200 (round 2) two NCCL ranks reproduce the single-rank iterates to
3e-17 (`tools/sharded_run.py mf-parity`, profiles/r02_sharded_mf.md).

One process per GPU.  Rank g owns the functions of its block: x[f,.,.], c[f,.], y1[f,.], y3[f,.], yS[f,.,.]
are local; the 2N multipliers of the coupling rows (y2: C2 memory, y4: C4 CPU) are replicated.  ONE all-reduce of
2N doubles per iteration -- [C4 activity of the pass that just ran | C2 activity of the c columns just updated] --
and nothing of the matrix is stored: the per-GPU share of C4 (2000 nodes x 25 functions) is 4 x 0.8 GB of state
instead of 9.6 GB of CSR.  Measured on 2 x B200: 1.40 ms per iteration = 4.6 TB/s per GPU (0.70 of the measured
copy bandwidth), the all-reduce 19 us of it (1.4 %).
"""
from __future__ import annotations

import copy
import ctypes as C

import numpy as np
import torch
import torch.distributed as dist

from . import _lib, device
from ._lib import FLAG_STRENGTHEN, check
from .device import _ptr as _p, _stream
from .sharding import shard_range, world

EPS = 1e-6


def slice_functions(data, lo, hi):
    """`Data` restricted to functions [lo, hi) (nodes, delays, node capacities unchanged)."""
    d = copy.copy(data)
    d.functions = list(data.functions[lo:hi])
    for k in ("function_memory_matrix", "max_delay_matrix"):
        setattr(d, k, np.asarray(getattr(data, k))[lo:hi])
    for k in ("workload_matrix", "core_per_req_matrix", "old_allocations_matrix", "cores_matrix"):
        setattr(d, k, np.asarray(getattr(data, k))[lo:hi])
    return d


class ShardedMF:
    def __init__(self, data, eta=0.99):
        self.rank, self.world = world()
        F, N = len(data.functions), len(data.nodes)
        self.f_lo, self.f_hi = shard_range(F, self.rank, self.world)
        self.N, self.Fg, self.eta = N, self.f_hi - self.f_lo, eta
        self.inst = inst = device.InstanceBatch.from_datas([slice_functions(data, self.f_lo, self.f_hi)])
        self.lib = _lib.load()
        dev = inst.d.device
        f64 = dict(dtype=torch.float64, device=dev)
        Fg = self.Fg
        self.X, self.Cn = Fg * N * N, Fg * N
        self.rows, self.cols, _ = device.model_sizes(N, Fg, 0, FLAG_STRENGTHEN)
        self.r2, self.r3, self.r4, self.rs = 2 * self.Cn, 2 * self.Cn + N, 3 * self.Cn + N, 3 * self.Cn + 2 * N
        # global Pock-Chambolle row sums of the coupling rows: sum_f |m|, sum_{f,i} |w r|
        s2 = inst.m.abs().sum(dim=1)                                                     # [1]
        s4 = (inst.w.abs().sum(dim=2, keepdim=True) * inst.r.abs()).sum(dim=1)           # [1,N]
        both = torch.cat([s2.reshape(1, 1), s4], dim=1).contiguous()
        self.allreduce(both)
        self.S2 = torch.where(both[:, :1] > 0, 1.0 / both[:, :1], torch.ones_like(both[:, :1])).reshape(1).contiguous()
        self.S4 = torch.where(both[:, 1:] > 0, 1.0 / both[:, 1:], torch.ones_like(both[:, 1:])).contiguous()
        self.x = torch.zeros((1, self.cols), **f64)
        self.y = torch.zeros((1, self.rows), **f64)
        self.xsum = torch.zeros((1, self.cols), **f64)
        self.ysum = torch.zeros((1, self.rows), **f64)
        self.coupling = torch.zeros((1, 2 * N), **f64)
        need = C.c_int64()
        check(self.lib.neptune_pdhg_mf_step_bytes(1, N, Fg, C.byref(need)), "neptune_pdhg_mf_step_bytes")
        self.ws = torch.empty(need.value, dtype=torch.uint8, device=dev)
        self.tau = self.sigma = eta
        self._sigma_prev = 0.0
        self._have_pass = 0
        self.iters = 0
        self.exchanged_doubles = 0
        self._column_sums()

    # -- plumbing --------------------------------------------------------------------------------------
    def allreduce(self, t):
        if self.world == 1:
            return
        if dist.get_backend() == "nccl":
            dist.all_reduce(t)                       # NVLink / NVSwitch, on the current stream
        else:                                        # gloo (single-GPU test boxes): through host memory
            h = t.cpu()
            dist.all_reduce(h)
            t.copy_(h)

    def _state(self):
        return [_p(self.x), _p(self.y), _p(self.xsum), _p(self.ysum), _p(self.S4), _p(self.S2)]

    def _column_sums(self):
        i = self.inst
        check(self.lib.neptune_pdhg_mf_column_sums(1, self.N, self.Fg, _p(i.w), _p(i.r), _p(i.m), *self._state(),
                                                   _p(self.ws), self.ws.numel(), _stream()), "neptune_pdhg_mf_column_sums")

    # -- the iteration ---------------------------------------------------------------------------------
    def iterate(self, n=1):
        """n iterations; the state is a consistent PDHG iterate afterwards (the last C4 dual is flushed)."""
        i, lib, N, Fg = self.inst, self.lib, self.N, self.Fg
        for _ in range(n):
            check(lib.neptune_pdhg_mf_local_step(1, N, Fg, _p(i.w), _p(i.r), _p(i.m), C.c_double(self.tau),
                                                 C.c_double(self._sigma_prev), self._have_pass, 1, *self._state(),
                                                 _p(self.ws), self.ws.numel(), _p(self.coupling), _stream()),
                  "neptune_pdhg_mf_local_step")
            self.allreduce(self.coupling)
            self.exchanged_doubles += 2 * N
            check(lib.neptune_pdhg_mf_pass(1, N, Fg, _p(i.d), _p(i.w), _p(i.r), _p(i.m), _p(i.Mj), _p(i.Kj),
                                           C.c_double(self.tau), C.c_double(self.sigma), C.c_double(self._sigma_prev),
                                           self._have_pass, 1, *self._state(), _p(self.ws), self.ws.numel(),
                                           _p(self.coupling), _stream()), "neptune_pdhg_mf_pass")
            self._sigma_prev, self._have_pass = self.sigma, 1
        if n > 0:
            self._flush()
        self.iters += n

    def _flush(self):
        i, lib, N, Fg = self.inst, self.lib, self.N, self.Fg
        check(lib.neptune_pdhg_mf_local_step(1, N, Fg, _p(i.w), _p(i.r), _p(i.m), C.c_double(self.tau),
                                             C.c_double(self._sigma_prev), 1, 0, *self._state(), _p(self.ws),
                                             self.ws.numel(), _p(self.coupling), _stream()), "neptune_pdhg_mf_local_step")
        self.allreduce(self.coupling)
        self.exchanged_doubles += 2 * N
        check(lib.neptune_pdhg_mf_pass(1, N, Fg, _p(i.d), _p(i.w), _p(i.r), _p(i.m), _p(i.Mj), _p(i.Kj),
                                       C.c_double(self.tau), C.c_double(self.sigma), C.c_double(self._sigma_prev), 1, 0,
                                       *self._state(), _p(self.ws), self.ws.numel(), _p(self.coupling), _stream()),
              "neptune_pdhg_mf_pass")
        self._have_pass = 0

    # -- views of the canonical vectors ----------------------------------------------------------------
    def _parts(self, x, y):
        N, Fg, X, Cn = self.N, self.Fg, self.X, self.Cn
        xs = x[0, :X].reshape(Fg, N, N)
        c = x[0, X:X + Cn].reshape(Fg, N)
        y1 = y[0, 1:2 * Cn:2].reshape(Fg, N)
        y2 = y[0, self.r2:self.r2 + N]
        y3 = y[0, self.r3:self.r3 + Cn].reshape(Fg, N)
        y4 = y[0, self.r4:self.r4 + N]
        yS = y[0, self.rs:self.rs + X].reshape(Fg, N, N)
        return xs, c, y1, y2, y3, y4, yS

    def _kkt(self, x, y):
        """(primal residual^2, dual residual^2, primal objective, dual objective) of (x, y), global; the terms of
        the replicated rows are added once (rank 0)."""
        i = self.inst
        xs, c, y1, y2, y3, y4, yS = self._parts(x, y)
        w, r, m, d = i.w[0], i.r[0], i.m[0], i.d[0]
        wr = w[:, :, None] * r[:, None, :]
        obj = d[None, :, :] * w[:, :, None]
        act = torch.cat([(wr * xs).sum(dim=(0, 1)), m @ c]).reshape(1, -1).contiguous()
        self.allreduce(act)
        a4, a2 = act[0, :self.N], act[0, self.N:]
        p2 = (torch.clamp(xs.sum(dim=1) - c + EPS, max=0.0) ** 2).sum() + ((xs.sum(dim=2) - 1.0) ** 2).sum() \
            + (torch.clamp(xs - c[:, None, :], min=0.0) ** 2).sum()
        d2 = (torch.clamp(y1, min=0.0) ** 2).sum() + (torch.clamp(yS, max=0.0) ** 2).sum()
        dobj = EPS * torch.clamp(y1, max=0.0).sum() - y3.sum()
        rcx = obj + y1[:, None, :] + y3[:, :, None] + wr * y4[None, None, :] + yS
        rcc = -y1 + m[:, None] * y2[None, :] - yS.sum(dim=1)
        dobj = dobj + torch.clamp(rcx, max=0.0).sum() + torch.clamp(rcc, max=0.0).sum()
        pobj = (obj * xs).sum()
        if self.rank == 0:
            Mj, Kj = i.Mj[0], i.Kj[0]
            p2 = p2 + (torch.clamp(a2 - Mj, min=0.0) ** 2).sum() + (torch.clamp(a4 - Kj, min=0.0) ** 2).sum()
            d2 = d2 + (torch.clamp(y2, max=0.0) ** 2).sum() + (torch.clamp(y4, max=0.0) ** 2).sum()
            dobj = dobj - (Mj * torch.clamp(y2, min=0.0)).sum() - (Kj * torch.clamp(y4, min=0.0)).sum()
        v = torch.stack([p2, d2, pobj, dobj]).reshape(1, 4).contiguous()
        self.allreduce(v)
        return [float(t) for t in v[0].cpu()]

    def _norms(self):
        """global ||b||, ||c|| (plain) and their Pock-Chambolle-weighted versions (initial primal weight)"""
        i, N = self.inst, self.N
        w, r, d = i.w[0], i.r[0], i.d[0]
        obj = d[None, :, :] * w[:, :, None]
        Tx = 1.0 / (3.0 + (w[:, :, None] * r[:, None, :]).abs())
        loc = torch.stack([(obj * obj).sum(), (obj * obj * Tx).sum(),
                           torch.tensor(float(self.Cn), dtype=torch.float64, device=obj.device)]).reshape(1, 3).contiguous()
        self.allreduce(loc)
        nc2, ncs2, C_all = float(loc[0, 0]), float(loc[0, 1]), float(loc[0, 2])
        Mj, Kj = i.Mj[0], i.Kj[0]
        m2, k2 = float((Mj * Mj).sum()), float((Kj * Kj).sum())
        nb2 = EPS * EPS * C_all + m2 + C_all + k2
        nbs2 = EPS * EPS * C_all / (N + 1) + m2 * float(self.S2[0]) + C_all / N + float((Kj * Kj * self.S4[0]).sum())
        return nb2 ** 0.5, nc2 ** 0.5, nbs2 ** 0.5, ncs2 ** 0.5

    def _move2(self, xr, yr):
        """squared preconditioned norms of the displacement since the last restart point, global"""
        i, N = self.inst, self.N
        w, r, m = i.w[0], i.r[0], i.m[0]
        dxs, dc, dy1, dy2, dy3, dy4, dyS = self._parts(self.x - xr, self.y - yr)
        Tx = 1.0 / (3.0 + (w[:, :, None] * r[:, None, :]).abs())
        Tc = (1.0 / (1.0 + m.abs() + N))[:, None]
        dx2 = (dxs * dxs / Tx).sum() + (dc * dc / Tc).sum()
        dy2v = (dy1 * dy1).sum() * (N + 1) + (dy3 * dy3).sum() * N + (dyS * dyS).sum() * 2.0
        if self.rank == 0:
            dy2v = dy2v + (dy2 * dy2).sum() / self.S2[0] + (dy4 * dy4 / self.S4[0]).sum()
        v = torch.stack([dx2, dy2v]).reshape(1, 2).contiguous()
        self.allreduce(v)
        return float(v[0, 0]), float(v[0, 1])

    # -- restarted solve: every rank sees the same all-reduced numbers, hence takes the same decisions --------
    def solve(self, max_iters=20000, check_every=128, eps_rel=1e-6, eps_abs=1e-9):
        norm_b, norm_c, nbs, ncs = self._norms()
        omega = ncs / nbs if nbs > 1e-10 and ncs > 1e-10 else 1.0
        kkt_restart = kkt_prev = float("inf")
        xr, yr = self.x.clone(), self.y.clone()
        since = restarts = total = 0
        self.xsum.zero_(); self.ysum.zero_()
        info = {}
        while total < max_iters:
            self.tau, self.sigma = self.eta / omega, self.eta * omega
            self.iterate(check_every)
            total += check_every; since += check_every
            cands = []
            for (cx, cy) in ((self.x, self.y), (self.xsum / since, self.ysum / since)):
                p2, d2, po, do = self._kkt(cx, cy)
                gap = abs(po - do)
                k = (omega * omega * p2 + d2 / (omega * omega) + gap * gap) ** 0.5
                ok = p2 ** 0.5 <= eps_abs + eps_rel * norm_b and d2 ** 0.5 <= eps_abs + eps_rel * norm_c and \
                    gap <= eps_abs + eps_rel * (abs(po) + abs(do))
                cands.append((k, ok, po, do, p2 ** 0.5, d2 ** 0.5))
            pick = 1 if (cands[1][1] and not cands[0][1]) else (0 if (cands[0][1] and not cands[1][1])
                                                                 else (1 if cands[1][0] < cands[0][0] else 0))
            k, ok, po, do, pr, dr = cands[pick]
            info = dict(primal_obj=po, dual_obj=do, primal_res=pr, dual_res=dr, iters=total, restarts=restarts,
                        converged=bool(cands[0][1] or cands[1][1]), primal_weight=omega)
            done = info["converged"] or total >= max_iters
            act = done or k <= 0.2 * kkt_restart or (k <= 0.8 * kkt_restart and k > kkt_prev) or \
                (since >= 0.36 * total and restarts > 0) or (restarts == 0 and since >= 4 * check_every)
            kkt_prev = k
            if act:
                if pick == 1:
                    self.x.copy_(self.xsum / since); self.y.copy_(self.ysum / since)
                    self._column_sums()                      # yS was replaced: its column sums feed the next c update
                if done:
                    break
                kkt_restart = k; restarts += 1
                dx2, dy2 = self._move2(xr, yr)
                if dx2 > 1e-20 and dy2 > 1e-20:
                    nw = (dy2 / dx2) ** 0.25 * omega ** 0.5
                    omega = min(max(nw, 0.5 * omega), 2.0 * omega)
                xr.copy_(self.x); yr.copy_(self.y)
                self.xsum.zero_(); self.ysum.zero_(); since = 0
        return info


def bench_record(rank, world_size, peak_gbs, n_nodes=2000, n_funcs=200, iters=64, seed=0):
    """BASELINE config 4 inside bench.py (called by every rank of an initialised NCCL group): the sharded
    matrix-free iteration on one n_nodes x n_funcs instance -- us per iteration (max over ranks), algorithmic GB/s
    per GPU, the share of the all-reduce, and the drift of the sharded iterates from the single-GPU ones."""
    from . import sharding, synth
    from .core.utils import data_to_solver_input
    data = data_to_solver_input(synth.random_payload(n_nodes, n_funcs, seed, node_cores=None), 1, with_db=False)
    lp = ShardedMF(data)
    N = n_nodes
    lp.iterate(4)
    torch.cuda.synchronize()
    if world_size > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); lp.iterate(iters); e1.record(); e1.synchronize()
    ms = sharding.max_over_ranks(e0.elapsed_time(e1), device="cuda")
    # the exchange alone: the same number of all-reduces of 2N doubles, back to back
    e0.record()
    for _ in range(iters):
        lp.allreduce(lp.coupling)
    e1.record(); e1.synchronize()
    ms_ar = sharding.max_over_ranks(e0.elapsed_time(e1), device="cuda")
    by = 64 * lp.X + 112 * lp.Cn + 8 * N * N
    kkt = lp._kkt(lp.x, lp.y)                                  # collective
    rec = {"workload": f"C4: {n_nodes} nodes x {n_funcs} functions, one instance, functions sharded over {world_size} ranks "
                       f"({lp.Fg} on rank 0), matrix-free PDHG", "iterations": iters,
           "us_per_iteration": 1e3 * ms / iters, "gbs_per_gpu": by * iters / ms / 1e6,
           "frac_of_measured_hbm": by * iters / ms / 1e6 / peak_gbs, "aggregate_gbs": world_size * by * iters / ms / 1e6,
           "collective": "one NCCL all-reduce of 2N doubles per iteration (C4 activity | C2 activity), on the launch stream",
           "allreduce_bytes_per_iteration": 16 * N, "allreduce_us": 1e3 * ms_ar / iters,
           "allreduce_share_of_iteration": ms_ar / ms, "kkt_after": kkt}
    return rec
