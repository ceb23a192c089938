"""Neptune step-1 classes (reference `core/solvers/neptune/neptune_step1.py:5-77`) on the GPU path.

`load_data` assembles the reference's MIP matrix on device (kernel group (a)); `solve` runs
LP relaxation by PDHG (b) for the bound and the rounding guide, the EFTTC greedy (d) for seeds, the
batched local search (c2), and the exact checkers/scorers (c1) on the winner.
"""
from __future__ import annotations

import numpy as np
import torch

from .... import device
from ..gpu_step import GpuStepMixin
from ..solver import Solver


class NeptuneStepBase(GpuStepMixin, Solver):
    """`lp_iters` > 0 by default: the drop-in path always solves the LP relaxation (matrix-free PDHG) and reports
    its bound and the gap of the returned placement (`lp_bound`, `mip_gap`).  `keep_model=True` additionally
    assembles the reference's matrix on device in `load_data` (kernel group (a)); nothing on the solve path reads
    it, so it is off by default (C4 would need 2 x 38 GB for it)."""

    def __init__(self, chains: int = 64, sweeps: int = 300, lp_iters: int = 20000, rng_seed: int = 1,
                 keep_model: bool = False, lns_chains: int = 384, lns_rounds: int = 8000, lns_k: int = 3,
                 lns_noise: float = 0.1, lns_final_k4: int = 1500, elites: int = 32, search: str = "auto", **kwargs):
        super().__init__(**kwargs)
        self.chains, self.sweeps, self.lp_iters, self.rng_seed = chains, sweeps, lp_iters, rng_seed
        self.lns_chains, self.lns_rounds, self.lns_k, self.lns_noise = lns_chains, lns_rounds, lns_k, lns_noise
        self.elites, self.search, self.lns_final_k4 = elites, search, lns_final_k4
        self.keep_model = keep_model
        self.model = None
        self.lp_bound = None
        self.mip_gap = None
        self.lp_result = None
        self._x = self._c = self._n = None

    def init_vars(self):
        self._upload()

    def init_constraints(self):
        # the reference builds rows here; on request so do we (on device), flags=0 is the as-written matrix
        if self.keep_model:
            self.model = device.assemble(self.inst, self.kind, self._alpha())

    def init_objective(self):
        pass                        # objective coefficients are part of `assemble`

    def results(self):
        self.data.prev_x = self._x
        self.data.prev_c = self._c
        return self._x, self._c


class NeptuneStep1CPUBase(NeptuneStepBase):
    def solve(self):
        """LP relaxation (bound, rounding guide, CPU-row prices) -> search -> exact routing LP -> the reference's
        checkers, all through `batch.solve_batch` (the path bench.py times) with a batch of one.  Min-delay instances too
        large for the searches with shared-memory chain state (N > 1066, BASELINE config 4) take the greedy ->
        pod-exchange search -> two-choice routing path instead."""
        from ....batch import BatchParams, solve_batch
        self.init_objective()
        prm = BatchParams(kind=self.kind, alpha=self._alpha(), lp_iters=self.lp_iters, lp_check_every=256,
                          chains=self.chains, sweeps=self.sweeps, rng_seed=self.rng_seed, search=self.search,
                          lns_chains=self.lns_chains, lns_rounds=self.lns_rounds, lns_k=self.lns_k,
                          lns_noise=self.lns_noise, elites=self.elites, lns_final_k4=self.lns_final_k4)
        res = solve_batch(self.inst, prm)
        self._take(res.c, res.x, res.n, res.flags, res.scores)
        if res.lp is not None:
            self.lp_result = res.lp[0]
            # a dual bound only once the dual residual is small; PDHG's dual objective is a bound at convergence
            self.lp_bound = float(res.lp[0]["dual_obj"])
            sc = float(self._kind_score())
            self.mip_gap = (sc - self.lp_bound) / max(abs(sc), 1e-12) if self.kind == "min_delay" else None
        self.log(f"step 1 ({res.search_path}): score {self._kind_score()} flags {self.flags:06b} "
                 f"lp bound {self.lp_bound} gap {self.mip_gap}")
        return self.feasible

    def score(self):
        return self._kind_score()


class NeptuneStep1CPUMinUtilization(NeptuneStep1CPUBase):
    kind = "min_util"

    def results(self):
        x, c = super().results()
        self.data.prev_n = self._n
        return x, c


class NeptuneStep1CPUMinDelay(NeptuneStep1CPUBase):
    kind = "min_delay"


class NeptuneStep1CPUMinDelayAndUtilization(NeptuneStep1CPUMinUtilization):
    kind = "min_delay_util"

    def __init__(self, alpha=0.5, **kwargs):
        super().__init__(**kwargs)
        self.alpha = alpha

    def load_data(self, data):
        data.alpha = self.alpha
        super().load_data(data)
