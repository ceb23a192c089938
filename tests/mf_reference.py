"""TEST INFRASTRUCTURE -- numpy reference of the MATRIX-FREE PDHG iteration of csrc/pdhg_mf.cu.

The constraint matrix of the strengthened min-delay placement model (reference rows
`core/solvers/neptune/utils/constraints_step1.py:5-65`, objective `objectives.py:4-11`, plus the valid rows
x[i,f,j] <= c[f,j]) is a closed formula of (N, F, w, r, m), so one PDHG iteration can be written as one pass
over the x-shaped arrays plus O(F*N) work on the small vectors.  This module states
  * `MatrixFree`  -- that iteration, in the order the CUDA kernels take it, and
  * `Generic`     -- the same algorithm on the oracle's CSR matrix (the matrix the reference's own builders
                     emit, `oracle/model.py`) with the same Pock-Chambolle step sizes,
so that tests can prove (on the CPU) that the matrix-free form IS the CSR iteration, and (on the GPU) that
the kernels reproduce it.  Used by tests/ and tools/ only.
"""
import numpy as np
import scipy.sparse as sp

EPS = 1e-6


def node_cut_bigm(a):
    """M of row C5a per node for the "node cut": the pods node j can hold, floor(Mj / min m) capped by F"""
    mm = a["m"].min()
    return np.clip(np.floor(a["Mj"] / mm + 1e-9), 0.0, float(a["F"])) if mm > 0 else np.full(a["N"], float(a["F"]))


def strengthened(a, kind="min_delay", alpha=0.5, bigm=None):
    from oracle import model as omodel
    m = omodel.build_step1(a, kind, alpha)
    N, F = a["N"], a["F"]; X = F * N * N
    if bigm is not None:                                      # C5a rows: sum_f c[f,j] - M_j n[j] <= 0 with the caller's M_j
        A = m["A"].tolil()
        r5 = 3 * F * N + 2 * N
        for jj in range(N):
            A[r5 + 2 * jj, X + F * N + jj] = -float(bigm[jj])
        m = dict(m); m["A"] = A.tocsr()
    q = np.arange(X); f = q // (N * N); j = q % N
    S = sp.csr_matrix((np.tile([1.0, -1.0], X), np.stack([q, X + f * N + j], 1).reshape(-1),
                       np.arange(0, 2 * X + 1, 2)), shape=(X, m["A"].shape[1]))
    m2 = dict(m); m2["A"] = sp.vstack([m["A"], S]).tocsr()
    m2["lo"] = np.concatenate([m["lo"], np.full(X, -np.inf)]); m2["hi"] = np.concatenate([m["hi"], np.zeros(X)])
    # as csrc/assemble.cu with NEPTUNE_FLAG_STRENGTHEN: C1a rows (even rows of the first 2*F*N) are free, x <= 1
    C = F * N
    m2["hi"][0:2 * C:2] = np.inf
    m2["ub"] = m2["ub"].copy(); m2["ub"][:X] = 1.0
    return m2


def pc_diag(m):
    """T = 1/colsum|A|, S = 1/rowsum|A| over the non-free rows: the Pock-Chambolle step sizes csrc/pdhg_mf.cu
    generates in closed form."""
    A = abs(m["A"]).tocsr()
    free = np.isinf(m["lo"]) & np.isinf(m["hi"])
    A = sp.diags((~free).astype(float)) @ A
    rs = np.asarray(A.sum(axis=1)).ravel(); cs = np.asarray(A.sum(axis=0)).ravel()
    return np.where(cs > 0, 1 / np.where(cs > 0, cs, 1), 1.0), np.where(rs > 0, 1 / np.where(rs > 0, rs, 1), 1.0)


class Generic:
    """The PDHG iteration on a CSR matrix with the step sizes of `pc_diag` (step and KKT pieces in the form the
    control logic of csrc/pdhg_ctl.cuh, k_ctl_decide / k_ctl_after_restart, reads them)."""

    def __init__(self, m, T, S):
        self.m, self.A, self.At, self.T, self.S = m, m["A"].tocsr(), m["A"].T.tocsr(), T, S
        fb = np.where(np.isfinite(m["lo"]), np.abs(m["lo"]), 0)
        fb = np.maximum(fb, np.where(np.isfinite(m["hi"]), np.abs(m["hi"]), 0))
        self.nb, self.nc = np.linalg.norm(fb), np.linalg.norm(m["obj"])
        nbs, ncs = np.sqrt(np.sum(fb * fb * S)), np.sqrt(np.sum(m["obj"] ** 2 * T))
        self.omega = ncs / nbs if nbs > 1e-10 and ncs > 1e-10 else 1.0
        self.eta = 0.99
        self.x = np.zeros(self.A.shape[1]); self.y = np.zeros(self.A.shape[0])

    def step(self):
        m = self.m
        tau, sig = self.eta / self.omega, self.eta * self.omega
        g = self.At @ self.y
        xn = np.clip(self.x - tau * self.T * (m["obj"] + g), m["lb"], m["ub"])
        xb = 2 * xn - self.x
        s = sig * self.S
        v = self.y + s * (self.A @ xb)
        yn = v - s * np.clip(v / s, m["lo"], m["hi"])
        self.x, self.y = xn, yn

    def kkt(self, x, y):
        m = self.m
        ax = self.A @ x
        p2 = np.sum((ax - np.clip(ax, m["lo"], m["hi"])) ** 2)
        dobj = 0.0; d2 = 0.0
        pos, neg = y > 0, y < 0
        fh, fl = np.isfinite(m["hi"]), np.isfinite(m["lo"])
        dobj -= np.sum(m["hi"][pos & fh] * y[pos & fh]); d2 += np.sum(y[pos & ~fh] ** 2)
        dobj -= np.sum(m["lo"][neg & fl] * y[neg & fl]); d2 += np.sum(y[neg & ~fl] ** 2)
        rc = m["obj"] + self.At @ y
        p, n = rc > 0, rc < 0
        fu = np.isfinite(m["ub"])
        dobj += np.sum(m["lb"][p] * rc[p]) + np.sum(m["ub"][n & fu] * rc[n & fu]); d2 += np.sum(rc[n & ~fu] ** 2)
        return p2, d2, float(m["obj"] @ x), dobj


class MatrixFree:
    """The same iteration without the matrix.  State in the canonical order: x[F,N,N] (f,i,j), c[F,N];
    y1[F,N] (C1b; C1a multipliers stay 0), y2[N], y3[F,N] (f,i), y4[N], yS[F,N,N]."""

    def __init__(self, a):
        N, F = a["N"], a["F"]
        self.N, self.F, self.a = N, F, a
        d, w, r, mm = a["d"], a["w"], a["r"], a["m"]
        self.wr = w[:, :, None] * r[:, None, :]                   # [f,i,j]
        self.obj = d[None, :, :] * w[:, :, None]
        self.Tx = 1.0 / (3.0 + self.wr)
        self.Tc = np.repeat((1.0 / (1.0 + mm + N))[:, None], N, 1)
        self.S1 = 1.0 / (N + 1); self.S3 = 1.0 / N; self.SS = 0.5
        sm = mm.sum(); self.S2 = 1.0 / sm if sm > 0 else 1.0
        s4 = self.wr.sum(axis=(0, 1)); self.S4 = np.where(s4 > 0, 1 / np.where(s4 > 0, s4, 1), 1.0)
        Mj, Kj = a["Mj"], a["Kj"]
        self.nb = np.sqrt(EPS ** 2 * F * N + np.sum(Mj ** 2) + F * N + np.sum(Kj ** 2))
        self.nc = np.linalg.norm(self.obj)
        nbs = np.sqrt(EPS ** 2 * self.S1 * F * N + np.sum(Mj ** 2) * self.S2 + self.S3 * F * N + np.sum(Kj ** 2 * self.S4))
        ncs = np.sqrt(np.sum(self.obj ** 2 * self.Tx))
        self.omega = ncs / nbs if nbs > 1e-10 and ncs > 1e-10 else 1.0
        self.eta = 0.99
        z = np.zeros
        self.x, self.c = z((F, N, N)), z((F, N))
        self.y1, self.y2, self.y3, self.y4, self.yS = z((F, N)), z(N), z((F, N)), z(N), z((F, N, N))
        self.sS = z((F, N))                                       # sum_i yS[f,i,j], maintained by the big pass

    def step(self):
        a, N = self.a, self.N
        tau, sig = self.eta / self.omega, self.eta * self.omega
        # ---- small kernel, part 1: c update (needs y of the previous iteration only) ----
        gc = -self.y1 + a["m"][:, None] * self.y2[None, :] - self.sS
        cn = np.clip(self.c - tau * self.Tc * gc, 0.0, 1.0)
        cb = 2 * cn - self.c
        self.c = cn
        # C2 dual (depends on c-bar only)
        s = sig * self.S2
        v = self.y2 + s * (a["m"] @ cb)
        y2n = v - s * np.minimum(v / s, a["Mj"])
        # ---- big fused pass over (f,i,j) ----
        g = self.obj + self.y1[:, None, :] + self.y3[:, :, None] + self.wr * self.y4[None, None, :] + self.yS
        xn = np.clip(self.x - tau * self.Tx * g, 0.0, 1.0)
        xb = 2 * xn - self.x
        s = sig * self.SS
        self.yS = np.maximum(self.yS + s * (xb - cb[:, None, :]), 0.0)
        self.x = xn
        A1 = xb.sum(axis=1)                      # [f,j]   sum over i
        A3 = xb.sum(axis=2)                      # [f,i]   sum over j
        A4 = (self.wr * xb).sum(axis=(0, 1))     # [j]
        self.sS = self.yS.sum(axis=1)
        # ---- small kernel, part 2 (start of the next launch): the remaining duals ----
        s = sig * self.S1
        v = self.y1 + s * (A1 - cb)
        self.y1 = v - s * np.maximum(v / s, -EPS)
        s = sig * self.S3
        v = self.y3 + s * A3
        self.y3 = v - s * 1.0
        s = sig * self.S4
        v = self.y4 + s * A4
        self.y4 = v - s * np.minimum(v / s, a["Kj"])
        self.y2 = y2n

    def pack(self):
        """canonical x / y vectors of the strengthened model"""
        F, N = self.F, self.N
        y1 = np.zeros((F * N, 2)); y1[:, 1] = self.y1.reshape(-1)
        return (np.concatenate([self.x.reshape(-1), self.c.reshape(-1)]),
                np.concatenate([y1.reshape(-1), self.y2, self.y3.reshape(-1), self.y4, self.yS.reshape(-1)]))

    def kkt(self, st):
        """closed-form KKT pieces of a state tuple (x,c,y1,y2,y3,y4,yS)"""
        a = self.a
        x, c, y1, y2, y3, y4, yS = st
        p2 = np.sum(np.minimum(x.sum(axis=1) - c + EPS, 0) ** 2) + np.sum(np.maximum(a["m"] @ c - a["Mj"], 0) ** 2)
        p2 += np.sum((x.sum(axis=2) - 1) ** 2) + np.sum(np.maximum((self.wr * x).sum(axis=(0, 1)) - a["Kj"], 0) ** 2)
        p2 += np.sum(np.maximum(x - c[:, None, :], 0) ** 2)
        d2 = np.sum(np.maximum(y1, 0) ** 2) + np.sum(np.minimum(y2, 0) ** 2) + np.sum(np.minimum(y4, 0) ** 2) + np.sum(np.minimum(yS, 0) ** 2)
        dobj = EPS * np.sum(np.minimum(y1, 0)) - np.sum(a["Mj"] * np.maximum(y2, 0)) - np.sum(y3) - np.sum(a["Kj"] * np.maximum(y4, 0))
        rcx = self.obj + y1[:, None, :] + y3[:, :, None] + self.wr * y4[None, None, :] + yS
        rcc = -y1 + a["m"][:, None] * y2[None, :] - yS.sum(axis=1)
        dobj += np.sum(np.minimum(rcx, 0)) + np.sum(np.minimum(rcc, 0))
        return p2, d2, float(np.sum(self.obj * x)), dobj

    def state(self):
        return (self.x, self.c, self.y1, self.y2, self.y3, self.y4, self.yS)

    def set_state(self, st):
        self.x, self.c, self.y1, self.y2, self.y3, self.y4, self.yS = [np.array(t, dtype=float) for t in st]
        self.sS = self.yS.sum(axis=1)

    def movement(self, st, rst):
        """distance from the last restart point in the preconditioned norms (primal, dual)"""
        Td = (self.Tx, self.Tc); Sd = (self.S1, self.S2, self.S3, self.S4, self.SS)
        dx2 = sum(np.sum((st[k] - rst[k]) ** 2 / Td[k]) for k in range(2))
        dy2 = sum(np.sum((st[2 + k] - rst[2 + k]) ** 2 / Sd[k]) for k in range(5))
        return np.sqrt(dx2), np.sqrt(dy2)


BIG_M = 1e6


def util_objective(a, kind, alpha):
    """(x-objective [F,N,N], n-objective scalar) of the models with node variables, reference `objectives.py:24-52`
    as oracle/model.py states them."""
    from oracle import model as omodel
    full = omodel.objective_step1(a, kind, alpha)
    N, F = a["N"], a["F"]; X = F * N * N
    return full[:X].reshape(F, N, N), float(full[X + F * N]) if N else 0.0


class MatrixFreeN(MatrixFree):
    """The iteration for the models with node variables n[j] (min-utilisation and the combined objective, reference
    `neptune_step1.py:38-77`): columns x, c, n; the rows of `MatrixFree` plus C5a (sum_f c[f,j] - M n[j] <= 0), C5b
    (sum_f c[f,j] - n[j] >= -eps) and C6 (cost_j n[j] <= budget), `constraints_step1.py:69-80, 101-103`.  Everything
    new is O(N) or O(F*N): it lives in the small-vector kernel; the pass over x only sees another objective."""

    def __init__(self, a, kind, alpha=0.5, bigm=None):
        super().__init__(a)
        N, F = self.N, self.F
        self.M = np.full(N, BIG_M) if bigm is None else np.asarray(bigm, dtype=float)
        self.obj, self.objn = util_objective(a, kind, alpha)
        self.cost, self.budget = a["cost"].astype(float), float(a["budget"])
        self.Tc = np.repeat((1.0 / (3.0 + a["m"] + N))[:, None], N, 1)
        self.Tn = 1.0 / (self.M + 1.0 + np.abs(self.cost))
        self.S5a, self.S5b = 1.0 / (F + self.M), 1.0 / (F + 1.0)
        self.S6 = np.where(self.cost != 0, 1.0 / np.where(self.cost != 0, np.abs(self.cost), 1.0), 1.0)
        Mj, Kj = a["Mj"], a["Kj"]
        bud2 = self.budget ** 2 if np.isfinite(self.budget) else 0.0
        self.nb = np.sqrt(EPS ** 2 * F * N + np.sum(Mj ** 2) + F * N + np.sum(Kj ** 2) + EPS ** 2 * N + bud2 * N)
        self.nc = np.sqrt(np.sum(self.obj ** 2) + self.objn ** 2 * N)
        nbs = np.sqrt(EPS ** 2 * self.S1 * F * N + np.sum(Mj ** 2) * self.S2 + self.S3 * F * N + np.sum(Kj ** 2 * self.S4)
                      + EPS ** 2 * self.S5b * N + bud2 * np.sum(self.S6))
        ncs = np.sqrt(np.sum(self.obj ** 2 * self.Tx) + self.objn ** 2 * np.sum(self.Tn))
        self.omega = ncs / nbs if nbs > 1e-10 and ncs > 1e-10 else 1.0
        z = np.zeros
        self.n, self.y5a, self.y5b, self.y6 = z(N), z(N), z(N), z(N)

    def step(self):
        a, N = self.a, self.N
        tau, sig = self.eta / self.omega, self.eta * self.omega
        # ---- small kernel, part 1: c and n columns from the duals of the previous iteration ----
        gc = -self.y1 + a["m"][:, None] * self.y2[None, :] - self.sS + (self.y5a + self.y5b)[None, :]
        cn = np.clip(self.c - tau * self.Tc * gc, 0.0, 1.0)
        cb = 2 * cn - self.c
        self.c = cn
        gn = self.objn - self.M * self.y5a - self.y5b + self.cost * self.y6
        nn = np.clip(self.n - tau * self.Tn * gn, 0.0, 1.0)
        nbar = 2 * nn - self.n
        self.n = nn
        # duals of the rows over (c, n) only
        s = sig * self.S2
        v = self.y2 + s * (a["m"] @ cb)
        y2n = v - s * np.minimum(v / s, a["Mj"])
        a5 = cb.sum(axis=0)
        s = sig * self.S5a
        v = self.y5a + s * (a5 - self.M * nbar)
        y5an = v - s * np.minimum(v / s, 0.0)
        s = sig * self.S5b
        v = self.y5b + s * (a5 - nbar)
        y5bn = v - s * np.maximum(v / s, -EPS)
        s = sig * self.S6
        v = self.y6 + s * (self.cost * nbar)
        y6n = v - s * np.minimum(v / s, self.budget)
        # ---- the pass over (f,i,j) and the remaining duals: as in the base class ----
        g = self.obj + self.y1[:, None, :] + self.y3[:, :, None] + self.wr * self.y4[None, None, :] + self.yS
        xn = np.clip(self.x - tau * self.Tx * g, 0.0, 1.0)
        xb = 2 * xn - self.x
        self.yS = np.maximum(self.yS + sig * self.SS * (xb - cb[:, None, :]), 0.0)
        self.x = xn
        A1, A3, A4 = xb.sum(axis=1), xb.sum(axis=2), (self.wr * xb).sum(axis=(0, 1))
        self.sS = self.yS.sum(axis=1)
        s = sig * self.S1
        v = self.y1 + s * (A1 - cb)
        self.y1 = v - s * np.maximum(v / s, -EPS)
        s = sig * self.S3
        self.y3 = self.y3 + s * A3 - s
        s = sig * self.S4
        v = self.y4 + s * A4
        self.y4 = v - s * np.minimum(v / s, a["Kj"])
        self.y2, self.y5a, self.y5b, self.y6 = y2n, y5an, y5bn, y6n

    def pack(self):
        F, N = self.F, self.N
        y1 = np.zeros((F * N, 2)); y1[:, 1] = self.y1.reshape(-1)
        y5 = np.stack([self.y5a, self.y5b], 1).reshape(-1)
        return (np.concatenate([self.x.reshape(-1), self.c.reshape(-1), self.n]),
                np.concatenate([y1.reshape(-1), self.y2, self.y3.reshape(-1), self.y4, y5, self.y6, self.yS.reshape(-1)]))

    def kkt(self, st):
        a = self.a
        x, c, y1, y2, y3, y4, yS, n, y5a, y5b, y6 = st
        p2, d2, _, dobj = super().kkt((x, c, y1, y2, y3, y4, yS))
        # super() priced the c columns without the C5 duals: redo that term
        rcc0 = -y1 + a["m"][:, None] * y2[None, :] - yS.sum(axis=1)
        rcc = rcc0 + (y5a + y5b)[None, :]
        dobj += np.sum(np.minimum(rcc, 0)) - np.sum(np.minimum(rcc0, 0))
        a5 = c.sum(axis=0)
        p2 += np.sum(np.maximum(a5 - self.M * n, 0) ** 2) + np.sum(np.minimum(a5 - n + EPS, 0) ** 2)
        p2 += np.sum(np.maximum(self.cost * n - self.budget, 0) ** 2)
        d2 += np.sum(np.minimum(y5a, 0) ** 2) + np.sum(np.maximum(y5b, 0) ** 2) + np.sum(np.minimum(y6, 0) ** 2)
        dobj += EPS * np.sum(np.minimum(y5b, 0)) - self.budget * np.sum(np.maximum(y6, 0))
        rcn = self.objn - self.M * y5a - y5b + self.cost * y6
        dobj += np.sum(np.minimum(rcn, 0))
        return p2, d2, float(np.sum(self.obj * x) + self.objn * np.sum(n)), dobj

    def state(self):
        return (self.x, self.c, self.y1, self.y2, self.y3, self.y4, self.yS, self.n, self.y5a, self.y5b, self.y6)

    def set_state(self, st):
        super().set_state(st[:7])
        self.n, self.y5a, self.y5b, self.y6 = [np.array(t, dtype=float) for t in st[7:]]

    def movement(self, st, rst):
        dx, dy = super().movement(st[:7], rst[:7])
        dx2 = dx ** 2 + np.sum((st[7] - rst[7]) ** 2 / self.Tn)
        dy2 = dy ** 2 + np.sum((st[8] - rst[8]) ** 2 / self.S5a) + np.sum((st[9] - rst[9]) ** 2 / self.S5b) + np.sum((st[10] - rst[10]) ** 2 / self.S6)
        return np.sqrt(dx2), np.sqrt(dy2)


def solve(mf: MatrixFree, max_iters=20000, check=64, eps=1e-6, verbose=False):
    """restart logic of csrc/pdhg_ctl.cuh (k_ctl_decide / k_ctl_after_restart) on the matrix-free state"""
    sums = [np.zeros_like(t) for t in mf.state()]
    rst = [np.array(t) for t in mf.state()]
    diag = None
    cnt = since = restarts = it = 0
    kr = kp = np.inf
    while it < max_iters:
        for _ in range(check):
            mf.step()
            for s_, t in zip(sums, mf.state()):
                s_ += t
            cnt += 1
        it += check; since += check
        cands = []
        for st in (mf.state(), tuple(s_ / cnt for s_ in sums)):
            p2, d2, po, do = mf.kkt(st)
            gap = abs(po - do)
            k = np.sqrt(mf.omega ** 2 * p2 + d2 / mf.omega ** 2 + gap ** 2)
            ok = np.sqrt(p2) <= 1e-9 + eps * mf.nb and np.sqrt(d2) <= 1e-9 + eps * mf.nc and gap <= 1e-9 + eps * (abs(po) + abs(do))
            cands.append((k, ok, p2, d2, po, do))
        pick = 1 if (cands[1][1] and not cands[0][1]) else (0 if (cands[0][1] and not cands[1][1]) else (1 if cands[1][0] < cands[0][0] else 0))
        if cands[0][1] or cands[1][1]:
            if pick == 1:
                mf.set_state(tuple(s_ / cnt for s_ in sums))
            return dict(primal=cands[pick][4], dual=cands[pick][5], iters=it, restarts=restarts, converged=True)
        cand = cands[pick][0]
        act = False
        if cand <= 0.2 * kr: act = True
        elif cand <= 0.8 * kr and cand > kp: act = True
        elif since >= 0.36 * it and restarts > 0: act = True
        elif restarts == 0 and since >= 4 * check: act = True
        kp = cand
        if verbose and (it // check) % 20 == 0:
            print(it, pick, f"kkt={cand:.3e} pres={np.sqrt(cands[pick][2]):.2e} dres={np.sqrt(cands[pick][3]):.2e} "
                  f"po={cands[pick][4]:.4f} do={cands[pick][5]:.4f} om={mf.omega:.3e} r={restarts}")
        if act:
            kr = cand; restarts += 1
            if pick == 1:
                mf.set_state(tuple(s_ / cnt for s_ in sums))
            st = mf.state()
            dx, dy = mf.movement(st, rst)
            if dx > 1e-10 and dy > 1e-10:
                nw = np.exp(0.5 * np.log(dy / dx) + 0.5 * np.log(mf.omega))
                mf.omega = min(max(nw, 0.5 * mf.omega), 2.0 * mf.omega)
            rst = [np.array(t) for t in st]
            for s_ in sums: s_[:] = 0
            cnt = since = 0
    return dict(primal=cands[pick][4], dual=cands[pick][5], iters=it, restarts=restarts, converged=False)


def solve_ctl(mf: MatrixFree, max_iters, check_every, eps_abs, eps_rel):
    """The restarted solve exactly as `neptune_pdhg_mf_solve` takes it: chunks of `check_every` iterations (the last
    one cut at max_iters), then the decision of k_ctl_decide and the primal-weight update of k_ctl_after_restart.
    Unlike `solve`, the final check (converged or out of iterations) takes no restart and leaves the better candidate
    in the state, and the absolute and relative tolerances are separate.

    Returns (info, log).  info: the device's result record (primal_obj, dual_obj, primal_res, dual_res,
    primal_weight, iters, restarts, converged).  log: one dict per check with the KKT errors of both candidates, the
    pick, the action (0 none, 1 restart to the average, 2 restart at the current iterate) and `decisions`, the
    floating-point comparisons the device evaluated at that check as (label, value, threshold) -- in the order and
    with the short-circuits of k_ctl_decide, so that a test can ask how far each was from going the other way."""
    omega = mf.omega
    sums = [np.zeros_like(t) for t in mf.state()]
    rst = [np.array(t) for t in mf.state()]
    iters = since = count = restarts = 0
    kr = kp = np.inf
    log = []
    while True:
        chunk = min(check_every, max_iters - iters)
        for _ in range(chunk):
            mf.step()
            for s_, t in zip(sums, mf.state()):
                s_ += t
        iters += chunk; since += chunk; count += chunk
        avg = tuple(s_ / count for s_ in sums)
        decisions, kkt, ok, nums = [], [], [], []
        for st in (mf.state(), avg):
            p2, d2, po, do = mf.kkt(st)
            gap = abs(po - do)
            kkt.append(np.sqrt(omega * omega * p2 + d2 / (omega * omega) + gap * gap))
            tests = [("primal residual", np.sqrt(p2), eps_abs + eps_rel * mf.nb),
                     ("dual residual", np.sqrt(d2), eps_abs + eps_rel * mf.nc),
                     ("gap", gap, eps_abs + eps_rel * (abs(po) + abs(do)))]
            good = True
            for t in tests:                                   # && of k_ctl_decide: stops at the first failure
                decisions.append(t)
                if not t[1] <= t[2]:
                    good = False
                    break
            ok.append(good)
            nums.append((po, do, np.sqrt(p2), np.sqrt(d2)))
        if ok[0] == ok[1]:
            decisions.append(("average vs current KKT", kkt[1], kkt[0]))
            pick = 1 if kkt[1] < kkt[0] else 0
        else:
            pick = 1 if ok[1] else 0
        done = ok[0] or ok[1]
        last = done or iters >= max_iters
        cand = kkt[pick]
        action = 0
        if not last:
            decisions.append(("sufficient decay", cand, 0.2 * kr))
            if cand <= 0.2 * kr:
                action = 1 + (pick == 0)
            else:
                decisions.append(("necessary decay", cand, 0.8 * kr))
                if cand <= 0.8 * kr:
                    decisions.append(("no progress", cand, kp))
                if cand <= 0.8 * kr and cand > kp:
                    action = 1 + (pick == 0)
                elif since >= 0.36 * iters and iters > 0 and restarts > 0:
                    action = 1 + (pick == 0)
                elif restarts == 0 and since >= 4 * chunk:
                    action = 1 + (pick == 0)
        kp = cand
        if action:
            kr = cand; restarts += 1
        log.append(dict(iters=iters, kkt=tuple(kkt), ok=tuple(ok), pick=pick, action=action if not last else 0,
                        decisions=decisions))
        po, do, pres, dres = nums[pick]
        info = dict(primal_obj=po, dual_obj=do, primal_res=pres, dual_res=dres, primal_weight=omega, iters=iters,
                    restarts=restarts, converged=int(done))
        if last:
            if pick == 1:                                     # the average is materialised into x, y
                mf.set_state(avg)
            return info, log
        if action:
            if action == 1:
                mf.set_state(avg)
            st = mf.state()
            dx, dy = mf.movement(st, rst)
            if dx > 1e-10 and dy > 1e-10 and np.isfinite(dx) and np.isfinite(dy):
                nw = np.exp(0.5 * np.log(dy / dx) + 0.5 * np.log(omega))
                omega = min(max(nw, 0.5 * omega), 2.0 * omega)
            mf.omega = omega                                  # MatrixFree.step takes tau, sigma from it
            rst = [np.array(t) for t in st]
            for s_ in sums:
                s_[:] = 0
            since = count = 0


def run_fixed(a, iters, kind="min_delay", alpha=0.5, bigm=None):
    """What `neptune_pdhg_mf_solve(max_iters = check_every = iters)` returns with unreachable tolerances:
    `iters` iterations, then the better (smaller KKT error) of the current iterate and the running average.
    Returns (x, y, info) with x / y in the canonical layout of the strengthened model."""
    mf = MatrixFree(a) if kind == "min_delay" else MatrixFreeN(a, kind, alpha, bigm)
    sums = [np.zeros_like(t) for t in mf.state()]
    for _ in range(iters):
        mf.step()
        for s_, t in zip(sums, mf.state()):
            s_ += t
    cands = []
    for st in (mf.state(), tuple(s_ / iters for s_ in sums)):
        p2, d2, po, do = mf.kkt(st)
        cands.append((np.sqrt(mf.omega ** 2 * p2 + d2 / mf.omega ** 2 + (po - do) ** 2), p2, d2, po, do))
    pick = 1 if cands[1][0] < cands[0][0] else 0
    if pick:
        mf.set_state(tuple(s_ / iters for s_ in sums))
    x, y = mf.pack()
    _, p2, d2, po, do = cands[pick]
    return x, y, dict(pick=pick, primal_obj=po, dual_obj=do, primal_res=float(np.sqrt(p2)), dual_res=float(np.sqrt(d2)),
                      omega=mf.omega, kkt=(cands[0][0], cands[1][0]))


class ShardedMatrixFree:
    """Function-block-sharded form of `MatrixFree` (SURVEY.md section 8(e); the plan for C4 on 8 GPUs): a rank
    owns the functions [f0, f1), i.e. x[f,:,:], c[f,:], y1[f,:], y3[f,:], yS[f,:,:] of those functions; the 2N
    multipliers of the coupling rows (y2: memory, y4: CPU) are replicated.  ONE exchange per iteration: the
    all-reduce of [sum_{own f,i} w r xbar (N) | sum_{own f} m cbar (N)] -- the C4 activity of the pass that just
    ran and the C2 activity of the c columns just updated.  `allreduce(vec)` sums a numpy vector over the ranks
    in place.  The KKT evaluation all-reduces the two activity vectors and four scalars; the replicated rows'
    terms are added once (by the rank with f0 == 0)."""

    def __init__(self, a, f0, f1, allreduce):
        self.full = MatrixFree(a)                      # closed-form tables and norms of the whole instance (host)
        self.f0, self.f1, self.allreduce = f0, f1, allreduce
        self.a, self.N = a, a["N"]
        sl = slice(f0, f1)
        F = self.full
        self.wr, self.obj, self.Tx, self.Tc = F.wr[sl], F.obj[sl], F.Tx[sl], F.Tc[sl]
        self.m = a["m"][sl]
        self.S1, self.S2, self.S3, self.S4, self.SS = F.S1, F.S2, F.S3, F.S4, F.SS
        self.omega, self.eta, self.nb, self.nc = F.omega, F.eta, F.nb, F.nc   # global numbers: every rank computes them alike
        Fg, N = f1 - f0, self.N
        z = np.zeros
        self.x, self.c = z((Fg, N, N)), z((Fg, N))
        self.y1, self.y3, self.yS = z((Fg, N)), z((Fg, N)), z((Fg, N, N))
        self.y2, self.y4 = z(N), z(N)                 # replicated
        self.sS = z((Fg, N))
        self.a4_part = z(N)                           # C4 activity of the last pass, own functions
        self.first = True
        self.exchanged_doubles = 0

    def step(self):
        a, N = self.a, self.N
        tau, sig = self.eta / self.omega, self.eta * self.omega
        # boundary work of the previous pass that is local: nothing pending on the very first step
        # c columns of this iteration (y1, sS local; y2 replicated and already global)
        gc = -self.y1 + self.m[:, None] * self.y2[None, :] - self.sS
        cn = np.clip(self.c - tau * self.Tc * gc, 0.0, 1.0)
        cb = 2 * cn - self.c
        self.c = cn
        # the one exchange: C4 activity of the previous pass | C2 activity of the new c columns
        buf = np.concatenate([self.a4_part, self.m @ cb])
        self.allreduce(buf)
        self.exchanged_doubles += buf.size
        a4, a2 = buf[:N], buf[N:]
        if not self.first:                            # y4 of the previous iteration (replicated update)
            s = self._sig_prev * self.S4
            v = self.y4 + s * a4
            self.y4 = v - s * np.minimum(v / s, a["Kj"])
        s = sig * self.S2
        v = self.y2 + s * a2
        y2n = v - s * np.minimum(v / s, a["Mj"])
        # the pass over the own functions
        g = self.obj + self.y1[:, None, :] + self.y3[:, :, None] + self.wr * self.y4[None, None, :] + self.yS
        xn = np.clip(self.x - tau * self.Tx * g, 0.0, 1.0)
        xb = 2 * xn - self.x
        self.yS = np.maximum(self.yS + sig * self.SS * (xb - cb[:, None, :]), 0.0)
        self.x = xn
        self.sS = self.yS.sum(axis=1)
        # local duals of this iteration; the C4 activity waits for the next exchange
        s = sig * self.S1
        v = self.y1 + s * (xb.sum(axis=1) - cb)
        self.y1 = v - s * np.maximum(v / s, -EPS)
        s = sig * self.S3
        self.y3 = self.y3 + s * xb.sum(axis=2) - s
        self.a4_part = (self.wr * xb).sum(axis=(0, 1))
        self.y2 = y2n
        self._sig_prev = sig
        self.first = False

    def flush(self):
        """apply the pending C4 dual update (end of a chunk: the state becomes a consistent PDHG iterate)"""
        if self.first:
            return
        buf = self.a4_part.copy()
        self.allreduce(buf)
        self.exchanged_doubles += buf.size
        s = self._sig_prev * self.S4
        v = self.y4 + s * buf
        self.y4 = v - s * np.minimum(v / s, self.a["Kj"])
        self.a4_part[:] = 0.0
        self.first = True

    def kkt(self):
        """global KKT pieces of the current iterate (same numbers on every rank)"""
        a = self.a
        x, c, y1, y2, y3, y4, yS = self.x, self.c, self.y1, self.y2, self.y3, self.y4, self.yS
        act = np.concatenate([(self.wr * x).sum(axis=(0, 1)), self.m @ c])
        self.allreduce(act)
        a4, a2 = act[:self.N], act[self.N:]
        p2 = np.sum(np.minimum(x.sum(axis=1) - c + EPS, 0) ** 2) + np.sum((x.sum(axis=2) - 1) ** 2)
        p2 += np.sum(np.maximum(x - c[:, None, :], 0) ** 2)
        d2 = np.sum(np.maximum(y1, 0) ** 2) + np.sum(np.minimum(yS, 0) ** 2)
        dobj = EPS * np.sum(np.minimum(y1, 0)) - np.sum(y3)
        rcx = self.obj + y1[:, None, :] + y3[:, :, None] + self.wr * y4[None, None, :] + yS
        rcc = -y1 + self.m[:, None] * y2[None, :] - yS.sum(axis=1)
        dobj += np.sum(np.minimum(rcx, 0)) + np.sum(np.minimum(rcc, 0))
        pobj = float(np.sum(self.obj * x))
        if self.f0 == 0:                              # replicated rows: counted once
            p2 += np.sum(np.maximum(a2 - a["Mj"], 0) ** 2) + np.sum(np.maximum(a4 - a["Kj"], 0) ** 2)
            d2 += np.sum(np.minimum(y2, 0) ** 2) + np.sum(np.minimum(y4, 0) ** 2)
            dobj += -np.sum(a["Mj"] * np.maximum(y2, 0)) - np.sum(a["Kj"] * np.maximum(y4, 0))
        v = np.array([p2, d2, pobj, dobj])
        self.allreduce(v)
        return tuple(float(t) for t in v)
