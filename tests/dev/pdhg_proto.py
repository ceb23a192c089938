"""Historical numpy prototype of the round-1 PDHG on the assembled CSR matrix (csrc/pdhg.cu, since retired in favour
of the matrix-free solver, DESIGN.md section 3(b')); kept as the record of how its Ruiz scaling and restarts were tuned."""
import sys, time
sys.path.insert(0, '/root/repo'); sys.path.insert(0, '/root/repo/tests')
import numpy as np, scipy.sparse as sp
from helpers import arrays_of
from neptune_mip_b200 import synth
from oracle import model as omodel, mip as omip

def strengthened(a, kind, alpha):
    m = omodel.build_step1(a, kind, alpha)
    N, F = a["N"], a["F"]; X = F*N*N
    q = np.arange(X); f = q // (N*N); j = q % N
    S = sp.csr_matrix((np.tile([1.0,-1.0], X), np.stack([q, X + f*N + j],1).reshape(-1), np.arange(0, 2*X+1, 2)), shape=(X, m["A"].shape[1]))
    m2 = dict(m); m2["A"] = sp.vstack([m["A"], S]).tocsr()
    m2["lo"] = np.concatenate([m["lo"], np.full(X, -np.inf)]); m2["hi"] = np.concatenate([m["hi"], np.zeros(X)])
    return m2

def scale(A, ruiz=10):
    rows, cols = A.shape
    dr = np.ones(rows); dc = np.ones(cols)
    Aabs = abs(A)
    for it in range(ruiz+1):
        S = sp.diags(dr) @ Aabs @ sp.diags(dc)
        if it < ruiz:
            rm = S.max(axis=1).toarray().ravel(); cm = S.max(axis=0).toarray().ravel()
        else:
            rm = np.asarray(S.sum(axis=1)).ravel(); cm = np.asarray(S.sum(axis=0)).ravel()
        dr = np.where(rm > 0, dr/np.sqrt(np.where(rm>0,rm,1)), dr); dc = np.where(cm > 0, dc/np.sqrt(np.where(cm>0,cm,1)), dc)
    return dr, dc

def kkt(A, m, x, y):
    ax = A @ x
    pres2 = np.sum((ax - np.clip(ax, m["lo"], m["hi"]))**2)
    dobj = 0.0; dres2 = 0.0
    pos = y > 0; neg = y < 0
    fin_h = np.isfinite(m["hi"]); fin_l = np.isfinite(m["lo"])
    dobj -= np.sum(m["hi"][pos & fin_h] * y[pos & fin_h]); dres2 += np.sum(y[pos & ~fin_h]**2)
    dobj -= np.sum(m["lo"][neg & fin_l] * y[neg & fin_l]); dres2 += np.sum(y[neg & ~fin_l]**2)
    rc = m["obj"] + A.T @ y
    p = rc > 0; n = rc < 0
    fu = np.isfinite(m["ub"])
    dobj += np.sum(m["lb"][p]*rc[p]); dobj += np.sum(m["ub"][n & fu]*rc[n & fu]); dres2 += np.sum(rc[n & ~fu]**2)
    return pres2, dres2, float(m["obj"] @ x), dobj

def pdhg(m, max_iters=60000, check=64, eps=1e-6, adaptive=False, verbose=False, eta0=0.99):
    A = m["A"].tocsr(); At = A.T.tocsr()
    dr, dc = scale(A)
    T = dc**2; S = dr**2
    fb = np.where(np.isfinite(m["lo"]), np.abs(m["lo"]), 0); fb = np.maximum(fb, np.where(np.isfinite(m["hi"]), np.abs(m["hi"]), 0))
    nb = np.linalg.norm(fb); nc = np.linalg.norm(m["obj"])
    omega = nc/nb if nb > 1e-10 and nc > 1e-10 else 1.0
    eta = eta0
    x = np.zeros(A.shape[1]); y = np.zeros(A.shape[0])
    xs = np.zeros_like(x); ys = np.zeros_like(y); xr = x.copy(); yr = y.copy()
    cnt = 0; since = 0; restarts = 0; kr = np.inf; kp = np.inf
    it = 0
    while it < max_iters:
        for _ in range(check):
            tau = eta/omega; sig = eta*omega
            g = At @ y
            xn = np.clip(x - tau*T*(m["obj"] + g), m["lb"], m["ub"])
            xb = 2*xn - x
            s = sig*S
            v = y + s*(A @ xb)
            yn = v - s*np.clip(v/s, m["lo"], m["hi"])
            x, y = xn, yn
            xs += x; ys += y; cnt += 1
        it += check; since += check
        cands = []
        for (cx, cy) in ((x, y), (xs/cnt, ys/cnt)):
            p2, d2, po, do = kkt(A, m, cx, cy)
            gap = abs(po - do)
            k = np.sqrt(omega**2*p2 + d2/omega**2 + gap**2)
            ok = np.sqrt(p2) <= 1e-9 + eps*nb and np.sqrt(d2) <= 1e-9 + eps*nc and gap <= 1e-9 + eps*(abs(po)+abs(do))
            cands.append((k, ok, p2, d2, po, do))
        pick = 1 if cands[1][0] < cands[0][0] else 0
        if cands[0][1] or cands[1][1]:
            pick = 1 if cands[1][1] else 0
            if verbose: print("converged", it, cands[pick][4], cands[pick][5])
            return cands[pick][4], cands[pick][5], it
        cand = cands[pick][0]
        act = False
        if cand <= 0.2*kr: act = True
        elif cand <= 0.8*kr and cand > kp: act = True
        elif since >= 0.36*it and restarts > 0: act = True
        kp = cand
        if verbose and (it // check) % 50 == 0:
            print(it, pick, f"kkt={cand:.3e} pres={np.sqrt(cands[pick][2]):.2e} dres={np.sqrt(cands[pick][3]):.2e} po={cands[pick][4]:.4f} do={cands[pick][5]:.4f} om={omega:.3e} r={restarts}")
        if act:
            kr = cand; restarts += 1
            if pick == 1: x, y = xs/cnt, ys/cnt
            dx = np.sqrt(np.sum((x-xr)**2/T)); dy = np.sqrt(np.sum((y-yr)**2/S))
            if dx > 1e-10 and dy > 1e-10: omega = np.exp(0.5*np.log(dy/dx) + 0.5*np.log(omega))
            xr, yr = x.copy(), y.copy(); xs[:] = 0; ys[:] = 0; cnt = 0; since = 0
    return cands[pick][4], cands[pick][5], it

if __name__ == "__main__":
    p = synth.random_payload(12, 5, 1, node_cores=25)
    a = arrays_of(p)
    m = strengthened(a, "min_delay", 0.5)
    lp = omip.solve_model(m, relax=True)
    print("highs", lp["objective"])
    t = time.time()
    print(pdhg(m, verbose=True), time.time()-t)
