"""numpy statement of the pod-exchange search of csrc/site_search.cu (`neptune_site_search`), term for term.

Objective: obj(c) = sum_f sum_i w[f,i] * d1[f,i], d1 = delay from source i to the nearest open pod of f.  Per function
and source the search keeps the nearest and second-nearest open pod (a1, d1, a2, d2; lowest node among equal delays).
One round:
  G[f,j] = sum_i w * max(0, d1 - d[i,j])              gain of adding pod (f, j)
  L[f,j] = sum_{i: a1 = j} w * (d2 - d1)              loss of removing open pod (f, j); +inf when f has one pod
  node j proposes the best of   add (f, j)            m[f] <= memfree[j] + 1e-9,            delta = -G[f,j]
                                exchange f_out -> f_in m[f_in] <= memfree[j] + m[f_out] + 1e-9, delta = L[f_out,j] - G[f_in,j]
      (enumerated add first, then f_out ascending; f ascending inside; a later candidate must be strictly better)
  function f proposes the best relocation j_out -> j_in: j_in among the 4 nodes with the largest G[f,.] (lowest node
      among equals) that have memory for f, j_out among its pods; delta = sum_i w * (min(dwo, d[i,j_in]) - d1),
      dwo = d2 where a1 = j_out else d1 (enumerated j_out ascending, then j_in ascending)
  proposals with delta < -1e-12 * (1 + obj) sorted by (delta, nodes before functions, lower index); a proposal is
  accepted when none of its functions and nodes was touched by an accepted one in this round.
Moves on disjoint functions and nodes are independent (the objective separates by function, memory by node), so the
objective after a round is the one before plus the accepted deltas.  Sums run over i in ascending order with a separate
multiply and add, as the kernels do: placements, counters and objectives compare bit for bit.
"""
from __future__ import annotations

import numpy as np

K_CAND = 4
MEM_TOL = 1e-9


def nearest_two(d, c):
    """(a1, d1, a2, d2) [F, N]: nearest / second-nearest open pod of every (f, source); -1 / +inf where there is none."""
    F, N = c.shape
    a1 = np.full((F, N), -1, dtype=np.int64); a2 = np.full((F, N), -1, dtype=np.int64)
    d1 = np.full((F, N), np.inf); d2 = np.full((F, N), np.inf)
    rows = np.arange(N)
    for f in range(F):
        pods = np.flatnonzero(c[f])
        if pods.size == 0:
            continue
        dd = d[:, pods]
        order = np.argsort(dd, axis=1, kind="stable")                    # lowest node among equal delays
        a1[f] = pods[order[:, 0]]; d1[f] = dd[rows, order[:, 0]]
        if pods.size > 1:
            a2[f] = pods[order[:, 1]]; d2[f] = dd[rows, order[:, 1]]
    return a1, d1, a2, d2


def objective(w, d1):
    """sum over i ascending per function, then over f ascending"""
    F, N = w.shape
    objf = np.zeros(F)
    for i in range(N):
        objf = objf + w[:, i] * d1[:, i]
    obj = 0.0
    for f in range(F):
        obj = obj + objf[f]
    return float(obj)


def free_memory(Mj, m, c):
    mf = np.asarray(Mj, dtype=np.float64).copy()
    for f in range(c.shape[0]):
        mf = np.where(c[f] > 0, mf - m[f], mf)
    return mf


def tables(d, w, c, a1, d1, d2):
    F, N = w.shape
    G = np.zeros((F, N)); L = np.zeros((F, N))
    ar = np.arange(F)
    with np.errstate(invalid="ignore"):
        for i in range(N):
            G = G + w[:, i, None] * np.maximum(d1[:, i, None] - d[i][None, :], 0.0)
            L[ar, a1[:, i]] = L[ar, a1[:, i]] + w[:, i] * (d2[:, i] - d1[:, i])
    L[c.sum(axis=1) <= 1] = np.inf
    return G, L


def node_proposals(m, c, memfree, G, L):
    """[(delta, f_in, f_out)] per node; f_out = -1 for an add, delta = +inf when the node has nothing to propose"""
    F, N = c.shape
    out = []
    for j in range(N):
        free = c[:, j] == 0
        best = (np.inf, -1, -1)
        cand = np.where(free & (m <= memfree[j] + MEM_TOL), -G[:, j], np.inf)
        k = int(np.argmin(cand))
        if cand[k] < best[0]:
            best = (float(cand[k]), k, -1)
        for fo in np.flatnonzero(c[:, j]):
            cand = np.where(free & (m <= memfree[j] + m[fo] + MEM_TOL), L[fo, j] - G[:, j], np.inf)
            k = int(np.argmin(cand))
            if cand[k] < best[0]:
                best = (float(cand[k]), k, int(fo))
        out.append(best)
    return out


def relocation_candidates(m_f, c_f, memfree, G_f):
    ok = np.flatnonzero((c_f == 0) & (m_f <= memfree + MEM_TOL))
    order = np.lexsort((ok, -G_f[ok]))                                   # largest gain, lowest node among equals
    return np.sort(ok[order[:K_CAND]])


def function_proposals(d, w, m, c, memfree, G, a1, d1, d2):
    """[(delta, j_out, j_in)] per function"""
    F, N = c.shape
    out = []
    for f in range(F):
        cand = relocation_candidates(m[f], c[f], memfree, G[f])
        pods = np.flatnonzero(c[f])
        if cand.size == 0 or pods.size == 0:
            out.append((np.inf, -1, -1))
            continue
        JO = np.repeat(pods, cand.size); JI = np.tile(cand, pods.size)       # pair p = q * ncand + k
        acc = np.zeros(JO.size)
        for i in range(N):
            dwo = np.where(a1[f, i] == JO, d2[f, i], d1[f, i])
            acc = acc + w[f, i] * (np.minimum(dwo, d[i, JI]) - d1[f, i])
        p = int(np.argmin(acc))
        out.append((float(acc[p]), int(JO[p]), int(JI[p])))
    return out


def exchange_search(a, c0, max_rounds=None):
    """Best-improvement pod-exchange search from placement c0 [F, N] (every function with a pod).  Returns a dict:
    c (uint8 [F, N]), info = [rounds that accepted a move, adds, exchanges, relocations], objs = objective at the start
    and after every such round, deltas = sum of the accepted deltas of every such round."""
    N, F = a["N"], a["F"]
    d, w, m, Mj = a["d"], a["w"], a["m"], a["Mj"]
    c = (np.asarray(c0) > 0).astype(np.uint8).copy()
    assert (c.sum(axis=1) >= 1).all(), "every function needs a pod"
    a1, d1, a2, d2 = nearest_two(d, c)
    obj = objective(w, d1)
    info = [0, 0, 0, 0]
    objs, deltas = [obj], []
    for _ in range(max_rounds or N * F):
        memfree = free_memory(Mj, m, c)
        G, L = tables(d, w, c, a1, d1, d2)
        props = [(dl, p, ("node", j, fi, fo)) for p, (j, (dl, fi, fo)) in enumerate(enumerate(node_proposals(m, c, memfree, G, L)))]
        props += [(dl, N + f, ("func", f, jo, ji))
                  for f, (dl, jo, ji) in enumerate(function_proposals(d, w, m, c, memfree, G, a1, d1, d2))]
        thr = -1e-12 * (1.0 + obj)
        props = sorted((p for p in props if p[0] < thr), key=lambda p: (p[0], p[1]))
        tf = np.zeros(F, dtype=bool); tn = np.zeros(N, dtype=bool)
        acc = 0
        dsum = 0.0
        for dl, _, mv in props:
            if mv[0] == "node":
                _, j, fi, fo = mv
                if tn[j] or tf[fi] or (fo >= 0 and tf[fo]):
                    continue
                c[fi, j] = 1; tn[j] = True; tf[fi] = True
                if fo >= 0:
                    c[fo, j] = 0; tf[fo] = True
                    info[2] += 1
                else:
                    info[1] += 1
            else:
                _, f, jo, ji = mv
                if tf[f] or tn[jo] or tn[ji]:
                    continue
                c[f, jo] = 0; c[f, ji] = 1; tf[f] = True; tn[jo] = True; tn[ji] = True
                info[3] += 1
            acc += 1
            dsum += dl
        if acc == 0:
            break
        info[0] += 1
        a1, d1, a2, d2 = nearest_two(d, c)
        obj = objective(w, d1)
        objs.append(obj)
        deltas.append(dsum)
    return dict(c=c, info=info, objs=objs, deltas=deltas)
