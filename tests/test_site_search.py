"""Pod-exchange search (`neptune_site_search`, csrc/site_search.cu) and the min-delay solve path built on it.

CPU: the numpy statement (tests/site_search_reference.py) keeps the memory rows and a pod per function after every
round, its objective moves by exactly the accepted deltas and never up, and at termination no add, exchange or
relocation found by brute force improves it; the size rule that sends min-delay instances to this path.
GPU: the device equals the numpy statement bit for bit, in a batch and alone; on the C2 seeds with HiGHS optima the path
is no worse than greedy + two-choice and never below the optimum; at BASELINE config 4 the drop-in class returns."""
import json
import os

import numpy as np
import pytest

import site_search_reference as ref
from helpers import arrays_of, cuda_batch, float_payload
from neptune_mip_b200 import synth
from oracle import site as osite

SHAPES = [("8x4", lambda s: synth.random_payload(8, 4, s, node_cores=30)),
          ("12x5", lambda s: synth.random_payload(12, 5, s, node_cores=25)),
          ("20x5", lambda s: synth.random_payload(20, 5, s, node_cores=100)),
          ("50x10", lambda s: synth.random_payload(50, 10, s, node_cores=200)),
          ("300x7", lambda s: synth.random_payload(300, 7, s, node_cores=None)),
          ("7x3-float", lambda s: float_payload(7, 3, 5 + s))]
IDS = [s[0] for s in SHAPES]


def random_start(a, seed):
    """a feasible placement that is not the greedy's: one pod per function on a random node with room, then random
    extra pods while memory lasts"""
    rng = np.random.default_rng(1000 + seed)
    F, N, m = a["F"], a["N"], a["m"]
    c = np.zeros((F, N), dtype=np.uint8)
    free = a["Mj"].astype(np.float64).copy()
    for f in rng.permutation(F):
        j = rng.choice(np.flatnonzero(m[f] <= free + ref.MEM_TOL))
        c[f, j] = 1; free[j] -= m[f]
    for _ in range(F * N // 3):
        f, j = int(rng.integers(F)), int(rng.integers(N))
        if not c[f, j] and m[f] <= free[j] + ref.MEM_TOL:
            c[f, j] = 1; free[j] -= m[f]
    return c


def starts(a, seed):
    return {"greedy": osite.solve(a)[0], "random": random_start(a, seed)}


def best_neighbour(a, c):
    """smallest objective change of any add, exchange or relocation, by direct evaluation"""
    d, w, m = a["d"], a["w"], a["m"]
    F, N = c.shape
    free = ref.free_memory(a["Mj"], m, c)
    best = np.inf
    add = np.zeros((F, N)); rem = np.full((F, N), np.inf); base = {}
    for f in range(F):
        pods = np.flatnonzero(c[f])
        D = d[:, pods]
        s = np.sort(D, axis=1)
        m1 = s[:, 0]; m2 = s[:, 1] if pods.size > 1 else np.full(N, np.inf)
        add[f] = (w[f][:, None] * (np.minimum(m1[:, None], d) - m1[:, None])).sum(axis=0)
        for q, j in enumerate(pods):
            base[f, j] = np.where(D[:, q] == m1, m2, m1)             # nearest delay without pod j
            if pods.size > 1:
                rem[f, j] = float((w[f] * (base[f, j] - m1)).sum())
        elig = np.flatnonzero((c[f] == 0) & (m[f] <= free + ref.MEM_TOL))
        best = min(best, add[f, elig].min(initial=np.inf))
        for j in pods:
            if elig.size:
                rel = (w[f][:, None] * (np.minimum(base[f, j][:, None], d[:, elig]) - m1[:, None])).sum(axis=0)
                best = min(best, rel.min())
    for j in range(N):
        for fo in np.flatnonzero(c[:, j]):
            ok = (c[:, j] == 0) & (m <= free[j] + m[fo] + ref.MEM_TOL)
            if ok.any() and np.isfinite(rem[fo, j]):
                best = min(best, rem[fo, j] + add[ok, j].min())
    return best


@pytest.mark.parametrize("name,make", SHAPES, ids=IDS)
def test_reference_rounds_keep_the_rows_and_move_by_the_accepted_deltas(name, make):
    a = arrays_of(make(0))
    for start, c0 in starts(a, 0).items():
        run = ref.exchange_search(a, c0)
        # the search keeps no state beyond the placement: one round at a time retraces the same run
        c = c0
        for r in range(run["info"][0]):
            step = ref.exchange_search(a, c, max_rounds=1)
            c = step["c"]
            assert step["info"][0] == 1
            assert (c.sum(axis=1) >= 1).all(), (name, start, r)
            assert ((a["m"][:, None] * c).sum(axis=0) <= a["Mj"] + 1e-9).all(), (name, start, r)
            before, after = run["objs"][r], run["objs"][r + 1]
            assert step["objs"] == [before, after]
            assert abs(after - (before + run["deltas"][r])) <= 1e-9 * abs(before), (name, start, r)
            assert after < before
        assert np.array_equal(c, run["c"])
        assert run["objs"][-1] == ref.objective(a["w"], ref.nearest_two(a["d"], run["c"])[1])
        assert sum(run["info"][1:]) >= run["info"][0]
        # a local optimum of the three moves
        obj = run["objs"][-1]
        assert best_neighbour(a, run["c"]) >= -2e-12 * (1.0 + obj), (name, start)
        again = ref.exchange_search(a, c0)
        assert np.array_equal(again["c"], run["c"]) and again["info"] == run["info"] and again["objs"] == run["objs"]


def test_reference_improves_random_starts_with_every_move_kind():
    """several memory sizes and free memory: adds, exchanges and relocations all occur somewhere"""
    tot = np.zeros(3, dtype=int)
    for s in range(4):
        a = arrays_of(float_payload(7, 3, 5 + s))
        tot += ref.exchange_search(a, random_start(a, s))["info"][1:]
        a = arrays_of(synth.random_payload(20, 5, s, node_cores=100))
        tot += ref.exchange_search(a, random_start(a, s))["info"][1:]
    assert (tot > 0).all(), tot


def test_local_search_size_rule():
    """the add/drop/swap search keeps a row of N doubles per warp (24 warps above N = 128) in 200 KiB of shared
    memory: N = 1066 fits, N = 1067 does not; the min-delay solve path takes the pod-exchange search beyond"""
    from neptune_mip_b200 import device
    for F in (1, 200):
        assert device.local_search_fits(1066, F) and not device.local_search_fits(1067, F)
        assert device.local_search_fits(128, F) and device.local_search_fits(129, F)
        assert not device.local_search_fits(2000, F)


@pytest.mark.gpu
@pytest.mark.parametrize("name,make", SHAPES, ids=IDS)
def test_device_equals_the_reference(name, make):
    import torch
    from neptune_mip_b200 import device
    payloads = [make(s) for s in range(3)]
    inst = cuda_batch(payloads)
    arrays = [arrays_of(p) for p in payloads]
    for start in ("greedy", "random"):
        c0 = np.stack([starts(a, b)[start] for b, a in enumerate(arrays)])
        c_in = torch.from_numpy(c0).cuda().contiguous()
        c, info, obj = device.site_search(inst, c_in)
        assert torch.equal(c_in.cpu(), torch.from_numpy(c0))                # the start is kept
        for b, a in enumerate(arrays):
            want = ref.exchange_search(a, c0[b])
            assert np.array_equal(c[b].cpu().numpy(), want["c"]), (name, start, b)
            assert info[b].cpu().tolist() == want["info"], (name, start, b)
            assert obj[b].cpu().tolist() == [want["objs"][0], want["objs"][-1]], (name, start, b)
            alone = cuda_batch([payloads[b]])
            c1, info1, obj1 = device.site_search(alone, c_in[b:b + 1].contiguous())
            assert torch.equal(c1[0], c[b]) and torch.equal(info1[0], info[b]) and torch.equal(obj1[0], obj[b])


@pytest.mark.gpu
def test_device_refuses_a_function_without_a_pod():
    import torch
    from neptune_mip_b200 import device
    from neptune_mip_b200._lib import NeptuneError
    p = synth.random_payload(8, 4, 0, node_cores=30)
    c0 = osite.solve(arrays_of(p))[0]
    c0[2] = 0
    with pytest.raises(NeptuneError, match="invalid argument"):
        device.site_search(cuda_batch([p]), torch.from_numpy(c0[None]).cuda().contiguous())


@pytest.mark.gpu
def test_c2_site_path_against_highs_optima():
    """`solve_batch(search="site")` on the C2 seeds with proven optima: the model's checks pass, the routed objective is
    no worse than greedy + two-choice on every seed and never below the optimum"""
    from neptune_mip_b200 import device
    from neptune_mip_b200.batch import MIN_DELAY_FLAGS, BatchParams, solve_batch
    gold = {r["seed"]: r for r in json.load(open(os.path.join(os.path.dirname(__file__), "golden", "mip_optima.json")))
            if r["config"] == "C2" and r["optimal"]}
    seeds = sorted(gold)
    assert len(seeds) == 15
    inst = cuda_batch([synth.config_payload("C2", s) for s in seeds])
    res = solve_batch(inst, BatchParams(search="site", lp_iters=0))
    assert res.search_path == "site"
    fl = res.flags.cpu().numpy()
    assert np.all((fl & MIN_DELAY_FLAGS) == MIN_DELAY_FLAGS), fl
    got = res.scores[:, 0].cpu().numpy()
    cg, _ = device.site_greedy(inst)
    cg2, x, n, _, _, _ = device.route_two_choice(inst, cg)
    _, sg = device.check_solution(inst, x, device.u8_to_f64(cg2), n)
    greedy = sg[:, 0].cpu().numpy()
    opt = np.array([gold[s]["objective"] for s in seeds])
    assert np.all(got <= greedy * (1 + 1e-12)), (got - greedy)             # the checkers sum the score with atomics
    assert np.all(got >= opt - 1e-6 * opt), (got, opt)
    assert np.any(got < greedy)
    res2 = solve_batch(inst, BatchParams(search="site", lp_iters=0))
    assert np.array_equal(res2.c.cpu().numpy(), res.c.cpu().numpy())


@pytest.mark.gpu
def test_c4_min_delay_class_returns():
    """BASELINE config 4 (2000 x 200) through the drop-in class: the min-delay model's checks pass, the score is no
    worse than greedy + two-choice, two solves agree, the LP bound lies below.  With the adapter's default budget (60
    nodes at cost 5) the budget flag is unset, as for the greedy; with the budget raised `solve()` returns True."""
    import torch
    from neptune_mip_b200 import device
    from neptune_mip_b200._lib import OK_BUDGET
    from neptune_mip_b200.batch import MIN_DELAY_FLAGS
    from neptune_mip_b200.core.solvers import NeptuneStep1CPUMinDelay
    from neptune_mip_b200.core.utils import data_to_solver_input
    payload = synth.config_payload("C4", 0)

    def solve(budget=None):
        data = data_to_solver_input(payload, 1, with_db=False)
        if budget is not None:
            data.node_budget = budget
        s = NeptuneStep1CPUMinDelay(lp_iters=256, verbose=False)
        s.load_data(data)
        ok = s.solve()
        return s, ok

    s1, ok1 = solve()
    assert s1.flags & MIN_DELAY_FLAGS == MIN_DELAY_FLAGS, bin(s1.flags)
    used = float((s1._n * np.asarray(s1.data.node_costs, dtype=float)).sum())
    assert bool(s1.flags & OK_BUDGET) == (used <= s1.data.node_budget + 1e-6)
    assert ok1 == (s1.flags == 63)
    inst = s1.inst
    cg, _ = device.site_greedy(inst)
    cg2, x, n, _, _, _ = device.route_two_choice(inst, cg)
    _, sg = device.check_solution(inst, x, device.u8_to_f64(cg2), n)
    del x
    torch.cuda.empty_cache()
    assert s1.score() <= float(sg[0, 0].cpu()) * (1 + 1e-12)
    assert s1.lp_bound is not None and s1.lp_bound <= s1.score()
    c1 = s1._c
    del s1
    s2, _ = solve()
    assert np.array_equal(s2._c, c1)
    del s2
    s3, ok3 = solve(budget=1e9)
    assert ok3 and s3.flags == 63
    assert np.array_equal(s3._c, c1)
