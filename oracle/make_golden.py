"""TEST INFRASTRUCTURE ONLY -- regenerate tests/golden/*.json:   python -m oracle.make_golden [--only NAME] [--jobs J]
The steps that run the unmodified reference need its tree (oracle/refshim, NEPTUNE_REFERENCE_ROOT).

Sources of truth written into the fixtures
  alibaba_case0.json   the reference's own shipped outputs testing/alibaba/alibaba_test/output_*_case0.json
                       (input payload, scores, allocations, routing for the Efttc solvers)
  c1_test_py.json      output-mip.json (reference's hand-kept expected output of test.py) + the response
                       of the unmodified reference code run here through oracle.refshim
  simulated.json       score tables published in testing/simulated/simulated_report_finale.pdf +
                       responses of the unmodified reference code (EFTTC: all 10 cases, MIP: cases 0-6)
  model_hashes.json    sha256 of indptr/indices/data/lo/hi/obj of the matrices the reference's own
                       builders emit (through the shim) for C1, C2, 20x5 and the Alibaba case
  random_small.json    unmodified reference on random-workload instances: EFTTC placements (with the
                       documented discard fallback where it raises KeyError) and Neptune* scores
  payload_json.json    the reference's payload.json sample (no matrices: every default) through six solvers
  mip_optima.json      step-1 optima by HiGHS on the oracle model (C2 seeds, C5 subsample), with the placements
  lp_cut.json          HiGHS optima of the slot-cut LP relaxation (oracle.relax) the matrix-free PDHG solves
  reference_vectors.json  input-adapter arrays, response shaping, step-1 matrix digests and EFTTC results on the small
                       payloads of tests/helpers.py (see make_reference_vectors)
"""
from __future__ import annotations

import argparse
import ast
import contextlib
import hashlib
import io
import json
import os
import sys
import time
from concurrent.futures import ProcessPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
GOLD = os.path.join(ROOT, "tests", "golden")
REF = "/root/reference"


def _dump(name, obj, indent=1):
    os.makedirs(GOLD, exist_ok=True)
    with open(os.path.join(GOLD, name), "w") as fh:
        json.dump(obj, fh, indent=indent, sort_keys=True)
    print("wrote", name)


def _clean(resp):
    return {k: v for k, v in resp.items() if not k.startswith("_")}


def _np_to_py(o):
    if isinstance(o, dict):
        return {k: _np_to_py(v) for k, v in o.items()}
    if isinstance(o, (list, tuple)):
        return [_np_to_py(v) for v in o]
    if isinstance(o, np.generic):
        return o.item()
    return o


def make_alibaba():
    d = os.path.join(REF, "testing", "alibaba", "alibaba_test")
    out = {"outputs": {}}
    for s in ["EfttcMinDelay", "EfttcMinUtilization", "EfttcMinDelayAndUtilization",
              "NeptuneMinDelay", "NeptuneMinUtilization", "NeptuneMinDelayAndUtilization"]:
        g = json.load(open(os.path.join(d, f"output_{s}_case0.json")))
        inp = dict(g["input"]); solver = inp.pop("solver")
        if "input" not in out:
            out["input"] = inp
        assert out["input"] == inp
        rec = {"score": g["score"], "cpu_allocations": g["cpu_allocations"],
               "processing_time": g["processing_time"], "alpha": solver["args"].get("alpha", 0.5)}
        if s.startswith("Efttc"):
            rec["cpu_routing_rules"] = g["cpu_routing_rules"]
        out["outputs"][s] = rec
    _dump("alibaba_case0.json", out)


def make_c1():
    from neptune_mip_b200 import synth
    from oracle.refshim import load_reference as L
    expected = ast.literal_eval(open(os.path.join(REF, "output-mip.json")).read())
    resp = _clean(L.serve(synth.test_py_payload()))
    resp.pop("processing_time")
    assert resp["score"] == expected["score"] and resp["cpu_allocations"] == expected["cpu_allocations"]
    assert resp["cpu_routing_rules"] == expected["cpu_routing_rules"]
    out = {"expected_output_mip_json": expected, "reference_response": resp, "per_solver": {}}
    for s in ["EfttcMinDelay", "EfttcMinUtilization", "EfttcMinDelayAndUtilization",
              "NeptuneMinDelay", "NeptuneMinUtilization", "NeptuneMinDelayAndUtilization",
              "NeptuneWithEFTTCMinDelay", "NeptuneWithEFTTCMinUtilization", "NeptuneWithEFTTCMinDelayAndUtilization"]:
        for alpha in (1, 0.5):
            r = _clean(L.serve(synth.test_py_payload(s, {"alpha": alpha, "verbose": False, "soften_step1_sol": 1.3})))
            r.pop("processing_time")
            out["per_solver"][f"{s}|{alpha}"] = _np_to_py(r)
    _dump("c1_test_py.json", out)


def make_payload_json():
    """payload.json of the reference (comments stripped, with_db false): no matrices -> all defaults."""
    from neptune_mip_b200 import synth
    from oracle.refshim import load_reference as L
    out = {}
    for s in ["NeptuneMinDelayAndUtilization", "NeptuneMinDelay", "NeptuneMinUtilization",
              "EfttcMinDelay", "EfttcMinUtilization", "EfttcMinDelayAndUtilization"]:
        p = synth.payload_json_sample()
        p["solver"] = {"type": s, "args": {"alpha": 1.0, "verbose": False}}
        r = _clean(L.serve(p))
        r.pop("processing_time")
        out[s] = _np_to_py(r)
    _dump("payload_json.json", out)


PDF_SCORES = {   # testing/simulated/simulated_report_finale.pdf "Score Table" (SURVEY.md section 6)
    "MinUtil": [1, 1, 1, 1, 1, 2, 1, 5, 2, 5],
    "MinDelay": [0.0] * 10,
}


def _serve_case(args):
    k, solver, alpha = args
    sys.path.insert(0, ROOT)
    from neptune_mip_b200 import synth
    from oracle.refshim import load_reference as L
    t0 = time.time()
    r = _clean(L.serve(synth.simulated_case(k, solver, alpha)))
    return k, solver, {"score": _np_to_py(r["score"]), "cpu_allocations": r["cpu_allocations"],
                       "seconds": time.time() - t0}


def make_simulated(jobs):
    tasks = []
    for k in range(10):
        for s in ["EfttcMinDelay", "EfttcMinUtilization", "EfttcMinDelayAndUtilization"]:
            tasks.append((k, s, 0.0))
        if k <= 6:
            for s in ["NeptuneMinDelay", "NeptuneMinUtilization", "NeptuneMinDelayAndUtilization"]:
                tasks.append((k, s, 0.0))
    out = {"pdf_scores": PDF_SCORES, "reference_run": {}}
    with ProcessPoolExecutor(jobs) as ex:
        for k, s, rec in ex.map(_serve_case, tasks):
            out["reference_run"][f"{s}|case{k}"] = rec
            print(k, s, rec["score"], f"{rec['seconds']:.1f}s", flush=True)
    for k in range(10):
        assert out["reference_run"][f"EfttcMinUtilization|case{k}"]["score"]["step1"] == PDF_SCORES["MinUtil"][k]
    _dump("simulated.json", out)


def _hash(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def model_digest(A, lo, hi, obj, lb, ub, integ):
    return {"shape": list(A.shape), "nnz": int(A.nnz),
            "pattern": _hash(A.indptr.astype(np.int64), A.indices.astype(np.int64)),
            "data": _hash(A.data.astype(np.float64) + 0.0),
            "rows": _hash(lo.astype(np.float64) + 0.0, hi.astype(np.float64) + 0.0),   # + 0.0: -0.0 == 0.0
            "cols": _hash(obj.astype(np.float64) + 0.0, lb.astype(np.float64) + 0.0, ub.astype(np.float64) + 0.0,
                          integ.astype(np.uint8))}


def make_model_hashes():
    from neptune_mip_b200 import synth
    from oracle.refshim import load_reference as L
    core = L.load_reference()
    solvers = sys.modules["core.solvers"]
    ali = json.load(open(os.path.join(GOLD, "alibaba_case0.json")))["input"]
    cases = {"C1": (synth.test_py_payload(), 1), "C2": (synth.config_payload("C2"), 0.5),
             "C5s0": (synth.config_payload("C5", 0), 0.5), "r8x4s1": (synth.random_payload(8, 4, 1, node_cores=30), 0.5),
             "alibaba": (ali, 0.5)}
    cls = {"min_delay": "NeptuneStep1CPUMinDelay", "min_util": "NeptuneStep1CPUMinUtilization",
           "min_delay_util": "NeptuneStep1CPUMinDelayAndUtilization"}
    out = {}
    for name, (pl, alpha) in cases.items():
        for kind, cn in cls.items():
            with contextlib.redirect_stdout(io.StringIO()):
                data = core.data_to_solver_input(pl, with_db=False, workload_coeff=1)
                kw = dict(verbose=False)
                if kind == "min_delay_util":
                    kw["alpha"] = alpha
                s = getattr(solvers, cn)(**kw)
                s.load_data(data); s.init_objective()
            out[f"{name}|{kind}"] = dict(alpha=alpha, **model_digest(*s.solver.export()))
            print(name, kind, out[f"{name}|{kind}"]["shape"], flush=True)
    _dump("model_hashes.json", out)


def _random_case(args):
    N, F, seed, cores = args
    sys.path.insert(0, ROOT)
    from neptune_mip_b200 import synth
    from oracle.refshim import load_reference as L
    core = L.load_reference()
    solvers = sys.modules["core.solvers"]
    rec = {"N": N, "F": F, "seed": seed, "node_cores": cores, "efttc": {}, "neptune": {}}
    pl = synth.random_payload(N, F, seed, node_cores=cores)
    cls = {"min_delay": "EfttcStep1CPUMinDelay", "min_util": "EfttcStep1CPUMinUtilization",
           "min_delay_util": "EfttcStep1CPUMinDelayAndUtilization"}
    for kind, cn in cls.items():
        raised = False
        for patched in (False, True):
            L.enable_efttc_discard_patch(patched)
            with contextlib.redirect_stdout(io.StringIO()):
                data = core.data_to_solver_input(pl, with_db=False, workload_coeff=1)
                kw = dict(verbose=False)
                if kind == "min_delay_util":
                    kw["alpha"] = 0.5
                s = getattr(solvers, cn)(**kw)
                s.load_data(data)
                try:
                    s.solve()
                except KeyError:
                    raised = True
                    continue
                x, c = s.results()
                rec["efttc"][kind] = {"c": c.astype(int).tolist(), "score": float(s.score()),
                                      "reference_raised_keyerror": raised}
                break
        L.enable_efttc_discard_patch(False)
    for solver in ["NeptuneMinDelay", "NeptuneMinUtilization", "NeptuneMinDelayAndUtilization"]:
        if N * F > 60 and solver != "NeptuneMinDelay":
            continue
        pl2 = dict(pl); pl2["solver"] = {"type": solver, "args": {"alpha": 0.5, "verbose": False}}
        t0 = time.time()
        r = L.serve(pl2)
        rec["neptune"][solver] = {"score": _np_to_py(r["score"]), "solved": r["_solved"],
                                  "pods": sum(len(v) for v in r["cpu_allocations"].values()),
                                  "seconds": time.time() - t0}
    return rec


def make_random_small(jobs):
    tasks = [(8, 4, s, 30) for s in range(4)] + [(12, 5, s, 25) for s in range(3)] + [(20, 5, s, 100) for s in range(4)]
    out = []
    with ProcessPoolExecutor(jobs) as ex:
        for rec in ex.map(_random_case, tasks):
            out.append(rec)
            print(rec["N"], rec["F"], rec["seed"], {k: v["score"] for k, v in rec["neptune"].items()}, flush=True)
    _dump("random_small.json", out)


def _mip_case(args):
    name, seed, kind, tl = args
    sys.path.insert(0, ROOT)
    from neptune_mip_b200 import synth
    from neptune_mip_b200.core.utils import data_to_solver_input
    from oracle import mip, model
    pl = synth.config_payload(name, seed)
    a = model.arrays_from_data(data_to_solver_input(pl, 1, with_db=False))
    o = mip.solve_step1(a, kind, 0.5, time_limit=tl)
    return {"config": name, "seed": seed, "kind": kind, "objective": o["objective"], "optimal": bool(o["optimal"]),
            "seconds": o["seconds"], "dual_bound": o["dual_bound"], "gap": o["gap"],
            "pods": int((o["c"] > 0.5).sum()) if o["sol"] is not None else None, "time_limit": tl,
            # the incumbent placement as [f, j] pairs: lets a test price a known-optimal placement with the device routing
            "placement": [[int(f), int(j)] for f, j in zip(*np.nonzero(o["c"] > 0.5))] if o["sol"] is not None else None}


def make_mip_optima(jobs, c2_seeds=16, c5_seeds=64):
    path = os.path.join(GOLD, "mip_optima.json")
    have = {}
    if os.path.exists(path):
        for r in json.load(open(path)):
            have[(r["config"], r["seed"], r["kind"])] = r
    tasks = [("C5", s, "min_delay", 120) for s in range(c5_seeds)] + [("C2", s, "min_delay", 900) for s in range(c2_seeds)]
    tasks = [t for t in tasks if (t[0], t[1], t[2]) not in have]
    with ProcessPoolExecutor(jobs) as ex:
        for rec in ex.map(_mip_case, tasks):
            have[(rec["config"], rec["seed"], rec["kind"])] = rec
            print(rec, flush=True)
            _dump("mip_optima.json", sorted(have.values(), key=lambda r: (r["config"], r["kind"], r["seed"])))


def make_reference_vectors():
    """What tests/test_oracle_vs_reference.py and the edge-case test of tests/test_host_logic.py hold the project to, on
    the payloads of tests/helpers.py: the input adapter's arrays, the response shaping of a seeded random solution,
    digests of the step-1 matrices and the EFTTC results (strict, and with the `discard` fallback).  Those tests used to
    import the unmodified reference and require equality with it; these values are computed by the project's
    restatements (core.utils adapter, core.solvers.output, oracle.model, oracle.efttc) as they stood when those tests
    held them equal to the reference, so that the comparison no longer needs the reference tree."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from helpers import DATA_FIELDS, arrays_of, data_of, edge_payloads, shaping_solution, small_payloads
    from neptune_mip_b200.core.solvers.output import convert_c_matrix, convert_x_matrix
    from oracle import efttc, model
    out = {"data": {}, "shaping": {}, "model": {}, "efttc": {}}
    edges = edge_payloads()
    for name, p in [(n, p) for n, p, _ in small_payloads()] + list(edges.items()):
        d = data_of(p)
        out["data"][name] = dict({k: np.asarray(getattr(d, k)).tolist() for k in DATA_FIELDS},
                                 nodes=d.nodes, functions=d.functions, node_budget=_np_to_py(d.node_budget))
        if name in edges:
            x, c = shaping_solution(len(d.nodes), len(d.functions))
            out["shaping"][name] = {"x": convert_x_matrix(x, d.nodes, d.functions), "c": convert_c_matrix(c, d.functions, d.nodes)}
    for name, p, alpha in small_payloads():
        a = arrays_of(p)
        for kind in ("min_delay", "min_util", "min_delay_util"):
            m = model.build_step1(a, kind, alpha)
            out["model"][f"{name}|{kind}"] = model_digest(m["A"], m["lo"], m["hi"], m["obj"], m["lb"], m["ub"], m["integ"])
            for strict in (True, False):
                try:
                    res = efttc.solve(a, kind, alpha, strict=strict)
                except KeyError:
                    rec = {"keyerror": True}
                else:
                    nz = np.flatnonzero(res.x)
                    rec = {"keyerror": False, "c": res.c.astype(int).tolist(), "x_shape": list(res.x.shape),
                           "x_index": nz.tolist(), "x_value": res.x.ravel()[nz].tolist(),
                           "score": float(efttc.score(a, kind, alpha, res))}
                out["efttc"][f"{name}|{kind}|{'strict' if strict else 'discard'}"] = rec
    _dump("reference_vectors.json", out, indent=None)


def make_lp_cut():
    """HiGHS optima of the slot-cut relaxation (oracle.relax) for the C2 seeds and a C5 subsample: pins the
    bound the matrix-free PDHG reports."""
    from neptune_mip_b200 import synth
    from neptune_mip_b200.core.utils import data_to_solver_input
    from oracle import model, relax
    out = []
    for name, seeds in (("C2", range(16)), ("C5", range(8))):
        for s in seeds:
            a = model.arrays_from_data(data_to_solver_input(synth.config_payload(name, s), 1, with_db=False))
            v1, _, lam = relax.strengthened_lp(a, slot_cut=True)
            v0, _, _ = relax.strengthened_lp(a, slot_cut=False)
            out.append({"config": name, "seed": s, "lp_slot_cut": v1, "lp_memory_rows": v0,
                        "cpu_duals": [float(x) for x in lam]})
            print(name, s, v1, v0, flush=True)
    _dump("lp_cut.json", out)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default=None)
    ap.add_argument("--jobs", type=int, default=4)
    a = ap.parse_args()
    steps = {"alibaba": make_alibaba, "c1": make_c1, "payload_json": make_payload_json, "simulated": lambda: make_simulated(a.jobs),
             "model_hashes": make_model_hashes, "random_small": lambda: make_random_small(a.jobs),
             "mip_optima": lambda: make_mip_optima(a.jobs), "lp_cut": make_lp_cut, "reference_vectors": make_reference_vectors}
    for name, fn in steps.items():
        if a.only in (None, name):
            fn()
