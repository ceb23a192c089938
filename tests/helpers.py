"""Shared test helpers: payload -> Data -> oracle arrays / device batch."""
import functools
import json
import os

import numpy as np

from neptune_mip_b200 import synth
from neptune_mip_b200.core.utils import data_to_solver_input
from oracle import model as omodel

KIND_NAMES = ("min_delay", "min_util", "min_delay_util")


def data_of(payload):
    return data_to_solver_input(payload, payload.get("workload_coeff", 1), with_db=False)


def arrays_of(payload):
    return omodel.arrays_from_data(data_of(payload))


def small_payloads():
    """(name, payload, alpha) triples covering the shapes the reference tests (and ragged ones)."""
    out = [("C1", synth.test_py_payload(), 1.0)]
    for k in (0, 1, 2, 3, 4, 5, 6):
        out.append((f"sim{k}", synth.simulated_case(k), 0.0))
    for s in range(3):
        out.append((f"r8x4s{s}", synth.random_payload(8, 4, s, node_cores=30), 0.5))
        out.append((f"r12x5s{s}", synth.random_payload(12, 5, s, node_cores=25), 0.3))
    out.append(("r7x3float", float_payload(7, 3, 5), 0.4))
    return out


DATA_FIELDS = ["node_memory_matrix", "function_memory_matrix", "node_delay_matrix", "workload_matrix", "max_delay_matrix",
               "node_cores_matrix", "cores_matrix", "old_allocations_matrix", "core_per_req_matrix", "node_costs"]


def edge_payloads():
    """Input-adapter edge cases: defaults only, a workload coefficient, empty / false allocations, x/0 and 0/0, 1x1."""
    out = {"payload_json": synth.payload_json_sample()}
    p = synth.test_py_payload(); p["workload_coeff"] = 2.5; out["workload_coeff"] = p
    p = synth.random_payload(6, 3, 0, node_cores=10); p["actual_cpu_allocations"] = {"ns/fn_0": {}, "ns/fn_2": {"node_3": False}}
    out["empty_and_false_allocations"] = p
    p = synth.random_payload(5, 2, 1, node_cores=10)
    p["workload_on_destination_matrix"] = [[0, 1, 0, 2, 0], [0, 0, 0, 0, 0]]      # x/0 -> DBL_MAX, 0/0 -> 0
    p["cores_matrix"] = [[0, 1, 3, 2, 0], [0, 0, 0, 0, 1]]
    out["division_by_zero"] = p
    p = synth.simulated_case(0); out["one_by_one"] = p
    return out


@functools.lru_cache(maxsize=None)
def reference_vectors():
    """What the unmodified reference computes on small_payloads() and edge_payloads() (oracle/make_golden.py)."""
    with open(os.path.join(os.path.dirname(__file__), "golden", "reference_vectors.json")) as fh:
        return json.load(fh)


def shaping_solution(N, F):
    """The random routing / placement the response-shaping comparisons convert (seeded)."""
    rng = np.random.default_rng(0)
    x = rng.random((N, F, N)) * (rng.random((N, F, N)) < 0.3)
    c = (rng.random((F, N)) < 0.4).astype(float)
    return x, c


def float_payload(N, F, seed):
    """Non-integer delays / workloads / memories: exercises rounding order."""
    rng = np.random.default_rng(seed)
    p = synth.random_payload(N, F, seed, node_cores=20)
    D = rng.uniform(0.5, 40.0, (N, N)); D = (D + D.T) / 2; np.fill_diagonal(D, 0.0)
    p["node_delay_matrix"] = D.tolist()
    p["workload_on_source_matrix"] = rng.uniform(0.0, 9.0, (F, N)).tolist()
    p["function_memories"] = rng.uniform(0.1, 0.49, F).round(2).tolist()
    p["node_memories"] = [1.0] * N
    return p


def cuda_batch(payloads):
    from neptune_mip_b200.device import InstanceBatch
    return InstanceBatch.from_datas([data_of(p) for p in payloads])
