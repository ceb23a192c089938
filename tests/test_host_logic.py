"""Host-side logic on CPU: the input adapter's defaults and edge cases, response shaping, error behaviour."""
import json

import numpy as np
import pytest

from helpers import DATA_FIELDS, data_of, edge_payloads, reference_vectors, shaping_solution
from neptune_mip_b200 import synth
from neptune_mip_b200.core import check_input, data_to_solver_input
from neptune_mip_b200.core.solvers.output import convert_c_matrix, convert_x_matrix


def test_defaults_without_reference():
    d = data_to_solver_input(synth.payload_json_sample(), 1, with_db=False)
    N, F = 5, 4
    assert np.array_equal(d.node_delay_matrix, 1 - np.eye(N, dtype=int))            # input_to_data.py:156
    assert d.workload_matrix.shape == (F, N) and not d.workload_matrix.any()         # :164
    assert np.array_equal(d.max_delay_matrix, [1000] * F)                            # :136, function_max_delays ignored
    assert np.array_equal(d.node_costs, [5] * N) and d.node_budget == 300            # :185-187
    assert d.old_allocations_matrix.sum() == 5 and d.old_allocations_matrix[1, 1] == 1
    assert not np.asarray(d.core_per_req_matrix).any()                               # 0/0 -> 0
    empty = synth.simulated_case(2)                                                  # nothing allocated -> all ones (:275-276)
    assert data_to_solver_input(empty, 1, with_db=False).old_allocations_matrix.all()
    with pytest.raises(RuntimeError):
        data_to_solver_input(synth.payload_json_sample(), 1, with_db=True)           # Postgres pull: out of scope, loud


def test_check_input_asserts_like_the_reference():
    p = synth.test_py_payload()
    check_input(p)
    for key in ("community", "node_cores", "function_max_delays", "actual_gpu_allocations"):
        q = dict(p); q.pop(key)
        with pytest.raises(AssertionError, match=key):
            check_input(q)
    q = dict(p); q["function_memories"] = [5]
    with pytest.raises(AssertionError):
        check_input(q)
    q = dict(p); q["gpu_node_names"] = ["nowhere"]; q["gpu_node_memories"] = [1]
    with pytest.raises(AssertionError):
        check_input(q)


def test_response_shaping():
    nodes, funcs = ["a", "b"], ["ns/f", "ns/g"]
    x = np.zeros((2, 2, 2)); x[0, 0, 1] = 1.0; x[1, 1, 0] = 0.33349; x[1, 1, 1] = 0.0009; x[0, 1, 0] = 0.6665
    c = np.array([[0.0, 1.0], [1.0, 0.0005]])
    rx, rc = convert_x_matrix(x, nodes, funcs), convert_c_matrix(c, funcs, nodes)
    assert rx == {"a": {"ns/f": {"b": 1.0}, "ns/g": {"a": 0.666}}, "b": {"ns/g": {"a": 0.333}}}      # > 0.001, 3 decimals
    assert rc == {"ns/f": {"b": True}, "ns/g": {"a": True}}
    assert json.loads(json.dumps(rx)) == rx
    with pytest.raises(AssertionError):
        convert_x_matrix(x[:1], nodes, funcs)


@pytest.mark.parametrize("name", list(edge_payloads()))
def test_adapter_and_shaping_equal_the_reference_on_edge_cases(name):
    """the reference's Data arrays and its convert_* responses on a random solution (golden/reference_vectors.json)"""
    payload = edge_payloads()[name]
    rd, shaped = reference_vectors()["data"][name], reference_vectors()["shaping"][name]
    check_input(payload)
    md = data_of(payload)
    for k in DATA_FIELDS:
        assert np.array_equal(np.asarray(rd[k]), np.asarray(getattr(md, k))), k
    assert rd["nodes"] == md.nodes and rd["functions"] == md.functions and rd["node_budget"] == md.node_budget
    x, c = shaping_solution(len(md.nodes), len(md.functions))
    assert convert_x_matrix(x, md.nodes, md.functions) == shaped["x"]
    assert convert_c_matrix(c, md.functions, md.nodes) == shaped["c"]
