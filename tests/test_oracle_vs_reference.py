"""Input adapter and oracle vs what the UNMODIFIED reference computes on the payloads of helpers.py: its Data arrays, the
digests of the step-1 matrices its builders emit, its EFTTC x, c, score and KeyError behaviour.  The reference's values are
stored in golden/reference_vectors.json (oracle/make_golden.py: make_reference_vectors)."""
import numpy as np
import pytest

from helpers import DATA_FIELDS, arrays_of, data_of, reference_vectors, small_payloads
from oracle import efttc as oefttc, model as omodel
from oracle.make_golden import model_digest

KINDS = ["min_delay", "min_util", "min_delay_util"]


@pytest.mark.parametrize("name,payload,alpha", small_payloads(), ids=lambda v: v if isinstance(v, str) else None)
def test_input_adapter_equals_reference(name, payload, alpha):
    want, md = reference_vectors()["data"][name], data_of(payload)
    for k in DATA_FIELDS:
        assert np.array_equal(np.asarray(want[k]), np.asarray(getattr(md, k))), k
    assert want["node_budget"] == md.node_budget and want["nodes"] == md.nodes and want["functions"] == md.functions


@pytest.mark.parametrize("name,payload,alpha", small_payloads(), ids=lambda v: v if isinstance(v, str) else None)
@pytest.mark.parametrize("kind", KINDS)
def test_model_equals_reference_built_matrix(name, payload, alpha, kind):
    want = reference_vectors()["model"][f"{name}|{kind}"]
    m = omodel.build_step1(arrays_of(payload), kind, alpha)
    got = model_digest(m["A"], m["lo"], m["hi"], m["obj"], m["lb"], m["ub"], m["integ"])
    for k in ("shape", "nnz", "pattern", "data", "rows", "cols"):
        assert got[k] == want[k], k


@pytest.mark.parametrize("name,payload,alpha", small_payloads(), ids=lambda v: v if isinstance(v, str) else None)
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("strict", [True, False])
def test_efttc_equals_reference(name, payload, alpha, kind, strict):
    """strict: the reference as shipped; otherwise with `remaining_functions.remove` behaving like `discard`"""
    want = reference_vectors()["efttc"][f"{name}|{kind}|{'strict' if strict else 'discard'}"]
    a = arrays_of(payload)
    if want["keyerror"]:
        with pytest.raises(KeyError):
            oefttc.solve(a, kind, alpha, strict=strict)
        return
    res = oefttc.solve(a, kind, alpha, strict=strict)
    x = np.zeros(want["x_shape"])
    x.ravel()[want["x_index"]] = want["x_value"]
    assert np.array_equal(np.array(want["c"]), res.c) and np.array_equal(x, res.x)
    got = oefttc.score(a, kind, alpha, res)
    assert got == want["score"] or np.isclose(got, want["score"], rtol=1e-15, atol=0)
