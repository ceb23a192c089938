"""BASELINE.json's full sizes, checked through size-independent properties (the oracle is only run on
subsamples / closed forms there): C5 = 4096 x (20x5) in one launch, C3 = 500x50."""
import numpy as np
import pytest

from helpers import arrays_of, cuda_batch, data_of
from neptune_mip_b200 import synth
from oracle import efttc as oefttc

pytestmark = pytest.mark.gpu


def test_c5_sweep_4096_instances_one_launch():
    import torch
    from neptune_mip_b200 import device
    from neptune_mip_b200._lib import OK_ALL, OK_CPU, OK_MEMORY, OK_N_C, OK_BUDGET
    B = 4096
    payloads = [synth.config_payload("C5", s) for s in range(B)]
    inst = cuda_batch(payloads)
    for kind in ("min_delay", "min_util"):
        c, n, info = device.efttc(inst, kind)
        x, nn = device.route_placements(inst, c)
        flags, scores = device.check_solution(inst, x, device.u8_to_f64(c), nn)
        c_h, flags_h, info_h = c.cpu().numpy(), flags.cpu().numpy(), info.cpu().numpy()
        # properties that hold for every EFTTC output, whatever the instance: memory, CPU, n<->c, budget
        must = OK_MEMORY | OK_CPU | OK_N_C | OK_BUDGET
        assert np.all((flags_h & must) == must)
        assert np.all(c_h.reshape(B, 5, 20).sum(axis=1).max(axis=1) <= 3)          # 3 x 30 <= 100 memory units
        assert np.all(info_h[:, 1] == c_h.reshape(B, -1).sum(axis=1))
        if kind == "min_util":
            assert np.all(flags_h == OK_ALL)                                         # every function placed
        # idempotence: the same batch again gives the same placements (deterministic kernel)
        c2, _, _ = device.efttc(inst, kind)
        assert torch.equal(c, c2)
        # oracle on a subsample
        for b in np.random.default_rng(0).choice(B, 24, replace=False):
            ref = oefttc.solve(arrays_of(payloads[b]), kind, 0.5, strict=False)
            assert np.array_equal(c_h[b], ref.c.astype(np.uint8)), (kind, b)


def test_c3_assembly_closed_form_properties_and_exact_transpose():
    """500 x 50: 50 075 000 non-zeros.  Row/column counts and checksums against closed forms, spot rows
    against the oracle's formulae, the stored transpose equal to A^T entry for entry."""
    import torch
    from neptune_mip_b200 import device
    p = synth.config_payload("C3")
    a = arrays_of(p)
    N, F = a["N"], a["F"]
    inst = cuda_batch([p])
    mdl = device.assemble(inst, "min_delay")
    assert (mdl.rows, mdl.cols, mdl.nnz) == (76000, 12525000, 50075000)
    rp = mdl.row_ptr
    lens = (rp[1:] - rp[:-1]).cpu().numpy()
    assert np.all(lens[:2 * F * N] == N + 1) and np.all(lens[2 * F * N:2 * F * N + N] == F)
    assert np.all(lens[2 * F * N + N:3 * F * N + N] == N) and np.all(lens[3 * F * N + N:] == F * N)
    X = F * N * N
    # checksum of checksums: every x column appears exactly 4 times, every c column 3 times
    counts = torch.bincount(mdl.col_idx.long(), minlength=mdl.cols)
    assert bool((counts[:X] == 4).all()) and bool((counts[X:] == 3).all())
    val = mdl.val[0]
    # C4 block: sum of coefficients == sum_j sum_{f,i} w[f,i] r[f,j]
    c4 = val[int(rp[3 * F * N + N]):]
    want = float((a["w"].sum(axis=1)[:, None] * a["r"]).sum())
    assert abs(float(c4.sum()) - want) <= 1e-9 * abs(want)
    # spot rows of every family against the closed form
    rng = np.random.default_rng(1)
    cols_h = lambda r0: mdl.col_idx[int(rp[r0]):int(rp[r0 + 1])].cpu().numpy()      # noqa: E731
    vals_h = lambda r0: val[int(rp[r0]):int(rp[r0 + 1])].cpu().numpy()               # noqa: E731
    for _ in range(20):
        f, j, i = int(rng.integers(F)), int(rng.integers(N)), int(rng.integers(N))
        r0 = 2 * (f * N + j)
        assert np.array_equal(cols_h(r0), np.concatenate([f * N * N + np.arange(N) * N + j, [X + f * N + j]]))
        assert np.array_equal(vals_h(r0), np.concatenate([np.ones(N), [-1e6]])) and vals_h(r0 + 1)[-1] == -1.0
        r3 = 2 * F * N + N + f * N + i
        assert np.array_equal(cols_h(r3), f * N * N + i * N + np.arange(N))
        r4 = 3 * F * N + N + j
        assert np.array_equal(vals_h(r4), (a["w"] * a["r"][:, j][:, None]).reshape(-1))
    # the stored transpose is A^T exactly: A's entries taken column by column, rows ascending within a column
    rows = torch.repeat_interleave(torch.arange(mdl.rows, dtype=torch.int32, device="cuda"), rp[1:] - rp[:-1])
    order = torch.argsort(mdl.col_idx, stable=True)
    assert torch.equal(mdl.colT_idx, rows[order])
    assert torch.equal(mdl.valT[0], val[order])
    assert torch.equal(mdl.rowT_ptr, torch.cat([counts.new_zeros(1), torch.cumsum(counts, 0)]))
    # objective vector: d[i,j] * w[f,i]
    obj = mdl.obj[0, :X].reshape(F, N, N).cpu().numpy()
    assert np.array_equal(obj, a["d"][None, :, :] * a["w"][:, :, None])


def test_c3_routing_and_checkers_at_full_size():
    """One pod of every function on every node it fits round-robin: nearest routing must satisfy
    handle_all / c<->x / n<->c, and routing the same placement twice is idempotent."""
    import torch
    from neptune_mip_b200 import device
    p = synth.config_payload("C3")
    N, F = 500, 50
    inst = cuda_batch([p])
    c = np.zeros((1, F, N), dtype=np.uint8)
    for j in range(N):
        for k in range(3):
            c[0, (3 * j + k) % F, j] = 1
    ct = torch.from_numpy(c).cuda()
    x, n = device.route_placements(inst, ct)
    flags, scores = device.check_solution(inst, x, device.u8_to_f64(ct), n)
    fl = int(flags.cpu()[0])
    from neptune_mip_b200._lib import OK_C_X, OK_HANDLE, OK_MEMORY, OK_N_C
    assert fl & OK_HANDLE and fl & OK_MEMORY and fl & OK_N_C and fl & OK_C_X
    assert float((x.sum(dim=3) - 1).abs().max()) <= 1e-12
    x2, _ = device.route_placements(inst, ct)
    assert torch.equal(x, x2)
    # delay score == sum_f sum_i w[f,i] * min over open pods d[i,j] (closed form, numpy)
    a = arrays_of(p)
    want = sum(float((a["w"][f] * a["d"][:, c[0, f] > 0].min(axis=1)).sum()) for f in range(F))
    assert abs(float(scores.cpu()[0, 0]) - want) <= 1e-9 * want


def test_c5_neptune_quality_against_highs_optima():
    """The add/drop/swap search + heuristic capacity-aware routing (the path of the model kinds and memory layouts the
    slot-count search does not take; tests/test_lns_gpu.py covers the default path: 64 of 64) on the first 64 instances
    of the C5 sweep vs the proven HiGHS optima: every answer passes the six checkers, none is below the optimum, at
    least 55 of 64 are within 1e-4 relative of it and none is more than 5 % above.  Two runs are bit-identical."""
    import json
    import os

    import torch
    from neptune_mip_b200 import device
    gold = {r["seed"]: r for r in json.load(open(os.path.join(os.path.dirname(__file__), "golden", "mip_optima.json")))
            if r["config"] == "C5" and r["optimal"]}
    seeds = sorted(s for s in gold if s < 64)
    payloads = [synth.config_payload("C5", s) for s in seeds]
    inst = cuda_batch(payloads)
    sd = torch.stack([device.efttc(inst, k)[0] for k in ("min_delay", "min_util", "min_delay_util")], dim=1).contiguous()
    bc, bo, _ = device.local_search(inst, "min_delay", sd, chains=32, sweeps=300)
    bc2, bo2, _ = device.local_search(inst, "min_delay", sd, chains=32, sweeps=300)
    assert torch.equal(bc, bc2) and torch.equal(bo, bo2)          # fixed-point load deltas, ordered pod compaction
    c2, x, n, obj, feas = device.route_capacitated(inst, bc)
    flags, scores = device.check_solution(inst, x, device.u8_to_f64(c2), n)
    flags, got = flags.cpu().numpy(), scores[:, 0].cpu().numpy()
    ref = np.array([gold[s]["objective"] for s in seeds])
    assert np.all(flags == 63)
    rel = (got - ref) / np.abs(ref)
    assert np.all(rel >= -1e-6), rel.min()
    assert (rel <= 1e-4).sum() >= 55, (rel <= 1e-4).sum()
    assert rel.max() <= 0.05
