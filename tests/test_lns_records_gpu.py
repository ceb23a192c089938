"""(c2) Records of the slot-count search (`neptune_lns_search`, csrc/lns.cu) pinned bit for bit: every chain's two
records (placement, both bounds, round) on fixed inputs equal tests/golden/lns_records.json.  The kernel's launch
shape and shared-memory layout may change; what a chain computes may not.  The search is called directly, without
an LP guide, so that the golden does not depend on the relaxation.

The cases cover both template widths of the kernel (8 and 12 chains per block) at k = 3 and k = 4, annealed and cold
rounds (the last eighth of a chain's rounds is cold), starts from randomised roundings and from seed placements, an
instance with N <= 32 (more dual-ascent passes) and one whose slot counts do not fit k nodes (trailing nodes dropped).

Regenerate (on a GPU, only when a change is meant to alter the search):  python tests/test_lns_records_gpu.py --write"""
import hashlib
import json
import os
import sys

import pytest

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden", "lns_records.json")

# name -> (instances, k, chains, rounds, block mode, rng seed, seeds from the records of this case or None)
CASES = {
    "c2_k3": ("c2", 3, 24, 600, 0, 11, None),
    "c2_k4": ("c2", 4, 24, 600, 0, 12, None),
    "c2_k3_wide": ("c2", 3, 24, 600, 2, 11, None),
    "c2_k4_wide": ("c2", 4, 24, 600, 2, 12, None),
    "c2_k4_from_records": ("c2", 4, 48, 300, 0, 13, "c2_k3"),
    "c5_k3": ("c5", 3, 24, 600, 0, 14, None),
    "c5_k4": ("c5", 4, 24, 600, 0, 15, None),
    "sim6_k3": ("sim6", 3, 16, 400, 0, 16, None),
    "sim6_k4": ("sim6", 4, 16, 400, 0, 17, None),
}


def _instances(name):
    from helpers import cuda_batch
    from neptune_mip_b200 import synth
    if name == "c2":
        return cuda_batch([synth.config_payload("C2", s) for s in (0, 6)])
    if name == "c5":
        return cuda_batch([synth.config_payload("C5", s) for s in (0, 1, 2, 3)])
    return cuda_batch([synth.simulated_case(6)])        # 20 x 5, ten slots per node capped at F = 5: only two nodes fit


def _run_all():
    from neptune_mip_b200 import device
    insts, raw, out = {}, {}, {}
    for case, (iname, k, chains, rounds, mode, rng, seeds_from) in CASES.items():
        inst = insts.setdefault(iname, _instances(iname))
        seeds = raw[seeds_from][0].contiguous() if seeds_from else None
        device.lns_block_mode(mode)
        try:
            c, g, rnd = device.lns_search(inst, "min_delay", chains=chains, rounds=rounds, k=k, noise_coef=0.1,
                                          rng_seed=rng, seeds_u8=seeds)
            lb = device.lns_search.last_other_bound
        finally:
            device.lns_block_mode(0)
        raw[case] = (c, g, lb, rnd)
        out[case] = {"out_c_sha256": hashlib.sha256(c.cpu().numpy().tobytes()).hexdigest(),
                     "out_g": [float(v).hex() for v in g.cpu().flatten().tolist()],
                     "out_lb": [float(v).hex() for v in lb.cpu().flatten().tolist()],
                     "out_round": [int(v) for v in rnd.cpu().flatten().tolist()]}
    return out


def test_records_equal_the_golden_bit_for_bit():
    want = json.load(open(GOLD))
    got = _run_all()
    assert sorted(got) == sorted(want)
    for case in CASES:
        for key in ("out_round", "out_g", "out_lb", "out_c_sha256"):
            assert got[case][key] == want[case][key], (case, key)


if __name__ == "__main__":
    sys.path[:0] = [HERE, os.path.dirname(HERE)]
    if sys.argv[1:] == ["--write"]:
        json.dump(_run_all(), open(GOLD, "w"), indent=0)
        print("wrote", GOLD)
