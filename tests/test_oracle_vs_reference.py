"""The oracle restatement (oracle/paf_oracle.c) against the reference's OWN parser:
  * committed goldens: human_t lists that /root/reference/src/paf.cpp (compiled verbatim
    into oracle/_ref) produced on the seeded synthetic frames -- runs anywhere;
  * random / noise / sweep inputs: what oracle/_ref returned on them (committed as ref_live.npz), and the live oracle/_ref
    as well where it is built."""
import os

import numpy as np
import pytest

import oracle
from hyperpose_b200 import synthetic as syn
from tests.golden.make_golden import (AREA_FRAME_CASES, FRAME_CASES, RANDOM_SEEDS, SWEEP_SEEDS, noise_case, random_case, sha,
                                      sweep_case)


@pytest.fixture(scope="module")
def ref_humans(golden_dir):
    return np.load(os.path.join(golden_dir, "ref_humans.npz"))


@pytest.fixture(scope="module")
def live(golden_dir):
    return np.load(os.path.join(golden_dir, "ref_live.npz"))


@pytest.mark.parametrize("case", FRAME_CASES, ids=[c[0] for c in FRAME_CASES])
def test_oracle_matches_reference_golden(ref_humans, case):
    name, seed, P, hf, wf, rw, rh, ct, pt = case
    conf, paf = syn.make_frame_tensors(seed, P, hf, wf)
    assert sha(conf) + sha(paf) == str(ref_humans[name + "_in_sha"]), "synthetic generator drifted from the goldens"
    got = oracle.oracle_process(conf, paf, ct, pt, rw, rh)["humans"]
    want = ref_humans[name + "_humans"]
    assert len(got) == len(want)
    assert got.tobytes() == want.tobytes()      # byte-identical human_t records, same order


@pytest.mark.parametrize("case", AREA_FRAME_CASES, ids=[c[0] for c in AREA_FRAME_CASES])
def test_oracle_matches_reference_golden_on_shrinking_resolutions(golden_dir, case):
    """A5 beyond pure up-scaling: resolutions that shrink an axis (mixed 2-tap regime, integer and fractional area averaging).
    Goldens = the reference's own src/paf.cpp over the cv2-pinned resize (tests/golden/make_golden.py area)."""
    ref = np.load(os.path.join(golden_dir, "ref_humans_area.npz"))
    name, seed, P, hf, wf, rw, rh, ct, pt = case
    conf, paf = syn.make_frame_tensors(seed, P, hf, wf)
    assert sha(conf) + sha(paf) == str(ref[name + "_in_sha"]), "synthetic generator drifted from the goldens"
    o = oracle.oracle_process(conf, paf, ct, pt, rw, rh)
    assert o["humans"].tobytes() == ref[name + "_humans"].tobytes()
    if oracle.ref_available():
        rp = oracle.RefParser(ct, pt, rw, rh)
        assert rp.process(conf, paf).tobytes() == o["humans"].tobytes()
        rp.close()


def test_goldens_are_not_vacuous(ref_humans):
    assert len(ref_humans["cfg1_p1_humans"]) == 1
    assert len(ref_humans["cfg1_p3_humans"]) >= 2
    assert len(ref_humans["cfg4_crowd_humans"]) >= 10
    assert len(ref_humans["empty_humans"]) == 0
    h = ref_humans["cfg1_p1_humans"][0]
    assert int(h["parts"]["has_value"].sum()) == 18


def _vs_reference(live, key, conf, paf, ct=0.05, pt=0.05, rw=-1, rh=-1):
    """(oracle humans, reference humans): the reference's output stored in ref_live.npz, held equal to the live oracle/_ref
    where that is built"""
    assert sha(conf) + sha(paf) == str(live[key + "_in_sha"]), "synthetic generator drifted from the goldens"
    want = live[key + "_humans"]
    if oracle.ref_available():
        rp = oracle.RefParser(ct, pt, rw, rh)
        assert rp.process(conf, paf).tobytes() == want.tobytes()
        rp.close()
    return oracle.oracle_process(conf, paf, ct, pt, rw, rh), want


@pytest.mark.parametrize("seed", RANDOM_SEEDS)
def test_oracle_matches_live_reference_random(live, seed):
    o, want = _vs_reference(live, f"random{seed}", *random_case(seed))
    assert o["humans"].tobytes() == want.tobytes()


def test_oracle_matches_live_reference_noise_field(live):
    # structureless input (many spurious peaks, few/no humans): exercises the candidate filter
    o, want = _vs_reference(live, "noise", *noise_case())
    assert len(o["peaks"]) > 50
    assert o["humans"].tobytes() == want.tobytes()


def test_peak_ids_are_scan_ordered():
    conf, paf = syn.make_frame_tensors(3, (10, 20), 46, 54)
    pk = oracle.oracle_process(conf, paf)["peaks"]
    assert np.array_equal(pk["id"], np.arange(len(pk)))
    key = pk["part_id"].astype(np.int64) * (1 << 32) + pk["y"].astype(np.int64) * (1 << 16) + pk["x"]
    assert np.all(np.diff(key) > 0)


@pytest.mark.parametrize("seed", SWEEP_SEEDS)
def test_oracle_matches_live_reference_sweep(live, seed):
    """wider sweep of what pins the oracle: odd feature sizes, both thresholds, custom parser resolutions (non-integer
    up-scaling factors -> the 2-tap INTER_AREA path), empty frames and crowds, noise levels around the thresholds.
    Two regions are left out because the reference itself leaves them open, not because the restatement differs:
      * noise-free fields: their plateaus give limb candidates with EXACTLY equal scores, and paf.cpp:246 orders
        candidates with an unstable std::sort -- the greedy assignment then depends on the sort's tie order (the
        restatement freezes score desc, idx1, idx2; seen on seeds 114 / 117 with noise 0: peaks identical, two
        limbs assigned differently among equal-score candidates);
      * feature maps wider than 4:1 (the default resolution then shrinks an axis) are covered separately by
        test_oracle_matches_reference_golden_on_shrinking_resolutions."""
    conf, paf, ct, pt, rw, rh = sweep_case(seed)
    o, want = _vs_reference(live, f"sweep{seed}", conf, paf, ct, pt, rw, rh)
    got = o["humans"]
    assert got.tobytes() == want.tobytes(), (conf.shape, ct, pt, rw, rh, len(got), len(want))
