"""OpenPifPaf decode path (SURVEY 8a A12, BASELINE config 5).
Checker = the reference's OWN decoder (src/pifpaf.cpp + src/pifpaf_decoder/*.cpp compiled verbatim into oracle/_ref):
its outputs on the seeded synthetic fields are committed as tests/golden/ref_pifpaf.npz.
  * CPU: goldens are non-vacuous, the synthetic generator still reproduces their inputs, live _ref == goldens;
  * GPU: the CUDA decoder, through the C ABI, equals the goldens byte-for-byte (keypoint pixels are integers, part scores
    are forced to 1 by the reference, so only the instance score is a free float -- held to bit equality as well)."""
import os

import numpy as np
import pytest

import oracle
from hyperpose_b200 import capi, synthetic as syn
from tests.golden.make_golden import PIFPAF_CASES, pifpaf_batch_case, sha


@pytest.fixture(scope="module")
def gold(golden_dir):
    return np.load(os.path.join(golden_dir, "ref_pifpaf.npz"))


def test_goldens_not_vacuous(gold):
    assert len(gold["pp_p2_humans"]) == 2 and len(gold["pp_p5_humans"]) == 5 and len(gold["pp_empty_humans"]) == 0
    assert len(gold["pp_crowd_humans"]) >= 4
    h = gold["pp_p2_humans"][0]
    assert int(h["parts"]["has_value"].sum()) == 18 and np.all(h["parts"]["score"][h["parts"]["has_value"] == 1] == 1.0)


@pytest.mark.parametrize("case", PIFPAF_CASES, ids=[c[0] for c in PIFPAF_CASES])
def test_generator_matches_golden_inputs(gold, case):
    name, seed, P, h, w, thr = case
    pif, paf = syn.make_pifpaf_fields(seed, P, h, w)
    assert sha(pif) + sha(paf) == str(gold[name + "_in_sha"])


@pytest.mark.skipif(not oracle.pifpaf_ref_available(), reason="oracle/_ref/libref_pifpaf.so not built")
@pytest.mark.parametrize("case", PIFPAF_CASES[:3], ids=[c[0] for c in PIFPAF_CASES[:3]])
def test_live_reference_matches_golden(gold, case):
    name, seed, P, h, w, thr = case
    pif, paf = syn.make_pifpaf_fields(seed, P, h, w)
    got = oracle.ref_pifpaf_process(pif, paf, (h - 1) * 8 + 1, (w - 1) * 8 + 1, thr)
    assert got.tobytes() == gold[name + "_humans"].tobytes()


def _diff(a, b):
    if len(a) != len(b):
        return f"{len(a)} humans vs {len(b)}"
    for i, (x, y) in enumerate(zip(a, b)):
        if x.tobytes() != y.tobytes():
            return f"human {i}:\n gpu={x}\n ref={y}"
    return None


@pytest.mark.gpu
@pytest.mark.parametrize("case", PIFPAF_CASES, ids=[c[0] for c in PIFPAF_CASES])
def test_gpu_decoder_equals_reference_golden(gold, case):
    name, seed, P, h, w, thr = case
    pif, paf = syn.make_pifpaf_fields(seed, P, h, w)
    dec = capi.PifPafParser((h - 1) * 8 + 1, (w - 1) * 8 + 1, thr)
    got = dec.process(pif, paf)
    d = _diff(got, gold[name + "_humans"])
    assert d is None, f"{name}: {d}"
    dec.close()


@pytest.mark.gpu
def test_gpu_decoder_batched_vs_live_reference(golden_dir):
    """against what oracle/_ref returned on these frames (ref_live.npz), and against the live oracle/_ref as well where it is built"""
    live = np.load(os.path.join(golden_dir, "ref_live.npz"))
    pif, paf = pifpaf_batch_case()
    assert sha(pif) + sha(paf) == str(live["pp_batch_in_sha"]), "synthetic generator drifted from the goldens"
    dec = capi.PifPafParser(385, 385, 0.1)
    got = dec.process_batch(pif, paf)
    for i in range(len(pif)):
        want = live[f"pp_batch{i}_humans"]
        if oracle.pifpaf_ref_available():
            assert oracle.ref_pifpaf_process(pif[i], paf[i], 385, 385, 0.1).tobytes() == want.tobytes()
        d = _diff(got[i], want)
        assert d is None, f"frame {i}: {d}"
    dec.close()
