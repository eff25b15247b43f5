"""Pose Proposal Network parse path (SURVEY 8f rank 3; hyperpose::parser::pose_proposal, src/pose_proposal.cpp:68-337).
Checker = the reference's OWN source compiled verbatim (oracle/_ref/libref_ppn.so); its outputs on seeded synthetic tensors
are committed as tests/golden/ref_ppn.npz, and oracle/ppn_oracle.py restates the algorithm for boxes without the reference.
  * CPU: goldens are non-vacuous, the generator reproduces their inputs, the restatement == goldens (== live reference where
    oracle/_ref is built);
  * GPU: the CUDA parser, through the C ABI, equals the goldens and the restatement byte-for-byte."""
import os

import numpy as np
import pytest

import oracle
from hyperpose_b200 import capi, synthetic as syn
from tests.golden.make_golden import PPN_CASES, PPN_RANDOM_ITERS, ppn_random_case, sha


@pytest.fixture(scope="module")
def gold(golden_dir):
    return np.load(os.path.join(golden_dir, "ref_ppn.npz"))


def _tensors(case):
    name, seed, P, net_w, net_h, gh, gw, nh, nw, pt, lt, nt, nd = case
    return syn.make_ppn_tensors(seed, P, net_h, net_w, gh, gw, nh, nw, nd)


def _as_records(humans):
    """oracle.ppn_process output -> HUMAN_DT array (the byte layout of hp_human / the goldens)"""
    out = np.zeros(len(humans), capi.HUMAN_DT)
    for i, h in enumerate(humans):
        out[i]["score"] = h["score"]
        for k, (has, x, y, s) in enumerate(h["parts"]):
            out[i]["parts"][k] = (has, x, y, s)
    return out


def _diff(a, b):
    if len(a) != len(b):
        return f"{len(a)} humans vs {len(b)}"
    for i, (x, y) in enumerate(zip(a, b)):
        if x.tobytes() != y.tobytes():
            return f"human {i}:\n got={x}\n ref={y}"
    return None


def test_goldens_not_vacuous(gold):
    assert len(gold["ppn_p1_humans"]) == 1 and len(gold["ppn_empty_humans"]) == 0
    assert len(gold["ppn_p4_humans"]) >= 3 and len(gold["ppn_crowd_humans"]) >= 6 and len(gold["ppn_dense_humans"]) >= 40
    h = gold["ppn_p1_humans"][0]
    assert float(h["score"]) == 18.0 and int(h["parts"]["has_value"].sum()) == 18


@pytest.mark.parametrize("case", PPN_CASES, ids=[c[0] for c in PPN_CASES])
def test_generator_matches_golden_inputs(gold, case):
    assert "".join(sha(a) for a in _tensors(case)) == str(gold[case[0] + "_in_sha"])


@pytest.mark.parametrize("case", PPN_CASES, ids=[c[0] for c in PPN_CASES])
def test_restatement_equals_reference_golden(gold, case):
    name, seed, P, net_w, net_h, gh, gw, nh, nw, pt, lt, nt, nd = case
    got = _as_records(oracle.ppn_process(*_tensors(case), net_w, net_h, pt, lt, nt))
    d = _diff(got, gold[name + "_humans"])
    assert d is None, f"{name}: {d}"


@pytest.mark.skipif(not oracle.ppn_ref_available(), reason="oracle/_ref/libref_ppn.so not built")
@pytest.mark.parametrize("case", PPN_CASES, ids=[c[0] for c in PPN_CASES])
def test_live_reference_matches_golden(gold, case):
    name, seed, P, net_w, net_h, gh, gw, nh, nw, pt, lt, nt, nd = case
    got = oracle.ref_ppn_process(*_tensors(case), net_w, net_h, pt, lt, nt)
    assert got.tobytes() == gold[name + "_humans"].tobytes()


def test_restatement_vs_live_reference_random(golden_dir):
    """the restatement against what oracle/_ref returned on these inputs (ref_live.npz), and against the live oracle/_ref
    as well where it is built"""
    live = np.load(os.path.join(golden_dir, "ref_live.npz"))
    rng = np.random.default_rng(7)
    for it in range(PPN_RANDOM_ITERS):
        t, (pt, lt, nt) = ppn_random_case(it, rng)
        assert "".join(sha(a) for a in t) == str(live[f"ppn_random{it}_in_sha"]), "synthetic generator drifted from the goldens"
        want = live[f"ppn_random{it}_humans"]
        if oracle.ppn_ref_available():
            assert oracle.ref_ppn_process(*t, 384, 384, pt, lt, nt).tobytes() == want.tobytes()
        got = _as_records(oracle.ppn_process(*t, 384, 384, pt, lt, nt))
        d = _diff(got, want)
        assert d is None, f"seed {1000 + it} thr {(pt, lt, nt)}: {d}"


@pytest.mark.gpu
@pytest.mark.parametrize("case", PPN_CASES, ids=[c[0] for c in PPN_CASES])
def test_gpu_parser_equals_reference_golden(gold, case):
    name, seed, P, net_w, net_h, gh, gw, nh, nw, pt, lt, nt, nd = case
    t = _tensors(case)
    p = capi.PoseProposalParser((net_w, net_h), pt, lt, nt)
    got = p.process(*t)
    d = _diff(got, gold[name + "_humans"])
    assert d is None, f"{name}: {d}"
    # one launch; the dense case overflows the shared-memory human capacity once and is re-run by the global-scratch variant
    assert p.launch_count == (2 if name == "ppn_dense" else 1)
    if name == "ppn_dense":
        assert _diff(p.process(*t), gold[name + "_humans"]) is None and p.launch_count == 3   # sticky: no second fast attempt
    p.close()


@pytest.mark.gpu
def test_gpu_parser_batched_vs_restatement():
    N = 24
    frames = [syn.make_ppn_tensors(500 + i, (0, 9), distractors=5 * i) for i in range(N)]
    p = capi.PoseProposalParser((384, 384))
    stacked = [np.stack([f[k] for f in frames]) for k in (0, 2, 3, 4, 5, 6)]
    for thr in [(0.10, 0.05, 0.3), (0.06, 0.03, 0.2), (0.10, 0.05, 0.05)]:
        p.set_point_thresh(thr[0]); p.set_limb_thresh(thr[1]); p.set_nms_thresh(thr[2])
        got = p.process_batch(*stacked, cap=512)
        for i in range(N):
            want = _as_records(oracle.ppn_process(*frames[i], 384, 384, *thr))
            d = _diff(got[i], want)
            assert d is None, f"frame {i} thr {thr}: {d}"
    p.close()


@pytest.mark.gpu
def test_gpu_parser_argument_errors():
    p = capi.PoseProposalParser((384, 384))
    t = syn.make_ppn_tensors(1, 1)
    with pytest.raises(capi.HyperposeError) as e:      # the COCO limb table needs 18 key-point maps (key_points.at() throws in the reference)
        p.process_batch(*[a[None, :17] for a in (t[0], t[2], t[3], t[4], t[5])], t[6][None])
    assert e.value.status == capi.HP_ERR_ARG
    with pytest.raises(capi.HyperposeError) as e:      # caller capacity smaller than the result
        p.process(*syn.make_ppn_tensors(22, (6, 10), distractors=40), cap=2)
    assert e.value.status == capi.HP_ERR_CAPACITY
    p.close()
