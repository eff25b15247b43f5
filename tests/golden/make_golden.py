"""Generates tests/golden/*.npz.  Run in the BUILD container only (needs Python cv2 and
/root/reference; neither is required at test time):

    python tests/golden/make_golden.py

1. cv_pin.npz      -- outputs of the real OpenCV (Python cv2) for the two third-party
                      primitives on the reference's path: cv::resize(INTER_AREA) upscale
                      (src/post_process.hpp:50) and cv::GaussianBlur(17x17, sigma=3)
                      (post_process.hpp:66-67), on seeded inputs; small cases stored in full,
                      full-size cases as sha256 of the output bytes.
2. ref_humans.npz  -- human_t lists produced by the reference's OWN src/paf.cpp (compiled
                      verbatim into oracle/_ref by oracle/Makefile) on the seeded synthetic
                      frames of hyperpose_b200/synthetic.py (SURVEY 8d configs).
3. ref_live.npz    -- (`python tests/golden/make_golden.py live`) the reference parsers' outputs
                      on the random / sweep inputs of the tests that compare against them.
"""
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
HERE = os.path.dirname(os.path.abspath(__file__))

# (name, seed, persons, hf, wf, res_w, res_h, conf_thresh, paf_thresh)
FRAME_CASES = [
    ("cfg1_p1", 0, 1, 46, 54, -1, -1, 0.05, 0.05),
    ("cfg1_p3", 1, 3, 46, 54, -1, -1, 0.05, 0.05),
    ("cfg3_p5", 2, 5, 46, 82, -1, -1, 0.05, 0.05),
    ("cfg4_crowd", 3, (10, 20), 46, 54, -1, -1, 0.05, 0.05),
    ("cfg3_crowd", 5, 12, 46, 82, -1, -1, 0.05, 0.05),
    ("square", 6, 4, 46, 46, -1, -1, 0.05, 0.05),
    ("user_res", 7, 3, 46, 54, 216, 184, 0.05, 0.05),       # untransposed 4x resolution set by the user
    ("user_res_odd", 8, 3, 46, 54, 300, 200, 0.1, 0.08),
    ("empty", 9, 0, 46, 54, -1, -1, 0.05, 0.05),
    ("tiny", 10, 1, 12, 16, -1, -1, 0.05, 0.05),
]


# (src_h, src_w, dst_h, dst_w) of the frame-resize pin
RESIZE_CASES = [(360, 640, 368, 656), (480, 640, 368, 656), (720, 1280, 368, 656), (736, 1312, 368, 656), (100, 80, 368, 432),
                (1080, 1920, 368, 656), (368, 656, 368, 656), (300, 500, 207, 344), (37, 53, 64, 48)]


# (name, seed, persons, h, w, keypoint_thresh) of the PifPaf decode pin (BASELINE config 5: 385x385 -> 49x49 fields)
PIFPAF_CASES = [("pp_p2", 4, 2, 49, 49, 0.1), ("pp_p5", 5, 5, 49, 49, 0.1), ("pp_crowd", 6, (6, 12), 49, 49, 0.1), ("pp_empty", 7, 0, 49, 49, 0.1),
                ("pp_rect", 8, 3, 47, 55, 0.1), ("pp_thr", 9, 4, 49, 49, 0.3), ("pp_small", 10, 2, 25, 33, 0.1)]


# (name, seed, persons, net_w, net_h, gh, gw, nh, nw, point_thresh, limb_thresh, nms_thresh, distractors) of the Pose Proposal pin
PPN_CASES = [("ppn_p1", 20, 1, 384, 384, 12, 12, 9, 9, 0.10, 0.05, 0.3, 12), ("ppn_p4", 21, 4, 384, 384, 12, 12, 9, 9, 0.10, 0.05, 0.3, 12),
             ("ppn_crowd", 22, (6, 10), 384, 384, 12, 12, 9, 9, 0.10, 0.05, 0.3, 40), ("ppn_empty", 23, 0, 384, 384, 12, 12, 9, 9, 0.10, 0.05, 0.3, 0),
             ("ppn_rect", 24, 3, 512, 384, 12, 16, 7, 9, 0.10, 0.05, 0.3, 12), ("ppn_thr", 25, 4, 384, 384, 12, 12, 9, 9, 0.30, 0.20, 0.5, 12),
             ("ppn_dense", 26, 5, 384, 384, 12, 12, 9, 9, 0.05, 0.03, 0.3, 60)]


# (src_h, src_w, dst_h, dst_w) of the INTER_AREA pin for the regimes beyond pure up-scaling (A5): mixed (one axis shrinks: 2-tap
# area-mode lerp on both), integer factors (resizeAreaFast_, incl. the 2x2 SIMD kernel and its scalar tail), fractional (DecimateAlpha)
AREA_CASES = [(46, 82, 100, 60), (46, 82, 30, 200), (46, 200, 800, 184), (46, 82, 23, 41), (48, 84, 16, 28), (48, 84, 12, 21), (46, 82, 46, 41),
              (46, 82, 23, 82), (40, 84, 20, 41), (46, 82, 30, 50), (46, 82, 45, 81), (46, 82, 20, 82), (54, 46, 13, 17), (46, 82, 46, 50), (46, 82, 11, 19)]

# parser cases whose up-map shrinks an axis: (name, seed, persons, hf, wf, res_w, res_h, conf_thresh, paf_thresh)
AREA_FRAME_CASES = [
    # default resolution (width 4*Hf, height 4*Wf) = (120, 520): width 120 < Wf = 130 -> mixed regime.  (Much wider maps, e.g. 24x120,
    # stretch rows ~20x: the plateaus give limb candidates with EXACTLY equal scores and the reference's unstable std::sort
    # (paf.cpp:246) then picks among them arbitrarily -- the region test_oracle_matches_live_reference_sweep documents.)
    ("wide_default", 11, 3, 30, 130, -1, -1, 0.05, 0.05),
    ("user_mixed", 12, 3, 46, 54, 40, 300, 0.05, 0.05),      # x shrinks, y grows
    ("user_half", 13, 3, 46, 54, 27, 23, 0.05, 0.05),        # exact 2x2 reduction (SIMD kernel + tail)
    ("user_third", 14, 2, 48, 54, 18, 16, 0.05, 0.05),       # 3x3 integer reduction
    ("user_frac", 15, 3, 46, 54, 41, 33, 0.05, 0.05),        # fractional reduction on both axes
    ("user_keep_x", 16, 3, 46, 54, 54, 30, 0.05, 0.05),      # one axis kept (scale 1), the other shrinks: area regime
]


def random_case(seed):
    """frame of test_oracle_matches_live_reference_random: (conf, paf)"""
    rng = np.random.default_rng(seed)
    hf, wf = [(46, 54), (46, 82), (32, 32), (23, 40)][seed % 4]
    P = int(rng.integers(0, 16))
    from hyperpose_b200 import synthetic as syn
    return syn.make_frame_tensors(seed, P, hf, wf)


def noise_case():
    """structureless input (many spurious peaks, few/no humans): (conf, paf)"""
    rng = np.random.default_rng(99)
    conf = rng.random((19, 24, 30), dtype=np.float32) * 0.3
    paf = (rng.random((38, 24, 30), dtype=np.float32) - 0.5)
    return conf, paf


def sweep_case(seed):
    """frame and parser settings of test_oracle_matches_live_reference_sweep: (conf, paf, ct, pt, rw, rh)"""
    from hyperpose_b200 import synthetic as syn
    rng = np.random.default_rng(seed)
    hf = int(rng.integers(9, 50))
    wf = int(rng.integers(9, min(90, 4 * hf) + 1))
    P = int(rng.integers(0, 13))
    noise = float(rng.choice([0.005, 0.02, 0.06]))
    conf, paf = syn.make_frame_tensors(seed, P, hf, wf, noise=noise)
    ct, pt = float(rng.choice([0.05, 0.1, 0.3])), float(rng.choice([0.02, 0.05, 0.2]))
    if seed % 3 == 0:      # user resolution (w, h) >= the feature map
        rw, rh = int(hf * rng.uniform(1.0, 4.6)) + 1, int(wf * rng.uniform(1.0, 4.6)) + 1
        rw, rh = max(rw, wf), max(rh, hf)
    else:
        rw = rh = -1
    return conf, paf, ct, pt, rw, rh


RANDOM_SEEDS, SWEEP_SEEDS = range(20, 32), range(100, 140)
PPN_RANDOM_ITERS = 40


def ppn_random_case(it, rng):
    """iteration `it` of test_restatement_vs_live_reference_random (rng: default_rng(7), advanced once per iteration)"""
    from hyperpose_b200 import synthetic as syn
    thr = [(0.10, 0.05, 0.3), (0.06, 0.03, 0.2), (0.2, 0.1, 0.6), (0.10, 0.05, 0.05)][it % 4]
    return syn.make_ppn_tensors(1000 + it, (0, 8), distractors=int(rng.integers(0, 80))), thr


def pifpaf_batch_case():
    """the 8 frames of test_gpu_decoder_batched_vs_live_reference: (pif [8,17,5,49,49], paf [8,19,9,49,49])"""
    from hyperpose_b200 import synthetic as syn
    fields = [syn.make_pifpaf_fields(100 + i, (1, 9), 49, 49) for i in range(8)]
    return np.stack([f[0] for f in fields]), np.stack([f[1] for f in fields])


def pifpaf_handoff_case():
    """the 2 frames of test_pifpaf_fields_hand_off: (pif [2,17,5,49,49], paf [2,19,9,49,49])"""
    from hyperpose_b200 import synthetic as syn
    fields = [syn.make_pifpaf_fields(20 + i, (2, 3), 49, 49) for i in range(2)]
    return np.stack([f[0] for f in fields]).astype(np.float32), np.stack([f[1] for f in fields]).astype(np.float32)


def make_live():
    """tests/golden/ref_live.npz: what the reference's own parsers (oracle/_ref) return on the inputs of the tests that compare
    against them, so that those comparisons run where the reference sources are absent"""
    import oracle
    assert oracle.ref_available() and oracle.pifpaf_ref_available() and oracle.ppn_ref_available()
    out = {}

    def paf_entry(key, conf, paf, ct=0.05, pt=0.05, rw=-1, rh=-1):
        rp = oracle.RefParser(ct, pt, rw, rh)
        out[key + "_humans"] = rp.process(conf, paf)
        out[key + "_in_sha"] = np.array(sha(conf) + sha(paf))
        rp.close()

    for seed in RANDOM_SEEDS:
        paf_entry(f"random{seed}", *random_case(seed))
    paf_entry("noise", *noise_case())
    for seed in SWEEP_SEEDS:
        paf_entry(f"sweep{seed}", *sweep_case(seed))
    rng = np.random.default_rng(7)
    for it in range(PPN_RANDOM_ITERS):
        t, thr = ppn_random_case(it, rng)
        out[f"ppn_random{it}_humans"] = oracle.ref_ppn_process(*t, 384, 384, *thr)
        out[f"ppn_random{it}_in_sha"] = np.array("".join(sha(a) for a in t))
    for key, (pif, paf) in (("pp_batch", pifpaf_batch_case()), ("pp_handoff", pifpaf_handoff_case())):
        for i in range(len(pif)):
            out[f"{key}{i}_humans"] = oracle.ref_pifpaf_process(pif[i], paf[i], 385, 385, 0.1)
        out[key + "_in_sha"] = np.array(sha(pif) + sha(paf))
    np.savez_compressed(os.path.join(HERE, "ref_live.npz"), **out)
    print({k: len(v) for k, v in out.items() if k.endswith("_humans")})


def make_area():
    """tests/golden/cv_pin_area.npz (real cv2) + ref_humans_area.npz (the reference's own paf.cpp over the pinned resize)"""
    import cv2
    import oracle
    from hyperpose_b200 import synthetic as syn
    oracle.build()
    out = {"cv2_version": np.array(cv2.__version__)}
    for i, (sh, sw, dh, dw) in enumerate(AREA_CASES):
        img = np.random.default_rng(300 + i).random((sh, sw), dtype=np.float32)
        ref = cv2.resize(img, (dw, dh), interpolation=cv2.INTER_AREA)
        out[f"area{i}_sha"] = np.array(sha(ref))
        if ref.size <= 4096:
            out[f"area{i}_out"] = ref
    np.savez_compressed(os.path.join(HERE, "cv_pin_area.npz"), **out)
    ref = {}
    for (name, seed, P, hf, wf, rw, rh, ct, pt) in AREA_FRAME_CASES:
        conf, paf = syn.make_frame_tensors(seed, P, hf, wf)
        rp = oracle.RefParser(ct, pt, rw, rh)
        ref[name + "_humans"] = rp.process(conf, paf)
        ref[name + "_in_sha"] = np.array(sha(conf) + sha(paf))
        rp.close()
    np.savez_compressed(os.path.join(HERE, "ref_humans_area.npz"), **ref)
    print({k: len(v) for k, v in ref.items() if k.endswith("_humans")})


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def main():
    import cv2
    from hyperpose_b200 import synthetic as syn
    import oracle

    out = {"cv2_version": np.array(cv2.__version__)}
    out["gauss_kernel"] = cv2.getGaussianKernel(17, 3.0, cv2.CV_32F).ravel()
    rng = np.random.default_rng(1234)
    small = [(23, 27, 108, 92), (12, 16, 64, 48), (9, 9, 36, 36), (10, 7, 31, 40), (5, 20, 80, 20)]
    for i, (sh, sw, dh, dw) in enumerate(small):
        img = rng.random((sh, sw), dtype=np.float32) * 2 - 0.5
        up = cv2.resize(img, (dw, dh), interpolation=cv2.INTER_AREA)
        out[f"small{i}_in"] = img
        out[f"small{i}_shape"] = np.array([dh, dw])
        out[f"small{i}_up"] = up
        out[f"small{i}_blur"] = cv2.GaussianBlur(up, (17, 17), 3.0)
    big = [(46, 54, 216, 184), (46, 82, 328, 184), (46, 46, 184, 184), (46, 54, 184, 216)]
    for i, (sh, sw, dh, dw) in enumerate(big):
        img = np.random.default_rng(100 + i).random((sh, sw), dtype=np.float32)
        up = cv2.resize(img, (dw, dh), interpolation=cv2.INTER_AREA)
        out[f"big{i}_dims"] = np.array([sh, sw, dh, dw])
        out[f"big{i}_up_sha"] = np.array(sha(up))
        out[f"big{i}_blur_sha"] = np.array(sha(cv2.GaussianBlur(up, (17, 17), 3.0)))
    # cv::resize(INTER_LINEAR) on u8 frames (src/tensorrt.cpp:451) and the letterbox path (src/data.cpp:53-69)
    for i, (sh, sw, dh, dw) in enumerate(RESIZE_CASES):
        img = np.random.default_rng(200 + i).integers(0, 256, (sh, sw, 3), dtype=np.uint8)
        out[f"rz{i}_sha"] = np.array(sha(cv2.resize(img, (dw, dh))))
        h1 = dw * (sh / float(sw)); w2 = dh * (sw / float(sh))
        rw, rh = (dw, int(h1)) if h1 <= dh else (int(w2), dh)
        lb = cv2.copyMakeBorder(cv2.resize(img, (rw, rh)), 0, dh - rh, 0, dw - rw, cv2.BORDER_CONSTANT, value=(0, 0, 0))
        out[f"lb{i}_sha"] = np.array(sha(lb))
    np.savez_compressed(os.path.join(HERE, "cv_pin.npz"), **out)

    ref = {}
    for (name, seed, P, hf, wf, rw, rh, ct, pt) in FRAME_CASES:
        conf, paf = syn.make_frame_tensors(seed, P, hf, wf)
        rp = oracle.RefParser(ct, pt, rw, rh)
        ref[name + "_humans"] = rp.process(conf, paf)
        ref[name + "_in_sha"] = np.array(sha(conf) + sha(paf))
        rp.close()
    np.savez_compressed(os.path.join(HERE, "ref_humans.npz"), **ref)
    pp = {}
    for (name, seed, P, h, w, thr) in PIFPAF_CASES:
        pif, paf = syn.make_pifpaf_fields(seed, P, h, w)
        pp[name + "_humans"] = oracle.ref_pifpaf_process(pif, paf, (h - 1) * 8 + 1, (w - 1) * 8 + 1, thr)
        pp[name + "_in_sha"] = np.array(sha(pif) + sha(paf))
    np.savez_compressed(os.path.join(HERE, "ref_pifpaf.npz"), **pp)
    make_ppn()


def make_ppn():
    """goldens of the reference's own src/pose_proposal.cpp (oracle/_ref/libref_ppn.so) on seeded synthetic tensors"""
    from hyperpose_b200 import synthetic as syn
    import oracle
    pn = {}
    for (name, seed, P, net_w, net_h, gh, gw, nh, nw, pt, lt, nt, nd) in PPN_CASES:
        t = syn.make_ppn_tensors(seed, P, net_h, net_w, gh, gw, nh, nw, nd)
        pn[name + "_humans"] = oracle.ref_ppn_process(*t, net_w, net_h, pt, lt, nt)
        pn[name + "_in_sha"] = np.array("".join(sha(a) for a in t))
    np.savez_compressed(os.path.join(HERE, "ref_ppn.npz"), **pn)
    print("wrote", os.listdir(HERE))


if __name__ == "__main__" and "area" in sys.argv[1:]:
    make_area()
    sys.exit(0)

if __name__ == "__main__" and "live" in sys.argv[1:]:
    make_live()
    sys.exit(0)

if __name__ == "__main__":
    if "ppn" in sys.argv[1:]:
        make_ppn()
    else:
        main()
