"""CPU suite, part 1: pin the ORACLE.
  * the NumPy Farneback restatement against the installed cv2 (the dependency the reference calls, F:878)
  * the motion-function restatements against golden vectors recorded from the reference itself, and
    live against the AST-loaded reference when oracle/ref_loader.py finds it."""
import json
import os

import numpy as np
import pytest

from funscript_flow_b200.synth import make_clip
from oracle import farneback_np as fb
from oracle import motion_np as mo
from oracle import ref_loader

cv2 = pytest.importorskip("cv2")


def test_known_constants():
    c = fb.poly_exp_constants()
    assert np.allclose(c["g"], [0.332452744, 0.234927148, 0.0828978196, 0.0146069536, 0.00128523575, 5.64693182e-05], rtol=1e-6)
    assert abs(c["ig11"] - 0.6944863966880652) < 1e-8 and abs(c["ig03"] + 0.3474535354408236) < 1e-8
    assert abs(c["ig33"] - 0.2413017476222371) < 1e-8 and abs(c["ig55"] - 0.4823113437926379) < 1e-8
    for ks, sg in [(3, 0.0), (3, 0.5), (9, 1.5), (19, 3.5)]:
        assert np.array_equal(fb.gaussian_kernel(ks, sg), cv2.getGaussianKernel(ks, sg, cv2.CV_32F).ravel())
    assert [(l["w"], l["h"], l["ksize"]) for l in fb.level_plan(1920, 1080)] == [(240, 135, 19), (480, 270, 9), (960, 540, 3), (1920, 1080, 3)]
    assert len(fb.level_plan(333, 217)) == 3 and len(fb.level_plan(96, 64)) == 2


@pytest.mark.parametrize("size", [(256, 256), (333, 217), (160, 120)])
def test_farneback_oracle_vs_cv2(size):
    w, h = size
    clip = make_clip(w, h, 8, seed=1, period=12.0, amplitude=0.3)
    ref = cv2.calcOpticalFlowFarneback(clip[2], clip[3], None, 0.5, 3, 15, 3, 5, 1.2, 0)
    mine = fb.farneback(clip[2], clip[3])
    d = np.abs(ref - mine)
    assert np.median(d) < 1e-6 and np.percentile(d, 99) < 1e-2 and (d > 0.05).mean() < 2e-3


def test_imgproc_primitives_vs_cv2():
    rng = np.random.default_rng(0)
    img = (rng.random((75, 101)) * 255).astype(np.float32)
    for ks, sg in [(3, 0.0), (3, 0.5), (9, 1.5), (19, 3.5)]:
        assert np.abs(fb.gaussian_blur_f32(img, ks, sg) - cv2.GaussianBlur(img, (ks, ks), sg)).max() < 1e-3
    for dw, dh in [(50, 37), (51, 38), (25, 19)]:
        assert np.abs(fb.resize_linear_f32(img, dw, dh) - cv2.resize(img, (dw, dh), interpolation=cv2.INTER_LINEAR)).max() < 1e-3
    fl = rng.standard_normal((40, 30, 2)).astype(np.float32)
    assert np.abs(fb.resize_linear_f32(fl, 60, 81) - cv2.resize(fl, (60, 81), interpolation=cv2.INTER_LINEAR)).max() < 1e-5


def test_motion_oracle_vs_golden(golden_dir):
    kat = json.load(open(os.path.join(golden_dir, "kat_motion.json")))
    for case in kat["cases"]:
        h, w = case["shape"]
        flow = np.random.default_rng(case["seed"]).standard_normal((h, w, 2)).astype(np.float32)
        x, y, v = mo.max_divergence(flow)
        assert [x, y] == case["max_divergence"][:2] and float(v) == case["max_divergence"][2]
        for r in case["radial"]:
            assert mo.radial_motion_weighted(flow, r["center"], False, r["pov"]) == pytest.approx(r["value"], rel=1e-12, abs=1e-15)
        assert mo.radial_motion_weighted(flow, [1, 1], True) == case["radial_cut"] == 0.0
    # survey-time known answers (SURVEY.md 8(c))
    flow = np.random.default_rng(0).standard_normal((8, 10, 2)).astype(np.float32)
    assert mo.max_divergence(flow)[:2] == (3, 0) and float(mo.max_divergence(flow)[2]) == pytest.approx(-2.8610074520111084)
    assert mo.radial_motion_weighted(flow, [4.5, 3.25], False) == pytest.approx(0.010646933131429252, rel=1e-12)
    assert mo.radial_motion_weighted(flow, [4.5, 3.25], False, True) == pytest.approx(-0.5006550564896315, rel=1e-12)
    assert mo.radial_motion_weighted(flow, [4.0, 3.0], False) == pytest.approx(0.012627041735249806, rel=1e-12)


def test_pair_oracle_vs_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "pairs.npz"))
    for name in "abc":
        info = mo.precompute_flow_info(g[f"{name}_p0"], g[f"{name}_p1"], {})
        assert np.array_equal(info["flow"], g[f"{name}_flow"])          # same cv2 build => bit-identical
        assert tuple(info["pos_center"]) == tuple(g[f"{name}_center"])
        assert info["val_pos"] == g[f"{name}_val"] and info["mean_mag"] == g[f"{name}_mean_mag"] and info["cut"] == g[f"{name}_cut"]
        # and the NumPy Farneback restatement against the recorded cv2 flow
        d = np.abs(fb.farneback(g[f"{name}_p0"], g[f"{name}_p1"]) - g[f"{name}_flow"])
        assert np.median(d) < 1e-6


def test_bracket_oracle_vs_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "bracket.npz"))
    vals, cuts, infos = mo.process_bracket(list(g["frames"]), {"cut_threshold": float(g["cut_threshold"])})
    assert np.array_equal(cuts, g["cut"]) and cuts.sum() == 1
    assert np.array_equal(np.array([i["pos_center"] for i in infos]), g["centers_raw"])
    assert np.allclose(vals, g["scalar"], rtol=1e-12, atol=1e-15)
    assert np.allclose(mo.smooth_centers([i["pos_center"] for i in infos]), g["centers"], rtol=0, atol=1e-12)


def test_postproc_vs_golden(golden_dir):
    from parity_checks import check_postproc_golden
    check_postproc_golden(golden_dir)


def test_oracle_vs_live_reference(golden_dir):
    """precompute_flow_info / radial_motion_weighted on four pairs and one post-processed series: the oracle against
    the records of tests/golden/reference_records.json, and against the AST-loaded reference
    itself when oracle/ref_loader.py finds FunscriptFlow.pyw."""
    import parity_checks as pc
    want = json.load(open(os.path.join(golden_dir, "reference_records.json")))["pairs_and_postprocess"]
    assert pc.record_pairs_and_postprocess(mo, pc.oracle_postprocess) == want
    if ref_loader.available():
        ref = ref_loader.load("ffref_live", serial_pools=True)
        assert pc.record_pairs_and_postprocess(ref, pc.reference_postprocess(ref)) == want


def test_preprocess_oracle_bit_exact_vs_cv2():
    """Row N2: cv2.resize (uint8 fixed point) + RGB2GRAY restated; integer work => bit-exact."""
    from oracle import preproc_np as pp
    rng = np.random.default_rng(1)
    for (h, w, dw, dh) in [(360, 640, 512, 512), (256, 256, 512, 512), (300, 200, 512, 512), (200, 300, 256, 256),
                           (1080, 1920, 256, 256), (97, 131, 256, 256), (480, 854, 256, 256)]:
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        assert np.array_equal(cv2.resize(img, (dw, dh)), pp.resize_u8_linear(img, dw, dh)), (h, w, dw, dh)
    for (h, w) in [(360, 640), (1080, 1920), (256, 256), (300, 200)]:
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        rgb = cv2.cvtColor(img, cv2.COLOR_BGR2RGB)
        assert np.array_equal(cv2.cvtColor(cv2.resize(rgb, (256, 256)), cv2.COLOR_RGB2GRAY), pp.frame_to_gray(img, False))
        assert np.array_equal(cv2.cvtColor(cv2.resize(rgb, (512, 512))[256:, :256], cv2.COLOR_RGB2GRAY), pp.frame_to_gray(img, True))
    # row N4: any target / window, including the identity target (cv2.resize returns the frame itself)
    import parity_checks as pc
    for (h, w, target, (x, y, ww, hh)) in pc.WINDOW_PLANS:
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        rgb = cv2.cvtColor(img, cv2.COLOR_BGR2RGB)
        want = cv2.cvtColor(np.ascontiguousarray(cv2.resize(rgb, target)[y:y + hh, x:x + ww]), cv2.COLOR_RGB2GRAY)
        assert np.array_equal(want, pp.frame_window_to_gray(img, target, (x, y, ww, hh))), (h, w, target)


def _mode_clip(case):
    from funscript_flow_b200.synth import ClipGenerator, ClipSpec
    sp = case["spec"]
    return ClipGenerator(ClipSpec(sp["width"], sp["height"], sp["n_frames"], seed=sp["seed"], amplitude=sp["amplitude"],
                                  period=sp["period"])).stack()


def test_oracle_pipeline_vs_golden_video_modes(golden_dir):
    """The whole oracle chain (pre-processing restatement -> cv2 flow -> motion functions -> post-processing)
    reproduces the funscripts the reference's process_video() wrote in VR mode, POV mode and from a 60 fps
    container (tests/golden/video_modes.json, recorded from the reference itself).  FFV1 is lossless, so the
    decoded frames are the generated clip."""
    import math
    from oracle import preproc_np as pp
    g = json.load(open(os.path.join(golden_dir, "video_modes.json")))
    for case in g["cases"]:
        st = case["settings"]
        clip = _mode_clip(case)
        step = max(1, int(math.ceil(case["fps"] / 30.0)))
        idx = list(range(0, len(clip), step))
        gray = [pp.frame_to_gray(cv2.cvtColor(clip[i], cv2.COLOR_GRAY2BGR), st["vr_mode"]) for i in idx]
        vals, cuts, _ = mo.process_bracket(gray, st)
        acts = mo.postprocess([(float(vals[j]), bool(cuts[j]), idx[j]) for j in range(len(vals))], case["fps"], st)
        assert acts == case["actions"], case["name"]


def test_postproc_product_equals_oracle_on_random_series(golden_dir):
    """Row N1 beyond the five golden cases: 60 random series (parity_checks.random_postproc_cases) through the
    shipped post-processing and through the oracle restatement, against the actions recorded in
    tests/golden/reference_records.json -- and through the reference's own statements when oracle/ref_loader.py
    finds FunscriptFlow.pyw."""
    import parity_checks as pc
    from funscript_flow_b200 import postproc
    recorded = json.load(open(os.path.join(golden_dir, "reference_records.json")))["random_postprocess"]
    cases = list(pc.random_postproc_cases())
    assert len(recorded) == len(cases)
    for case, ((vals, cuts, idx, fps, step, prm), want) in enumerate(zip(cases, recorded)):
        ffl = [(float(vals[i]), bool(cuts[i]), idx[i]) for i in range(len(vals))]
        assert mo.postprocess(ffl, fps, prm) == want, (case, len(vals), fps, prm)
        got = postproc.scalars_to_actions(vals.tolist(), cuts.tolist(), idx, fps, prm)
        assert got == want, (case, len(vals), fps, prm)
    if ref_loader.available():
        ref = ref_loader.load("ffref_pp", serial_pools=True)
        assert pc.record_random_postprocess(pc.reference_postprocess(ref)) == recorded


def test_motion_oracle_equals_live_reference_on_random_fields(golden_dir):
    """The restated max_divergence / radial_motion_weighted on the field families of parity_checks.check_reductions_random
    (ties, zero divergence, centres on and off the frame) against the records of
    tests/golden/reference_records.json, and against the reference's own functions when oracle/ref_loader.py finds
    FunscriptFlow.pyw."""
    import parity_checks as pc
    want = json.load(open(os.path.join(golden_dir, "reference_records.json")))["random_fields"]
    assert pc.record_random_fields(mo) == want and all(r["radial_cut"] == 0.0 for r in want)
    if ref_loader.available():
        assert pc.record_random_fields(ref_loader.load("ffref_rand", serial_pools=True)) == want
