"""Shared parity checks: the same assertions run against the g++ emulation (small sizes, CPU suite)
and against the real sm_100a library (`-m gpu`, larger sizes).  Every check compares the CUDA path,
called through the C ABI, with the oracle (oracle/) and/or golden vectors recorded from the
reference itself (tests/golden/)."""
from __future__ import annotations

import hashlib
import json
import os

import numpy as np

from funscript_flow_b200 import api, postproc
from funscript_flow_b200.synth import ClipGenerator, ClipSpec, make_clip
from oracle import farneback_np as fb
from oracle import motion_np as mo

# ---- stated tolerances ------------------------------------------------------------------------
# north_star: median |dflow| < 0.05 px.  We hold the kernels to far tighter numbers and keep the
# north-star bound as the outer gate.
FLOW_MEDIAN_TOL = 1e-5          # px, vs cv2 / the float64-accumulating oracle
FLOW_P99_TOL = 1e-2             # px (isolated border pixels flip the in-bounds test of step 6)
FLOW_BAD_FRACTION = 2e-3        # fraction of pixels allowed beyond 0.05 px
NORTH_STAR_MEDIAN = 0.05
SCALAR_RTOL = 1e-3              # north_star: per-frame scalars within 1e-3 relative
ARGMAX_MARGIN = 1e-4            # exact (x, y) is asserted when the reference's top1-top2 gap >= this
MEAN_MAG_RTOL = 2e-3            # a handful of border pixels flip step 6's in-bounds test (up to ~0.1 px each) and
MEAN_MAG_ATOL = 5e-4            # each flip perturbs its 15x15 blur footprint over 3 iterations (~600 px by ~1e-3..5e-2 px);
                                # on a 128x96 frame that is ~3e-4 px of mean magnitude (profiles/r1_parity_sensitivity.txt)


def flow_stats(a, b):
    d = np.abs(a.astype(np.float64) - b.astype(np.float64))
    return float(np.median(d)), float(np.percentile(d, 99)), float(d.max()), float((d > 0.05).mean())


def assert_flow_close(got, ref, what=""):
    med, p99, mx, bad = flow_stats(got, ref)
    msg = f"{what}: median {med:.3e} p99 {p99:.3e} max {mx:.3e} frac>0.05px {bad:.3e}"
    assert med < NORTH_STAR_MEDIAN, msg
    assert med < FLOW_MEDIAN_TOL, msg
    assert p99 < FLOW_P99_TOL, msg
    assert bad < FLOW_BAD_FRACTION, msg
    return msg


def argmax_margin(flow):
    """(x, y, top1, top1 - best |div| outside the argmax pixel) of the reference's quantity."""
    d = np.abs(mo.divergence_field(flow))
    flat = int(np.argmax(d))
    top1 = float(d.flat[flat])
    d2 = d.copy()
    d2.flat[flat] = -1.0
    return flat % d.shape[1], flat // d.shape[1], top1, top1 - float(d2.max())


def assert_argmax(got_xy, got_val, ref_flow, what=""):
    """Bit-exact location when the reference's own margin is >= ARGMAX_MARGIN, else value parity."""
    x, y, top1, gap = argmax_margin(ref_flow)
    if gap >= ARGMAX_MARGIN:
        assert (int(got_xy[0]), int(got_xy[1])) == (x, y), f"{what}: argmax {got_xy} != {(x, y)} (gap {gap:.2e})"
    else:
        assert abs(abs(float(got_val)) - top1) <= 1e-5, f"{what}: |div| {got_val} vs top1 {top1} (gap {gap:.2e})"
    return gap


def scalar_tol(flow, center):
    """1e-3 relative with an absolute floor tied to the mean |term| (the balanced weights cancel
    global motion, so the scalar can be tiny next to its terms)."""
    h, w = flow.shape[:2]
    xs = np.arange(w)[None, :] - center[0]
    ys = np.arange(h)[:, None] - center[1]
    # floor = 1e-4 x mean |term|: the flow itself only agrees with cv2 to ~1e-5 px at p99 (plus a few
    # border pixels at ~0.1 px), and near-stationary pairs have scalars 1000x smaller than their terms
    return 1e-4 * float(np.mean(np.abs(flow[..., 0] * xs) + np.abs(flow[..., 1] * ys)))


# ---- stage-wise checks -----------------------------------------------------------------------
def check_stages(ctx, width, height, seed=3):
    clip = make_clip(width, height, 4, seed=seed, period=10.0, amplitude=0.3)
    p0, p1 = clip[1], clip[2]
    plan = fb.level_plan(width, height)
    for lvl in plan:
        got = ctx.stage_pyramid(p0, lvl["k"])
        ref = fb.pyramid_level(p0, lvl)
        assert got.shape == ref.shape
        assert np.abs(got - ref).max() < 1e-3, f"pyramid k={lvl['k']}: {np.abs(got - ref).max()}"   # values ~0..255
    top = plan[-1]
    I0, I1 = fb.pyramid_level(p0, top), fb.pyramid_level(p1, top)
    R0, R1 = fb.poly_exp(I0), fb.poly_exp(I1)
    got = ctx.stage_polyexp(I0)
    assert np.abs(got - R0).max() < 2e-4 * max(1.0, np.abs(R0).max()), f"polyexp {np.abs(got - R0).max()}"
    rng = np.random.default_rng(seed)
    flow = (rng.standard_normal((height, width, 2)) * 1.5).astype(np.float32)
    for f_in in (flow, None):
        f_ref = flow if f_in is not None else np.zeros_like(flow)
        M = fb.update_matrices(R0, R1, f_ref)
        got = ctx.stage_update_matrices(R0, R1, f_in)
        assert np.abs(got - M).max() < 1e-4 * max(1.0, np.abs(M).max()), f"update_matrices {np.abs(got - M).max()}"
        got = ctx.stage_flow_iter(R0, R1, f_in)
        ref = fb.blur_solve(M)
        assert np.abs(got - ref).max() < 1e-4, f"flow_iter {np.abs(got - ref).max()}"
    hc, wc = plan[0]["h"], plan[0]["w"]
    fc = rng.standard_normal((hc, wc, 2)).astype(np.float32)
    got = ctx.stage_upsample_flow(fc, width, height)
    assert np.abs(got - fb.upsample_flow(fc, width, height)).max() < 1e-5


def check_farneback_vs_cv2(ctx, width, height, seed=1, period=12.0, amplitude=0.3):
    import cv2
    clip = make_clip(width, height, 8, seed=seed, period=period, amplitude=amplitude)
    p0, p1 = clip[2], clip[3]
    ref = cv2.calcOpticalFlowFarneback(p0, p1, None, 0.5, 3, 15, 3, 5, 1.2, 0)
    got = ctx.farneback(p0, p1)
    return assert_flow_close(got, ref, f"farneback {width}x{height}")


def check_reductions_kat(ctx, golden_dir):
    """max_divergence / radial_motion_weighted known answers recorded from the reference."""
    kat = json.load(open(os.path.join(golden_dir, "kat_motion.json")))
    for case in kat["cases"]:
        h, w = case["shape"]
        if min(h, w) < 16:
            continue   # ffb_configure refuses frames under 16 px; the oracle test covers the 8x10 case
        flow = np.random.default_rng(case["seed"]).standard_normal((h, w, 2)).astype(np.float32)
        x, y, v = ctx.max_divergence(flow)
        assert [x, y] == case["max_divergence"][:2]
        assert np.float32(v) == np.float32(case["max_divergence"][2])   # bit-exact: same fp32 ops on the same input
        for r in case["radial"]:
            got = ctx.radial_motion(flow, r["center"], False, r["pov"])
            assert abs(got - r["value"]) <= 1e-6 * max(1.0, abs(r["value"])), (r, got)
        assert ctx.radial_motion(flow, [1.0, 1.0], True, False) == 0.0 == case["radial_cut"]
    exp = kat["expansion_640x360"]
    ys, xs = np.mgrid[0:360, 0:640].astype(np.float32)
    flow = np.stack([0.01 * (xs - 352), 0.01 * (ys - 162)], axis=-1).astype(np.float32)
    got = ctx.radial_motion(flow, [352, 162], False, False)
    assert abs(got - exp["radial"]) <= 1e-6 * abs(exp["radial"])
    x, y, v = ctx.max_divergence(flow)
    assert [x, y] == exp["max_divergence"][:2]


def check_reductions_random(ctx, n_cases=24, max_side=97, seed=123):
    """Device reductions against the oracle on random flow fields of random (odd, non-square) sizes: integer centres
    on a pixel column / row (the `x == cx` branch), fractional centres, centres on the border and outside the frame,
    POV mode, a constant field (all |div| == 0: the first pixel wins), duplicated maxima (first in C order wins)."""
    from oracle import motion_np as mo
    rng = np.random.default_rng(seed)
    for case in range(n_cases):
        w, h = int(rng.integers(16, max_side)), int(rng.integers(16, max_side))
        kind = case % 4
        if kind == 0:
            flow = rng.standard_normal((h, w, 2)).astype(np.float32)
        elif kind == 1:
            flow = (rng.standard_normal((h, w, 2)) * 8).astype(np.float32).round()      # many exact ties
        elif kind == 2:
            flow = np.full((h, w, 2), np.float32(rng.uniform(-2, 2)), np.float32)       # zero divergence everywhere
        else:   # the left half repeated on the right: every interior maximum exists twice, the first in C order wins
            flow = rng.standard_normal((h, w, 2)).astype(np.float32)
            flow[:, w // 2: 2 * (w // 2)] = flow[:, : w // 2]
        x, y, v = ctx.max_divergence(flow)
        rx, ry, rv = mo.max_divergence(flow)
        assert (x, y) == (int(rx), int(ry)), (case, w, h, (x, y), (rx, ry))
        assert np.float32(v) == np.float32(rv), (case, v, rv)
        mm = ctx.mean_magnitude(flow) if hasattr(ctx, "mean_magnitude") else None
        if mm is not None:
            ref_mm = mo.mean_magnitude(flow)
            assert abs(mm - ref_mm) <= 1e-6 * max(1.0, abs(ref_mm)), (case, mm, ref_mm)
        centres = [[float(rng.integers(0, w)), float(rng.integers(0, h))], [rng.uniform(0, w - 1), rng.uniform(0, h - 1)],
                   [0.0, 0.0], [float(w - 1), float(h - 1)], [-3.5, h + 2.25], [w / 2, h - 1]]
        for c in centres:
            for pov in (False, True):
                got = ctx.radial_motion(flow, c, False, pov)
                ref = mo.radial_motion_weighted(flow, c, False, pov)
                assert abs(got - ref) <= 1e-6 * max(1.0, abs(ref)) + 1e-9, (case, w, h, c, pov, got, ref)


def check_golden_pairs(ctx, golden_dir, names=("a", "b", "c")):
    """precompute_flow_info() outputs recorded from the reference (cv2 Farneback + NumPy)."""
    g = np.load(os.path.join(golden_dir, "pairs.npz"))
    api.set_context(ctx)
    for name in names:
        p0, p1, flow = g[f"{name}_p0"], g[f"{name}_p1"], g[f"{name}_flow"]
        info = api.precompute_flow_info(p0, p1, {"backend": "CUDA"})
        assert set(info) == {"flow", "pos_center", "neg_center", "val_pos", "val_neg", "cut", "cut_center", "mean_mag"}
        assert_flow_close(info["flow"], flow, f"golden pair {name}")
        assert_argmax(info["pos_center"], info["val_pos"], flow, f"golden pair {name}")
        assert info["cut"] == bool(g[f"{name}_cut"])
        assert abs(float(info["mean_mag"]) - float(g[f"{name}_mean_mag"])) <= MEAN_MAG_RTOL * float(g[f"{name}_mean_mag"]) + MEAN_MAG_ATOL
        pov = api.precompute_flow_info(p0, p1, {"pov_mode": True})
        assert tuple(pov["pos_center"]) == tuple(int(v) for v in g[f"{name}_pov_center"]) and pov["val_pos"] == 0


def check_golden_bracket(ctx, golden_dir, batch_frames=5):
    """A 28-frame bracket with one hard cut: per-pair centres, cut flags and scalars recorded from
    the reference's functions driven like F:1188-1242."""
    g = np.load(os.path.join(golden_dir, "bracket.npz"))
    frames = g["frames"]
    params = {"cut_threshold": float(g["cut_threshold"]), "pov_mode": False}
    r = api.process_bracket(frames, params, ctx=ctx, batch_frames=batch_frames, return_flows=True)
    n = len(frames) - 1
    assert r["n_pairs"] == n
    assert np.array_equal(r["cut"], g["cut"]), "scene-cut flags differ"
    assert np.allclose(r["mean_mag"], g["mean_mag"], rtol=MEAN_MAG_RTOL, atol=MEAN_MAG_ATOL)
    import cv2
    guarded = 0
    for j in range(n):
        flow = cv2.calcOpticalFlowFarneback(frames[j], frames[j + 1], None, 0.5, 3, 15, 3, 5, 1.2, 0)
        gap = assert_argmax((r["cx"][j], r["cy"][j]), r["val"][j], flow, f"pair {j}")
        guarded += gap < ARGMAX_MARGIN
        # scalar parity with the *device's* smoothed centre against the oracle formula on cv2's flow
        ref_local = mo.radial_motion_weighted(flow, r["centers"][j], bool(g["cut"][j]))
        assert abs(r["scalar"][j] - ref_local) <= SCALAR_RTOL * abs(ref_local) + scalar_tol(flow, r["centers"][j]), j
    # The generating script asserted that every pair of this clip has an argmax margin >= 3e-4 in the reference and
    # that cv2 and the NumPy restatement agree on every centre, so nothing here is conditional: raw centres, smoothed
    # centres (A5, F:1201-1214) and scalars must equal what the reference's functions produced.
    print(f"golden bracket: {guarded} of {n} pairs fell under the {ARGMAX_MARGIN:g} argmax margin guard "
          f"(smallest recorded margin {float(g['argmax_gap'].min()):.2e})")
    assert guarded == 0, "the golden clip lost its argmax margin"
    assert np.array_equal(np.stack([r["cx"], r["cy"]], 1), g["centers_raw"]), "raw centres differ from the reference's"
    assert np.array_equal(r["centers"], mo.smooth_centers(np.stack([r["cx"], r["cy"]], 1))), "A5: smoothed centres differ from the oracle"
    assert np.allclose(r["centers"], g["centers"], rtol=0, atol=1e-12)
    assert np.allclose(r["scalar"], g["scalar"], rtol=SCALAR_RTOL, atol=1e-6)
    return r


def check_bracket_vs_oracle(ctx, clip, params=None, batch_frames=8, min_clear=None, what="bracket"):
    """A bracket against the oracle driven like F:1188-1242 on cv2 flows: cut flags, margin-guarded raw centres,
    A5 (the device's smoothed centres equal oracle.motion_np.smooth_centers of the device's raw centres --
    unconditionally), scalars with the device's centre against the oracle formula, and -- for every pair whose whole
    +-6 window has clear argmax margins -- the scalar the oracle's own bracket loop produced.  Prints how many pairs
    the margin guard covered; fails if fewer than `min_clear` pairs were compared without the guard."""
    params = params or {}
    vals, cuts, infos = mo.process_bracket(list(clip), params)
    r = api.process_bracket(clip, params, ctx=ctx, batch_frames=batch_frames, return_flows=True)
    n = len(infos)
    assert r["n_pairs"] == n and np.array_equal(r["cut"], cuts), f"{what}: scene-cut flags differ"
    gaps = np.zeros(n)
    for j, info in enumerate(infos):
        if j >= r["flow_first"]:
            assert_flow_close(r["flows"][j - r["flow_first"]], info["flow"], f"{what} pair {j}")
        gaps[j] = assert_argmax((r["cx"][j], r["cy"][j]), r["val"][j], info["flow"], f"{what} pair {j}")
        ref = mo.radial_motion_weighted(info["flow"], r["centers"][j], info["cut"], bool(params.get("pov_mode", False)))
        assert abs(r["scalar"][j] - ref) <= SCALAR_RTOL * abs(ref) + scalar_tol(info["flow"], r["centers"][j]), (what, j)
    raw = np.stack([r["cx"], r["cy"]], 1)
    assert np.array_equal(r["centers"], mo.smooth_centers(raw)), f"{what}: A5 smoothed centres differ from the oracle"
    clear = gaps >= ARGMAX_MARGIN
    window_clear = np.array([clear[max(0, j - 6):j + 7].all() for j in range(n)])
    ref_raw = np.array([i["pos_center"] for i in infos])
    assert np.array_equal(raw[clear], ref_raw[clear]), f"{what}: raw centres differ where the margin is clear"
    for j in np.flatnonzero(window_clear):
        assert abs(r["scalar"][j] - vals[j]) <= SCALAR_RTOL * abs(vals[j]) + scalar_tol(infos[j]["flow"], r["centers"][j]), (what, j)
    print(f"{what}: {int((~clear).sum())} of {n} pairs under the argmax margin guard; {int(window_clear.sum())} scalars compared "
          f"with the oracle's own bracket loop")
    need = n // 2 if min_clear is None else min_clear
    assert int(clear.sum()) >= need, f"{what}: only {int(clear.sum())} pairs with a clear argmax margin (need {need})"
    return r, vals, cuts


def check_batch_independence(ctx, width, height, n_frames=14, seed=9):
    """Size-independent property: the per-pair results do not depend on how frames are batched or
    pushed (same kernels, per-pair reductions) -> bit-identical."""
    clip = make_clip(width, height, n_frames, seed=seed, period=11.0, amplitude=0.3)
    a = api.process_bracket(clip, {}, ctx=ctx, batch_frames=n_frames)
    b = api.process_bracket(clip, {}, ctx=ctx, batch_frames=3)
    for k in ("scalar", "cut", "cx", "cy", "val", "mean_mag", "centers"):
        assert np.array_equal(a[k], b[k]), k
    # pushing in ragged pieces
    ctx.configure(width, height, 4, n_frames)
    ctx.bracket_begin(False, 7.0)
    ctx.bracket_push(clip[:1]); ctx.bracket_push(clip[1:6]); ctx.bracket_push(clip[6:7]); ctx.bracket_push(clip[7:])
    c = ctx.bracket_finish()
    for k in ("scalar", "cx", "cy", "val", "mean_mag"):
        assert np.array_equal(a[k], c[k]), k
    return a


def check_edge_brackets(ctx, width=96, height=64):
    """Empty and ragged inputs: 0 / 1 frame -> no pairs; 2 frames -> one pair; identical frames -> zero flow."""
    clip = make_clip(width, height, 3, seed=2)
    ctx.configure(width, height, 4, 8)
    ctx.bracket_begin(False, 7.0)
    assert ctx.bracket_finish()["n_pairs"] == 0
    ctx.bracket_begin(False, 7.0)
    ctx.bracket_push(clip[:1])
    assert ctx.bracket_finish()["n_pairs"] == 0
    still = np.stack([clip[0], clip[0]])
    r = api.process_bracket(still, {}, ctx=ctx, return_flows=True)
    assert r["n_pairs"] == 1 and not r["cut"][0]
    # identical frames do NOT give exactly zero flow in the reference either: the last row/column
    # takes step 6's out-of-bounds fallback.  Parity, not zero, is the requirement.
    import cv2
    ref = cv2.calcOpticalFlowFarneback(clip[0], clip[0], None, 0.5, 3, 15, 3, 5, 1.2, 0)
    assert np.abs(r["flows"][0] - ref).max() < 1e-4 and np.abs(np.median(r["flows"][0])) < 1e-6
    # POV mode: fixed centre, unweighted mean (F:880-882, F:776-777)
    r = api.process_bracket(clip, {"pov_mode": True}, ctx=ctx, return_flows=True)
    assert list(r["cx"]) == [width // 2] * 2 and list(r["cy"]) == [height - 1] * 2 and not r["val"].any()
    for j in range(2):
        ref = mo.radial_motion_weighted(r["flows"][j], r["centers"][j], False, True)
        assert abs(r["scalar"][j] - ref) <= SCALAR_RTOL * abs(ref) + 1e-6


def check_postproc_golden(golden_dir):
    data = json.load(open(os.path.join(golden_dir, "postproc.json")))
    for case in data["cases"]:
        got = postproc.scalars_to_actions(case["values"], case["cuts"], case["frame_indices"], case["fps"], case["params"])
        assert got == case["actions"]
        ffl = list(zip(case["values"], case["cuts"], case["frame_indices"]))
        assert mo.postprocess(ffl, case["fps"], case["params"]) == case["actions"]


def check_preprocess(ctx, sizes=((360, 640), (300, 200), (256, 256))):
    """Row N2: BGR frame -> 256x256 gray on the device, bit-exact with the oracle (and so with cv2)."""
    from oracle import preproc_np as pp
    rng = np.random.default_rng(3)
    for (h, w) in sizes:
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        for vr in (False, True):
            assert np.array_equal(ctx.stage_preprocess(img, vr), pp.frame_to_gray(img, vr)), (h, w, vr)


WINDOW_PLANS = (   # (src h, src w, target (w, h), window (x, y, w, h))
    (120, 160, (160, 120), (0, 0, 160, 120)),        # native resolution: no resampling
    (120, 160, (160, 120), (0, 60, 80, 60)),         # native VR, left eye, lower half
    (120, 160, (160, 120), (80, 60, 80, 60)),        # native VR, right eye
    (200, 300, (512, 512), (256, 256, 256, 256)),    # reference VR geometry, right eye
    (97, 131, (200, 90), (13, 7, 150, 70)),          # arbitrary target and window
    (90, 70, (333, 77), (300, 0, 33, 77)),           # window touching the right edge, odd sizes
)


def check_preprocess_window(ctx, plans=WINDOW_PLANS):
    """Row N4: the windowed pre-processing (any resize target, any kept window) is bit-exact with the
    oracle; the identity target returns the plain gray conversion of the frame."""
    from oracle import preproc_np as pp
    rng = np.random.default_rng(5)
    for (h, w, target, window) in plans:
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        got = ctx.stage_preprocess_window(img, target, window)
        assert np.array_equal(got, pp.frame_window_to_gray(img, target, window)), (h, w, target, window)
        if target == (w, h):
            x, y, ww, hh = window
            assert np.array_equal(got, pp.rgb_to_gray(img[y:y + hh, x:x + ww, ::-1]))


def check_native_resolution_bracket(ctx, width=160, height=120, n=6, vr=False, eye="left"):
    """Colour frames pushed with a native-resolution plan give exactly the result of converting them on
    the host (oracle arithmetic) and pushing the gray window."""
    import cv2
    from funscript_flow_b200 import runner
    from oracle import preproc_np as pp
    clip = make_clip(width, height, n, seed=8)
    bgr = np.stack([cv2.cvtColor(f, cv2.COLOR_GRAY2BGR) for f in clip])
    bgr[..., 2] = (bgr[..., 2].astype(int) * 2 // 3).astype(np.uint8)
    target, window, cut_scale = runner.preprocess_plan(width, height, {"native_resolution": True, "vr_mode": vr, "vr_eye": eye})
    assert target == (width, height) and abs(cut_scale - np.sqrt(window[2] * window[3]) / 256.0) < 1e-12
    gray = np.stack([pp.frame_window_to_gray(f, target, window) for f in bgr])
    ra = api.process_bracket(gray, {"cut_threshold": 7.0 * cut_scale}, ctx=ctx, batch_frames=3)
    ctx.configure(window[2], window[3], 3, n - 1)
    ctx.preprocess_configure_window(width, height, target, window)
    ctx.bracket_begin(False, 7.0 * cut_scale)
    ctx.bracket_push_bgr(bgr)
    rb = ctx.bracket_finish()
    for k in ("scalar", "cut", "cx", "cy", "val", "mean_mag"):
        assert np.array_equal(ra[k], rb[k]), k


def check_bgr_push_equals_gray_push(ctx, width=320, height=200, n=7):
    """The fused upload path (colour frames -> device pre-processing -> hot path) gives exactly the
    result of pre-processing on the host and pushing gray frames."""
    import cv2
    from oracle import preproc_np as pp
    clip = make_clip(width, height, n, seed=4)
    bgr = np.stack([cv2.cvtColor(f, cv2.COLOR_GRAY2BGR) for f in clip])
    bgr[..., 0] = (bgr[..., 0].astype(int) * 3 // 4).astype(np.uint8)      # make the channels differ
    gray = np.stack([pp.frame_to_gray(f) for f in bgr])
    ra = api.process_bracket(gray, {}, ctx=ctx, batch_frames=3)
    ctx.configure(256, 256, 3, n - 1)
    ctx.preprocess_configure(width, height, False)
    ctx.bracket_begin(False, 7.0)
    ctx.bracket_push_bgr(bgr[:4])
    ctx.bracket_push_bgr(bgr[4:])
    rb = ctx.bracket_finish()
    for k in ("scalar", "cut", "cx", "cy", "val", "mean_mag"):
        assert np.array_equal(ra[k], rb[k]), k


# ---- records of the comparisons with the reference ----------------------------------------------
# The reference (FunscriptFlow.pyw) is not part of the repository.  Each record_* function runs one implementation of
# the reference's functions on the inputs of one test and returns what that test compares, in a form JSON stores
# exactly (Python floats round-trip, flow fields as SHA-256 of their float32 bytes).  tests/golden/reference_records.json
# holds the records (tests/golden/make_golden_reference_records.py); the tests compare the oracle and the product with
# them, and the reference's own functions too when oracle/ref_loader.py finds the file.

def flow_digest(flow):
    a = np.ascontiguousarray(flow, np.float32)
    return f"{a.shape[0]}x{a.shape[1]}x{a.shape[2]}:" + hashlib.sha256(a.tobytes()).hexdigest()


def record_pairs_and_postprocess(impl, postprocess):
    """precompute_flow_info / radial_motion_weighted on four pairs of a 128x96 clip, and one post-processed series.
    `postprocess(final_flow_list, fps, step, params) -> actions`."""
    clip = make_clip(128, 96, 10, seed=4, period=9.0, amplitude=0.3)
    pairs = []
    for j in range(4):
        info = impl.precompute_flow_info(clip[j], clip[j + 1], {"backend": "CPU"})
        pairs.append({"flow": flow_digest(info["flow"]), "pos_center": [int(v) for v in info["pos_center"]],
                      "val_pos": float(info["val_pos"]), "mean_mag": float(info["mean_mag"]), "cut": bool(info["cut"]),
                      "radial": [float(impl.radial_motion_weighted(info["flow"], c, False, pov))
                                 for c in ([40.5, 30.25], [64.0, 48.0]) for pov in (False, True)]})
    rng = np.random.default_rng(3)
    vals = rng.standard_normal(200).cumsum() * 0.1
    ffl = [(float(vals[i]), i == 77, i) for i in range(200)]
    prm = {"detrend_window": 1.5, "norm_window": 4, "keyframe_reduction": True}
    return {"pairs": pairs, "actions": postprocess(ffl, 30.0, 1, prm)}


def record_random_fields(impl):
    """max_divergence / radial_motion_weighted on the field families of check_reductions_random (ties, zero
    divergence, centres on and off the frame)."""
    rng = np.random.default_rng(123)
    out = []
    for case in range(30):
        w, h = int(rng.integers(2, 80)), int(rng.integers(2, 80))
        flow = rng.standard_normal((h, w, 2)).astype(np.float32)
        if case % 3 == 1:
            flow = (flow * 8).round()
        elif case % 3 == 2:
            flow[:] = np.float32(rng.uniform(-2, 2))
        x, y, v = impl.max_divergence(flow)
        centres = ([float(rng.integers(0, w)), float(rng.integers(0, h))], [rng.uniform(0, w), rng.uniform(0, h)], [-3.5, h + 2.25])
        out.append({"max_divergence": [int(x), int(y), float(np.float32(v))],
                    "radial": [float(impl.radial_motion_weighted(flow, c, False, pov)) for c in centres for pov in (False, True)],
                    "radial_cut": float(impl.radial_motion_weighted(flow, [1.0, 1.0], True, False))})
    return out


def random_postproc_cases():
    """60 random series (lengths 2..500, random cut positions incl. adjacent cuts and cuts at both ends, 24..120 fps
    containers, both keyframe modes, short and long windows): (vals, cuts, frame indices, fps, step, params)."""
    rng = np.random.default_rng(11)
    for case in range(60):
        n = int(rng.choice([2, 3, 4, 5, 7, 12, 40, 150, 500]))
        fps = float(rng.choice([23.976, 24.0, 25.0, 29.97, 30.0, 50.0, 59.94, 60.0, 120.0]))
        step = max(1, int(np.ceil(fps / 30.0)))
        kind = case % 3
        if kind == 0:
            vals = rng.standard_normal(n).cumsum() * 0.2
        elif kind == 1:
            vals = np.sin(np.arange(n) * rng.uniform(0.05, 0.9)) * rng.uniform(0.1, 6) + rng.standard_normal(n) * 0.05
        else:
            vals = np.zeros(n) if case % 2 else np.full(n, 0.37)          # flat series: the normalisation's degenerate case
        cuts = rng.random(n) < rng.choice([0.0, 0.02, 0.2])
        if n > 3 and case % 5 == 0:
            cuts[0] = cuts[-1] = True
            cuts[1] = True
        idx = [i * step for i in range(n)]
        prm = {"detrend_window": float(rng.choice([0.5, 1.5, 2.0, 5.0])), "norm_window": float(rng.choice([1.0, 3.0, 4.0, 10.0])),
               "keyframe_reduction": bool(case % 2)}
        yield vals, cuts, idx, fps, step, prm


def oracle_postprocess(final_flow_list, fps, step, params):
    return mo.postprocess(final_flow_list, fps, params)


def reference_postprocess(ref):
    """The reference's post-processing statements (oracle/ref_loader.postproc_function) in the form of oracle_postprocess."""
    from oracle import ref_loader
    pp = ref_loader.postproc_function(ref)
    return lambda final_flow_list, fps, step, params: pp(final_flow_list, fps, fps / step, params, lambda *_: None)


def record_random_postprocess(postprocess):
    """The actions of every random_postproc_cases() series; `postprocess(final_flow_list, fps, step, params)`."""
    return [postprocess([(float(v), bool(c), i) for v, c, i in zip(vals, cuts, idx)], fps, step, prm)
            for vals, cuts, idx, fps, step, prm in random_postproc_cases()]


def record_process_video_logs(process_video, tmp_dir):
    """The log lines of process_video on a 96x64 FFV1 clip, then of a second call that finds the output; the
    directory reads <dir>, the backend name and the elapsed time are dropped.  None without an FFV1 writer."""
    import cv2
    clip = make_clip(96, 64, 8, seed=12, period=5.0, amplitude=0.3)
    path = os.path.join(tmp_dir, "log.avi")
    vw = cv2.VideoWriter(path, cv2.VideoWriter_fourcc(*"FFV1"), 30.0, (96, 64), True)
    if not vw.isOpened():
        return None
    for f in clip:
        vw.write(cv2.cvtColor(f, cv2.COLOR_GRAY2BGR))
    vw.release()
    prm = {"threads": 1, "detrend_window": 2.0, "norm_window": 3.0, "batch_size": 3000, "overwrite": True, "vr_mode": False,
           "pov_mode": True, "keyframe_reduction": False, "backend": "CPU"}
    first, again = [], []
    err = bool(process_video(path, prm, first.append))
    process_video(path, dict(prm, overwrite=False), again.append)

    def shape(lines):
        out = []
        for ln in lines:
            for prefix in ("Using backend:", "Processing time:"):
                if ln.startswith(prefix):
                    ln = prefix
            out.append(ln.replace(tmp_dir, "<dir>"))
        return out
    return {"error_occurred": err, "lines": shape(first), "lines_when_output_exists": shape(again)}
