"""Farneback with caller-chosen parameters (pyr_scale, levels, winsize, iterations, poly_n, poly_sigma).

CPU part: the oracle's stage functions composed for any parameter set against cv2; the kernel sources (g++ emulation)
against cv2 and against the oracle stages; the parameter domain, the C ABI's set / get semantics, batching and
sharding invariance, the settings keys at every entry point and the CLI.  `-m gpu` part: the sm_100a library against
cv2 up to 4K, a bracket against the oracle, allocation and bit-identity of the reference parameters on the device."""
import os

import numpy as np
import pytest

import parity_checks as pc
from funscript_flow_b200 import _native, api, runner
from funscript_flow_b200.synth import make_clip
from oracle import farneback_np as fb
from oracle import motion_np as mo

REF = (0.5, 3, 15, 3, 5, 1.2)
# (pyr_scale, levels, winsize, iterations, poly_n, poly_sigma): every row of the parameter domain -- even winsize,
# winsize 3 and 63, poly_n 7, poly_sigma 0, pyr_scale 0.3 / 0.8, levels 0 and more than 4 levels, iterations 1 and 6
GRID = [
    (0.5, 3, 14, 3, 5, 1.2),
    (0.5, 3, 21, 3, 7, 1.5),
    (0.8, 6, 9, 1, 5, 0.0),
    (0.3, 2, 3, 6, 7, 1.1),
    (0.6, 0, 63, 2, 5, 1.2),
]
# the emulated kernels run the same rows on frames of ~100 px, where winsize 3 with 6 iterations is ill-conditioned
# (the float64 oracle itself puts 0.35 % of a 97 x 70 frame beyond 0.05 px of cv2): that row takes 2 iterations there
EMU_GRID = [p if p[2] != 3 else p[:3] + (2,) + p[4:] for p in GRID] + [REF]


def oracle_farneback(p0, p1, pyr_scale, levels, winsize, iterations, poly_n, poly_sigma):
    """calcOpticalFlowFarneback(p0, p1, None, ..., 0) composed from the oracle's stage functions."""
    flow = None
    h, w = p0.shape
    for lvl in fb.level_plan(w, h, levels, pyr_scale):
        R0 = fb.poly_exp(fb.pyramid_level(p0, lvl), poly_n, poly_sigma)
        R1 = fb.poly_exp(fb.pyramid_level(p1, lvl), poly_n, poly_sigma)
        if flow is None:
            flow = np.zeros((lvl["h"], lvl["w"], 2), np.float32)
        else:
            flow = fb.upsample_flow(flow, lvl["w"], lvl["h"], pyr_scale)
        for _ in range(iterations):
            flow = fb.blur_solve(fb.update_matrices(R0, R1, flow), winsize)
    return flow


def cv2_flow(p0, p1, prm):
    import cv2
    return cv2.calcOpticalFlowFarneback(p0, p1, None, *prm, 0)


def settings(prm):
    return {k: v for k, v in zip(api.FARNEBACK_SETTINGS, prm)}


def pair(width, height, seed=1):
    clip = make_clip(width, height, 4, seed=seed, period=12.0, amplitude=0.3)
    return clip[1], clip[2]


# ---- oracle ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("size", [(256, 256), (333, 217), (640, 360)])
@pytest.mark.parametrize("prm", GRID)
def test_oracle_vs_cv2(size, prm):
    p0, p1 = pair(*size)
    pc.assert_flow_close(oracle_farneback(p0, p1, *prm), cv2_flow(p0, p1, prm), f"oracle {size} {prm}")


def test_oracle_composition_is_the_reference_farneback():
    p0, p1 = pair(160, 120)
    assert np.array_equal(oracle_farneback(p0, p1, *REF), fb.farneback(p0, p1))


# ---- emulated kernels ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("size", [(160, 120), (97, 70)])
@pytest.mark.parametrize("prm", EMU_GRID)
def test_emu_farneback_vs_cv2(emu_ctx, size, prm):
    p0, p1 = pair(*size, seed=2)
    emu_ctx.set_farneback(*prm)
    pc.assert_flow_close(emu_ctx.farneback(p0, p1), cv2_flow(p0, p1, prm), f"emu {size} {prm}")


def test_emu_calc_optical_flow_farneback(emu_ctx):
    p0, p1 = pair(128, 96)
    prm = (0.6, 4, 11, 2, 7, 1.3)
    got = api.calc_optical_flow_farneback(p0, p1, None, *prm, 0, ctx=emu_ctx)
    assert got.dtype == np.float32 and got.shape == (96, 128, 2)
    pc.assert_flow_close(got, cv2_flow(p0, p1, prm), "cv2 signature")
    with pytest.raises(ValueError):
        api.calc_optical_flow_farneback(p0, p1, np.zeros((96, 128, 2), np.float32), *prm, 0, ctx=emu_ctx)
    with pytest.raises(_native.FFBError, match="OPTFLOW_FARNEBACK_GAUSSIAN"):
        api.calc_optical_flow_farneback(p0, p1, None, *prm, 256, ctx=emu_ctx)


def test_emu_stage_hooks(emu_ctx):
    """Large-radius pyramid, N = 7 expansion, box solve at winsize 9 / 14 / 21 and a 1 / pyr_scale up-sampling
    against the oracle stages."""
    clip = make_clip(400, 360, 3, seed=4, period=10.0, amplitude=0.3)
    p0, p1 = clip[1], clip[2]
    emu_ctx.set_farneback(0.3, 2, 15, 3, 5, 1.2)        # level 2: scale 0.09, ksize 25 (radius 12 > 9)
    plan = fb.level_plan(400, 360, 2, 0.3)
    assert [(l["w"], l["h"], l["ksize"]) for l in plan] == [(l["w"], l["h"], l["ksize"])
                                                            for l in _native.level_plan_ex(400, 360, 0.3, 2, emu_ctx.lib_path)]
    assert plan[0]["ksize"] // 2 > 9
    for lvl in plan:
        got = emu_ctx.stage_pyramid(p0, lvl["k"])
        ref = fb.pyramid_level(p0, lvl)
        assert got.shape == ref.shape and np.abs(got - ref).max() < 1e-3, (lvl, np.abs(got - ref).max())
    I0, I1 = fb.pyramid_level(p0, plan[1]), fb.pyramid_level(p1, plan[1])
    emu_ctx.set_farneback(0.5, 3, 15, 3, 7, 1.5)
    R0, R1 = fb.poly_exp(I0, 7, 1.5), fb.poly_exp(I1, 7, 1.5)
    got = emu_ctx.stage_polyexp(I0)
    assert np.abs(got - R0).max() < 2e-4 * max(1.0, np.abs(R0).max()), f"polyexp N=7 {np.abs(got - R0).max()}"
    rng = np.random.default_rng(5)
    h, w = I0.shape
    flow = (rng.standard_normal((h, w, 2)) * 1.5).astype(np.float32)
    for win in (9, 14, 21):
        emu_ctx.set_farneback(0.5, 3, win, 3, 7, 1.5)
        for f_in in (flow, None):
            M = fb.update_matrices(R0, R1, flow if f_in is not None else np.zeros_like(flow))
            got = emu_ctx.stage_flow_iter(R0, R1, f_in)
            assert np.abs(got - fb.blur_solve(M, win)).max() < 1e-4, (win, np.abs(got - fb.blur_solve(M, win)).max())
    emu_ctx.set_farneback(0.6, 3, 15, 3, 5, 1.2)
    fc = rng.standard_normal((30, 40, 2)).astype(np.float32)
    got = emu_ctx.stage_upsample_flow(fc, 67, 50)
    assert np.abs(got - fb.upsample_flow(fc, 67, 50, 0.6)).max() < 1e-5
    emu_ctx.set_farneback(*REF)


# ---- parameter domain and the set / get contract -------------------------------------------------------------------
BAD = [
    dict(pyr_scale=0.0), dict(pyr_scale=1.0), dict(pyr_scale=float("nan")), dict(levels=-1), dict(winsize=2),
    dict(winsize=64), dict(iterations=0), dict(iterations=21), dict(poly_n=6), dict(poly_n=3), dict(poly_sigma=-0.1),
    dict(poly_sigma=float("inf")), dict(flags=4), dict(flags=256), dict(flags=1),
    dict(pyr_scale=0.99, levels=100),       # a plan of more than 16 levels at 120 x 96
]


def test_domain_refused(emu_lib):
    ctx = _native.FlowContext(0, emu_lib)
    try:
        good = (0.6, 4, 11, 2, 7, 1.3)
        ctx.set_farneback(*good)
        ctx.configure(120, 96, 4, 8)
        before = (ctx.farneback_params, ctx.geometry, ctx.alloc_counts())
        for bad in BAD:
            kw = dict(zip(("pyr_scale", "levels", "winsize", "iterations", "poly_n", "poly_sigma"), good), **bad)
            with pytest.raises(_native.FFBError):
                ctx.set_farneback(**kw)
            assert (ctx.farneback_params, ctx.geometry, ctx.alloc_counts()) == before, bad
        with pytest.raises(_native.FFBError):
            _native.level_plan_ex(120, 96, 0.99, 100, emu_lib)
        # equal parameters: nothing allocated
        ctx.set_farneback(*good)
        assert ctx.alloc_counts() == before[2]
        # refused inside a bracket, the bracket stays usable
        ctx.bracket_begin(False, 7.0)
        with pytest.raises(_native.FFBError, match="inside a bracket"):
            ctx.set_farneback(*REF)
        ctx.bracket_abort()
        assert ctx.farneback_params == before[0]
        ctx.set_farneback(*REF)
        assert ctx.farneback_params == dict(zip(("pyr_scale", "levels", "winsize", "iterations", "poly_n", "poly_sigma"), REF),
                                            flags=0)
        assert ctx.geometry == before[1]
    finally:
        ctx.close()


def test_level_plan_ex_matches_oracle(emu_lib):
    for (w, h, s, lv) in [(256, 256, 0.5, 3), (1920, 1080, 0.5, 5), (333, 217, 0.8, 6), (640, 360, 0.3, 3), (100, 40, 0.5, 3)]:
        got = _native.level_plan_ex(w, h, s, lv, emu_lib)
        ref = fb.level_plan(w, h, lv, s)
        assert [(g["k"], g["w"], g["h"], g["ksize"]) for g in got] == [(r["k"], r["w"], r["h"], r["ksize"]) for r in ref]
        assert np.allclose([g["sigma"] for g in got], [r["sigma"] for r in ref], rtol=0, atol=0)
    # the 4-entry reference contract of ffb_level_plan is unchanged
    assert _native.level_plan(1920, 1080, emu_lib) == [{k: v for k, v in g.items() if k != "k"}
                                                      for g in _native.level_plan_ex(1920, 1080, 0.5, 3, emu_lib)]


def test_reference_parameters_set_explicitly_are_identical(emu_lib):
    """A context switched to other parameters and back computes the same bits with the same launches as a new one."""
    clip = make_clip(112, 80, 7, seed=8, period=9.0, amplitude=0.3)
    a, b = _native.FlowContext(0, emu_lib), _native.FlowContext(0, emu_lib)
    try:
        ra = api.process_bracket(clip, {}, ctx=a, batch_frames=4, return_flows=True)
        b.set_farneback(0.6, 5, 21, 2, 7, 1.5)
        api.process_bracket(clip, {}, ctx=b, batch_frames=4)     # no flow_* keys: back to the reference's
        assert b.farneback_params["winsize"] == 15
        a.profile_reset(); b.profile_reset()
        ra = api.process_bracket(clip, {}, ctx=a, batch_frames=4, return_flows=True)
        rb = api.process_bracket(clip, {}, ctx=b, batch_frames=4, return_flows=True)
        for k in ("scalar", "cut", "cx", "cy", "val", "mean_mag", "centers", "flows"):
            assert np.array_equal(ra[k], rb[k]), k
        assert a.kernel_stats() == b.kernel_stats()
        assert a.flow_iter_level_stats() == b.flow_iter_level_stats()
    finally:
        a.close(); b.close()


def test_non_default_batching_and_sharding(emu_lib):
    """A non-default set is bit-identical across batch sizes and across 1 vs 3 frame-range shards."""
    clip = make_clip(96, 72, 10, seed=9, period=11.0, amplitude=0.3)
    prm = settings((0.6, 4, 9, 2, 7, 1.4))
    ctxs = [_native.FlowContext(0, emu_lib) for _ in range(3)]
    try:
        a = api.process_bracket(clip, prm, ctx=ctxs[0], batch_frames=10)
        b = api.process_bracket(clip, prm, ctx=ctxs[0], batch_frames=3)
        one = api.process_bracket_on_contexts(clip, prm, ctxs[:1], batch_frames=4)
        three = api.process_bracket_on_contexts(clip, prm, ctxs, batch_frames=2)
        for k in ("scalar", "cut", "cx", "cy", "val", "mean_mag", "centers"):
            assert np.array_equal(a[k], b[k]) and np.array_equal(a[k], one[k]) and np.array_equal(a[k], three[k]), k
        assert all(c.farneback_params["winsize"] == 9 for c in ctxs)
        ref = api.process_bracket(clip, {}, ctx=ctxs[1], batch_frames=10)
        assert not np.array_equal(a["scalar"], ref["scalar"])     # the parameters did reach the kernels
    finally:
        for c in ctxs:
            c.close()


def test_settings_reach_every_entry_point(emu_ctx, tmp_path):
    api.set_context(emu_ctx)
    clip = make_clip(96, 64, 9, seed=6, period=7.0, amplitude=0.3)
    prm = {"batch_size": 4, "detrend_window": 2.0, "norm_window": 3.0, "keyframe_reduction": False, "flow_winsize": 21,
           "flow_poly_n": 7}
    want = dict(api.REFERENCE_FARNEBACK, winsize=21, poly_n=7)
    assert api.farneback_params(prm) == want and api.farneback_params({}) == api.REFERENCE_FARNEBACK
    # the series of process_frames (brackets pipelined over two contexts) = brackets of flows made with those parameters
    _, series = runner.process_frames(clip, 30.0, prm, ctx=emu_ctx, return_series=True)
    direct = []
    for a in range(0, 9, 4):
        if 9 - a >= 2:
            direct.extend(api.process_bracket(clip[a:a + 4], prm, ctx=emu_ctx)["scalar"].tolist())
    assert series["values"].tolist() == direct
    ref_series = runner.process_frames(clip, 30.0, dict(prm, flow_winsize=None, flow_poly_n=None), ctx=emu_ctx,
                                       return_series=True)[1]
    assert ref_series["values"].tolist() != direct
    # the drop-in shares the context: a reference-parameter call returns the reference result after a non-default one
    p0, p1 = clip[2], clip[3]
    ref = api.precompute_flow_info(p0, p1, {})["flow"]
    got = api.precompute_flow_info(p0, p1, {"flow_winsize": 21})["flow"]
    pc.assert_flow_close(got, cv2_flow(p0, p1, (0.5, 3, 21, 3, 5, 1.2)), "precompute_flow_info winsize 21")
    assert np.array_equal(api.precompute_flow_info(p0, p1, {})["flow"], ref)
    # process_video_series: both eyes' contexts take the parameters
    import cv2
    path = str(tmp_path / "tiny.avi")
    vw = cv2.VideoWriter(path, cv2.VideoWriter_fourcc(*"FFV1"), 30.0, (96, 64), True)
    if not vw.isOpened():
        pytest.skip("FFV1 writer unavailable")
    for f in clip:
        vw.write(cv2.cvtColor(f, cv2.COLOR_GRAY2BGR))
    vw.release()
    vprm = dict(prm, batch_size=3000, native_resolution=True, gpu_batch_frames=4, overwrite=True, vr_mode=False)
    res = runner.process_video_series(path, vprm, ctx=emu_ctx)
    direct = api.process_bracket(clip, dict(prm, cut_threshold=7.0 * np.sqrt(96 * 64) / 256.0), ctx=emu_ctx, batch_frames=4)
    assert res[0] == direct["scalar"].tolist()
    runner.process_video_series(path, dict(vprm, vr_mode=True, vr_eye="both"), ctx=emu_ctx)
    assert api.get_aux_context(emu_ctx).farneback_params["winsize"] == 21
    emu_ctx.set_farneback(*REF)


def test_cli_options():
    from funscript_flow_b200 import __main__ as cli
    default = cli.settings_from_args(cli.build_parser().parse_args(["x.mp4"]))
    assert default == {"threads": 8, "detrend_window": 2.0, "norm_window": 3.0, "batch_size": 3000, "overwrite": False,
                       "vr_mode": False, "pov_mode": False, "keyframe_reduction": False, "backend": "CUDA"}
    args = cli.build_parser().parse_args(["x.mp4", "--flow_winsize", "21", "--flow_poly_n", "7", "--flow_levels", "5",
                                          "--flow_pyr_scale", "0.5", "--flow_iterations", "4", "--flow_poly_sigma", "1.5"])
    s = cli.settings_from_args(args)
    assert {k: v for k, v in s.items() if k.startswith("flow_")} == {"flow_winsize": 21, "flow_poly_n": 7, "flow_levels": 5,
                                                                      "flow_iterations": 4, "flow_poly_sigma": 1.5}
    assert api.farneback_params(s) == dict(pyr_scale=0.5, levels=5, winsize=21, iterations=4, poly_n=7, poly_sigma=1.5)
    with pytest.raises(SystemExit):
        cli.build_parser().parse_args(["x.mp4", "--flow_poly_n", "6"])


# ---- GPU -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("size", [(256, 256), (640, 360), (1920, 1080)])
@pytest.mark.parametrize("prm", GRID)
def test_gpu_farneback_vs_cv2(gpu_ctx, size, prm):
    p0, p1 = pair(*size)
    gpu_ctx.set_farneback(*prm)
    try:
        pc.assert_flow_close(gpu_ctx.farneback(p0, p1), cv2_flow(p0, p1, prm), f"gpu {size} {prm}")
    finally:
        gpu_ctx.set_farneback(*REF)


@pytest.mark.gpu
def test_gpu_deep_plan_4k(gpu_ctx):
    """levels 5 at 3840 x 2160: levels 4 and 5 take the large-radius pyramid (ksize 39 and 79)."""
    prm = (0.5, 5, 21, 3, 5, 1.2)
    assert len(_native.level_plan_ex(3840, 2160, 0.5, 5)) == 6
    p0, p1 = pair(3840, 2160)
    gpu_ctx.set_farneback(*prm)
    try:
        pc.assert_flow_close(gpu_ctx.farneback(p0, p1), cv2_flow(p0, p1, prm), "gpu 4K levels 5")
    finally:
        gpu_ctx.set_farneback(*REF)


@pytest.mark.gpu
def test_gpu_bracket_vs_oracle(gpu_ctx):
    """Bracket scalars, centres and cut flags with a non-default set against the oracle's bracket loop on the
    composed oracle's flows, under the argmax-margin guard of parity_checks.check_bracket_vs_oracle."""
    prm_t = (0.6, 4, 21, 2, 7, 1.5)
    params = settings(prm_t)
    clip = make_clip(256, 256, 14, seed=21, period=9.0, amplitude=0.35)
    vals, cuts, infos = mo.process_bracket(list(clip), {}, flow_fn=lambda a, b: oracle_farneback(a, b, *prm_t))
    r = api.process_bracket(clip, params, ctx=gpu_ctx, batch_frames=5, return_flows=True)
    gpu_ctx.set_farneback(*REF)
    n = len(infos)
    assert r["n_pairs"] == n and np.array_equal(r["cut"], cuts)
    gaps = np.zeros(n)
    for j, info in enumerate(infos):
        if j >= r["flow_first"]:
            pc.assert_flow_close(r["flows"][j - r["flow_first"]], info["flow"], f"pair {j}")
        gaps[j] = pc.assert_argmax((r["cx"][j], r["cy"][j]), r["val"][j], info["flow"], f"pair {j}")
        ref = mo.radial_motion_weighted(info["flow"], r["centers"][j], info["cut"], False)
        assert abs(r["scalar"][j] - ref) <= pc.SCALAR_RTOL * abs(ref) + pc.scalar_tol(info["flow"], r["centers"][j]), j
    raw = np.stack([r["cx"], r["cy"]], 1)
    assert np.array_equal(r["centers"], mo.smooth_centers(raw))
    clear = gaps >= pc.ARGMAX_MARGIN
    ref_raw = np.array([i["pos_center"] for i in infos])
    assert np.array_equal(raw[clear], ref_raw[clear])
    for j in range(n):
        if clear[max(0, j - 6):j + 7].all():
            assert abs(r["scalar"][j] - vals[j]) <= pc.SCALAR_RTOL * abs(vals[j]) + pc.scalar_tol(infos[j]["flow"], r["centers"][j]), j
    assert int(clear.sum()) >= n // 2


@pytest.mark.gpu
def test_gpu_no_allocation_after_first_bracket(gpu_ctx):
    params = settings((0.5, 5, 21, 3, 7, 1.5))
    clip = make_clip(640, 360, 9, seed=3)
    api.process_bracket(clip, params, ctx=gpu_ctx, batch_frames=4)
    before = gpu_ctx.alloc_counts()
    for _ in range(2):
        api.process_bracket(clip, params, ctx=gpu_ctx, batch_frames=4)
    assert gpu_ctx.alloc_counts() == before
    gpu_ctx.set_farneback(*REF)


@pytest.mark.gpu
def test_gpu_reference_parameters_bit_identical():
    clip = make_clip(1920, 1080, 6, seed=5)
    a, b = _native.FlowContext(0), _native.FlowContext(0)
    try:
        ra = api.process_bracket(clip, {}, ctx=a, batch_frames=3, return_flows=True)
        b.set_farneback(0.6, 5, 21, 2, 7, 1.5)
        b.set_farneback(*REF)
        b.profile_reset()
        a.profile_reset()
        ra = api.process_bracket(clip, {}, ctx=a, batch_frames=3, return_flows=True)
        rb = api.process_bracket(clip, {}, ctx=b, batch_frames=3, return_flows=True)
        for k in ("scalar", "cut", "cx", "cy", "val", "mean_mag", "centers", "flows"):
            assert np.array_equal(ra[k], rb[k]), k
        assert {k: v["launches"] for k, v in a.kernel_stats().items()} == {k: v["launches"] for k, v in b.kernel_stats().items()}
    finally:
        a.close(); b.close()
