"""Backward flows and a forward-backward consistency mask along a sequence of frames, each frame expanded once
(ffb_farneback_sequence_bidir, ffb_stage_fb_check, FlowContext.farneback_sequence_bidir / stage_fb_check,
api.calc_optical_flow_farneback_sequence_bidirectional).

CPU part (emulated kernels): forward flows bit-identical to the sequence call, backward flows bit-identical to the
per-pair call on the reversed pair, masks and counts equal to the NumPy float32 restatement of the check below, for
three parameter sets while the rings wrap; invariance to the batch size (the host-input ramp included); every forced
k_flow_iter variant; the check on hand-built flows (edges, NaN, alpha = beta = 0, a huge beta); each output alone,
pitched / strided outputs, refusals, nothing to do, no allocation on a repeated call, bracket bits around a call; the
cv2-order function against cv2.  `-m gpu` part: the sm_100a library against cv2 at three sizes, bit-identity and exact
masks at 1080p with a small batch into device, pinned and pageable buffers, torch tensors on a non-default stream, no
allocation after the first 1080p call, and the sequence call unchanged around a bidirectional call."""

import numpy as np
import pytest

import parity_checks as pc
from funscript_flow_b200 import _native, api
from funscript_flow_b200.synth import make_clip

REF = (0.5, 3, 15, 3, 5, 1.2)
UNFUSED = (0.6, 4, 21, 2, 7, 1.5)          # winsize 21: k_flow_matrices + k_box_solve
NO_FUSED_UP = (0.8, 3, 15, 3, 5, 1.2)      # winsize 15, pyr_scale 0.8: k_flow_iter with a separate k_upsample_flow
ALPHA, BETA = 0.01, 0.5


def np_check(fw, bw, alpha=ALPHA, beta=BETA):
    """The forward-backward check of one pair in float32, one rounding per operation in the kernel's order:
    (mask bool [h, w], count)."""
    f32 = np.float32
    fw = np.asarray(fw, f32)
    bw = np.asarray(bw, f32)
    h, w = fw.shape[:2]
    ys, xs = np.mgrid[0:h, 0:w].astype(f32)
    fx, fy = fw[..., 0], fw[..., 1]
    with np.errstate(invalid="ignore", over="ignore"):
        tx, ty = xs + fx, ys + fy
        inside = (tx >= 0) & (tx <= f32(w - 1)) & (ty >= 0) & (ty <= f32(h - 1))
        tx, ty = np.where(inside, tx, f32(0)), np.where(inside, ty, f32(0))
        x0f, y0f = np.floor(tx), np.floor(ty)
        x0, y0 = x0f.astype(np.int64), y0f.astype(np.int64)
        x1, y1 = np.minimum(x0 + 1, w - 1), np.minimum(y0 + 1, h - 1)
        ax, ay = tx - x0f, ty - y0f
        rx, ry = f32(1) - ax, f32(1) - ay
        b = [(bw[y0, x0, c] * rx + bw[y0, x1, c] * ax) * ry + (bw[y1, x0, c] * rx + bw[y1, x1, c] * ax) * ay for c in (0, 1)]
        ex, ey = fx + b[0], fy + b[1]
        e = ex * ex + ey * ey
        nf = fx * fx + fy * fy
        nb = b[0] * b[0] + b[1] * b[1]
        ok = inside & (e <= f32(alpha) * (nf + nb) + f32(beta))
    return ok, int(ok.sum())


def assert_check_matches(r, alpha=ALPHA, beta=BETA):
    for j in range(r["flow"].shape[0]):
        want, n = np_check(r["flow"][j], r["flow_bw"][j], alpha, beta)
        assert np.array_equal(r["mask"][j], want), j
        assert r["n_consistent"][j] == n, (j, r["n_consistent"][j], n)


def cv2_flow(p0, p1, prm):
    import cv2
    return cv2.calcOpticalFlowFarneback(p0, p1, None, *prm, 0)


def clip(width, height, n, seed=7):
    return np.ascontiguousarray(make_clip(width, height, n, seed=seed, period=9.0, amplitude=0.3))


@pytest.fixture
def ectx(emu_lib):
    """A fresh emulated context, installed as the drop-in functions' context for the duration of the test."""
    saved = dict(api._contexts)
    ctx = _native.FlowContext(0, emu_lib)
    api.set_context(ctx)
    yield ctx
    api._contexts.clear()
    api._contexts.update(saved)
    ctx.close()


# ---- CPU: emulated kernels -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("size", [(160, 120), (97, 70)])
@pytest.mark.parametrize("prm", [REF, UNFUSED, NO_FUSED_UP])
def test_bidir_equals_sequence_farneback_and_check(ectx, size, prm):
    frames = clip(*size, 25)
    ectx.set_farneback(*prm)
    ectx.configure(*size, 4, 24)       # 24 pairs in batches of at most 4 through rings of 16 slots
    r = ectx.farneback_sequence_bidir(frames)
    assert ectx.flow_ring_size == 16
    assert r["flow_bw"].shape == (24,) + frames.shape[1:] + (2,) and r["flow_bw"].dtype == np.float32
    assert r["mask"].shape == (24,) + frames.shape[1:] and r["mask"].dtype == np.bool_
    assert r["n_consistent"].shape == (24,) and r["n_consistent"].dtype == np.int64
    assert np.array_equal(r["flow"], ectx.farneback_sequence(frames)["flow"]), prm
    for j in range(24):
        assert np.array_equal(r["flow_bw"][j], ectx.farneback(frames[j + 1], frames[j])), (prm, j)
    assert_check_matches(r)
    assert 0 < r["n_consistent"].sum() < r["mask"].size     # the clip has pixels of both kinds


def test_batch_size_does_not_matter(ectx):
    frames = clip(96, 72, 25)
    out = []
    for batch in (4, 7, 64):         # 64: host input ramps up (17 frames, then 8)
        ectx.configure(96, 72, batch, 24)
        out.append(ectx.farneback_sequence_bidir(frames, alpha=0.02, beta=0.3))
    for r in out[1:]:
        for k in ("flow", "flow_bw", "mask", "n_consistent"):
            assert np.array_equal(r[k], out[0][k]), k
    assert_check_matches(out[0], 0.02, 0.3)


@pytest.mark.parametrize("variant", ["256x4x8", "128x2x4", "160x2x4", "96x2x4", "64x2x4"])
def test_every_forced_variant(emu_lib, variant, monkeypatch):
    monkeypatch.setenv("FFB_ITER_CFG", variant)
    ctx = _native.FlowContext(0, emu_lib)
    try:
        frames = clip(97, 70, 6)
        ctx.configure(97, 70, 2, 8)
        r = ctx.farneback_sequence_bidir(frames, mask=False, counts=False)
        for j in range(5):
            assert np.array_equal(r["flow_bw"][j], ctx.farneback(frames[j + 1], frames[j])), (variant, j)
    finally:
        ctx.close()


def test_each_frame_is_expanded_once(ectx):
    """The backward pass re-uses the forward pass's expansions: the same pyramid and expansion launches as the sequence
    call, twice its flow-iteration bytes, and one check launch per batch."""
    frames = clip(96, 72, 9)
    ectx.configure(96, 72, 4, 8)
    ectx.profile_reset()
    ectx.farneback_sequence(frames)
    seq = ectx.kernel_stats()
    ectx.profile_reset()
    ectx.farneback_sequence_bidir(frames)
    bid = ectx.kernel_stats()
    for k in ("pyramid", "polyexp"):
        assert bid[k] == seq[k], k
    for k in ("upsample", "flow_iter"):
        assert bid[k]["launches"] == 2 * seq[k]["launches"] and bid[k]["alg_bytes"] == 2 * seq[k]["alg_bytes"], k
    assert bid["fb_check"]["launches"] == 2 and bid["fb_check"]["alg_bytes"] == 8 * 96 * 72 * 17
    assert bid["divmag"]["launches"] == bid["radial"]["launches"] == bid["small"]["launches"] == 0
    ectx.profile_reset()
    ectx.farneback_sequence_bidir(frames, backward=False, mask=False, counts=False)
    assert ectx.kernel_stats() == seq                       # forward flows only: the sequence call's launches


def test_stage_fb_check_on_hand_built_flows(ectx):
    h, w = 37, 53
    rng = np.random.default_rng(3)
    ys, xs = np.mgrid[0:h, 0:w].astype(np.float32)
    cases = []
    # a pure translation: consistent where the target stays inside
    fw = np.zeros((h, w, 2), np.float32)
    fw[..., 0], fw[..., 1] = 2.5, -1.25
    cases.append((fw, -fw, ALPHA, BETA))
    # targets exactly on column w-1 and row h-1, and just below 0 (outside)
    fw = rng.normal(0, 0.3, (h, w, 2)).astype(np.float32)
    fw[:, ::3, 0] = np.float32(w - 1) - xs[:, ::3]
    fw[::4, :, 1] = np.float32(h - 1) - ys[::4, :]
    fw[1::5, :, 0] = -xs[1::5, :] - np.float32(1e-6)
    fw[:, 2::7, 1] = np.nextafter(-ys[:, 2::7], np.float32(-np.inf))
    bw = rng.normal(0, 0.5, (h, w, 2)).astype(np.float32)
    cases.append((fw, bw, ALPHA, BETA))
    # NaN in the forward flow (target undefined) and in the backward flow (sample undefined)
    fn, bn = fw.copy(), bw.copy()
    fn[5, 7, 0] = np.nan
    fn[9, :, 1] = np.nan
    bn[::2, ::2] = np.nan
    cases.append((fn, bn, ALPHA, BETA))
    # alpha = beta = 0: only exact cancellations pass (the translation's); a huge beta: every target inside passes
    cases.append((cases[0][0], cases[0][1], 0.0, 0.0))
    cases.append((fw, bw, 0.0, 0.0))
    cases.append((fw, bw * 50, ALPHA, 1e30))
    for i, (f, b, a, be) in enumerate(cases):
        got, n = ectx.stage_fb_check(f, b, a, be)
        want, m = np_check(f, b, a, be)
        assert np.array_equal(got, want), i
        assert n == m == int(got.sum()), (i, n, m)
    inside = np_check(cases[-1][0], cases[-1][1], ALPHA, 1e30)[0]
    with np.errstate(invalid="ignore"):
        tx, ty = xs + cases[-1][0][..., 0], ys + cases[-1][0][..., 1]
        assert np.array_equal(inside, (tx >= 0) & (tx <= w - 1) & (ty >= 0) & (ty <= h - 1))
    assert 0 < np_check(*cases[1])[1] < h * w and np_check(*cases[3])[1] > 0
    with pytest.raises(_native.FFBError, match="alpha"):
        ectx.stage_fb_check(fw, bw, -0.1, BETA)


def test_each_output_alone(ectx):
    frames = clip(97, 70, 9)
    ectx.configure(97, 70, 3, 8)
    full = ectx.farneback_sequence_bidir(frames)
    only_mask = ectx.farneback_sequence_bidir(frames, forward=False, backward=False, counts=False)
    assert only_mask["flow"] is None and only_mask["flow_bw"] is None and only_mask["n_consistent"] is None
    assert np.array_equal(only_mask["mask"], full["mask"])
    only_counts = ectx.farneback_sequence_bidir(frames, forward=False, backward=False, mask=False)
    assert np.array_equal(only_counts["n_consistent"], full["n_consistent"]) and only_counts["mask"] is None
    only_bw = ectx.farneback_sequence_bidir(frames, forward=False, mask=False, counts=False)
    assert np.array_equal(only_bw["flow_bw"], full["flow_bw"]) and only_bw["flow"] is None
    only_fw = ectx.farneback_sequence_bidir(frames, backward=False, mask=False, counts=False)
    assert np.array_equal(only_fw["flow"], full["flow"])


def test_pitched_and_strided_outputs(ectx):
    frames = clip(97, 70, 9)
    ectx.configure(97, 70, 3, 8)
    ref = ectx.farneback_sequence_bidir(frames)
    # frames inside wider rows with a gap between frames; flows and masks inside wider rows with a gap between pairs
    wide = np.zeros((9, 72, 128), np.uint8)
    wide[:, :70, 5:102] = frames
    fw = np.full((8, 73, 100, 2), np.nan, np.float32)
    bw = np.full((8, 73, 100, 2), np.nan, np.float32)
    mask = np.full((8, 72, 101), 7, np.uint8)
    cnt = ectx.farneback_sequence_bidir_ptr(wide.ctypes.data + 5, 9, 97, 70, 128, 72 * 128, fw.ctypes.data, bw.ctypes.data,
                                            100 * 8, 73 * 100 * 8, mask.ctypes.data, 101, 72 * 101, counts=True)
    assert np.array_equal(fw[:, :70, :97], ref["flow"]) and np.array_equal(bw[:, :70, :97], ref["flow_bw"])
    assert np.array_equal(mask[:, :70, :97], ref["mask"].view(np.uint8)) and np.array_equal(cnt, ref["n_consistent"])
    for a in (fw, bw):
        assert np.isnan(a[:, 70:]).all() and np.isnan(a[:, :, 97:]).all()
    assert (mask[:, 70:] == 7).all() and (mask[:, :, 97:] == 7).all()
    # evenly spaced rows: one copy per run of ring slots into larger preallocated arrays
    fw = np.full((10, 70, 97, 2), np.nan, np.float32)
    mask = np.full((10, 70, 97), 7, np.uint8)
    assert ectx.farneback_sequence_bidir_ptr(frames.ctypes.data, 9, 97, 70, 97, 97 * 70, fw[1:].ctypes.data, 0, 97 * 8,
                                             97 * 70 * 8, mask[1:].ctypes.data, 97, 97 * 70) is None
    assert np.array_equal(fw[1:9], ref["flow"]) and np.isnan(fw[0]).all() and np.isnan(fw[9]).all()
    assert np.array_equal(mask[1:9], ref["mask"].view(np.uint8)) and (mask[0] == 7).all() and (mask[9] == 7).all()


def test_refusals_leave_the_context_usable(ectx):
    frames = clip(97, 70, 6)
    before = api.process_bracket(frames, {}, ctx=ectx, batch_frames=3, return_flows=True)
    lib, h = ectx._lib, ectx._h
    p = frames.ctypes.data
    flow = np.empty((5, 70, 97, 2), np.float32)
    mask = np.empty((5, 70, 97), np.uint8)
    f, m = flow.ctypes.data, mask.ctypes.data
    fs, ms = 97 * 70 * 8, 97 * 70
    ok = (p, 6, 97, 70, 97, 97 * 70, None, f, 97 * 8, fs, m, 97, ms, ALPHA, BETA)
    bad = [
        dict(n=-1),                      # n_frames < 0
        dict(pitch=96),                  # pitch below the width
        dict(fstride=97 * 69),           # frames overlap
        dict(flow_pitch=97 * 8 - 1),     # flow_pitch below 8 * width (backward flow only)
        dict(flow_stride=97 * 69 * 8),   # flows overlap
        dict(mask_pitch=96),             # mask_pitch below the width
        dict(mask_stride=97 * 69),       # masks overlap
        dict(alpha=-0.01), dict(alpha=float("nan")), dict(beta=float("inf")), dict(beta=-1.0),
    ]
    keys = dict(n=1, pitch=4, fstride=5, flow_pitch=8, flow_stride=9, mask_pitch=11, mask_stride=12, alpha=13, beta=14)
    for change in bad:
        args = list(ok)
        for k, v in change.items():
            args[keys[k]] = v
        assert lib.ffb_farneback_sequence_bidir(h, *args, None, None) == -1, change
        assert b"ffb_farneback_sequence_bidir" in lib.ffb_last_error(h), change
    cnt = np.full(5, -7, np.int64)
    for n in (0, 1):          # nothing to do
        args = list(ok)
        args[1] = n
        assert lib.ffb_farneback_sequence_bidir(h, *args, cnt.ctypes.data_as(_native.C.POINTER(_native.C.c_int64)), None) == 0
    assert (cnt == -7).all()
    ectx.bracket_begin(False, 7.0)
    with pytest.raises(_native.FFBError, match="inside a bracket"):
        ectx.farneback_sequence_bidir(frames)
    with pytest.raises(_native.FFBError, match="inside a bracket"):
        api.calc_optical_flow_farneback_sequence_bidirectional(frames, None, *REF, 0, ctx=ectx)
    ectx.bracket_abort()
    r = ectx.farneback_sequence_bidir(frames)
    assert_check_matches(r)
    with pytest.raises(_native.FFBError):      # the call replaced the bracket's flows in the final-flow ring
        ectx.get_flow(0)
    after = api.process_bracket(frames, {}, ctx=ectx, batch_frames=3, return_flows=True)
    for k in ("scalar", "cut", "cx", "cy", "val", "mean_mag", "centers", "flows"):
        assert np.array_equal(before[k], after[k]), k


def test_allocation_only_when_needed_and_not_on_a_repeated_call(ectx):
    frames = clip(96, 72, 12)
    ectx.configure(96, 72, 4, 11)
    ectx.farneback_sequence(frames)
    base = ectx.alloc_counts()
    ectx.farneback_sequence_bidir(frames, backward=False, mask=False, counts=False)
    assert ectx.alloc_counts() == base                     # forward flows only: the sequence's buffers
    ectx.farneback_sequence_bidir(frames)
    grown = ectx.alloc_counts()
    assert grown[0] == base[0] + 3 and grown[1] == base[1]   # backward ring, mask ring, counts
    ectx.farneback_sequence_bidir(frames)
    ectx.farneback_sequence_bidir(frames[:5], forward=False)
    ectx.farneback_sequence_bidir(frames, mask=False)
    ectx.farneback_sequence(frames)
    assert ectx.alloc_counts() == grown


def test_calc_optical_flow_farneback_sequence_bidirectional(ectx):
    frames = clip(128, 96, 5, seed=3)
    prm = (0.6, 4, 11, 2, 7, 1.3)
    fw, bw, mask = api.calc_optical_flow_farneback_sequence_bidirectional(frames, None, *prm, 0, ctx=ectx)
    for a in (fw, bw):
        assert isinstance(a, np.ndarray) and a.dtype == np.float32 and a.shape == (4, 96, 128, 2)
    assert isinstance(mask, np.ndarray) and mask.dtype == np.bool_ and mask.shape == (4, 96, 128)
    assert np.array_equal(fw, api.calc_optical_flow_farneback_sequence(frames, None, *prm, 0, ctx=ectx))
    for j in range(4):
        pc.assert_flow_close(fw[j], cv2_flow(frames[j], frames[j + 1], prm), f"forward pair {j}")
        pc.assert_flow_close(bw[j], cv2_flow(frames[j + 1], frames[j], prm), f"backward pair {j}")
        assert np.array_equal(mask[j], np_check(fw[j], bw[j])[0]), j
    _, _, m2 = api.calc_optical_flow_farneback_sequence_bidirectional(frames, None, *prm, 0, alpha=0.0, beta=0.0, ctx=ectx)
    assert m2.sum() < mask.sum()
    empty = api.calc_optical_flow_farneback_sequence_bidirectional(frames[:1], None, *prm, 0, ctx=ectx)
    assert [a.shape for a in empty] == [(0, 96, 128, 2), (0, 96, 128, 2), (0, 96, 128)]
    with pytest.raises(ValueError):
        api.calc_optical_flow_farneback_sequence_bidirectional(frames[0], None, *prm, 0, ctx=ectx)
    with pytest.raises(ValueError):
        api.calc_optical_flow_farneback_sequence_bidirectional(frames, np.zeros((4, 96, 128, 2), np.float32), *prm, 0,
                                                               ctx=ectx)
    with pytest.raises(TypeError):
        api.calc_optical_flow_farneback_sequence_bidirectional(frames.astype(np.float32), None, *prm, 0, ctx=ectx)
    with pytest.raises(_native.FFBError, match="OPTFLOW_USE_INITIAL_FLOW"):
        api.calc_optical_flow_farneback_sequence_bidirectional(frames, None, *prm, 4, ctx=ectx)
    with pytest.raises(_native.FFBError, match="OPTFLOW_FARNEBACK_GAUSSIAN"):
        api.calc_optical_flow_farneback_sequence_bidirectional(frames, None, *prm, 256, ctx=ectx)


def test_strided_numpy_views_equal_their_contiguous_copies(ectx):
    """Every other frame, one channel of a colour clip and a reversed clip are views with other strides; the call reads
    them as the dense frames they stand for."""
    gray = clip(64, 48, 9, seed=5)
    colour = np.ascontiguousarray(np.stack([gray, gray[:, ::-1], 255 - gray], axis=-1))
    for view in (gray[::2], colour[..., 0], colour[..., 2], gray[::-1]):
        assert not view.flags.c_contiguous
        got = api.calc_optical_flow_farneback_sequence_bidirectional(view, None, *REF, 0, ctx=ectx)
        want = api.calc_optical_flow_farneback_sequence_bidirectional(np.ascontiguousarray(view), None, *REF, 0, ctx=ectx)
        for g, w in zip(got, want):
            assert np.array_equal(g, w)
        assert np.array_equal(got[0], api.calc_optical_flow_farneback_sequence(view, None, *REF, 0, ctx=ectx))


# ---- GPU -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("size", [(256, 256), (640, 360), (1920, 1080)])
def test_gpu_forward_and_backward_vs_cv2(gpu_ctx, size):
    frames = clip(*size, 4, seed=11)
    fw, bw, mask = api.calc_optical_flow_farneback_sequence_bidirectional(frames, None, *REF, 0, ctx=gpu_ctx)
    for j in range(3):
        pc.assert_flow_close(fw[j], cv2_flow(frames[j], frames[j + 1], REF), f"gpu {size} forward pair {j}")
        pc.assert_flow_close(bw[j], cv2_flow(frames[j + 1], frames[j], REF), f"gpu {size} backward pair {j}")
        assert np.array_equal(mask[j], np_check(fw[j], bw[j])[0]), (size, j)


@pytest.mark.gpu
def test_gpu_rings_wrap_into_device_pinned_and_pageable_buffers(gpu_ctx):
    """Batches of 4 frames through rings of 16 pairs wrap them twice; a slot overwritten before its copy-out would show
    in every kind of destination.  A context of its own: the rings only grow, so the shared context may already hold
    larger ones from an earlier test."""
    torch = pytest.importorskip("torch")
    W, H, n = 1920, 1080, 34
    frames = clip(W, H, n, seed=13)
    gpu_ctx.configure(W, H, 4, 8)
    ref_bw = np.stack([gpu_ctx.farneback(frames[j + 1], frames[j]) for j in range(n - 1)])
    ctx = _native.FlowContext(gpu_ctx.device)
    pin = _native.PinnedBuffer((2 * (n - 1) * H * W * 8 + (n - 1) * H * W,))
    try:
        ctx.configure(W, H, 4, 8)
        pageable = ctx.farneback_sequence_bidir(frames)
        assert ctx.flow_ring_size == 16
        assert np.array_equal(pageable["flow_bw"], ref_bw)
        assert np.array_equal(pageable["flow"], ctx.farneback_sequence(frames)["flow"])
        assert_check_matches(pageable)
        nb = (n - 1) * H * W * 8
        fw_p = pin.array[:nb].view(np.float32).reshape(n - 1, H, W, 2)
        bw_p = pin.array[nb:2 * nb].view(np.float32).reshape(n - 1, H, W, 2)
        m_p = pin.array[2 * nb:].reshape(n - 1, H, W)
        cnt = ctx.farneback_sequence_bidir_ptr(frames.ctypes.data, n, W, H, W, W * H, fw_p.ctypes.data, bw_p.ctypes.data,
                                               W * 8, W * H * 8, m_p.ctypes.data, W, W * H, counts=True)
        assert np.array_equal(fw_p, pageable["flow"]) and np.array_equal(bw_p, ref_bw)
        assert np.array_equal(m_p, pageable["mask"].view(np.uint8)) and np.array_equal(cnt, pageable["n_consistent"])
        dev = torch.device("cuda", ctx.device)
        f_t = torch.from_numpy(frames).to(dev)
        fw_t = torch.empty((n - 1, H, W, 2), dtype=torch.float32, device=dev)
        bw_t = torch.empty_like(fw_t)
        m_t = torch.empty((n - 1, H, W), dtype=torch.uint8, device=dev)
        cnt = ctx.farneback_sequence_bidir_ptr(f_t.data_ptr(), n, W, H, W, W * H, fw_t.data_ptr(), bw_t.data_ptr(), W * 8,
                                               W * H * 8, m_t.data_ptr(), W, W * H, counts=True)
        assert np.array_equal(bw_t.cpu().numpy(), ref_bw) and np.array_equal(fw_t.cpu().numpy(), pageable["flow"])
        assert np.array_equal(m_t.cpu().numpy(), pageable["mask"].view(np.uint8))
        assert np.array_equal(cnt, pageable["n_consistent"])
        assert ctx.flow_ring_size == 16
    finally:
        pin.free()
        ctx.close()


@pytest.mark.gpu
def test_gpu_torch_tensors_on_a_side_stream(gpu_ctx):
    torch = pytest.importorskip("torch")
    frames = clip(640, 360, 20, seed=17)
    want = api.calc_optical_flow_farneback_sequence_bidirectional(frames, None, *REF, 0, ctx=gpu_ctx)
    dev = torch.device("cuda", gpu_ctx.device)
    side = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(side):
        # the frames are written on the side stream by a torch op, read there by the call, and the outputs read there
        f_t = torch.from_numpy(frames.astype(np.int16)).to(dev).add_(0).to(torch.uint8)
        got = api.calc_optical_flow_farneback_sequence_bidirectional(f_t, None, *REF, 0, ctx=gpu_ctx)
        host = [t.cpu() for t in got]
    side.synchronize()
    assert [t.device for t in got] == [dev] * 3 and [t.dtype for t in got] == [torch.float32, torch.float32, torch.bool]
    assert tuple(got[2].shape) == (19, 360, 640)
    for g, w in zip(host, want):
        assert np.array_equal(g.numpy(), w)
    with pytest.raises(TypeError):
        api.calc_optical_flow_farneback_sequence_bidirectional(f_t.cpu(), None, *REF, 0, ctx=gpu_ctx)


@pytest.mark.gpu
def test_gpu_no_allocation_after_first_call(gpu_ctx):
    frames = clip(1920, 1080, 20, seed=23)
    gpu_ctx.configure(1920, 1080, 8, 19)
    gpu_ctx.farneback_sequence_bidir(frames)
    before = gpu_ctx.alloc_counts()
    for _ in range(2):
        gpu_ctx.farneback_sequence_bidir(frames)
        gpu_ctx.farneback_sequence_bidir(frames[:5], forward=False, counts=False)
        gpu_ctx.farneback_sequence(frames)
    assert gpu_ctx.alloc_counts() == before


@pytest.mark.gpu
def test_gpu_sequence_unchanged_around_a_bidir_call(gpu_ctx):
    frames = clip(1920, 1080, 18, seed=29)
    gpu_ctx.configure(1920, 1080, 8, 17)
    before = gpu_ctx.farneback_sequence(frames, stats=True)
    gpu_ctx.farneback_sequence_bidir(frames)
    after = gpu_ctx.farneback_sequence(frames, stats=True)
    for k in ("flow", "scalar", "cut", "cx", "cy", "val", "mean_mag", "centers"):
        assert np.array_equal(before[k], after[k]), k
