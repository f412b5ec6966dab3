"""Farneback flow along a sequence of frames, each frame expanded once (ffb_farneback_sequence,
FlowContext.farneback_sequence, api.calc_optical_flow_farneback_sequence, api.process_sequence).

CPU part (emulated kernels): bit-identity with the per-pair ffb_farneback and with ffb_farneback_pairs for three
parameter sets while the final-flow ring wraps several times, invariance to the batch size (the host-input ramp
included), every forced k_flow_iter variant, per-pair results against a bracket with POV on and off, process_sequence
against process_bracket, pitched / strided frames and flows, refusals, bracket bits around a sequence call, no
allocation on a repeated call, the cv2-order function against cv2.  `-m gpu` part: the sm_100a library against cv2,
bit-identity at 1080p with a small batch into device, pinned and pageable flows, torch tensors on a non-default stream,
per-pair results against a bracket, and no allocation after the first 1080p call."""

import numpy as np
import pytest

import parity_checks as pc
from funscript_flow_b200 import _native, api
from funscript_flow_b200.synth import make_clip

REF = (0.5, 3, 15, 3, 5, 1.2)
UNFUSED = (0.6, 4, 21, 2, 7, 1.5)          # winsize 21: k_flow_matrices + k_box_solve
NO_FUSED_UP = (0.8, 3, 15, 3, 5, 1.2)      # winsize 15, pyr_scale 0.8: k_flow_iter with a separate k_upsample_flow
STATS = ("scalar", "cut", "cx", "cy", "val", "mean_mag", "centers")


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
def test_sequence_equals_farneback_and_pairs(ectx, size, prm):
    frames = clip(*size, 25)
    ectx.set_farneback(*prm)
    ectx.configure(*size, 4, 24)       # 24 pairs in batches of at most 4 through a final-flow ring of 16 slots
    r = ectx.farneback_sequence(frames)
    assert ectx.flow_ring_size == 16
    assert r["flow"].shape == (24,) + frames.shape[1:] + (2,) and r["flow"].dtype == np.float32
    pairs = ectx.farneback_pairs(frames[:-1], frames[1:])["flow"]
    assert np.array_equal(r["flow"], pairs), prm
    for j in range(24):
        assert np.array_equal(r["flow"][j], ectx.farneback(frames[j], frames[j + 1])), (prm, j)


def test_batch_size_does_not_matter(ectx):
    frames = clip(96, 72, 25)
    out = []
    for batch in (4, 7, 64):         # 64: host input ramps up (17 frames, then 8)
        ectx.configure(96, 72, batch, 24)
        out.append(ectx.farneback_sequence(frames, stats=True))
    for r in out[1:]:
        for k in STATS + ("flow",):
            assert np.array_equal(r[k], out[0][k]), k


@pytest.mark.parametrize("variant", ["256x4x8", "128x2x4", "160x2x4", "96x2x4", "64x2x4"])
def test_every_forced_variant(emu_lib, variant, monkeypatch):
    monkeypatch.setenv("FFB_ITER_CFG", variant)
    ctx = _native.FlowContext(0, emu_lib)
    try:
        frames = clip(97, 70, 6)
        ctx.configure(97, 70, 2, 8)
        r = ctx.farneback_sequence(frames)
        for j in range(5):
            assert np.array_equal(r["flow"][j], ctx.farneback(frames[j], frames[j + 1])), (variant, j)
    finally:
        ctx.close()


@pytest.mark.parametrize("pov", [False, True])
def test_per_pair_results_equal_the_bracket(ectx, pov):
    frames = clip(160, 120, 22, seed=5)
    frames[9:] = frames[9:, ::-1]          # a scene cut between frames 8 and 9
    mags = np.sort(api.process_bracket(frames, {}, ctx=ectx, batch_frames=4)["mean_mag"])
    thr = float(0.5 * (mags[-1] + mags[-2]))
    params = {"pov_mode": pov, "cut_threshold": thr}
    want = api.process_bracket(frames, params, ctx=ectx, batch_frames=4)
    assert 0 < want["cut"].sum() < len(want["cut"])
    ectx.configure(160, 120, 4, 21)
    got = ectx.farneback_sequence(frames, stats=True, pov=pov, cut_threshold=thr)
    assert got["n_pairs"] == want["n_pairs"] == 21
    for k in STATS:
        assert got[k].dtype == want[k].dtype and np.array_equal(got[k], want[k]), k
    for j in range(21):
        assert np.array_equal(got["flow"][j], ectx.farneback(frames[j], frames[j + 1])), j
    only = ectx.farneback_sequence(frames, flow=False, stats=True, pov=pov, cut_threshold=thr)
    assert only["flow"] is None
    for k in STATS:
        assert np.array_equal(only[k], want[k]), k


def test_process_sequence_is_process_bracket_plus_flows(ectx):
    frames = clip(97, 70, 15, seed=9)
    params = {"cut_threshold": 0.4, "flow_winsize": 13}
    want = api.process_bracket(frames, params, ctx=ectx, batch_frames=4)
    got = api.process_sequence(frames, params, ctx=ectx, batch_frames=4)
    assert set(got) == set(want) | {"flows"} and got["n_pairs"] == want["n_pairs"] == 14
    for k in STATS:
        assert got[k].dtype == want[k].dtype and np.array_equal(got[k], want[k]), k
    assert ectx.farneback_params["winsize"] == 13
    for j in range(14):
        assert np.array_equal(got["flows"][j], ectx.farneback(frames[j], frames[j + 1])), j
    one = api.process_sequence(frames[:1], {}, ctx=ectx)
    assert one["n_pairs"] == 0 and one["flows"].shape == (0, 70, 97, 2)


def test_pitched_frames_and_strided_flows(ectx):
    frames = clip(97, 70, 9)
    ectx.configure(97, 70, 3, 8)
    ref = ectx.farneback_sequence(frames, stats=True)
    # frames inside wider rows with a gap between frames, flows inside wider rows with a gap between pairs
    wide = np.zeros((9, 72, 128), np.uint8)
    wide[:, :70, 5:102] = frames
    flow = np.full((8, 73, 100, 2), np.nan, np.float32)
    s = ectx.farneback_sequence_ptr(wide.ctypes.data + 5, 9, 97, 70, 128, 72 * 128, flow.ctypes.data, 100 * 8,
                                    73 * 100 * 8, stats=True)
    assert np.array_equal(flow[:, :70, :97], ref["flow"])
    assert np.isnan(flow[:, 70:]).all() and np.isnan(flow[:, :, 97:]).all()
    for k in STATS:
        assert np.array_equal(s[k], ref[k]), k
    # evenly spaced rows: one copy per run of ring slots into a larger preallocated array
    flow = np.full((10, 70, 97, 2), np.nan, np.float32)
    assert ectx.farneback_sequence_ptr(frames.ctypes.data, 9, 97, 70, 97, 97 * 70, flow[1:].ctypes.data, 97 * 8,
                                       97 * 70 * 8) is None
    assert np.array_equal(flow[1:9], ref["flow"]) and np.isnan(flow[0]).all() and np.isnan(flow[9]).all()


def test_refusals_leave_the_context_usable(ectx):
    frames = clip(97, 70, 6)
    before = api.process_bracket(frames, {}, ctx=ectx, batch_frames=3, return_flows=True)
    lib, h = ectx._lib, ectx._h
    p = frames.ctypes.data
    flow = np.empty((5, 70, 97, 2), np.float32)
    f = flow.ctypes.data
    none = [None] * 7
    bad = [
        (p, -1, 97, 70, 97, 97 * 70, f, 97 * 8, 97 * 70 * 8),      # n_frames < 0
        (p, 6, 97, 70, 96, 97 * 70, f, 97 * 8, 97 * 70 * 8),       # pitch below the width
        (p, 6, 97, 70, 97, 97 * 69, f, 97 * 8, 97 * 70 * 8),       # frames overlap
        (p, 6, 97, 70, 97, 97 * 70, f, 97 * 8 - 1, 97 * 70 * 8),   # flow_pitch below 8 * width
        (p, 6, 97, 70, 97, 97 * 70, f, 97 * 8, 97 * 69 * 8),       # flows overlap
    ]
    for args in bad:
        assert lib.ffb_farneback_sequence(h, *args, 0, 7.0, *none, None) == -1, args
        assert b"ffb_farneback_sequence" in lib.ffb_last_error(h)
    for n in (0, 1):          # nothing to do
        assert lib.ffb_farneback_sequence(h, p, n, 97, 70, 97, 97 * 70, f, 97 * 8, 97 * 70 * 8, 0, 7.0, *none, None) == 0
    ectx.bracket_begin(False, 7.0)
    with pytest.raises(_native.FFBError, match="inside a bracket"):
        ectx.farneback_sequence(frames)
    with pytest.raises(_native.FFBError, match="inside a bracket"):
        api.calc_optical_flow_farneback_sequence(frames, None, *REF, 0, ctx=ectx)
    ectx.bracket_abort()
    ectx.farneback_sequence(frames)
    with pytest.raises(_native.FFBError):      # the sequence replaced the bracket's flows in the final-flow ring
        ectx.get_flow(0)
    after = api.process_bracket(frames, {}, ctx=ectx, batch_frames=3, return_flows=True)
    for k in STATS + ("flows",):
        assert np.array_equal(before[k], after[k]), k


def test_no_allocation_on_a_repeated_call(ectx):
    frames = clip(96, 72, 12)
    ectx.configure(96, 72, 4, 11)
    ectx.farneback_sequence(frames, stats=True)
    before = ectx.alloc_counts()
    ectx.farneback_sequence(frames, stats=True)
    ectx.farneback_sequence(frames)
    ectx.farneback_sequence(frames[:5], flow=False, stats=True)
    assert ectx.alloc_counts() == before


def test_flow_only_launches_no_reduction(ectx):
    """Without per-pair outputs the call runs the bracket's expansion and flow launches and nothing else; with them, the
    bracket's launches exactly."""
    frames = clip(96, 72, 9)
    ectx.configure(96, 72, 4, 8)
    ectx.profile_reset()
    api.process_bracket(frames, {"cut_threshold": float("inf")}, ctx=ectx, batch_frames=4)
    brk = ectx.kernel_stats()
    ectx.profile_reset()
    ectx.farneback_sequence(frames)
    seq = ectx.kernel_stats()
    for k in ("pyramid", "polyexp", "upsample", "flow_iter"):
        assert seq[k] == brk[k], k
    assert seq["divmag"]["launches"] == seq["radial"]["launches"] == seq["small"]["launches"] == 0
    ectx.profile_reset()
    ectx.farneback_sequence(frames, stats=True)
    assert ectx.kernel_stats() == brk


def test_calc_optical_flow_farneback_sequence(ectx):
    frames = clip(128, 96, 6, seed=3)
    prm = (0.6, 4, 11, 2, 7, 1.3)
    got = api.calc_optical_flow_farneback_sequence(frames, None, *prm, 0, ctx=ectx)
    assert isinstance(got, np.ndarray) and got.dtype == np.float32 and got.shape == (5, 96, 128, 2)
    for j in range(5):
        pc.assert_flow_close(got[j], cv2_flow(frames[j], frames[j + 1], prm), f"sequence pair {j}")
    assert api.calc_optical_flow_farneback_sequence(frames[:1], None, *prm, 0, ctx=ectx).shape == (0, 96, 128, 2)
    with pytest.raises(ValueError):
        api.calc_optical_flow_farneback_sequence(frames[0], None, *prm, 0, ctx=ectx)
    with pytest.raises(ValueError):
        api.calc_optical_flow_farneback_sequence(frames, np.zeros((5, 96, 128, 2), np.float32), *prm, 0, ctx=ectx)
    with pytest.raises(TypeError):
        api.calc_optical_flow_farneback_sequence(frames.astype(np.float32), None, *prm, 0, ctx=ectx)
    with pytest.raises(_native.FFBError, match="OPTFLOW_FARNEBACK_GAUSSIAN"):
        api.calc_optical_flow_farneback_sequence(frames, None, *prm, 256, ctx=ectx)


# ---- GPU -------------------------------------------------------------------------------------------------------------
GPU_SET = (0.6, 4, 21, 2, 7, 1.5)


@pytest.mark.gpu
@pytest.mark.parametrize("size", [(256, 256), (640, 360), (1920, 1080)])
@pytest.mark.parametrize("prm", [REF, GPU_SET])
def test_gpu_sequence_vs_cv2(gpu_ctx, size, prm):
    frames = clip(*size, 6, seed=11)
    try:
        got = api.calc_optical_flow_farneback_sequence(frames, None, *prm, 0, ctx=gpu_ctx)
        for j in range(5):
            pc.assert_flow_close(got[j], cv2_flow(frames[j], frames[j + 1], prm), f"gpu {size} {prm} pair {j}")
    finally:
        gpu_ctx.set_farneback(*REF)


@pytest.mark.gpu
def test_gpu_ring_wraps_into_device_pinned_and_pageable_flows(gpu_ctx):
    """Batches of 4 frames through a final-flow ring of 16 pairs wrap it three times; a slot overwritten before its
    copy-out would show in every kind of destination.  A context of its own: the ring only grows, so the shared
    context may already hold a larger one from an earlier test."""
    torch = pytest.importorskip("torch")
    frames = clip(1920, 1080, 50, seed=13)
    gpu_ctx.configure(1920, 1080, 4, 8)
    ref = np.stack([gpu_ctx.farneback(frames[j], frames[j + 1]) for j in range(49)])
    ctx = _native.FlowContext(gpu_ctx.device)
    pin = _native.PinnedBuffer((49, 1080, 1920, 8))
    try:
        ctx.configure(1920, 1080, 4, 8)
        pageable = ctx.farneback_sequence(frames)["flow"]
        assert ctx.flow_ring_size == 16
        assert np.array_equal(pageable, ref)
        pinned = pin.array.view(np.float32).reshape(49, 1080, 1920, 2)
        ctx.farneback_sequence_ptr(frames.ctypes.data, 50, 1920, 1080, 1920, 1920 * 1080, pinned.ctypes.data, 1920 * 8,
                                   1920 * 1080 * 8)
        assert np.array_equal(pinned, ref)
        dev = torch.device("cuda", ctx.device)
        f_t = torch.from_numpy(frames).to(dev)
        out = torch.empty((49, 1080, 1920, 2), dtype=torch.float32, device=dev)
        ctx.farneback_sequence_ptr(f_t.data_ptr(), 50, 1920, 1080, 1920, 1920 * 1080, out.data_ptr(), 1920 * 8,
                                   1920 * 1080 * 8)
        assert np.array_equal(out.cpu().numpy(), ref)
        assert ctx.flow_ring_size == 16
    finally:
        pin.free()
        ctx.close()


@pytest.mark.gpu
def test_gpu_torch_tensors_on_a_side_stream(gpu_ctx):
    torch = pytest.importorskip("torch")
    frames = clip(640, 360, 20, seed=17)
    gpu_ctx.configure(640, 360, 7, 19)
    ref = gpu_ctx.farneback_sequence(frames)["flow"]
    dev = torch.device("cuda", gpu_ctx.device)
    side = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(side):
        # the frames are written on the side stream by a torch op, read there by the call, and the flow is read there
        f_t = torch.from_numpy(frames.astype(np.int16)).to(dev).add_(0).to(torch.uint8)
        out = api.calc_optical_flow_farneback_sequence(f_t, None, *REF, 0, ctx=gpu_ctx)
        host = out.cpu()
    side.synchronize()
    assert out.device == dev and out.dtype == torch.float32 and tuple(out.shape) == (19, 360, 640, 2)
    assert np.array_equal(host.numpy(), ref)
    with pytest.raises(TypeError):
        api.calc_optical_flow_farneback_sequence(f_t.cpu(), None, *REF, 0, ctx=gpu_ctx)


@pytest.mark.gpu
def test_gpu_per_pair_results_equal_the_bracket(gpu_ctx):
    frames = clip(1920, 1080, 30, seed=19)
    params = {"cut_threshold": 0.5}
    want = api.process_bracket(frames, params, ctx=gpu_ctx, batch_frames=8)
    got = api.process_sequence(frames, params, ctx=gpu_ctx, batch_frames=8)
    for k in STATS:
        assert np.array_equal(got[k], want[k]), k
    for j in (0, 13, 28):
        assert np.array_equal(got["flows"][j], gpu_ctx.farneback(frames[j], frames[j + 1])), j


@pytest.mark.gpu
def test_gpu_no_allocation_after_first_call(gpu_ctx):
    frames = clip(1920, 1080, 20, seed=23)
    gpu_ctx.configure(1920, 1080, 8, 19)
    gpu_ctx.farneback_sequence(frames, stats=True)
    before = gpu_ctx.alloc_counts()
    for _ in range(2):
        gpu_ctx.farneback_sequence(frames, stats=True)
        gpu_ctx.farneback_sequence(frames)
        gpu_ctx.farneback_sequence(frames[:5], flow=False, stats=True)
    assert gpu_ctx.alloc_counts() == before
