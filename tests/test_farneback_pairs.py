"""Farneback flow for batches of independent frame pairs (ffb_farneback_pairs, FlowContext.farneback_pairs,
api.calc_optical_flow_farneback_batch, api.precompute_flow_info_batch).

CPU part (emulated kernels): bit-identity with the per-pair ffb_farneback for three parameter sets and every forced
k_flow_iter variant, invariance to the chunk size, per-pair results against precompute_flow_info, the cv2-order batch
function and its refusals, bracket state around a pairs call, no allocation on a repeated call.  `-m gpu` part: the
sm_100a library against cv2 and against gpu_ctx.farneback, torch CUDA tensors on a non-default stream, and no
allocation after the first 1080p call."""

import numpy as np
import pytest

import parity_checks as pc
from funscript_flow_b200 import _native, api
from funscript_flow_b200.synth import make_clip

REF = (0.5, 3, 15, 3, 5, 1.2)
UNFUSED = (0.6, 4, 21, 2, 7, 1.5)          # winsize 21: k_flow_matrices + k_box_solve
NO_FUSED_UP = (0.8, 3, 15, 3, 5, 1.2)      # winsize 15, pyr_scale 0.8: k_flow_iter with a separate k_upsample_flow
STATS = ("cx", "cy", "val", "mean_mag", "cut")


def cv2_flow(p0, p1, prm):
    import cv2
    return cv2.calcOpticalFlowFarneback(p0, p1, None, *prm, 0)


def unrelated_pairs(width, height):
    """5 pairs that are not consecutive frames of one clip: a pair, the same pair reversed, two frames 3 apart of
    another clip, one frame with itself, and two frames of different clips."""
    a = make_clip(width, height, 4, seed=11, period=12.0, amplitude=0.3)
    b = make_clip(width, height, 4, seed=12, period=9.0, amplitude=0.35)
    c = make_clip(width, height, 3, seed=13, period=14.0, amplitude=0.25)
    pairs = [(a[1], a[2]), (a[2], a[1]), (b[0], b[3]), (c[2], c[2]), (b[1], a[1])]
    return np.stack([p for p, _ in pairs]), np.stack([q for _, q in pairs])


def clip_pairs(width, height, n, seed=21):
    clip = make_clip(width, height, n + 1, seed=seed, period=10.0, amplitude=0.3)
    order = np.random.default_rng(seed).permutation(n + 1)
    return clip[order[:n]], clip[np.roll(order, 1)[:n]]


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
def test_pairs_equal_farneback(ectx, size, prm):
    prev, nxt = unrelated_pairs(*size)
    ectx.set_farneback(*prm)
    ectx.configure(*size, 4, 8)        # chunks of 2 pairs: 5 pairs take 3 chunks, both final-flow ring halves
    r = ectx.farneback_pairs(prev, nxt)
    assert r["flow"].shape == (5,) + prev.shape[1:] + (2,) and r["flow"].dtype == np.float32
    for i in range(5):
        assert np.array_equal(r["flow"][i], ectx.farneback(prev[i], nxt[i])), (prm, i)
    # one frame with itself: Farneback's border rule (the last row and column have no bilinear footprint) leaves a
    # small residual flow, in cv2 as here, instead of an exact zero
    assert r["mean_mag"][3] < 0.01 and r["mean_mag"][0] > 5 * r["mean_mag"][3]
    # the reversed pair moves the other way
    assert np.mean(r["flow"][0] * r["flow"][1]) < 0


@pytest.mark.parametrize("variant", ["256x4x8", "128x2x4", "160x2x4", "96x2x4", "64x2x4"])
def test_every_forced_variant_has_the_pair_stride(emu_lib, variant, monkeypatch):
    monkeypatch.setenv("FFB_ITER_CFG", variant)
    ctx = _native.FlowContext(0, emu_lib)
    try:
        prev, nxt = unrelated_pairs(97, 70)
        ctx.configure(97, 70, 3, 8)
        r = ctx.farneback_pairs(prev[:3], nxt[:3])
        for i in range(3):
            assert np.array_equal(r["flow"][i], ctx.farneback(prev[i], nxt[i])), (variant, i)
    finally:
        ctx.close()


def test_unknown_forced_variant_is_refused(emu_lib, monkeypatch):
    monkeypatch.setenv("FFB_ITER_CFG", "192x2x4")
    ctx = _native.FlowContext(0, emu_lib)
    try:
        prev, nxt = unrelated_pairs(97, 70)
        with pytest.raises(_native.FFBError, match="no k_flow_iter variant") as ei:
            ctx.farneback_pairs(prev[:2], nxt[:2])
        assert ei.value.code == -1
    finally:
        ctx.close()


def test_chunk_size_does_not_matter(ectx):
    prev, nxt = clip_pairs(96, 72, 9)
    out = []
    for batch in (4, 7, 64):
        ectx.configure(96, 72, batch, 16)
        out.append(ectx.farneback_pairs(prev, nxt))
    for r in out[1:]:
        for k in STATS + ("flow",):
            assert np.array_equal(r[k], out[0][k]), k


@pytest.mark.parametrize("pov", [False, True])
def test_per_pair_results_equal_precompute_flow_info(ectx, pov):
    prev, nxt = unrelated_pairs(160, 120)
    ref = [api.precompute_flow_info(p, q, {"pov_mode": pov}) for p, q in zip(prev, nxt)]
    mags = sorted(float(d["mean_mag"]) for d in ref)
    thr = 0.5 * (mags[1] + mags[2])           # cuts the two or three largest motions, not the others
    ref = [api.precompute_flow_info(p, q, {"pov_mode": pov, "cut_threshold": thr}) for p, q in zip(prev, nxt)]
    assert 0 < sum(d["cut"] for d in ref) < len(ref)
    ectx.configure(160, 120, 4, 8)
    r = ectx.farneback_pairs(prev, nxt, pov=pov, cut_threshold=thr)
    assert r["cx"].dtype == np.int32 and r["val"].dtype == np.float32 and r["cut"].dtype == bool
    for i, d in enumerate(ref):
        assert np.array_equal(r["flow"][i], d["flow"])
        assert bool(r["cut"][i]) == d["cut"] and r["mean_mag"][i] == d["mean_mag"]
        if not pov:
            assert (r["cx"][i], r["cy"][i]) == d["pos_center"] and r["val"][i] == d["val_pos"]
    batch = api.precompute_flow_info_batch(list(zip(prev, nxt)), {"pov_mode": pov, "cut_threshold": thr})
    assert len(batch) == len(ref)
    for got, want in zip(batch, ref):
        assert got.keys() == want.keys()
        for k in want:
            assert type(got[k]) is type(want[k]), k
            if k == "flow":
                assert np.array_equal(got[k], want[k]) and got[k].dtype == want[k].dtype
            elif isinstance(want[k], tuple):
                assert got[k] == want[k] and [type(v) for v in got[k]] == [type(v) for v in want[k]], k
            else:
                assert got[k] == want[k], k


def test_precompute_flow_info_batch_settings(ectx):
    prev, nxt = unrelated_pairs(97, 70)
    cfg = {"flow_winsize": 21, "flow_poly_n": 7, "cut_threshold": 0.0}
    got = api.precompute_flow_info_batch(zip(prev[:2], nxt[:2]), cfg)
    for g, p, q in zip(got, prev, nxt):
        want = api.precompute_flow_info(p, q, cfg)
        assert np.array_equal(g["flow"], want["flow"]) and g["cut"] is True
    assert ectx.farneback_params["winsize"] == 21
    assert api.precompute_flow_info_batch([], {}) == []
    with pytest.raises(ValueError):
        api.precompute_flow_info_batch([(prev[0], nxt[0]), (prev[0][:60], nxt[0][:60])], {})


def test_calc_optical_flow_farneback_batch(ectx):
    prev, nxt = unrelated_pairs(128, 96)
    prm = (0.6, 4, 11, 2, 7, 1.3)
    got = api.calc_optical_flow_farneback_batch(prev, nxt, None, *prm, 0, ctx=ectx)
    assert isinstance(got, np.ndarray) and got.dtype == np.float32 and got.shape == (5, 96, 128, 2)
    for i in range(5):
        pc.assert_flow_close(got[i], cv2_flow(prev[i], nxt[i], prm), f"batch pair {i}")
    empty = api.calc_optical_flow_farneback_batch(prev[:0], nxt[:0], None, *prm, 0, ctx=ectx)
    assert empty.shape == (0, 96, 128, 2)
    with pytest.raises(ValueError):
        api.calc_optical_flow_farneback_batch(prev, nxt[:4], None, *prm, 0, ctx=ectx)
    with pytest.raises(ValueError):
        api.calc_optical_flow_farneback_batch(prev[0], nxt[0], None, *prm, 0, ctx=ectx)
    with pytest.raises(ValueError):
        api.calc_optical_flow_farneback_batch(prev, nxt, np.zeros((5, 96, 128, 2), np.float32), *prm, 0, ctx=ectx)
    with pytest.raises(_native.FFBError, match="OPTFLOW_FARNEBACK_GAUSSIAN"):
        api.calc_optical_flow_farneback_batch(prev, nxt, None, *prm, 256, ctx=ectx)
    with pytest.raises(_native.FFBError, match="OPTFLOW_USE_INITIAL_FLOW"):
        api.calc_optical_flow_farneback_batch(prev, nxt, None, *prm, 4, ctx=ectx)
    ectx.set_farneback(*prm)
    ectx.bracket_begin(False, 7.0)
    with pytest.raises(_native.FFBError, match="inside a bracket"):
        api.calc_optical_flow_farneback_batch(prev, nxt, None, *prm, 0, ctx=ectx)
    with pytest.raises(_native.FFBError, match="inside a bracket"):
        ectx.farneback_pairs(prev, nxt)
    ectx.bracket_abort()


def test_refusals_leave_the_context_usable(ectx):
    prev, nxt = unrelated_pairs(97, 70)
    clip = make_clip(97, 70, 6, seed=4, period=9.0, amplitude=0.3)
    before = api.process_bracket(clip, {}, ctx=ectx, batch_frames=3, return_flows=True)
    lib, h = ectx._lib, ectx._h
    p, q = prev.ctypes.data, nxt.ctypes.data
    flow = np.empty((5, 70, 97, 2), np.float32)
    f = flow.ctypes.data
    none = [None] * 5
    bad = [
        (p, q, -1, 97, 70, 97, 97 * 70, f, 97 * 8, 97 * 70 * 8),     # n_pairs < 0
        (p, q, 5, 97, 70, 96, 97 * 70, f, 97 * 8, 97 * 70 * 8),      # pitch below the width
        (p, q, 5, 97, 70, 97, 97 * 70, f, 97 * 8 - 1, 97 * 70 * 8),  # flow_pitch below 8 * width
        (p, q, 5, 97, 70, 97, 97 * 69, f, 97 * 8, 97 * 70 * 8),      # frames overlap
    ]
    for args in bad:
        assert lib.ffb_farneback_pairs(h, *args, 0, 7.0, *none, None) == -1, args
        assert lib.ffb_last_error(h)
    assert lib.ffb_farneback_pairs(h, p, q, 0, 97, 70, 97, 97 * 70, f, 97 * 8, 97 * 70 * 8, 0, 7.0, *none, None) == 0
    ectx.farneback_pairs(prev, nxt)
    with pytest.raises(_native.FFBError):      # the pairs call replaced the bracket's flows in the final-flow ring
        ectx.get_flow(0)
    after = api.process_bracket(clip, {}, ctx=ectx, batch_frames=3, return_flows=True)
    for k in ("scalar", "cut", "cx", "cy", "val", "mean_mag", "centers", "flows"):
        assert np.array_equal(before[k], after[k]), k


def test_flow_strides_and_stats_only(ectx):
    prev, nxt = unrelated_pairs(97, 70)
    ectx.configure(97, 70, 3, 8)
    ref = ectx.farneback_pairs(prev, nxt)
    # frames inside wider rows, flows inside wider rows and with gaps between pairs
    wide = np.zeros((5, 70, 128), np.uint8)
    wide[:, :, 5:102] = prev
    wide_n = np.zeros((5, 70, 128), np.uint8)
    wide_n[:, :, 5:102] = nxt
    flow = np.full((5, 72, 100, 2), np.nan, np.float32)
    s = ectx.farneback_pairs_ptr(wide.ctypes.data + 5, wide_n.ctypes.data + 5, 5, 97, 70, 128, 70 * 128, flow.ctypes.data,
                                 100 * 8, 72 * 100 * 8, stats=True)
    assert np.array_equal(flow[:, :70, :97], ref["flow"]) and np.isnan(flow[:, 70:]).all() and np.isnan(flow[:, :, 97:]).all()
    for k in STATS:
        assert np.array_equal(s[k], ref[k]), k
    only = ectx.farneback_pairs(prev, nxt, flow=False)
    assert only["flow"] is None
    for k in STATS:
        assert np.array_equal(only[k], ref[k]), k


def test_no_allocation_on_a_covered_call(ectx):
    prev, nxt = clip_pairs(96, 72, 7)
    ectx.configure(96, 72, 6, 8)
    ectx.farneback_pairs(prev, nxt)
    before = ectx.alloc_counts()
    ectx.farneback_pairs(prev, nxt)
    ectx.farneback_pairs(prev[:3], nxt[:3], flow=False)
    api.calc_optical_flow_farneback_batch(prev[:2], nxt[:2], None, *REF, 0, ctx=ectx)
    assert ectx.alloc_counts() == before


def test_launch_counts_and_bytes(ectx):
    """A pairs call counts the same flow-phase launches and algorithmic bytes per pair as a bracket, and expands two
    frames per pair."""
    prev, nxt = clip_pairs(96, 72, 4)
    ectx.configure(96, 72, 8, 8)
    ectx.profile_reset()
    ectx.farneback_pairs(prev, nxt)
    pairs = ectx.kernel_stats()
    ectx.profile_reset()
    api.process_bracket(make_clip(96, 72, 5, seed=3), {}, ctx=ectx, batch_frames=8)
    brk = ectx.kernel_stats()
    for k in ("flow_iter", "divmag"):
        assert pairs[k] == brk[k], k
    for k in ("pyramid", "polyexp"):
        assert pairs[k]["launches"] == brk[k]["launches"] and pairs[k]["alg_bytes"] == pytest.approx(8 / 5 * brk[k]["alg_bytes"])


# ---- GPU -------------------------------------------------------------------------------------------------------------
GPU_SET = (0.6, 4, 21, 2, 7, 1.5)


@pytest.mark.gpu
@pytest.mark.parametrize("size", [(256, 256), (640, 360), (1920, 1080)])
@pytest.mark.parametrize("prm", [REF, GPU_SET])
def test_gpu_pairs_vs_cv2(gpu_ctx, size, prm):
    prev, nxt = unrelated_pairs(*size)
    try:
        got = api.calc_optical_flow_farneback_batch(prev, nxt, None, *prm, 0, ctx=gpu_ctx)
        for i in range(len(prev)):
            pc.assert_flow_close(got[i], cv2_flow(prev[i], nxt[i], prm), f"gpu {size} {prm} pair {i}")
    finally:
        gpu_ctx.set_farneback(*REF)


@pytest.mark.gpu
def test_gpu_pairs_bit_identical_to_farneback(gpu_ctx):
    prev, nxt = clip_pairs(1920, 1080, 7)
    gpu_ctx.configure(1920, 1080, 4, 8)
    r = gpu_ctx.farneback_pairs(prev, nxt)
    for i in range(7):
        assert np.array_equal(r["flow"][i], gpu_ctx.farneback(prev[i], nxt[i])), i
        d = api.precompute_flow_info(prev[i], nxt[i], {"cut_threshold": float("inf")})
        assert (r["cx"][i], r["cy"][i], r["val"][i], r["mean_mag"][i]) == (*d["pos_center"], d["val_pos"], d["mean_mag"])


@pytest.mark.gpu
def test_gpu_torch_tensors_on_a_side_stream(gpu_ctx):
    torch = pytest.importorskip("torch")
    prev, nxt = clip_pairs(640, 360, 9)
    gpu_ctx.configure(640, 360, 7, 16)
    ref = gpu_ctx.farneback_pairs(prev, nxt)["flow"]
    dev = torch.device("cuda", gpu_ctx.device)
    # pinned and pageable host input give the same flows as device input
    pin = [_native.PinnedBuffer(prev.shape), _native.PinnedBuffer(nxt.shape)]
    pin[0].array[...] = prev
    pin[1].array[...] = nxt
    assert np.array_equal(gpu_ctx.farneback_pairs(pin[0].array, pin[1].array)["flow"], ref)
    side = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(side):
        # the inputs are written on the side stream by a torch op, read there by the call, and the flow is read there
        p_t = torch.from_numpy(prev.astype(np.int16)).to(dev, non_blocking=False).add_(0).to(torch.uint8)
        n_t = torch.from_numpy(nxt.astype(np.int16)).to(dev).add_(0).to(torch.uint8)
        out = api.calc_optical_flow_farneback_batch(p_t, n_t, None, *REF, 0, ctx=gpu_ctx)
        host = out.cpu()
    side.synchronize()
    assert out.device == dev and out.dtype == torch.float32 and tuple(out.shape) == (9, 360, 640, 2)
    assert np.array_equal(host.numpy(), ref)
    # the host round trip of the device inputs gives the same flows
    assert np.array_equal(gpu_ctx.farneback_pairs(p_t.cpu().numpy(), n_t.cpu().numpy())["flow"], ref)
    with pytest.raises(TypeError):
        api.calc_optical_flow_farneback_batch(p_t, nxt, None, *REF, 0, ctx=gpu_ctx)
    with pytest.raises(TypeError):
        api.calc_optical_flow_farneback_batch(p_t.cpu(), n_t.cpu(), None, *REF, 0, ctx=gpu_ctx)
    for b in pin:
        b.free()


@pytest.mark.gpu
def test_gpu_no_allocation_after_first_call(gpu_ctx):
    prev, nxt = clip_pairs(1920, 1080, 6)
    gpu_ctx.configure(1920, 1080, 8, 8)
    gpu_ctx.farneback_pairs(prev, nxt)
    before = gpu_ctx.alloc_counts()
    for _ in range(2):
        gpu_ctx.farneback_pairs(prev, nxt)
        gpu_ctx.farneback_pairs(prev[:2], nxt[:2], flow=False)
    assert gpu_ctx.alloc_counts() == before
