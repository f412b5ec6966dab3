"""Backward flows and a forward-backward consistency mask for batches of independent frame pairs, each frame expanded
once (ffb_farneback_pairs_bidir, FlowContext.farneback_pairs_bidir, api.calc_optical_flow_farneback_batch_bidirectional).

CPU part (emulated kernels): forward flows bit-identical to the pairs call and to the per-pair call, backward flows
bit-identical to the per-pair call on the reversed pair, masks and counts equal to the NumPy float32 restatement of the
check, for three parameter sets while the chunks alternate ring halves; invariance to the chunk size; every forced
k_flow_iter variant; the launch set; every combination of outputs, pitched / strided outputs, the two eyes of
side-by-side frames, refusals, nothing to do, no allocation on a repeated call, bracket bits and the pairs call around a
call; the cv2-order function against cv2.  `-m gpu` part: the sm_100a library against cv2 at three sizes, bit-identity
and exact masks at 1080p with a small batch into device, pinned and pageable buffers, torch tensors on a non-default
stream, no allocation after the first 1080p call, and the pairs call unchanged around a bidirectional call."""

import itertools

import numpy as np
import pytest

import parity_checks as pc
from funscript_flow_b200 import _native, api
from funscript_flow_b200.synth import make_clip
from test_farneback_bidirectional import ALPHA, BETA, np_check

REF = (0.5, 3, 15, 3, 5, 1.2)
UNFUSED = (0.6, 4, 21, 2, 7, 1.5)          # winsize 21: k_flow_matrices + k_box_solve
NO_FUSED_UP = (0.8, 3, 15, 3, 5, 1.2)      # winsize 15, pyr_scale 0.8: k_flow_iter with a separate k_upsample_flow
OUTPUTS = ("flow", "flow_bw", "mask", "n_consistent")


def assert_check_matches(r, alpha=ALPHA, beta=BETA):
    for i in range(r["flow"].shape[0]):
        want, n = np_check(r["flow"][i], r["flow_bw"][i], alpha, beta)
        assert np.array_equal(r["mask"][i], want), i
        assert r["n_consistent"][i] == n, (i, r["n_consistent"][i], n)


def cv2_flow(p0, p1, prm):
    import cv2
    return cv2.calcOpticalFlowFarneback(p0, p1, None, *prm, 0)


def pairs(width, height, n, seed=21):
    """n independent pairs: frames of one clip in a shuffled order, so that the motion of a pair ranges from a frame
    step to several, and every pair has consistent and inconsistent pixels."""
    clip = make_clip(width, height, n + 1, seed=seed, period=9.0, amplitude=0.35)
    order = np.random.default_rng(seed).permutation(n + 1)
    return np.ascontiguousarray(clip[order[:n]]), np.ascontiguousarray(clip[np.roll(order, 1)[:n]])


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
def test_pairs_bidir_equals_farneback_and_check(ectx, size, prm):
    prev, nxt = pairs(*size, 9)
    ectx.set_farneback(*prm)
    ectx.configure(*size, 3, 8)        # chunks of 2 pairs: 9 pairs take 5 chunks, ring halves 0, 1, 0, 1, 0
    r = ectx.farneback_pairs_bidir(prev, nxt)
    assert r["flow_bw"].shape == (9,) + prev.shape[1:] + (2,) and r["flow_bw"].dtype == np.float32
    assert r["mask"].shape == (9,) + prev.shape[1:] and r["mask"].dtype == np.bool_
    assert r["n_consistent"].shape == (9,) and r["n_consistent"].dtype == np.int64
    assert np.array_equal(r["flow"], ectx.farneback_pairs(prev, nxt)["flow"]), prm
    for i in range(9):
        assert np.array_equal(r["flow"][i], ectx.farneback(prev[i], nxt[i])), (prm, i)
        assert np.array_equal(r["flow_bw"][i], ectx.farneback(nxt[i], prev[i])), (prm, i)
    assert_check_matches(r)
    assert 0 < r["n_consistent"].sum() < r["mask"].size     # the pairs have pixels of both kinds


def test_chunk_size_does_not_matter(ectx):
    prev, nxt = pairs(96, 72, 7)
    out = []
    for batch in (3, 4, 64):         # chunks of 2 pairs, of 2 pairs with a spare frame slot, one chunk of all 7
        ectx.configure(96, 72, batch, 8)
        out.append(ectx.farneback_pairs_bidir(prev, nxt, alpha=0.02, beta=0.3))
    for r in out[1:]:
        for k in OUTPUTS:
            assert np.array_equal(r[k], out[0][k]), k
    assert_check_matches(out[0], 0.02, 0.3)


@pytest.mark.parametrize("variant", ["256x4x8", "128x2x4", "160x2x4", "96x2x4", "64x2x4"])
def test_every_forced_variant(emu_lib, variant, monkeypatch):
    monkeypatch.setenv("FFB_ITER_CFG", variant)
    ctx = _native.FlowContext(0, emu_lib)
    try:
        prev, nxt = pairs(97, 70, 3)
        ctx.configure(97, 70, 3, 8)
        r = ctx.farneback_pairs_bidir(prev, nxt, mask=False, counts=False)
        for i in range(3):
            assert np.array_equal(r["flow"][i], ctx.farneback(prev[i], nxt[i])), (variant, i)
            assert np.array_equal(r["flow_bw"][i], ctx.farneback(nxt[i], prev[i])), (variant, i)
    finally:
        ctx.close()


def test_each_frame_is_expanded_once(ectx):
    """The backward pass re-uses the forward pass's expansions: the same pyramid and expansion launches as the pairs
    call, twice its flow-iteration launches and bytes, one check launch per chunk, and no k_divmag."""
    prev, nxt = pairs(96, 72, 5)
    ectx.configure(96, 72, 3, 8)
    ectx.profile_reset()
    ectx.farneback_pairs(prev, nxt, flow=True)
    fwd = ectx.kernel_stats()
    ectx.profile_reset()
    ectx.farneback_pairs_bidir(prev, nxt)
    bid = ectx.kernel_stats()
    for k in ("pyramid", "polyexp"):
        assert bid[k] == fwd[k], k
    for k in ("upsample", "flow_iter"):
        assert bid[k]["launches"] == 2 * fwd[k]["launches"] and bid[k]["alg_bytes"] == 2 * fwd[k]["alg_bytes"], k
    assert bid["fb_check"]["launches"] == 3 and bid["fb_check"]["alg_bytes"] == 5 * 96 * 72 * 17
    assert fwd["divmag"]["launches"] == 3
    assert bid["divmag"]["launches"] == bid["radial"]["launches"] == bid["small"]["launches"] == 0
    ectx.profile_reset()
    ectx.farneback_pairs_bidir(prev, nxt, backward=False, mask=False, counts=False)
    fwd_only = ectx.kernel_stats()
    assert fwd_only["fb_check"]["launches"] == 0 and fwd_only["divmag"]["launches"] == 0
    for k in ("pyramid", "polyexp", "upsample", "flow_iter"):
        assert fwd_only[k] == fwd[k], k


def test_every_combination_of_outputs(ectx):
    prev, nxt = pairs(97, 70, 5)
    ectx.configure(97, 70, 3, 8)
    full = ectx.farneback_pairs_bidir(prev, nxt)
    assert np.array_equal(full["n_consistent"], full["mask"].sum(axis=(1, 2)))
    for want in itertools.product((False, True), repeat=4):
        r = ectx.farneback_pairs_bidir(prev, nxt, forward=want[0], backward=want[1], mask=want[2], counts=want[3])
        for k, asked in zip(OUTPUTS, want):
            if asked:
                assert np.array_equal(r[k], full[k]), (want, k)
            else:
                assert r[k] is None, (want, k)


def test_pitched_and_strided_outputs(ectx):
    prev, nxt = pairs(97, 70, 5)
    ectx.configure(97, 70, 3, 8)
    ref = ectx.farneback_pairs_bidir(prev, nxt)
    # frames inside wider rows with a gap between frames; flows and masks inside wider rows with a gap between pairs
    wide = np.zeros((2, 5, 72, 128), np.uint8)
    wide[0, :, :70, 5:102] = prev
    wide[1, :, :70, 5:102] = nxt
    fw = np.full((5, 73, 100, 2), np.nan, np.float32)
    bw = np.full((5, 73, 100, 2), np.nan, np.float32)
    mask = np.full((5, 72, 101), 7, np.uint8)
    cnt = ectx.farneback_pairs_bidir_ptr(wide[0].ctypes.data + 5, wide[1].ctypes.data + 5, 5, 97, 70, 128, 72 * 128,
                                         fw.ctypes.data, bw.ctypes.data, 100 * 8, 73 * 100 * 8, mask.ctypes.data, 101,
                                         72 * 101, counts=True)
    assert np.array_equal(fw[:, :70, :97], ref["flow"]) and np.array_equal(bw[:, :70, :97], ref["flow_bw"])
    assert np.array_equal(mask[:, :70, :97], ref["mask"].view(np.uint8)) and np.array_equal(cnt, ref["n_consistent"])
    for a in (fw, bw):
        assert np.isnan(a[:, 70:]).all() and np.isnan(a[:, :, 97:]).all()
    assert (mask[:, 70:] == 7).all() and (mask[:, :, 97:] == 7).all()
    # evenly spaced rows: one copy per chunk into larger preallocated arrays
    bw = np.full((7, 70, 97, 2), np.nan, np.float32)
    mask = np.full((7, 70, 97), 7, np.uint8)
    assert ectx.farneback_pairs_bidir_ptr(prev.ctypes.data, nxt.ctypes.data, 5, 97, 70, 97, 97 * 70, 0, bw[1:].ctypes.data,
                                          97 * 8, 97 * 70 * 8, mask[1:].ctypes.data, 97, 97 * 70) is None
    assert np.array_equal(bw[1:6], ref["flow_bw"]) and np.isnan(bw[0]).all() and np.isnan(bw[6]).all()
    assert np.array_equal(mask[1:6], ref["mask"].view(np.uint8)) and (mask[0] == 7).all() and (mask[6] == 7).all()


def test_stereo_side_by_side_frames(ectx):
    """The two eyes of side-by-side frames: left -> right and right -> left flows and the left-right check.  NumPy views
    of the halves through the api function, and the halves read in place through the pointer call (pitch 2W)."""
    W, H, n = 64, 48, 4
    clip = make_clip(W + 6, H, n, seed=31, period=11.0, amplitude=0.3)
    sbs = np.ascontiguousarray(np.concatenate([clip[:, :, 6:], clip[:, :, :W]], axis=2))   # right eye 6 px apart
    left, right = sbs[:, :, :W], sbs[:, :, W:]
    assert not left.flags.c_contiguous
    got = api.calc_optical_flow_farneback_batch_bidirectional(left, right, None, *REF, 0, ctx=ectx)
    want = api.calc_optical_flow_farneback_batch_bidirectional(np.ascontiguousarray(left), np.ascontiguousarray(right),
                                                               None, *REF, 0, ctx=ectx)
    for g, w in zip(got, want):
        assert np.array_equal(g, w)
    assert np.array_equal(got[0], api.calc_optical_flow_farneback_batch(left, right, None, *REF, 0, ctx=ectx))
    fw = np.empty((n, H, W, 2), np.float32)
    bw = np.empty((n, H, W, 2), np.float32)
    mask = np.empty((n, H, W), np.uint8)
    cnt = ectx.farneback_pairs_bidir_ptr(sbs.ctypes.data, sbs.ctypes.data + W, n, W, H, 2 * W, 2 * W * H, fw, bw, mask=mask,
                                         counts=True)
    assert np.array_equal(fw, got[0]) and np.array_equal(bw, got[1]) and np.array_equal(mask.view(np.bool_), got[2])
    assert np.array_equal(cnt, got[2].sum(axis=(1, 2)))
    # the disparity is a horizontal shift: the left eye's flow points right, the right eye's left
    assert np.median(got[0][..., 0]) > 3 and np.median(got[1][..., 0]) < -3
    assert 0 < cnt.sum() < mask.size      # the strip the other eye does not see is inconsistent


def test_refusals_leave_the_context_usable(ectx):
    prev, nxt = pairs(97, 70, 5)
    clip = make_clip(97, 70, 6, seed=4, period=9.0, amplitude=0.3)
    before = api.process_bracket(clip, {}, ctx=ectx, batch_frames=3, return_flows=True)
    lib, h = ectx._lib, ectx._h
    p, q = prev.ctypes.data, nxt.ctypes.data
    flow = np.empty((5, 70, 97, 2), np.float32)
    mask = np.empty((5, 70, 97), np.uint8)
    f, m = flow.ctypes.data, mask.ctypes.data
    fs, ms = 97 * 70 * 8, 97 * 70
    ok = (p, q, 5, 97, 70, 97, 97 * 70, None, f, 97 * 8, fs, m, 97, ms, ALPHA, BETA)
    bad = [
        dict(prev=None),                 # no frames
        dict(width=0),                   # bad frame size
        dict(n=-1),                      # n_pairs < 0
        dict(pitch=96),                  # pitch below the width
        dict(fstride=97 * 69),           # frames overlap
        dict(flow_pitch=97 * 8 - 1),     # flow_pitch below 8 * width (backward flow only)
        dict(flow_stride=97 * 69 * 8),   # flows overlap
        dict(mask_pitch=96),             # mask_pitch below the width
        dict(mask_stride=97 * 69),       # masks overlap
        dict(alpha=-0.01), dict(alpha=float("nan")), dict(beta=float("inf")), dict(beta=-1.0),
    ]
    keys = dict(prev=0, n=2, width=3, pitch=5, fstride=6, flow_pitch=9, flow_stride=10, mask_pitch=12, mask_stride=13,
                alpha=14, beta=15)
    for change in bad:
        args = list(ok)
        for k, v in change.items():
            args[keys[k]] = v
        assert lib.ffb_farneback_pairs_bidir(h, *args, None, None) == -1, change
        assert b"ffb_farneback_pairs_bidir" in lib.ffb_last_error(h), change
    cnt = np.full(5, -7, np.int64)
    args = list(ok)
    args[2] = 0               # nothing to do
    assert lib.ffb_farneback_pairs_bidir(h, *args, cnt.ctypes.data_as(_native.C.POINTER(_native.C.c_int64)), None) == 0
    assert (cnt == -7).all()
    args[2], args[6], args[10], args[13] = 1, 0, 0, 0    # one pair: the strides are not read
    assert lib.ffb_farneback_pairs_bidir(h, *args, cnt.ctypes.data_as(_native.C.POINTER(_native.C.c_int64)), None) == 0
    assert cnt[0] == int(mask[0].sum()) and (cnt[1:] == -7).all()
    ectx.bracket_begin(False, 7.0)
    with pytest.raises(_native.FFBError, match="inside a bracket"):
        ectx.farneback_pairs_bidir(prev, nxt)
    with pytest.raises(_native.FFBError, match="inside a bracket"):
        api.calc_optical_flow_farneback_batch_bidirectional(prev, nxt, None, *REF, 0, ctx=ectx)
    ectx.bracket_abort()
    r = ectx.farneback_pairs_bidir(prev, nxt)
    assert_check_matches(r)
    with pytest.raises(_native.FFBError):      # the call replaced the bracket's flows in the final-flow ring
        ectx.get_flow(0)
    after = api.process_bracket(clip, {}, ctx=ectx, batch_frames=3, return_flows=True)
    for k in ("scalar", "cut", "cx", "cy", "val", "mean_mag", "centers", "flows"):
        assert np.array_equal(before[k], after[k]), k


def test_allocation_only_when_needed_and_not_on_a_repeated_call(ectx):
    prev, nxt = pairs(96, 72, 7)
    ectx.configure(96, 72, 4, 8)
    ectx.farneback_pairs(prev, nxt)
    base = ectx.alloc_counts()
    ectx.farneback_pairs_bidir(prev, nxt, backward=False, mask=False, counts=False)
    assert ectx.alloc_counts() == base                     # forward flows only: the pairs call's buffers
    ectx.farneback_pairs_bidir(prev, nxt)
    grown = ectx.alloc_counts()
    assert grown[0] == base[0] + 3 and grown[1] == base[1]   # backward ring, mask ring, counts
    ectx.farneback_pairs_bidir(prev, nxt)
    ectx.farneback_pairs_bidir(prev[:3], nxt[:3], forward=False)
    ectx.farneback_pairs_bidir(prev, nxt, mask=False)
    ectx.farneback_pairs(prev, nxt)
    assert ectx.alloc_counts() == grown


def test_bracket_and_pairs_call_around_a_call(ectx):
    """A bracket keeps its bits, and ffb_farneback_pairs its outputs and its launches per kernel, around a
    bidirectional call."""
    prev, nxt = pairs(96, 72, 5)
    clip = make_clip(96, 72, 6, seed=8, period=9.0, amplitude=0.3)
    ectx.configure(96, 72, 3, 8)
    brk0 = api.process_bracket(clip, {}, ctx=ectx, batch_frames=3, return_flows=True)
    ectx.configure(96, 72, 3, 8)
    ectx.profile_reset()
    before = ectx.farneback_pairs(prev, nxt)
    launches = ectx.kernel_stats()
    ectx.farneback_pairs_bidir(prev, nxt)
    brk1 = api.process_bracket(clip, {}, ctx=ectx, batch_frames=3, return_flows=True)
    ectx.configure(96, 72, 3, 8)
    ectx.profile_reset()
    after = ectx.farneback_pairs(prev, nxt)
    assert ectx.kernel_stats() == launches
    for k in ("flow", "cx", "cy", "val", "mean_mag", "cut"):
        assert np.array_equal(before[k], after[k]), k
    for k in ("scalar", "cut", "cx", "cy", "val", "mean_mag", "centers", "flows"):
        assert np.array_equal(brk0[k], brk1[k]), k


def test_calc_optical_flow_farneback_batch_bidirectional(ectx):
    prev, nxt = pairs(128, 96, 4, seed=3)
    prm = (0.6, 4, 11, 2, 7, 1.3)
    fw, bw, mask = api.calc_optical_flow_farneback_batch_bidirectional(prev, nxt, None, *prm, 0, ctx=ectx)
    for a in (fw, bw):
        assert isinstance(a, np.ndarray) and a.dtype == np.float32 and a.shape == (4, 96, 128, 2)
    assert isinstance(mask, np.ndarray) and mask.dtype == np.bool_ and mask.shape == (4, 96, 128)
    assert np.array_equal(fw, api.calc_optical_flow_farneback_batch(prev, nxt, None, *prm, 0, ctx=ectx))
    for i in range(4):
        pc.assert_flow_close(fw[i], cv2_flow(prev[i], nxt[i], prm), f"forward pair {i}")
        pc.assert_flow_close(bw[i], cv2_flow(nxt[i], prev[i], prm), f"backward pair {i}")
        assert np.array_equal(mask[i], np_check(fw[i], bw[i])[0]), i
    _, _, m2 = api.calc_optical_flow_farneback_batch_bidirectional(prev, nxt, None, *prm, 0, alpha=0.0, beta=0.0, ctx=ectx)
    assert m2.sum() < mask.sum()
    empty = api.calc_optical_flow_farneback_batch_bidirectional(prev[:0], nxt[:0], None, *prm, 0, ctx=ectx)
    assert [a.shape for a in empty] == [(0, 96, 128, 2), (0, 96, 128, 2), (0, 96, 128)]
    with pytest.raises(ValueError):
        api.calc_optical_flow_farneback_batch_bidirectional(prev, nxt[:3], None, *prm, 0, ctx=ectx)
    with pytest.raises(ValueError):
        api.calc_optical_flow_farneback_batch_bidirectional(prev[0], nxt[0], None, *prm, 0, ctx=ectx)
    with pytest.raises(ValueError):
        api.calc_optical_flow_farneback_batch_bidirectional(prev, nxt, np.zeros((4, 96, 128, 2), np.float32), *prm, 0,
                                                            ctx=ectx)
    with pytest.raises(TypeError):
        api.calc_optical_flow_farneback_batch_bidirectional(prev.astype(np.float32), nxt, None, *prm, 0, ctx=ectx)
    with pytest.raises(_native.FFBError, match="OPTFLOW_USE_INITIAL_FLOW"):
        api.calc_optical_flow_farneback_batch_bidirectional(prev, nxt, None, *prm, 4, ctx=ectx)
    with pytest.raises(_native.FFBError, match="OPTFLOW_FARNEBACK_GAUSSIAN"):
        api.calc_optical_flow_farneback_batch_bidirectional(prev, nxt, None, *prm, 256, ctx=ectx)
    with pytest.raises(_native.FFBError, match="alpha"):
        api.calc_optical_flow_farneback_batch_bidirectional(prev, nxt, None, *prm, 0, alpha=-1.0, ctx=ectx)


# ---- GPU -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("size", [(256, 256), (640, 360), (1920, 1080)])
def test_gpu_forward_and_backward_vs_cv2(gpu_ctx, size):
    prev, nxt = pairs(*size, 3, seed=11)
    fw, bw, mask = api.calc_optical_flow_farneback_batch_bidirectional(prev, nxt, None, *REF, 0, ctx=gpu_ctx)
    for i in range(3):
        pc.assert_flow_close(fw[i], cv2_flow(prev[i], nxt[i], REF), f"gpu {size} forward pair {i}")
        pc.assert_flow_close(bw[i], cv2_flow(nxt[i], prev[i], REF), f"gpu {size} backward pair {i}")
        assert np.array_equal(mask[i], np_check(fw[i], bw[i])[0]), (size, i)


@pytest.mark.gpu
def test_gpu_ring_halves_alternate_into_device_pinned_and_pageable_buffers(gpu_ctx):
    """Chunks of 2 pairs alternate between the two halves of the rings 5 times; a slot overwritten before its copy-out
    would show in every kind of destination.  A context of its own: the rings only grow, so the shared context may
    already hold larger ones from an earlier test."""
    torch = pytest.importorskip("torch")
    W, H, n = 1920, 1080, 11
    prev, nxt = pairs(W, H, n, seed=13)
    gpu_ctx.configure(W, H, 3, 8)
    ref_fw = np.stack([gpu_ctx.farneback(prev[i], nxt[i]) for i in range(n)])
    ref_bw = np.stack([gpu_ctx.farneback(nxt[i], prev[i]) for i in range(n)])
    ctx = _native.FlowContext(gpu_ctx.device)
    pin = _native.PinnedBuffer((2 * n * H * W * 8 + n * H * W,))
    try:
        ctx.configure(W, H, 3, 8)
        pageable = ctx.farneback_pairs_bidir(prev, nxt)
        assert np.array_equal(pageable["flow"], ref_fw) and np.array_equal(pageable["flow_bw"], ref_bw)
        assert_check_matches(pageable)
        assert 0 < pageable["n_consistent"].sum() < pageable["mask"].size
        nb = n * H * W * 8
        fw_p = pin.array[:nb].view(np.float32).reshape(n, H, W, 2)
        bw_p = pin.array[nb:2 * nb].view(np.float32).reshape(n, H, W, 2)
        m_p = pin.array[2 * nb:].reshape(n, H, W)
        cnt = ctx.farneback_pairs_bidir_ptr(prev.ctypes.data, nxt.ctypes.data, n, W, H, W, W * H, fw_p.ctypes.data,
                                            bw_p.ctypes.data, W * 8, W * H * 8, m_p.ctypes.data, W, W * H, counts=True)
        assert np.array_equal(fw_p, ref_fw) and np.array_equal(bw_p, ref_bw)
        assert np.array_equal(m_p, pageable["mask"].view(np.uint8)) and np.array_equal(cnt, pageable["n_consistent"])
        dev = torch.device("cuda", ctx.device)
        p_t, n_t = torch.from_numpy(prev).to(dev), torch.from_numpy(nxt).to(dev)
        fw_t = torch.empty((n, H, W, 2), dtype=torch.float32, device=dev)
        bw_t = torch.empty_like(fw_t)
        m_t = torch.empty((n, H, W), dtype=torch.uint8, device=dev)
        cnt = ctx.farneback_pairs_bidir_ptr(p_t.data_ptr(), n_t.data_ptr(), n, W, H, W, W * H, fw_t.data_ptr(),
                                            bw_t.data_ptr(), W * 8, W * H * 8, m_t.data_ptr(), W, W * H, counts=True)
        assert np.array_equal(fw_t.cpu().numpy(), ref_fw) and np.array_equal(bw_t.cpu().numpy(), ref_bw)
        assert np.array_equal(m_t.cpu().numpy(), pageable["mask"].view(np.uint8))
        assert np.array_equal(cnt, pageable["n_consistent"])
    finally:
        pin.free()
        ctx.close()


@pytest.mark.gpu
def test_gpu_torch_tensors_on_a_side_stream(gpu_ctx):
    torch = pytest.importorskip("torch")
    prev, nxt = pairs(640, 360, 9, seed=17)
    want = api.calc_optical_flow_farneback_batch_bidirectional(prev, nxt, None, *REF, 0, ctx=gpu_ctx)
    dev = torch.device("cuda", gpu_ctx.device)
    side = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(side):
        # the frames are written on the side stream by a torch op, read there by the call, and the outputs read there
        p_t = torch.from_numpy(prev.astype(np.int16)).to(dev).add_(0).to(torch.uint8)
        n_t = torch.from_numpy(nxt.astype(np.int16)).to(dev).add_(0).to(torch.uint8)
        got = api.calc_optical_flow_farneback_batch_bidirectional(p_t, n_t, None, *REF, 0, ctx=gpu_ctx)
        host = [t.cpu() for t in got]
    side.synchronize()
    assert [t.device for t in got] == [dev] * 3 and [t.dtype for t in got] == [torch.float32, torch.float32, torch.bool]
    assert tuple(got[2].shape) == (9, 360, 640)
    for g, w in zip(host, want):
        assert np.array_equal(g.numpy(), w)
    with pytest.raises(TypeError):
        api.calc_optical_flow_farneback_batch_bidirectional(p_t, nxt, None, *REF, 0, ctx=gpu_ctx)
    with pytest.raises(TypeError):
        api.calc_optical_flow_farneback_batch_bidirectional(p_t.cpu(), n_t.cpu(), None, *REF, 0, ctx=gpu_ctx)


@pytest.mark.gpu
def test_gpu_no_allocation_after_first_call(gpu_ctx):
    prev, nxt = pairs(1920, 1080, 6, seed=23)
    gpu_ctx.configure(1920, 1080, 8, 8)
    gpu_ctx.farneback_pairs_bidir(prev, nxt)
    before = gpu_ctx.alloc_counts()
    for _ in range(2):
        gpu_ctx.farneback_pairs_bidir(prev, nxt)
        gpu_ctx.farneback_pairs_bidir(prev[:2], nxt[:2], forward=False, counts=False)
        gpu_ctx.farneback_pairs(prev, nxt)
    assert gpu_ctx.alloc_counts() == before


@pytest.mark.gpu
def test_gpu_pairs_unchanged_around_a_bidir_call(gpu_ctx):
    prev, nxt = pairs(1920, 1080, 7, seed=29)
    gpu_ctx.configure(1920, 1080, 4, 8)
    before = gpu_ctx.farneback_pairs(prev, nxt)
    gpu_ctx.farneback_pairs_bidir(prev, nxt)
    after = gpu_ctx.farneback_pairs(prev, nxt)
    for k in ("flow", "cx", "cy", "val", "mean_mag", "cut"):
        assert np.array_equal(before[k], after[k]), k
