"""Warping images by dense flows on the device, bit-exact with cv2.remap's relative bilinear warp (ffb_remap_flow,
FlowContext.remap_flow, api.remap_by_flow).

CPU part (emulated kernels): equality with cv2.remap(..., INTER_LINEAR | WARP_RELATIVE_MAP) for gray and BGR images,
both borders and two border values, at sizes from 1 x 1 up, for random flows, flows far outside the image, flows on the
1/64 px rounding ties, flows around -1 .. 0 and non-finite or huge flows; flows of the library's own sequence call;
several chunks; pitched and strided buffers, one eye of side-by-side frames read in place, strided NumPy views, refusals,
nothing to do, no allocation on a repeated call, a bracket's flows, geometry and parameters around a call, the launch
set.  `-m gpu` part: the sm_100a library against cv2 from 256 x 256 to 4K, every combination of device, pinned and
pageable buffers at 1080p past one chunk, torch tensors on a side stream, no allocation after the first call, and a
sequence-then-remap pipeline on tensors."""

import itertools

import numpy as np
import pytest

from funscript_flow_b200 import _native, api
from funscript_flow_b200.synth import make_clip

cv2 = pytest.importorskip("cv2")

REF = (0.5, 3, 15, 3, 5, 1.2)
CHUNK_BYTES = 8 << 20      # ffb_remap_flow's staging chunk: source, flow and output of its images together


def cv_remap(src, flow, border=0, value=0):
    return cv2.remap(src, flow, None, cv2.INTER_LINEAR | cv2.WARP_RELATIVE_MAP,
                     borderMode=(cv2.BORDER_CONSTANT, cv2.BORDER_REPLICATE)[border], borderValue=(value,) * 3)


def cv_batch(src, flow, border=0, value=0):
    return np.stack([cv_remap(s, f, border, value) for s, f in zip(src, flow)])


def images(n, h, w, ch, seed):
    shape = (n, h, w) if ch == 1 else (n, h, w, 3)
    return np.random.default_rng(seed).integers(0, 256, shape, dtype=np.uint8)


def flow_cases(h, w, seed=0):
    """Five flows: random, far outside the image, on the +-0.5/32 rounding ties, around -1 .. 0, and non-finite or huge
    components (NaN, +-inf, +-1e30, beyond +-2^26 and just inside, where 32 f nears the int range)."""
    rng = np.random.default_rng(seed)
    shape = (h, w, 2)
    special = np.array([np.nan, np.inf, -np.inf, 1e30, -1e30, 2.0 ** 26, -2.0 ** 26, 2.0 ** 26 + 64, -2.0 ** 26 - 64,
                        2.0 ** 26 - 64, -2.0 ** 26 + 64, 40000.0, -40000.0, 0.0, -1.0, w, h, -w, -h], np.float32)
    return np.stack([
        rng.uniform(-12, 12, shape),
        rng.uniform(-3, 3, shape) * np.array([w, h]) + rng.choice([-1, 1], shape) * np.array([w, h]),
        rng.integers(-96, 96, shape) / 32 + rng.choice([-0.5, 0.5], shape) / 32,
        rng.uniform(-1.05, 0.05, shape),
        rng.choice(special, shape),
    ]).astype(np.float32)


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
@pytest.mark.parametrize("size", [(1, 1), (37, 1), (1, 29), (97, 70), (160, 120)])
@pytest.mark.parametrize("ch", [1, 3])
@pytest.mark.parametrize("border", [0, 1])
@pytest.mark.parametrize("value", [0, 7])
def test_equals_cv2(ectx, size, ch, border, value):
    w, h = size
    flow = flow_cases(h, w, seed=w * h)
    src = images(len(flow), h, w, ch, seed=w + h)
    got = ectx.remap_flow(src, flow, border, value)
    assert got.shape == src.shape and got.dtype == np.uint8
    assert np.array_equal(got, cv_batch(src, flow, border, value))


def test_ties_and_float_sums_where_cv2_rounds_after_adding_the_grid(ectx):
    """cv2 rounds 32 f and adds the grid in integers: a flow whose x + f rounds to a tie in float32 is not a tie for
    cv2, and a flow near 2^26 saturates at the far side rather than wrapping."""
    h, w = 8, 160
    flow = np.zeros((3, h, w, 2), np.float32)
    flow[0, ..., 0] = -17.484373           # x + f rounds to k + 0.515625 in float32; 32 f rounds to -559
    flow[1, ..., 0] = np.float32(2.0 ** 26 - 64)
    flow[2, ..., 1] = np.float32(-(2.0 ** 26 - 64))
    src = images(3, h, w, 1, seed=3)
    for border in (0, 1):
        assert np.array_equal(ectx.remap_flow(src, flow, border, 9), cv_batch(src, flow, border, 9))


@pytest.mark.parametrize("ch", [1, 3])
def test_flows_of_the_sequence_call(ectx, ch):
    """Warping each next frame onto its previous one with the library's own flows."""
    w, h = 97, 70
    clip = make_clip(w, h, 5, seed=9, period=9.0, amplitude=0.35)
    ectx.configure(w, h, 2, 8)
    flows = ectx.farneback_sequence(clip)["flow"]
    nxt = clip[1:] if ch == 1 else np.ascontiguousarray(np.stack([clip[1:], 255 - clip[1:], clip[1:] // 2], axis=-1))
    for border in (0, 1):
        got = api.remap_by_flow(nxt, flows, border, 7, ctx=ectx)
        assert np.array_equal(got, cv_batch(nxt, flows, border, 7))
    if ch == 1:   # the warp brings the next frame closer to the previous one
        warped = api.remap_by_flow(nxt, flows, 1, ctx=ectx)
        inner = (slice(None), slice(8, -8), slice(8, -8))
        err_warp = np.abs(warped[inner].astype(int) - clip[:-1][inner]).mean()
        err_raw = np.abs(nxt[inner].astype(int) - clip[:-1][inner]).mean()
        assert err_warp < 0.7 * err_raw, (err_warp, err_raw)


@pytest.mark.parametrize("ch", [1, 3])
def test_several_chunks_and_the_launch_set(ectx, ch):
    """Host buffers move in chunks: one k_remap_flow launch per chunk, with its algorithmic bytes, and nothing else."""
    w, h, n = 256, 256, 30
    per = w * h * (8 + 2 * ch)
    k = CHUNK_BYTES // per
    assert n > 2 * k
    src = images(n, h, w, ch, seed=ch)
    flow = np.concatenate([flow_cases(h, w, seed=s) for s in range(n // 5)])
    ectx.profile_reset()
    got = ectx.remap_flow(src, flow, 1)
    st = ectx.kernel_stats()
    assert st["remap"]["launches"] == -(-n // k)
    assert st["remap"]["alg_bytes"] == n * per
    assert all(v["launches"] == 0 for name, v in st.items() if name != "remap")
    assert np.array_equal(got, cv_batch(src, flow, 1))


@pytest.mark.parametrize("ch", [1, 3])
def test_pitched_and_strided_buffers(ectx, ch):
    w, h, n = 97, 70, 5
    flow = flow_cases(h, w, seed=4)
    src = images(n, h, w, ch, seed=5)
    want = cv_batch(src, flow, 0, 3)
    c = ch
    # images inside wider rows with a gap between images, flows likewise, output likewise
    s_wide = np.zeros((n, h + 2, (w + 9) * c), np.uint8)
    s_wide[:, :h, 5 * c:(5 + w) * c] = src.reshape(n, h, w * c)
    f_wide = np.zeros((n, h + 1, w + 3, 2), np.float32)
    f_wide[:, :h, :w] = flow
    out = np.full((n, h + 3, (w + 7) * c), 77, np.uint8)
    ectx.remap_flow_ptr(s_wide.ctypes.data + 5 * c, n, w, h, c, (w + 9) * c, (h + 2) * (w + 9) * c, f_wide.ctypes.data,
                        (w + 3) * 8, (h + 1) * (w + 3) * 8, out.ctypes.data, (w + 7) * c, (h + 3) * (w + 7) * c, 0, 3)
    assert np.array_equal(out[:, :h, :w * c], want.reshape(n, h, w * c))
    assert (out[:, h:] == 77).all() and (out[:, :, w * c:] == 77).all()
    # evenly spaced rows into a larger preallocated array: its neighbours stay untouched
    out = np.full((n + 2,) + src.shape[1:], 77, np.uint8)
    ectx.remap_flow_ptr(src.ctypes.data, n, w, h, c, w * c, w * h * c, flow.ctypes.data, w * 8, w * h * 8,
                        out[1:].ctypes.data, w * c, w * h * c, 0, 3)
    assert np.array_equal(out[1:-1], want) and (out[0] == 77).all() and (out[-1] == 77).all()
    # one image: the strides are not read
    one = np.empty_like(src[:1])
    ectx.remap_flow_ptr(src.ctypes.data, 1, w, h, c, w * c, 0, flow.ctypes.data, w * 8, 0, one.ctypes.data, w * c, 0, 0, 3)
    assert np.array_equal(one, want[:1])


def test_side_by_side_eye_in_place_and_strided_views(ectx):
    """One eye of side-by-side frames read in place (pitch 2W) and as a NumPy view; every other frame and every other
    flow as views: the same bits as their dense copies."""
    w, h, n = 64, 48, 6
    sbs = images(n, h, 2 * w, 1, seed=12)
    flow = np.concatenate([flow_cases(h, w, seed=s) for s in (2, 3, 4)])[:2 * n]
    right, fl = sbs[:, :, w:], flow[::2]
    assert not right.flags.c_contiguous and not fl.flags.c_contiguous
    want = cv_batch(np.ascontiguousarray(right), np.ascontiguousarray(fl), 1)
    assert np.array_equal(api.remap_by_flow(right, fl, 1, ctx=ectx), want)
    out = np.empty((n, h, w), np.uint8)
    ectx.remap_flow_ptr(sbs.ctypes.data + w, n, w, h, 1, 2 * w, 2 * w * h, fl.ctypes.data, w * 8, 2 * w * h * 8,
                        out.ctypes.data, w, w * h, 1, 0)
    assert np.array_equal(out, want)
    frames = images(2 * n, h, w, 3, seed=13)
    assert np.array_equal(api.remap_by_flow(frames[::2], fl, ctx=ectx),
                          api.remap_by_flow(np.ascontiguousarray(frames[::2]), np.ascontiguousarray(fl), ctx=ectx))


def test_refusals_and_nothing_to_do(ectx):
    w, h, n = 20, 10, 3
    src = images(n, h, w, 3, seed=1)
    flow = flow_cases(h, w)[:n]
    dst = np.full((n, h, w, 3), 5, np.uint8)
    lib, hd = ectx._lib, ectx._h
    s, f, d = src.ctypes.data, flow.ctypes.data, dst.ctypes.data
    ok = [s, n, w, h, 3, w * 3, w * h * 3, f, w * 8, w * h * 8, d, w * 3, w * h * 3, 0, 0]
    keys = dict(src=0, n=1, width=2, height=3, channels=4, src_pitch=5, src_stride=6, flow=7, flow_pitch=8,
                flow_stride=9, dst=10, dst_pitch=11, dst_stride=12, border=13, value=14)
    bad = [dict(n=-1), dict(src=None), dict(flow=None), dict(dst=None), dict(width=0), dict(height=0),
           dict(width=32767), dict(height=40000), dict(channels=2), dict(channels=4), dict(border=2), dict(border=-1),
           dict(value=-1), dict(value=256), dict(src_pitch=w * 3 - 1), dict(src_stride=w * (h - 1) * 3),
           dict(flow_pitch=w * 8 - 4), dict(flow_stride=w * (h - 1) * 8), dict(dst_pitch=w * 3 - 1),
           dict(dst_stride=w * (h - 1) * 3), dict(channels=1, src_pitch=w * 3, dst_pitch=w - 1)]
    for change in bad:
        args = list(ok)
        for k, v in change.items():
            args[keys[k]] = v
        assert lib.ffb_remap_flow(hd, *args, None) == -1, change
        assert b"ffb_remap_flow" in lib.ffb_last_error(hd), change
    assert (dst == 5).all()
    args = list(ok)
    args[1] = 0                        # nothing to do, whatever else is passed
    args[0] = args[7] = args[10] = None
    assert lib.ffb_remap_flow(hd, *args, None) == 0
    assert ectx.remap_flow(src[:0], flow[:0]).shape == (0, h, w, 3)
    ectx.configure(64, 48, 2, 8)
    ectx.bracket_begin(False, 7.0)
    with pytest.raises(_native.FFBError, match="ffb_remap_flow inside a bracket"):
        ectx.remap_flow(src, flow)
    ectx.bracket_abort()
    assert np.array_equal(ectx.remap_flow(src, flow), cv_batch(src, flow))


def test_api_shapes_and_errors(ectx):
    w, h = 33, 21
    flow = flow_cases(h, w, seed=8)
    gray, bgr = images(5, h, w, 1, seed=1), images(5, h, w, 3, seed=2)
    for src in (gray, bgr):
        batch = api.remap_by_flow(src, flow, 1, ctx=ectx)
        assert isinstance(batch, np.ndarray) and batch.shape == src.shape and batch.dtype == np.uint8
        one = api.remap_by_flow(src[2], flow[2], 1, ctx=ectx)
        assert one.shape == src.shape[1:] and np.array_equal(one, batch[2])
        assert np.array_equal(one, cv_remap(src[2], flow[2], 1))
    with pytest.raises(ValueError):
        api.remap_by_flow(gray[:4], flow, ctx=ectx)
    with pytest.raises(ValueError):
        api.remap_by_flow(gray[0], flow, ctx=ectx)
    with pytest.raises(ValueError):
        api.remap_by_flow(np.zeros((5, h, w, 4), np.uint8), flow, ctx=ectx)
    with pytest.raises(ValueError):
        api.remap_by_flow(gray, flow[..., :1], ctx=ectx)
    with pytest.raises(TypeError):
        api.remap_by_flow(gray.astype(np.float32), flow, ctx=ectx)
    with pytest.raises(TypeError):
        api.remap_by_flow(gray, flow.astype(np.float64), ctx=ectx)
    with pytest.raises(_native.FFBError, match="border"):
        api.remap_by_flow(gray, flow, 3, ctx=ectx)


def test_no_allocation_on_a_repeated_call(ectx):
    flow = flow_cases(70, 97, seed=1)
    src = images(5, 70, 97, 3, seed=1)
    ectx.remap_flow(src, flow)
    before = ectx.alloc_counts()
    for _ in range(2):
        ectx.remap_flow(src, flow, 1, 9)
        ectx.remap_flow(src[:2], flow[:2])
        ectx.remap_flow(src[..., 0], flow)                       # gray: fewer bytes than BGR
        ectx.remap_flow(src[:, :40, :50], flow[:, :40, :50])     # a smaller size
    assert ectx.alloc_counts() == before


def test_bracket_state_is_left_alone(ectx):
    """A remap call does not configure the context: the flows of the last bracket stay readable, and its geometry and
    Farneback parameters stay as they were."""
    w, h = 96, 72
    clip = make_clip(w, h, 6, seed=8, period=9.0, amplitude=0.3)
    ectx.set_farneback(0.6, 4, 11, 2, 7, 1.3)
    r = api.process_bracket(clip, {"flow_pyr_scale": 0.6, "flow_levels": 4, "flow_winsize": 11, "flow_iterations": 2,
                                   "flow_poly_n": 7, "flow_poly_sigma": 1.3}, ctx=ectx, batch_frames=3, return_flows=True)
    geometry, params, ring = ectx.geometry, ectx.farneback_params, ectx.flow_ring_size
    allocs = ectx.alloc_counts()
    src = images(4, 50, 130, 3, seed=4)
    ectx.remap_flow(src, flow_cases(50, 130)[:4], 1)
    ectx.remap_flow(clip[1:], r["flows"])
    assert ectx.geometry == geometry and ectx.farneback_params == params and ectx.flow_ring_size == ring
    for p in range(r["flow_first"], r["n_pairs"]):
        assert np.array_equal(ectx.get_flow(p), r["flows"][p - r["flow_first"]]), p
    assert ectx.alloc_counts()[0] > allocs[0]          # its own staging, not the context's geometry


# ---- GPU -------------------------------------------------------------------------------------------------------------
def smooth_flows(n, h, w, seed, amplitude=30.0):
    """Smooth flows of tens of pixels (a sum of low-frequency waves), with a sprinkle of non-finite and huge values."""
    rng = np.random.default_rng(seed)
    ys, xs = np.mgrid[0:h, 0:w].astype(np.float32)
    out = np.empty((n, h, w, 2), np.float32)
    for i in range(n):
        for c in range(2):
            k = rng.uniform(0.5, 3.0, 4) * 2 * np.pi
            out[i, ..., c] = amplitude * (np.sin(k[0] * xs / w + k[1] * ys / h + rng.uniform(0, 6)) +
                                          0.5 * np.cos(k[2] * xs / w - k[3] * ys / h))
    flat = out.reshape(-1)
    idx = rng.choice(flat.size, flat.size // 5000, replace=False)
    flat[idx] = rng.choice(np.array([np.nan, np.inf, -np.inf, 1e30, 2.0 ** 26 + 64], np.float32), idx.size)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("size", [(256, 256), (640, 360), (1920, 1080), (3840, 2160)])
@pytest.mark.parametrize("ch", [1, 3])
def test_gpu_equals_cv2(gpu_ctx, size, ch):
    w, h = size
    flow = smooth_flows(2, h, w, seed=w)
    src = images(2, h, w, ch, seed=h)
    for border, value in ((0, 0), (0, 7), (1, 0)):
        got = gpu_ctx.remap_flow(src, flow, border, value)
        assert np.array_equal(got, cv_batch(src, flow, border, value)), (size, ch, border, value)


@pytest.mark.gpu
@pytest.mark.parametrize("ch", [1, 3])
def test_gpu_device_pinned_and_pageable_buffers(gpu_ctx, ch):
    """Every combination of device, pinned and pageable source, flow and output at 1080p, with more images than one
    chunk holds; device flows also with rows 4-byte but not 32-byte aligned (read in place) and 2-byte aligned (staged
    first)."""
    torch = pytest.importorskip("torch")
    w, h, n = 1920, 1080, 3
    flow = smooth_flows(n, h, w, seed=ch)
    src = images(n, h, w, ch, seed=ch)
    want = cv_batch(src, flow, 1)
    dev = torch.device("cuda", gpu_ctx.device)
    c = ch
    pins = [_native.PinnedBuffer(src.shape), _native.PinnedBuffer(flow.shape + (4,)), _native.PinnedBuffer(src.shape)]
    try:
        pins[0].array[...] = src
        pins[1].array.view(np.float32).reshape(flow.shape)[...] = flow
        s_t, f_t = torch.from_numpy(src).to(dev), torch.from_numpy(flow).to(dev)
        srcs = dict(device=s_t.data_ptr(), pinned=pins[0].array.ctypes.data, pageable=src.ctypes.data)
        flows = dict(device=f_t.data_ptr(), pinned=pins[1].array.ctypes.data, pageable=flow.ctypes.data)
        for ks, kf, kd in itertools.product(("device", "pinned", "pageable"), repeat=3):
            d_t = torch.full(src.shape, 1, dtype=torch.uint8, device=dev)
            d_np = np.full(src.shape, 1, np.uint8)
            pins[2].array[...] = 1
            dsts = dict(device=d_t.data_ptr(), pinned=pins[2].array.ctypes.data, pageable=d_np.ctypes.data)
            gpu_ctx.remap_flow_ptr(srcs[ks], n, w, h, c, w * c, w * h * c, flows[kf], w * 8, w * h * 8, dsts[kd], w * c,
                                   w * h * c, 1, 0)
            got = dict(device=lambda: d_t.cpu().numpy(), pinned=lambda: pins[2].array, pageable=lambda: d_np)[kd]()
            assert np.array_equal(got, want), (ks, kf, kd)
        for extra in (4, 2):
            pitch = w * 8 + extra
            buf = torch.zeros(n * h * pitch + extra, dtype=torch.uint8, device=dev)
            host = np.zeros(buf.numel(), np.uint8)
            for i in range(n):
                rows = host[extra + i * h * pitch:extra + (i + 1) * h * pitch].reshape(h, pitch)
                rows[:, :w * 8] = flow[i].view(np.uint8).reshape(h, w * 8)
            buf.copy_(torch.from_numpy(host))
            d_t = torch.empty(src.shape, dtype=torch.uint8, device=dev)
            gpu_ctx.remap_flow_ptr(s_t.data_ptr(), n, w, h, c, w * c, w * h * c, buf.data_ptr() + extra, pitch, h * pitch,
                                   d_t.data_ptr(), w * c, w * h * c, 1, 0)
            assert np.array_equal(d_t.cpu().numpy(), want), extra
    finally:
        for p in pins:
            p.free()


@pytest.mark.gpu
def test_gpu_torch_tensors_on_a_side_stream(gpu_ctx):
    torch = pytest.importorskip("torch")
    w, h, n = 640, 360, 9
    flow = smooth_flows(n, h, w, seed=5)
    src = images(n, h, w, 3, seed=6)
    want = cv_batch(src, flow, 0, 7)
    dev = torch.device("cuda", gpu_ctx.device)
    side = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(side):
        # the inputs are written on the side stream by torch ops, read there by the call, and the output read there
        s_t = torch.from_numpy(src.astype(np.int16)).to(dev).add_(0).to(torch.uint8)
        f_t = torch.from_numpy(flow).to(dev).mul_(1.0)
        got = api.remap_by_flow(s_t, f_t, 0, 7, ctx=gpu_ctx)
        one = api.remap_by_flow(s_t[4], f_t[4], 0, 7, ctx=gpu_ctx)
        host, host_one = got.cpu(), one.cpu()
    side.synchronize()
    assert got.device == dev and got.dtype == torch.uint8 and tuple(got.shape) == src.shape
    assert np.array_equal(host.numpy(), want) and np.array_equal(host_one.numpy(), want[4])
    with pytest.raises(TypeError):
        api.remap_by_flow(s_t, flow, ctx=gpu_ctx)
    with pytest.raises(TypeError):
        api.remap_by_flow(s_t.cpu(), f_t.cpu(), ctx=gpu_ctx)
    with pytest.raises(TypeError):
        api.remap_by_flow(s_t.float(), f_t, ctx=gpu_ctx)


@pytest.mark.gpu
def test_gpu_no_allocation_after_first_call(gpu_ctx):
    w, h = 1920, 1080
    flow = smooth_flows(3, h, w, seed=7)
    src = images(3, h, w, 3, seed=7)
    gpu_ctx.remap_flow(src, flow)
    before = gpu_ctx.alloc_counts()
    for _ in range(2):
        gpu_ctx.remap_flow(src, flow, 1)
        gpu_ctx.remap_flow(src[..., 0], flow)
        gpu_ctx.remap_flow(src[:1, :360, :640], flow[:1, :360, :640])
    assert gpu_ctx.alloc_counts() == before


@pytest.mark.gpu
def test_gpu_sequence_then_remap_on_tensors(gpu_ctx):
    """calc_optical_flow_farneback_sequence then remap_by_flow(frames[1:], flows), all on the device, equal to cv2.remap
    on host copies of the same frames and flows."""
    torch = pytest.importorskip("torch")
    w, h, n = 1920, 1080, 6
    clip = make_clip(w, h, n, seed=21, period=9.0, amplitude=0.35)
    dev = torch.device("cuda", gpu_ctx.device)
    frames = torch.from_numpy(clip).to(dev)
    flows = api.calc_optical_flow_farneback_sequence(frames, None, *REF, 0, ctx=gpu_ctx)
    warped = api.remap_by_flow(frames[1:], flows, 1, ctx=gpu_ctx)
    torch.cuda.current_stream(dev).synchronize()
    f_host = flows.cpu().numpy()
    assert np.array_equal(warped.cpu().numpy(), cv_batch(clip[1:], f_host, 1))
