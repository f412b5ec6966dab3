"""ctypes binding of libffb.so (the C ABI in include/ffb.h).

There is deliberately no fallback: if the CUDA library is missing or no device is usable the
import of a context raises.  (`load(path)` accepts an explicit path only so the CPU test-suite
can point it at the g++-built emulation of the same sources under tests/emu/.)
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
DEFAULT_LIB = os.path.join(_HERE, "libffb.so")

K_NAMES = ["pyramid", "polyexp", "upsample", "flow_iter", "divmag", "radial", "small", "preprocess", "fb_check", "remap"]
K_FLOW_ITER = 3


class FFBError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"ffb error {code}: {msg}")
        self.code = code


_libs = {}


def load(path: Optional[str] = None) -> C.CDLL:
    path = os.path.abspath(path or DEFAULT_LIB)
    if path in _libs:
        return _libs[path]
    if not os.path.exists(path):
        raise FileNotFoundError(
            f"{path} not found: build it with `python -m funscript_flow_b200.build` (needs nvcc). "
            "There is no CPU fallback.")
    lib = C.CDLL(path)
    vp, i32, u8p, f32p, f64p, i32p, sz = (C.c_void_p, C.c_int, C.POINTER(C.c_uint8), C.POINTER(C.c_float),
                                          C.POINTER(C.c_double), C.POINTER(C.c_int32), C.c_size_t)
    sig = {
        "ffb_version": (i32, []),
        "ffb_device_count": (i32, [i32p]),
        "ffb_device_pci_bus_id": (i32, [i32, C.c_char_p, i32]),
        "ffb_device_name": (i32, [i32, C.c_char_p, i32]),
        "ffb_last_error": (C.c_char_p, [vp]),
        "ffb_create": (i32, [i32, C.POINTER(vp)]),
        "ffb_destroy": (None, [vp]),
        "ffb_host_alloc": (i32, [C.POINTER(vp), sz]),
        "ffb_host_free": (i32, [vp]),
        "ffb_configure": (i32, [vp, i32, i32, i32, i32]),
        "ffb_get_geometry": (i32, [vp, i32p, i32p, i32p, i32p]),
        "ffb_alloc_counts": (i32, [vp, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
        "ffb_bracket_begin": (i32, [vp, i32, C.c_double]),
        "ffb_bracket_begin_shard": (i32, [vp, i32, C.c_double, i32]),
        "ffb_bracket_phase1_finish": (i32, [vp, i32p, i32p, i32p, f32p, f32p, u8p]),
        "ffb_bracket_radial": (i32, [vp, i32p, i32p, i32, i32, f64p, f64p]),
        "ffb_bracket_push": (i32, [vp, vp, i32, sz, sz]),
        "ffb_bracket_finish": (i32, [vp, i32p, f64p, u8p, i32p, i32p, f32p, f32p, f64p]),
        "ffb_sync": (i32, [vp]),
        "ffb_chain_after": (i32, [vp, vp]),
        "ffb_bracket_abort": (i32, [vp]),
        "ffb_bracket_get_flow": (i32, [vp, i32, f32p]),
        "ffb_flow_ring_size": (i32, [vp]),
        "ffb_farneback": (i32, [vp, u8p, u8p, i32, i32, sz, f32p]),
        "ffb_farneback_pairs": (i32, [vp, vp, vp, i32, i32, i32, sz, sz, vp, sz, sz, i32, C.c_double, i32p, i32p, f32p, f32p,
                                      u8p, vp]),
        "ffb_farneback_sequence": (i32, [vp, vp, i32, i32, i32, sz, sz, vp, sz, sz, i32, C.c_double, f64p, u8p, i32p, i32p,
                                         f32p, f32p, f64p, vp]),
        "ffb_farneback_sequence_bidir": (i32, [vp, vp, i32, i32, i32, sz, sz, vp, vp, sz, sz, vp, sz, sz, C.c_double,
                                               C.c_double, C.POINTER(C.c_int64), vp]),
        "ffb_farneback_pairs_bidir": (i32, [vp, vp, vp, i32, i32, i32, sz, sz, vp, vp, sz, sz, vp, sz, sz, C.c_double,
                                            C.c_double, C.POINTER(C.c_int64), vp]),
        "ffb_remap_flow": (i32, [vp, vp, i32, i32, i32, i32, sz, sz, vp, sz, sz, vp, sz, sz, i32, i32, vp]),
        "ffb_max_divergence": (i32, [vp, f32p, i32, i32, i32p, i32p, f32p]),
        "ffb_mean_magnitude": (i32, [vp, f32p, i32, i32, f32p]),
        "ffb_radial_motion": (i32, [vp, f32p, i32, i32, C.c_double, C.c_double, i32, i32, f64p]),
        "ffb_level_plan": (i32, [i32, i32, i32p, i32p, i32p, i32p, f64p]),
        "ffb_set_farneback": (i32, [vp, C.c_double, i32, i32, i32, i32, C.c_double, i32]),
        "ffb_get_farneback": (i32, [vp, f64p, i32p, i32p, i32p, i32p, f64p, i32p]),
        "ffb_level_plan_ex": (i32, [i32, i32, C.c_double, i32, i32, i32p, i32p, i32p, i32p, f64p]),
        "ffb_stage_pyramid": (i32, [vp, u8p, i32, i32, sz, i32, f32p]),
        "ffb_stage_polyexp": (i32, [vp, f32p, i32, i32, f32p]),
        "ffb_stage_update_matrices": (i32, [vp, f32p, f32p, f32p, i32, i32, f32p]),
        "ffb_stage_flow_iter": (i32, [vp, f32p, f32p, f32p, i32, i32, f32p]),
        "ffb_stage_upsample_flow": (i32, [vp, f32p, i32, i32, i32, i32, f32p]),
        "ffb_stage_fb_check": (i32, [vp, f32p, f32p, i32, i32, C.c_double, C.c_double, u8p, C.POINTER(C.c_int64)]),
        "ffb_preprocess_configure": (i32, [vp, i32, i32, i32]),
        "ffb_bracket_push_bgr": (i32, [vp, vp, i32, sz, sz]),
        "ffb_stage_preprocess": (i32, [vp, u8p, i32, i32, sz, i32, u8p]),
        "ffb_preprocess_configure_window": (i32, [vp] + [i32] * 8),
        "ffb_stage_preprocess_window": (i32, [vp, u8p, i32, i32, sz] + [i32] * 6 + [u8p]),
        "ffb_profile": (i32, [vp, i32]),
        "ffb_profile_reset": (i32, [vp]),
        "ffb_kernel_stats": (i32, [vp, i32, C.POINTER(C.c_int64), f64p, f64p]),
        "ffb_flow_iter_level_stats": (i32, [vp, i32, C.POINTER(C.c_int64), f64p, f64p]),
        "ffb_launch_count": (C.c_int64, [vp]),
        "ffb_kernel_name": (C.c_char_p, [i32]),
        "ffb_timer_mark": (i32, [vp, i32]),
        "ffb_timer_elapsed": (i32, [vp, i32, i32, f64p]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)   # AttributeError here = the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    lib._ffb_symbols = sorted(sig)
    _libs[path] = lib
    return lib


def device_count(lib_path: Optional[str] = None) -> int:
    n = C.c_int32(0)
    load(lib_path).ffb_device_count(C.byref(n))
    return int(n.value)


def device_pci_bus_id(device: int = 0, lib_path: Optional[str] = None) -> Optional[str]:
    buf = C.create_string_buffer(32)
    if load(lib_path).ffb_device_pci_bus_id(int(device), buf, 32) != 0:
        return None
    return buf.value.decode().lower()


def device_name(device: int = 0, lib_path: Optional[str] = None) -> Optional[str]:
    buf = C.create_string_buffer(256)
    if load(lib_path).ffb_device_name(int(device), buf, 256) != 0:
        return None
    return buf.value.decode()


def level_plan(width: int, height: int, lib_path: Optional[str] = None):
    lib = load(lib_path)
    n = C.c_int32(0)
    w = (C.c_int32 * 4)()
    h = (C.c_int32 * 4)()
    ks = (C.c_int32 * 4)()
    sg = (C.c_double * 4)()
    rc = lib.ffb_level_plan(width, height, C.byref(n), w, h, ks, sg)
    if rc:
        raise FFBError(rc, "ffb_level_plan")
    return [dict(w=w[i], h=h[i], ksize=ks[i], sigma=sg[i]) for i in range(n.value)]


MAX_PLAN_LEVELS = 16


def level_plan_ex(width: int, height: int, pyr_scale: float, levels: int, lib_path: Optional[str] = None):
    """Level geometry (coarsest first) for any (pyr_scale, levels): list of dicts k, w, h, ksize, sigma."""
    lib = load(lib_path)
    n = C.c_int32(0)
    w, h, ks = ((C.c_int32 * MAX_PLAN_LEVELS)() for _ in range(3))
    sg = (C.c_double * MAX_PLAN_LEVELS)()
    rc = lib.ffb_level_plan_ex(int(width), int(height), float(pyr_scale), int(levels), MAX_PLAN_LEVELS, C.byref(n), w, h, ks, sg)
    if rc:
        raise FFBError(rc, f"ffb_level_plan_ex({width}, {height}, {pyr_scale}, {levels})")
    return [dict(k=n.value - 1 - i, w=w[i], h=h[i], ksize=ks[i], sigma=sg[i]) for i in range(n.value)]


def _u8(a):
    return a.ctypes.data_as(C.POINTER(C.c_uint8))


def _f32(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _bidir_outputs(n, width, height, flow, flow_bw, flow_pitch, flow_stride, mask, mask_pitch, mask_stride):
    """The output arguments of a bidirectional call, from pointers (0 = none) with their pitches and strides or from
    dense NumPy arrays: float32 [n, H, W, 2] flows, a uint8 / bool [n, H, W] mask."""
    ptrs = []
    for arr in (flow, flow_bw):
        if isinstance(arr, np.ndarray):
            assert arr.dtype == np.float32 and arr.flags.c_contiguous and arr.shape == (n, height, width, 2)
            flow_pitch, flow_stride = width * 8, width * height * 8
            ptrs.append(arr.ctypes.data)
        else:
            ptrs.append(int(arr or 0))
    if isinstance(mask, np.ndarray):
        assert mask.dtype in (np.uint8, np.bool_) and mask.flags.c_contiguous and mask.shape == (n, height, width)
        mask_ptr, mask_pitch, mask_stride = mask.ctypes.data, width, width * height
    else:
        mask_ptr = int(mask or 0)
    return (C.c_void_p(ptrs[0] or None), C.c_void_p(ptrs[1] or None), int(flow_pitch), int(flow_stride),
            C.c_void_p(mask_ptr or None), int(mask_pitch), int(mask_stride))


class PinnedBuffer:
    """Page-locked host memory exposed as a NumPy uint8 array (frames DMA straight out of it)."""

    def __init__(self, shape, lib_path: Optional[str] = None):
        self._lib = load(lib_path)
        self.nbytes = int(np.prod(shape))
        p = C.c_void_p()
        rc = self._lib.ffb_host_alloc(C.byref(p), self.nbytes)
        if rc:
            raise FFBError(rc, "ffb_host_alloc")
        self._ptr = p
        self.array = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(self.nbytes,)).reshape(shape)

    def free(self):
        if self._ptr:
            self.array = None
            self._lib.ffb_host_free(self._ptr)
            self._ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class FlowContext:
    """One GPU, one host thread.  Thin, allocation-free wrappers over the C ABI."""

    def __init__(self, device: int = 0, lib_path: Optional[str] = None):
        self._lib = load(lib_path)
        self.lib_path = lib_path
        h = C.c_void_p()
        rc = self._lib.ffb_create(int(device), C.byref(h))
        if rc:
            raise FFBError(rc, (self._lib.ffb_last_error(None) or b"").decode())
        self._h = h
        self.device = device

    # -- plumbing
    def _ck(self, rc: int):
        if rc:
            raise FFBError(rc, (self._lib.ffb_last_error(self._h) or b"").decode())

    def close(self):
        if getattr(self, "_h", None):
            self._lib.ffb_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # -- geometry / bracket API
    def configure(self, width: int, height: int, batch_frames: int = 16, max_bracket_pairs: int = 4096):
        """Incremental on the C side: unchanged or smaller requests touch nothing on the device."""
        self._ck(self._lib.ffb_configure(self._h, int(width), int(height), int(batch_frames), int(max_bracket_pairs)))

    @property
    def geometry(self):
        """(width, height, batch_frames, max_bracket_pairs) of the last successful configure, None before it."""
        v = [C.c_int32(0) for _ in range(4)]
        self._ck(self._lib.ffb_get_geometry(self._h, *(C.byref(x) for x in v)))
        geo = tuple(int(x.value) for x in v)
        return geo if geo[0] > 0 else None

    def alloc_counts(self):
        """(cudaMalloc calls, cudaHostAlloc calls) made for this context so far."""
        d, h = C.c_int64(0), C.c_int64(0)
        self._ck(self._lib.ffb_alloc_counts(self._h, C.byref(d), C.byref(h)))
        return int(d.value), int(h.value)

    def set_farneback(self, pyr_scale: float = 0.5, levels: int = 3, winsize: int = 15, iterations: int = 3,
                      poly_n: int = 5, poly_sigma: float = 1.2, flags: int = 0):
        """Parameters of every flow this context computes (cv2.calcOpticalFlowFarneback's, after `flow`); the defaults
        are the reference's call.  Equal parameters change nothing; refused inside a bracket."""
        self._ck(self._lib.ffb_set_farneback(self._h, float(pyr_scale), int(levels), int(winsize), int(iterations), int(poly_n),
                                             float(poly_sigma), int(flags)))

    @property
    def farneback_params(self) -> dict:
        """The parameters set_farneback took last (the reference's for a new context)."""
        ps, sg = C.c_double(), C.c_double()
        lv, ws, it, pn, fl = (C.c_int32() for _ in range(5))
        self._ck(self._lib.ffb_get_farneback(self._h, C.byref(ps), C.byref(lv), C.byref(ws), C.byref(it), C.byref(pn),
                                             C.byref(sg), C.byref(fl)))
        return dict(pyr_scale=ps.value, levels=lv.value, winsize=ws.value, iterations=it.value, poly_n=pn.value,
                    poly_sigma=sg.value, flags=fl.value)

    def bracket_begin(self, pov_mode: bool = False, cut_threshold: float = 7.0):
        self._ck(self._lib.ffb_bracket_begin(self._h, int(bool(pov_mode)), float(cut_threshold)))

    # -- frame-range shard of a bracket: phase 1 (flows, raw centres, cut test), exchange of the raw centres
    #    with the neighbouring shards on the host, phase 2 (radial scalars)
    def bracket_begin_shard(self, shard_pairs: int, pov_mode: bool = False, cut_threshold: float = 7.0):
        self._ck(self._lib.ffb_bracket_begin_shard(self._h, int(bool(pov_mode)), float(cut_threshold), int(shard_pairs)))

    def bracket_phase1_finish(self):
        m = self.geometry[3]
        out = dict(cx=np.empty(m, np.int32), cy=np.empty(m, np.int32), val=np.empty(m, np.float32),
                   mean_mag=np.empty(m, np.float32), cut=np.empty(m, np.uint8))
        n = C.c_int32(0)
        i32p = C.POINTER(C.c_int32)
        self._ck(self._lib.ffb_bracket_phase1_finish(self._h, C.byref(n), out["cx"].ctypes.data_as(i32p),
                                                     out["cy"].ctypes.data_as(i32p), _f32(out["val"]), _f32(out["mean_mag"]),
                                                     _u8(out["cut"])))
        k = n.value
        res = {key: v[:k].copy() for key, v in out.items()}
        res["cut"] = res["cut"].astype(bool)
        res["n_pairs"] = k
        return res

    def bracket_radial(self, cx_ext, cy_ext, first: int, n_pairs: int):
        """cx_ext / cy_ext: raw centres of the shard's pairs and of up to 6 neighbours on each side (clipped to the
        bracket), the shard's first pair at index `first`.  Returns (scalar f64[n], centers f64[n, 2])."""
        cx_ext = np.ascontiguousarray(cx_ext, np.int32)
        cy_ext = np.ascontiguousarray(cy_ext, np.int32)
        assert cx_ext.shape == cy_ext.shape and cx_ext.ndim == 1
        scalar = np.empty(max(n_pairs, 1), np.float64)
        centers = np.empty((max(n_pairs, 1), 2), np.float64)
        i32p, f64p = C.POINTER(C.c_int32), C.POINTER(C.c_double)
        self._ck(self._lib.ffb_bracket_radial(self._h, cx_ext.ctypes.data_as(i32p), cy_ext.ctypes.data_as(i32p), int(cx_ext.size),
                                              int(first), scalar.ctypes.data_as(f64p), centers.ctypes.data_as(f64p)))
        return scalar[:n_pairs].copy(), centers[:n_pairs].copy()

    def bracket_push(self, frames: np.ndarray):
        """frames: uint8 [n, H, W] (or [H, W]); the last axis must be contiguous."""
        if frames.ndim == 2:
            frames = frames[None]
        assert frames.dtype == np.uint8 and frames.ndim == 3 and frames.strides[2] == 1
        n = frames.shape[0]
        stride = frames.strides[0] if n > 1 else frames.strides[1] * frames.shape[1]
        self._ck(self._lib.ffb_bracket_push(self._h, frames.ctypes.data, n, frames.strides[1], stride))

    def bracket_push_ptr(self, ptr: int, n: int, pitch: int, frame_stride: int):
        """Raw pointer variant (device pointers, e.g. torch_tensor.data_ptr())."""
        self._ck(self._lib.ffb_bracket_push(self._h, C.c_void_p(ptr), int(n), int(pitch), int(frame_stride)))

    def preprocess_configure(self, src_width: int, src_height: int, vr_mode: bool = False):
        """Source geometry of decoded BGR frames for bracket_push_bgr (output is always 256x256)."""
        self._ck(self._lib.ffb_preprocess_configure(self._h, int(src_width), int(src_height), int(bool(vr_mode))))

    def preprocess_configure_window(self, src_width: int, src_height: int, target, window):
        """General form (row N4): resize to target=(w, h), keep window=(x, y, w, h) of the resized frame."""
        self._ck(self._lib.ffb_preprocess_configure_window(self._h, int(src_width), int(src_height), int(target[0]), int(target[1]),
                                                           *(int(v) for v in window)))

    def bracket_push_bgr(self, frames: np.ndarray):
        """frames: uint8 [n, H, W, 3] (or [H, W, 3]) BGR as decoded; resized + gray-converted on the GPU."""
        if frames.ndim == 3:
            frames = frames[None]
        assert frames.dtype == np.uint8 and frames.ndim == 4 and frames.shape[3] == 3
        assert frames.strides[3] == 1 and frames.strides[2] == 3
        n = frames.shape[0]
        stride = frames.strides[0] if n > 1 else frames.strides[1] * frames.shape[1]
        self._ck(self._lib.ffb_bracket_push_bgr(self._h, frames.ctypes.data, n, frames.strides[1], stride))

    def stage_preprocess(self, bgr: np.ndarray, vr_mode: bool = False) -> np.ndarray:
        bgr = np.ascontiguousarray(bgr, dtype=np.uint8)
        h, w = bgr.shape[:2]
        out = np.empty((256, 256), np.uint8)
        self._ck(self._lib.ffb_stage_preprocess(self._h, _u8(bgr), w, h, w * 3, int(bool(vr_mode)), _u8(out)))
        return out

    def stage_preprocess_window(self, bgr: np.ndarray, target, window) -> np.ndarray:
        bgr = np.ascontiguousarray(bgr, dtype=np.uint8)
        h, w = bgr.shape[:2]
        out = np.empty((int(window[3]), int(window[2])), np.uint8)
        self._ck(self._lib.ffb_stage_preprocess_window(self._h, _u8(bgr), w, h, w * 3, int(target[0]), int(target[1]),
                                                       *(int(v) for v in window), _u8(out)))
        return out

    def bracket_abort(self):
        """Drop the open bracket (error path / cancel); the context can be configured again afterwards."""
        self._ck(self._lib.ffb_bracket_abort(self._h))

    def bracket_finish(self):
        m = self.geometry[3]
        out = dict(scalar=np.empty(m, np.float64), cut=np.empty(m, np.uint8), cx=np.empty(m, np.int32),
                   cy=np.empty(m, np.int32), val=np.empty(m, np.float32), mean_mag=np.empty(m, np.float32),
                   centers=np.empty((m, 2), np.float64))
        n = C.c_int32(0)
        self._ck(self._lib.ffb_bracket_finish(
            self._h, C.byref(n), out["scalar"].ctypes.data_as(C.POINTER(C.c_double)), _u8(out["cut"]),
            out["cx"].ctypes.data_as(C.POINTER(C.c_int32)), out["cy"].ctypes.data_as(C.POINTER(C.c_int32)),
            _f32(out["val"]), _f32(out["mean_mag"]), out["centers"].ctypes.data_as(C.POINTER(C.c_double))))
        k = n.value
        res = {key: v[:k].copy() for key, v in out.items()}
        res["cut"] = res["cut"].astype(bool)
        res["n_pairs"] = k
        return res

    def chain_after(self, earlier: "FlowContext"):
        """Kernels queued on this context from now on start after everything `earlier` (same device) has queued."""
        self._ck(self._lib.ffb_chain_after(self._h, earlier._h))

    def sync(self):
        self._ck(self._lib.ffb_sync(self._h))

    def get_flow(self, pair: int) -> np.ndarray:
        w, h = self.geometry[:2]
        out = np.empty((h, w, 2), np.float32)
        self._ck(self._lib.ffb_bracket_get_flow(self._h, int(pair), _f32(out)))
        return out

    @property
    def flow_ring_size(self) -> int:
        return int(self._lib.ffb_flow_ring_size(self._h))

    # -- per-call functions
    def farneback(self, prev: np.ndarray, nxt: np.ndarray) -> np.ndarray:
        prev = np.ascontiguousarray(prev, dtype=np.uint8)
        nxt = np.ascontiguousarray(nxt, dtype=np.uint8)
        assert prev.shape == nxt.shape and prev.ndim == 2
        h, w = prev.shape
        out = np.empty((h, w, 2), np.float32)
        self._ck(self._lib.ffb_farneback(self._h, _u8(prev), _u8(nxt), w, h, w, _f32(out)))
        return out

    def farneback_pairs(self, prev: np.ndarray, nxt: np.ndarray, *, flow: bool = True, pov: bool = False,
                        cut_threshold: float = float("inf")) -> dict:
        """n independent pairs (prev[i], nxt[i]), uint8 [n, H, W] each, in one call (ffb_farneback_pairs): flow f32
        [n, H, W, 2] (None with flow=False), cx / cy (int32), val / mean_mag (float32) and cut (bool) per pair.  Each
        flow is bit-identical to farneback(prev[i], nxt[i]).  Pairs run in chunks of (batch_frames + 1) / 2 of the last
        configure(); a context never configured runs one pair per chunk, so configure it first (api's batch functions
        do)."""
        prev = np.ascontiguousarray(prev, dtype=np.uint8)
        nxt = np.ascontiguousarray(nxt, dtype=np.uint8)
        if prev.shape != nxt.shape or prev.ndim != 3:
            raise ValueError(f"farneback_pairs: prev and nxt must be uint8 [n, H, W] of one shape, not {prev.shape} and {nxt.shape}")
        n, h, w = prev.shape
        out = self.farneback_pairs_ptr(prev.ctypes.data, nxt.ctypes.data, n, w, h, w, w * h, stats=True, pov=pov,
                                       cut_threshold=cut_threshold,
                                       flow=np.empty((n, h, w, 2), np.float32) if flow else None)
        return out

    def farneback_pairs_ptr(self, prev_ptr: int, next_ptr: int, n: int, width: int, height: int, pitch: int,
                            frame_stride: int, flow=None, flow_pitch: int = 0, flow_stride: int = 0, stream: int = 0, *,
                            stats: bool = False, pov: bool = False, cut_threshold: float = float("inf")):
        """Raw-pointer variant of farneback_pairs, like bracket_push_ptr: frames anywhere (e.g. torch_tensor.data_ptr()),
        `flow` a pointer (int; 0 = no flow) or a float32 NumPy array, `stream` a cudaStream_t handle (0 = none; e.g.
        torch.cuda.current_stream().cuda_stream).  stats=True returns the per-pair dict (then the call waits for the
        device), otherwise None."""
        flow_arr = flow if isinstance(flow, np.ndarray) else None
        if flow_arr is not None:
            assert flow_arr.dtype == np.float32 and flow_arr.flags.c_contiguous and flow_arr.shape == (n, height, width, 2)
            flow_ptr, flow_pitch, flow_stride = flow_arr.ctypes.data, width * 8, width * height * 8
        else:
            flow_ptr = int(flow or 0)
        res = None
        args = [None] * 5
        if stats:
            res = dict(cx=np.empty(max(n, 1), np.int32), cy=np.empty(max(n, 1), np.int32), val=np.empty(max(n, 1), np.float32),
                       mean_mag=np.empty(max(n, 1), np.float32), cut=np.empty(max(n, 1), np.uint8))
            i32p = C.POINTER(C.c_int32)
            args = [res["cx"].ctypes.data_as(i32p), res["cy"].ctypes.data_as(i32p), _f32(res["val"]), _f32(res["mean_mag"]),
                    _u8(res["cut"])]
        self._ck(self._lib.ffb_farneback_pairs(self._h, C.c_void_p(prev_ptr), C.c_void_p(next_ptr), int(n), int(width),
                                               int(height), int(pitch), int(frame_stride), C.c_void_p(flow_ptr or None),
                                               int(flow_pitch), int(flow_stride), int(bool(pov)), float(cut_threshold), *args,
                                               C.c_void_p(int(stream) or None)))
        if res is None:
            return None
        res = {k: v[:n] for k, v in res.items()}
        res["cut"] = res["cut"].astype(bool)
        res["flow"] = flow_arr
        return res

    def farneback_sequence(self, frames: np.ndarray, *, flow: bool = True, stats: bool = False, pov: bool = False,
                           cut_threshold: float = float("inf")) -> dict:
        """The n - 1 pairs of consecutive frames of uint8 [n, H, W] in one call (ffb_farneback_sequence), each frame
        expanded once: {"flow": f32 [n - 1, H, W, 2]} (None with flow=False).  Each flow is bit-identical to
        farneback(frames[j], frames[j + 1]).  stats=True adds bracket_finish's per-pair arrays (scalar, cut, cx, cy, val,
        mean_mag, centers, n_pairs), bit-identical to a bracket of these frames with pov / cut_threshold.  Batches are
        those of the last configure(); a context never configured runs batches of 2 frames, so configure it first
        (api.calc_optical_flow_farneback_sequence does)."""
        frames = np.ascontiguousarray(frames, dtype=np.uint8)
        if frames.ndim != 3:
            raise ValueError(f"farneback_sequence: frames must be uint8 [n, H, W], not {frames.shape}")
        n, h, w = frames.shape
        out = np.empty((max(n - 1, 0), h, w, 2), np.float32) if flow else None
        res = self.farneback_sequence_ptr(frames.ctypes.data, n, w, h, w, w * h, out, stats=stats, pov=pov,
                                          cut_threshold=cut_threshold)
        return res if stats else {"flow": out}

    def farneback_sequence_ptr(self, frames_ptr: int, n_frames: int, width: int, height: int, pitch: int,
                               frame_stride: int, flow=None, flow_pitch: int = 0, flow_stride: int = 0, stream: int = 0, *,
                               stats: bool = False, pov: bool = False, cut_threshold: float = float("inf")):
        """Raw-pointer variant of farneback_sequence, like farneback_pairs_ptr: frames anywhere (e.g.
        torch_tensor.data_ptr()), `flow` a pointer (int; 0 = no flow) or a float32 NumPy array [n_frames - 1, H, W, 2],
        `stream` a cudaStream_t handle (0 = none).  stats=True returns the per-pair dict with "flow" (then the call waits
        for the device), otherwise None."""
        n = max(int(n_frames) - 1, 0)
        flow_arr = flow if isinstance(flow, np.ndarray) else None
        if flow_arr is not None:
            assert flow_arr.dtype == np.float32 and flow_arr.flags.c_contiguous and flow_arr.shape == (n, height, width, 2)
            flow_ptr, flow_pitch, flow_stride = flow_arr.ctypes.data, width * 8, width * height * 8
        else:
            flow_ptr = int(flow or 0)
        res = None
        args = [None] * 7
        if stats:
            m = max(n, 1)
            res = dict(scalar=np.empty(m, np.float64), cut=np.empty(m, np.uint8), cx=np.empty(m, np.int32),
                       cy=np.empty(m, np.int32), val=np.empty(m, np.float32), mean_mag=np.empty(m, np.float32),
                       centers=np.empty((m, 2), np.float64))
            i32p, f64p = C.POINTER(C.c_int32), C.POINTER(C.c_double)
            args = [res["scalar"].ctypes.data_as(f64p), _u8(res["cut"]), res["cx"].ctypes.data_as(i32p),
                    res["cy"].ctypes.data_as(i32p), _f32(res["val"]), _f32(res["mean_mag"]), res["centers"].ctypes.data_as(f64p)]
        self._ck(self._lib.ffb_farneback_sequence(self._h, C.c_void_p(frames_ptr), int(n_frames), int(width), int(height),
                                                  int(pitch), int(frame_stride), C.c_void_p(flow_ptr or None), int(flow_pitch),
                                                  int(flow_stride), int(bool(pov)), float(cut_threshold), *args,
                                                  C.c_void_p(int(stream) or None)))
        if res is None:
            return None
        res = {k: v[:n].copy() for k, v in res.items()}
        res["cut"] = res["cut"].astype(bool)
        res["n_pairs"] = n
        res["flow"] = flow_arr
        return res

    def farneback_sequence_bidir(self, frames: np.ndarray, *, forward: bool = True, backward: bool = True,
                                 mask: bool = True, counts: bool = True, alpha: float = 0.01, beta: float = 0.5) -> dict:
        """farneback_sequence plus, for pair j, the backward flow (frames[j + 1] -> frames[j]) and the forward-backward
        consistency check, in one call (ffb_farneback_sequence_bidir; each frame expanded once): {"flow": f32
        [n - 1, H, W, 2], "flow_bw": the same, "mask": bool [n - 1, H, W], "n_consistent": int64 [n - 1]}, an output
        not asked for is None.  "flow" is farneback_sequence's, flow_bw[j] is bit-identical to
        farneback(frames[j + 1], frames[j]), and mask[j] is True where |f + b|^2 <= alpha (|f|^2 + |b|^2) + beta with b
        the backward flow sampled bilinearly at the forward target (False for a target outside the frame).  Batches are
        those of the last configure(), as in farneback_sequence."""
        frames = np.ascontiguousarray(frames, dtype=np.uint8)
        if frames.ndim != 3:
            raise ValueError(f"farneback_sequence_bidir: frames must be uint8 [n, H, W], not {frames.shape}")
        n, h, w = frames.shape
        m = max(n - 1, 0)
        fw = np.empty((m, h, w, 2), np.float32) if forward else None
        bw = np.empty((m, h, w, 2), np.float32) if backward else None
        mk = np.empty((m, h, w), np.uint8) if mask else None
        cnt = self.farneback_sequence_bidir_ptr(frames.ctypes.data, n, w, h, w, w * h, fw, bw, mask=mk, counts=counts,
                                                alpha=alpha, beta=beta)
        return {"flow": fw, "flow_bw": bw, "mask": None if mk is None else mk.view(np.bool_), "n_consistent": cnt}

    def farneback_sequence_bidir_ptr(self, frames_ptr: int, n_frames: int, width: int, height: int, pitch: int,
                                     frame_stride: int, flow=None, flow_bw=None, flow_pitch: int = 0, flow_stride: int = 0,
                                     mask=None, mask_pitch: int = 0, mask_stride: int = 0, stream: int = 0, *,
                                     counts: bool = False, alpha: float = 0.01, beta: float = 0.5):
        """Raw-pointer variant of farneback_sequence_bidir, like farneback_sequence_ptr: `flow` / `flow_bw` pointers
        (0 = none) sharing flow_pitch / flow_stride, or float32 NumPy arrays [n_frames - 1, H, W, 2]; `mask` a pointer
        (0 = none) or a uint8 / bool NumPy array [n_frames - 1, H, W]; `stream` a cudaStream_t handle (0 = none).
        Returns the int64 consistent-pixel counts with counts=True (the call then waits for the device), else None."""
        n = max(int(n_frames) - 1, 0)
        out = _bidir_outputs(n, width, height, flow, flow_bw, flow_pitch, flow_stride, mask, mask_pitch, mask_stride)
        cnt = np.empty(max(n, 1), np.int64) if counts else None
        self._ck(self._lib.ffb_farneback_sequence_bidir(
            self._h, C.c_void_p(frames_ptr), int(n_frames), int(width), int(height), int(pitch), int(frame_stride), *out,
            float(alpha), float(beta), None if cnt is None else cnt.ctypes.data_as(C.POINTER(C.c_int64)),
            C.c_void_p(int(stream) or None)))
        return None if cnt is None else cnt[:n].copy()

    def farneback_pairs_bidir(self, prev: np.ndarray, nxt: np.ndarray, *, forward: bool = True, backward: bool = True,
                              mask: bool = True, counts: bool = True, alpha: float = 0.01, beta: float = 0.5) -> dict:
        """farneback_pairs plus, for pair i, the backward flow (nxt[i] -> prev[i]) and the forward-backward consistency
        check, in one call (ffb_farneback_pairs_bidir; each frame expanded once): {"flow": f32 [n, H, W, 2], "flow_bw":
        the same, "mask": bool [n, H, W], "n_consistent": int64 [n]}, an output not asked for is None.  "flow" is
        farneback_pairs', flow_bw[i] is bit-identical to farneback(nxt[i], prev[i]), and the mask and counts are
        farneback_sequence_bidir's.  Chunks are those of the last configure(), as in farneback_pairs."""
        prev = np.ascontiguousarray(prev, dtype=np.uint8)
        nxt = np.ascontiguousarray(nxt, dtype=np.uint8)
        if prev.shape != nxt.shape or prev.ndim != 3:
            raise ValueError(f"farneback_pairs_bidir: prev and nxt must be uint8 [n, H, W] of one shape, not {prev.shape} "
                             f"and {nxt.shape}")
        n, h, w = prev.shape
        fw = np.empty((n, h, w, 2), np.float32) if forward else None
        bw = np.empty((n, h, w, 2), np.float32) if backward else None
        mk = np.empty((n, h, w), np.uint8) if mask else None
        cnt = self.farneback_pairs_bidir_ptr(prev.ctypes.data, nxt.ctypes.data, n, w, h, w, w * h, fw, bw, mask=mk,
                                             counts=counts, alpha=alpha, beta=beta)
        return {"flow": fw, "flow_bw": bw, "mask": None if mk is None else mk.view(np.bool_), "n_consistent": cnt}

    def farneback_pairs_bidir_ptr(self, prev_ptr: int, next_ptr: int, n: int, width: int, height: int, pitch: int,
                                  frame_stride: int, flow=None, flow_bw=None, flow_pitch: int = 0, flow_stride: int = 0,
                                  mask=None, mask_pitch: int = 0, mask_stride: int = 0, stream: int = 0, *,
                                  counts: bool = False, alpha: float = 0.01, beta: float = 0.5):
        """Raw-pointer variant of farneback_pairs_bidir, like farneback_pairs_ptr: frames anywhere, `flow` / `flow_bw`
        pointers (0 = none) sharing flow_pitch / flow_stride, or float32 NumPy arrays [n, H, W, 2]; `mask` a pointer
        (0 = none) or a uint8 / bool NumPy array [n, H, W]; `stream` a cudaStream_t handle (0 = none).  Returns the int64
        consistent-pixel counts with counts=True (the call then waits for the device), else None."""
        n = int(n)
        out = _bidir_outputs(max(n, 0), width, height, flow, flow_bw, flow_pitch, flow_stride, mask, mask_pitch,
                             mask_stride)
        cnt = np.empty(max(n, 1), np.int64) if counts else None
        self._ck(self._lib.ffb_farneback_pairs_bidir(
            self._h, C.c_void_p(prev_ptr), C.c_void_p(next_ptr), n, int(width), int(height), int(pitch),
            int(frame_stride), *out, float(alpha), float(beta),
            None if cnt is None else cnt.ctypes.data_as(C.POINTER(C.c_int64)), C.c_void_p(int(stream) or None)))
        return None if cnt is None else cnt[:max(n, 0)].copy()

    def remap_flow(self, src: np.ndarray, flow: np.ndarray, border_mode: int = 0, border_value: int = 0) -> np.ndarray:
        """cv2.remap(src, flow, None, cv2.INTER_LINEAR | cv2.WARP_RELATIVE_MAP, border_mode, (v, v, v)) bit for bit
        (ffb_remap_flow), for one image or a batch: src uint8 [H, W], [H, W, 3], [n, H, W] or [n, H, W, 3], flow float32
        [H, W, 2] or [n, H, W, 2] (its ndim tells one image from a batch).  border_mode 0 is cv2.BORDER_CONSTANT (value
        border_value), 1 cv2.BORDER_REPLICATE.  Returns uint8 of src's shape."""
        src = np.ascontiguousarray(src)
        flow = np.ascontiguousarray(flow)
        if src.dtype != np.uint8 or flow.dtype != np.float32:
            raise TypeError(f"remap_flow: src must be uint8 and flow float32, not {src.dtype} and {flow.dtype}")
        single = flow.ndim == 3
        src_b, flow_b = (src[None], flow[None]) if single else (src, flow)
        if flow_b.ndim != 4 or flow_b.shape[3] != 2 or src_b.shape[:3] != flow_b.shape[:3] or src_b.ndim not in (3, 4) \
                or (src_b.ndim == 4 and src_b.shape[3] != 3):
            raise ValueError(f"remap_flow: src {src.shape} and flow {flow.shape} are not [n,] H, W[, 3] and [n,] H, W, 2")
        n, h, w = flow_b.shape[:3]
        ch = 3 if src_b.ndim == 4 else 1
        out = np.empty_like(src_b)
        self.remap_flow_ptr(src_b.ctypes.data, n, w, h, ch, w * ch, w * h * ch, flow_b.ctypes.data, w * 8, w * h * 8,
                            out.ctypes.data, w * ch, w * h * ch, border_mode, border_value)
        return out[0] if single else out

    def remap_flow_ptr(self, src_ptr: int, n: int, width: int, height: int, channels: int, src_pitch: int, src_stride: int,
                       flow_ptr: int, flow_pitch: int, flow_stride: int, dst_ptr: int, dst_pitch: int, dst_stride: int,
                       border_mode: int = 0, border_value: int = 0, stream: int = 0):
        """Raw-pointer variant of remap_flow, like farneback_pairs_ptr: buffers anywhere (e.g. torch_tensor.data_ptr()),
        pitches and strides in bytes, `stream` a cudaStream_t handle (0 = none)."""
        self._ck(self._lib.ffb_remap_flow(self._h, C.c_void_p(int(src_ptr) or None), int(n), int(width), int(height),
                                          int(channels), int(src_pitch), int(src_stride), C.c_void_p(int(flow_ptr) or None),
                                          int(flow_pitch), int(flow_stride), C.c_void_p(int(dst_ptr) or None),
                                          int(dst_pitch), int(dst_stride), int(border_mode), int(border_value),
                                          C.c_void_p(int(stream) or None)))

    def max_divergence(self, flow: np.ndarray):
        flow = np.ascontiguousarray(flow, dtype=np.float32)
        h, w = flow.shape[:2]
        x, y, v = C.c_int32(), C.c_int32(), C.c_float()
        self._ck(self._lib.ffb_max_divergence(self._h, _f32(flow), w, h, C.byref(x), C.byref(y), C.byref(v)))
        return x.value, y.value, np.float32(v.value)

    def mean_magnitude(self, flow: np.ndarray) -> np.float32:
        flow = np.ascontiguousarray(flow, dtype=np.float32)
        h, w = flow.shape[:2]
        v = C.c_float()
        self._ck(self._lib.ffb_mean_magnitude(self._h, _f32(flow), w, h, C.byref(v)))
        return np.float32(v.value)

    def radial_motion(self, flow: np.ndarray, center, is_cut: bool, pov_mode: bool = False) -> float:
        flow = np.ascontiguousarray(flow, dtype=np.float32)
        h, w = flow.shape[:2]
        v = C.c_double()
        self._ck(self._lib.ffb_radial_motion(self._h, _f32(flow), w, h, float(center[0]), float(center[1]),
                                             int(bool(is_cut)), int(bool(pov_mode)), C.byref(v)))
        return float(v.value)

    # -- stage hooks
    def stage_pyramid(self, img: np.ndarray, level_k: int) -> np.ndarray:
        img = np.ascontiguousarray(img, dtype=np.uint8)
        h, w = img.shape
        fp = self.farneback_params
        plan = level_plan_ex(w, h, fp["pyr_scale"], fp["levels"], self._lib._name)
        lv = plan[len(plan) - 1 - level_k]
        out = np.empty((lv["h"], lv["w"]), np.float32)
        self._ck(self._lib.ffb_stage_pyramid(self._h, _u8(img), w, h, w, int(level_k), _f32(out)))
        return out

    def stage_polyexp(self, img: np.ndarray) -> np.ndarray:
        """f32 [h, w] -> f32 [h, w, 5] (converted from the kernel's 5 planes)."""
        img = np.ascontiguousarray(img, dtype=np.float32)
        h, w = img.shape
        out = np.empty((5, h, w), np.float32)
        self._ck(self._lib.ffb_stage_polyexp(self._h, _f32(img), w, h, _f32(out)))
        return np.ascontiguousarray(out.transpose(1, 2, 0))

    @staticmethod
    def _planes(R: np.ndarray) -> np.ndarray:
        return np.ascontiguousarray(np.asarray(R, np.float32).transpose(2, 0, 1))

    def stage_update_matrices(self, R0, R1, flow) -> np.ndarray:
        h, w = R0.shape[:2]
        p0, p1 = self._planes(R0), self._planes(R1)
        fl = None if flow is None else np.ascontiguousarray(flow, np.float32)
        out = np.empty((5, h, w), np.float32)
        self._ck(self._lib.ffb_stage_update_matrices(self._h, _f32(p0), _f32(p1), None if fl is None else _f32(fl),
                                                     w, h, _f32(out)))
        return np.ascontiguousarray(out.transpose(1, 2, 0))

    def stage_flow_iter(self, R0, R1, flow_in) -> np.ndarray:
        h, w = R0.shape[:2]
        p0, p1 = self._planes(R0), self._planes(R1)
        fl = None if flow_in is None else np.ascontiguousarray(flow_in, np.float32)
        out = np.empty((h, w, 2), np.float32)
        self._ck(self._lib.ffb_stage_flow_iter(self._h, _f32(p0), _f32(p1), None if fl is None else _f32(fl),
                                               w, h, _f32(out)))
        return out

    def stage_upsample_flow(self, flow_c: np.ndarray, w: int, h: int) -> np.ndarray:
        fc = np.ascontiguousarray(flow_c, np.float32)
        hc, wc = fc.shape[:2]
        out = np.empty((h, w, 2), np.float32)
        self._ck(self._lib.ffb_stage_upsample_flow(self._h, _f32(fc), wc, hc, w, h, _f32(out)))
        return out

    def stage_fb_check(self, flow_fw: np.ndarray, flow_bw: np.ndarray, alpha: float = 0.01, beta: float = 0.5):
        """The forward-backward check of one pair (k_fb_check) on host flows f32 [h, w, 2]: (mask bool [h, w], count)."""
        fw = np.ascontiguousarray(flow_fw, np.float32)
        bw = np.ascontiguousarray(flow_bw, np.float32)
        assert fw.shape == bw.shape and fw.ndim == 3 and fw.shape[2] == 2
        h, w = fw.shape[:2]
        mask = np.empty((h, w), np.uint8)
        n = C.c_int64()
        self._ck(self._lib.ffb_stage_fb_check(self._h, _f32(fw), _f32(bw), w, h, float(alpha), float(beta), _u8(mask),
                                              C.byref(n)))
        return mask.view(np.bool_), int(n.value)

    # -- instrumentation
    def profile(self, enable: bool):
        self._ck(self._lib.ffb_profile(self._h, int(enable)))

    def profile_reset(self):
        self._ck(self._lib.ffb_profile_reset(self._h))

    def kernel_stats(self):
        out = {}
        for kid, name in enumerate(K_NAMES):
            n, ms, by = C.c_int64(), C.c_double(), C.c_double()
            self._ck(self._lib.ffb_kernel_stats(self._h, kid, C.byref(n), C.byref(ms), C.byref(by)))
            out[name] = dict(launches=int(n.value), ms=float(ms.value), alg_bytes=float(by.value))
        return out

    def flow_iter_level_stats(self, levels: int = 4):
        """Flow-iteration launches / device ms / algorithmic bytes per pyramid level k (0 = full resolution) for
        k < levels (at most 16; the reference's plans have 4)."""
        out = {}
        for k in range(levels):
            n, ms, by = C.c_int64(), C.c_double(), C.c_double()
            self._ck(self._lib.ffb_flow_iter_level_stats(self._h, k, C.byref(n), C.byref(ms), C.byref(by)))
            if n.value:
                out[k] = dict(launches=int(n.value), ms=float(ms.value), alg_bytes=float(by.value))
        return out

    def timer_mark(self, slot: int):
        self._ck(self._lib.ffb_timer_mark(self._h, int(slot)))

    def timer_elapsed_ms(self, slot_from: int, slot_to: int) -> float:
        ms = C.c_double()
        self._ck(self._lib.ffb_timer_elapsed(self._h, int(slot_from), int(slot_to), C.byref(ms)))
        return float(ms.value)

    @property
    def launch_count(self) -> int:
        return int(self._lib.ffb_launch_count(self._h))
