"""Drop-in processing functions with the reference's names, signatures and return shapes
(FunscriptFlow.pyw, "F:n" = line n), backed by the sm_100a kernels through the C ABI.

    precompute_flow_info(p0, p1, config)            F:843-907   (8-key dict, F:898-907)
    precompute_flow_info_gpu(p0, p1, cut_threshold) F:982-1017  (the slot this build fills)
    precompute_wrapper(p, params)                   F:1019-1021
    max_divergence(flow)                            F:748-758
    radial_motion_weighted(flow, center, is_cut, pov_mode=False)   F:761-785
    get_available_backends()                        F:32-63
    calc_optical_flow_farneback(prev, next, None, pyr_scale, levels, winsize, iterations, poly_n, poly_sigma, 0)
                                                    cv2's signature (F:878), any parameter set
    calc_optical_flow_farneback_batch(prev, next, None, ...)   the same for n independent pairs ([n, H, W]; NumPy
                                                    arrays or torch CUDA tensors, which stay on the device)
    calc_optical_flow_farneback_batch_bidirectional(prev, next, None, ...)   the same plus the backward flows and the
                                                    forward-backward consistency mask ([n, H, W] bool)
    precompute_flow_info_batch(pairs, config)       [precompute_wrapper(p, config) for p in pairs] in one call
    calc_optical_flow_farneback_sequence(frames, None, ...)    the same for every pair of consecutive frames ([n, H, W]
                                                    -> [n - 1, H, W, 2]; each frame expanded once)
    calc_optical_flow_farneback_sequence_bidirectional(frames, None, ...)   the same plus the backward flows and the
                                                    forward-backward consistency mask ([n - 1, H, W] bool)
    remap_by_flow(src, flow, border_mode, border_value)   cv2.remap(src, flow, None, INTER_LINEAR | WARP_RELATIVE_MAP,
                                                    ...) bit for bit, for one image or a batch (NumPy or torch CUDA)

Every entry point that configures a context first sets its Farneback parameters from the settings keys
flow_pyr_scale, flow_levels, flow_winsize, flow_iterations, flow_poly_n, flow_poly_sigma (farneback_params;
a missing key means the reference's value).

plus the batched entry the GPU runner uses, because per-pair calls from forked pool workers
(F:1190-1191) cannot drive a GPU:

    process_bracket(frames, params) -> dict of per-pair arrays   (F:1188-1242 in one call)
    process_sequence(frames, params)                the same dict plus the flow of every pair

There is no CPU path here: every function raises if libffb.so or a CUDA device is missing.
"""
from __future__ import annotations

import os
from typing import Dict, Optional, Sequence

import numpy as np

from . import _native

DEFAULT_CUT_THRESHOLD = 7          # F:876
DEFAULT_BATCH_FRAMES = 64

# cv2.calcOpticalFlowFarneback's parameters in the reference's call (F:878-879) and the settings keys that override them
REFERENCE_FARNEBACK = dict(pyr_scale=0.5, levels=3, winsize=15, iterations=3, poly_n=5, poly_sigma=1.2)
FARNEBACK_SETTINGS = {"flow_pyr_scale": "pyr_scale", "flow_levels": "levels", "flow_winsize": "winsize",
                      "flow_iterations": "iterations", "flow_poly_n": "poly_n", "flow_poly_sigma": "poly_sigma"}


def farneback_params(params: Optional[Dict]) -> Dict:
    """The Farneback parameters a settings dict asks for: the flow_* keys, the reference's value where one is missing."""
    params = params or {}
    out = dict(REFERENCE_FARNEBACK)
    for key, name in FARNEBACK_SETTINGS.items():
        if params.get(key) is not None:
            out[name] = type(REFERENCE_FARNEBACK[name])(params[key])
    return out


def apply_farneback(ctx: "_native.FlowContext", params: Optional[Dict]) -> None:
    """Set the context's Farneback parameters from a settings dict (a no-op when they are already set)."""
    ctx.set_farneback(**farneback_params(params))

_contexts: Dict[int, _native.FlowContext] = {}


def default_device() -> int:
    """FFB_DEVICE, else the torchrun LOCAL_RANK folded onto the visible devices (ranks may share a GPU), else 0."""
    if os.environ.get("FFB_DEVICE", "") != "":
        return int(os.environ["FFB_DEVICE"])
    if os.environ.get("LOCAL_RANK", "") != "":
        try:
            n = _native.device_count()
        except Exception:
            n = 0
        return int(os.environ["LOCAL_RANK"]) % max(1, n)
    return 0


def get_context(device: Optional[int] = None) -> _native.FlowContext:
    """Process-wide context per device (created lazily; raises without a GPU)."""
    dev = default_device() if device is None else int(device)
    ctx = _contexts.get(dev)
    if ctx is None:
        ctx = _native.FlowContext(dev)
        _contexts[dev] = ctx
    return ctx


_aux_contexts: Dict[int, _native.FlowContext] = {}


def get_aux_context(primary: _native.FlowContext) -> _native.FlowContext:
    """A second context on the device (and from the library) of `primary`, for work that runs beside it:
    the other eye of a side-by-side VR frame (runner, vr_eye="both")."""
    key = id(primary)
    ctx = _aux_contexts.get(key)
    if ctx is None:
        ctx = _native.FlowContext(primary.device, lib_path=primary.lib_path)
        _aux_contexts.clear()          # one auxiliary context at a time
        _aux_contexts[key] = ctx
    return ctx


def set_context(ctx: _native.FlowContext, device: int = 0) -> None:
    """Install an externally created context (tests use this to inject the emulated library)."""
    _contexts[int(device)] = ctx


def get_available_backends() -> Dict[str, bool]:
    """Shape of F:32-63's result.  Only the CUDA entry can be True: this build ships no CPU,
    OpenCL or DIS path."""
    try:
        n = _native.device_count()
    except Exception:
        n = 0
    return {"CPU": False, "CUDA": n > 0, "OpenCL": False, "DNN": False}


def get_gpu_info() -> str:
    """F:64-99: "CUDA: <device name>" for one GPU, "CUDA: <n> devices" for several, "CPU only" when there is none
    (the reference's wording for 'no accelerator'; this build cannot run in that case)."""
    try:
        n = _native.device_count()
    except Exception:
        n = 0
    if n <= 0:
        return "CPU only"
    if n == 1:
        return f"CUDA: {_native.device_name(0) or 'Device 0'}"
    return f"CUDA: {n} devices"


def _as_frames(frames) -> np.ndarray:
    if isinstance(frames, np.ndarray) and frames.ndim == 3:
        arr = frames
    else:
        arr = np.stack([np.asarray(f) for f in frames])
    if arr.dtype != np.uint8:
        raise TypeError("frames must be uint8 grayscale")
    return np.ascontiguousarray(arr)


def process_bracket(frames, params: Optional[Dict] = None, *, ctx: Optional[_native.FlowContext] = None,
                    batch_frames: int = DEFAULT_BATCH_FRAMES, return_flows: bool = False) -> Dict:
    """One bracket of N consecutive sampled frames -> N-1 pairs (F:1188-1242 as one GPU pass).

    Returns a dict with per-pair arrays: scalar (f64), cut (bool), cx / cy (int32), val (f32),
    mean_mag (f32), centers (f64 [N-1, 2], the +-6 smoothed centre) and n_pairs.  With
    return_flows=True also `flows` (f32 [k, H, W, 2]) for the last k <= ring pairs (tests).
    """
    params = params or {}
    ctx = ctx or get_context()
    arr = _as_frames(frames)
    n, h, w = arr.shape
    apply_farneback(ctx, params)
    ctx.configure(w, h, max(1, min(batch_frames, n)), max(n - 1, 1))
    ctx.bracket_begin(bool(params.get("pov_mode", False)), float(params.get("cut_threshold", DEFAULT_CUT_THRESHOLD)))
    try:
        ctx.bracket_push(arr)
    except BaseException:
        ctx.bracket_abort()      # leave the context usable
        raise
    res = ctx.bracket_finish()
    if return_flows:
        k = res["n_pairs"]
        first = max(0, k - ctx.flow_ring_size)
        res["flow_first"] = first
        res["flows"] = np.stack([ctx.get_flow(p) for p in range(first, k)]) if k else np.empty((0, h, w, 2), np.float32)
    return res


def shard_bounds(n_pairs: int, parts: int):
    """Contiguous, balanced pair ranges [a, b) of a bracket of n_pairs pairs for `parts` GPUs (SURVEY 8(e)): shard r
    needs frames a .. b (one frame of overlap with shard r+1).  Ranges may be empty when parts > n_pairs."""
    return [(n_pairs * r // parts, n_pairs * (r + 1) // parts) for r in range(parts)]


def shard_phase1(ctx: _native.FlowContext, frames, a: int, b: int, params: Optional[Dict] = None,
                 batch_frames: int = DEFAULT_BATCH_FRAMES) -> Dict:
    """Phase 1 of pairs [a, b) of the bracket `frames` on `ctx` (flows, raw centres, cut test; F:1188-1199).
    The shard's final flows stay resident in `ctx` until shard_phase2."""
    params = params or {}
    arr = _as_frames(frames[a:b + 1])
    n, h, w = arr.shape
    apply_farneback(ctx, params)
    ctx.configure(w, h, max(1, min(batch_frames, n)), max(n - 1, 1))
    ctx.bracket_begin_shard(n - 1, bool(params.get("pov_mode", False)), float(params.get("cut_threshold", DEFAULT_CUT_THRESHOLD)))
    try:
        ctx.bracket_push(arr)
        return ctx.bracket_phase1_finish()
    except BaseException:
        ctx.bracket_abort()
        raise


def shard_phase2(ctx: _native.FlowContext, cx_all: np.ndarray, cy_all: np.ndarray, a: int, b: int):
    """Phase 2 of pairs [a, b): cx_all / cy_all are the raw centres of ALL pairs of the bracket (gathered from the
    shards); the +-6 window (F:1201-1214) reads [a-6, b+6) clipped to the bracket.  Returns (scalar, centers)."""
    lo, hi = max(0, a - 6), min(len(cx_all), b + 6)
    return ctx.bracket_radial(cx_all[lo:hi], cy_all[lo:hi], a - lo, b - a)


def process_bracket_on_contexts(frames, params: Optional[Dict], ctxs: Sequence[_native.FlowContext],
                                batch_frames: int = DEFAULT_BATCH_FRAMES) -> Dict:
    """One bracket cut into len(ctxs) frame-range shards, shard r on ctxs[r] (several GPUs driven by one process, or
    several contexts of one GPU).  Same dict as process_bracket, bit for bit."""
    arr = _as_frames(frames)
    n_pairs = len(arr) - 1
    bounds = shard_bounds(n_pairs, len(ctxs))
    p1 = [shard_phase1(c, arr, a, b, params, batch_frames) if b > a else None for c, (a, b) in zip(ctxs, bounds)]
    cat = {k: np.concatenate([p[k] for p in p1 if p is not None]) for k in ("cx", "cy", "val", "mean_mag", "cut")}
    parts = [shard_phase2(c, cat["cx"], cat["cy"], a, b) for c, (a, b) in zip(ctxs, bounds) if b > a]
    cat["scalar"] = np.concatenate([p[0] for p in parts])
    cat["centers"] = np.concatenate([p[1] for p in parts])
    cat["n_pairs"] = n_pairs
    return cat


class BracketPipeline:
    """Consecutive brackets (of one video, or the clips of a library) pipelined over two contexts of one GPU: bracket
    i+1 is pushed -- its frames start uploading -- before the results of bracket i are fetched, so the upload of the
    first batch and the drain of the last one no longer sit between brackets.  The kernels of the two contexts are
    chained (ffb_chain_after), only uploads overlap.  Results are those of process_bracket, bit for bit.

        pipe = BracketPipeline(ctx)
        for frames in brackets:
            done = pipe.submit(frames, params)      # returns the result of the bracket submitted before, or None
        last = pipe.flush()

    Host frames (pinned or pageable) must stay valid until their bracket's result has been returned."""

    def __init__(self, ctx: Optional[_native.FlowContext] = None, batch_frames: int = DEFAULT_BATCH_FRAMES):
        primary = ctx or get_context()
        self.ctxs = [primary, get_aux_context(primary)]
        self.batch_frames = batch_frames
        self._turn = 0
        self._pending = None        # (context, keep-alive array) of the bracket whose result has not been fetched

    def submit(self, frames, params: Optional[Dict] = None):
        params = params or {}
        arr = _as_frames(frames)
        n, h, w = arr.shape
        ctx = self.ctxs[self._turn]
        other = self.ctxs[self._turn ^ 1]
        apply_farneback(ctx, params)
        ctx.configure(w, h, max(1, min(self.batch_frames, n)), max(n - 1, 1))
        if self._pending is not None:
            ctx.chain_after(other)
        ctx.bracket_begin(bool(params.get("pov_mode", False)), float(params.get("cut_threshold", DEFAULT_CUT_THRESHOLD)))
        try:
            ctx.bracket_push(arr)
        except BaseException:
            ctx.bracket_abort()
            raise
        done = self.flush()
        self._pending = (ctx, arr)
        self._turn ^= 1
        return done

    def flush(self):
        """Result of the bracket submitted last (None when there is none)."""
        if self._pending is None:
            return None
        ctx, _ = self._pending
        self._pending = None
        return ctx.bracket_finish()


def precompute_flow_info(p0: np.ndarray, p1: np.ndarray, config: Dict) -> Dict:
    """F:843-907.  `config["backend"]` is ignored (there is one backend); `pov_mode` and the
    hidden `cut_threshold` key are honoured like the CPU branch (F:876-894)."""
    ctx = get_context()
    p0 = np.ascontiguousarray(p0, dtype=np.uint8)
    p1 = np.ascontiguousarray(p1, dtype=np.uint8)
    if p0.shape != p1.shape or p0.ndim != 2:
        raise ValueError("p0 and p1 must be equal-sized 2-D uint8 arrays")
    h, w = p0.shape
    pov = bool(config.get("pov_mode"))
    apply_farneback(ctx, config)    # the context is shared: a call without flow_* keys switches back to the reference's
    ctx.configure(w, h, 2, 1)       # incremental: a context already configured for this frame size is left alone
    ctx.bracket_begin(pov, float(config.get("cut_threshold", DEFAULT_CUT_THRESHOLD)))
    try:
        ctx.bracket_push(p0)
        ctx.bracket_push(p1)
    except BaseException:
        ctx.bracket_abort()
        raise
    r = ctx.bracket_finish()
    flow = ctx.get_flow(0)
    if pov:   # F:882: plain Python ints and the int 0
        pos_center, val = (w // 2, h - 1), 0
    else:     # F:757-758: NumPy integer / float32 scalars
        pos_center, val = (np.int64(r["cx"][0]), np.int64(r["cy"][0])), np.float32(r["val"][0])
    return {
        "flow": flow,
        "pos_center": pos_center,
        "neg_center": pos_center,
        "val_pos": val,
        "val_neg": val,
        "cut": bool(r["cut"][0]),
        "cut_center": pos_center[0],
        "mean_mag": np.float32(r["mean_mag"][0]),
    }


def calc_optical_flow_farneback(prev: np.ndarray, next: np.ndarray, flow, pyr_scale: float, levels: int, winsize: int,
                                iterations: int, poly_n: int, poly_sigma: float, flags: int = 0, *,
                                ctx: Optional[_native.FlowContext] = None) -> np.ndarray:
    """cv2.calcOpticalFlowFarneback with cv2's positional order, on the GPU: float32 [H, W, 2] (x, y displacement).
    `flow` must be None (an initial flow, OPTFLOW_USE_INITIAL_FLOW, is not supported) and `flags` 0."""
    if flow is not None:
        raise ValueError("calc_optical_flow_farneback: flow must be None (an initial flow is not supported)")
    ctx = ctx or get_context()
    ctx.set_farneback(pyr_scale, levels, winsize, iterations, poly_n, poly_sigma, flags)
    return ctx.farneback(prev, next)


def _pairs_batch(width: int, height: int, n: int) -> int:
    """batch_frames for n independent pairs of width x height: the runner's batch for the frame size (chunks of
    (batch_frames + 1) / 2 pairs fill the GPU as a bracket's batches do), no more than n pairs need."""
    from .runner import default_batch_frames
    return max(1, min(default_batch_frames(width, height), 2 * n - 1))


def _is_torch_tensor(x) -> bool:
    return type(x).__module__.split(".")[0] == "torch"


def calc_optical_flow_farneback_batch(prev, next, flow, pyr_scale: float, levels: int, winsize: int, iterations: int,
                                      poly_n: int, poly_sigma: float, flags: int = 0, *,
                                      ctx: Optional[_native.FlowContext] = None):
    """calc_optical_flow_farneback for n independent pairs (prev[i], next[i]) in one call, cv2's order with a leading
    batch axis: uint8 [n, H, W] -> float32 [n, H, W, 2].  NumPy arrays give a NumPy array.  torch.uint8 CUDA tensors on
    the context's device give a tensor on that device, ordered on torch.cuda.current_stream(): the frames and the flow
    never pass through host memory.  `flow` must be None and `flags` 0.  Like precompute_flow_info, it (re)configures the
    context: this frame size, the runner's batch for it (at most 2n - 1 frames) and max_pairs n become its limits."""
    if flow is not None:
        raise ValueError("calc_optical_flow_farneback_batch: flow must be None (an initial flow is not supported)")
    ctx = ctx or get_context()
    tensors = _is_torch_tensor(prev), _is_torch_tensor(next)
    if tensors[0] != tensors[1]:
        raise TypeError("calc_optical_flow_farneback_batch: prev and next must both be NumPy arrays or both torch tensors")
    if tensors[0]:
        import torch
        if prev.dtype != torch.uint8 or next.dtype != torch.uint8 or not prev.is_cuda or not next.is_cuda:
            raise TypeError("calc_optical_flow_farneback_batch: tensors must be torch.uint8 on a CUDA device")
        if prev.device != next.device or prev.device.index != ctx.device:
            raise ValueError(f"calc_optical_flow_farneback_batch: tensors on {prev.device} / {next.device}, "
                             f"the context on cuda:{ctx.device}")
    else:
        prev, next = np.asarray(prev), np.asarray(next)
        if prev.dtype != np.uint8 or next.dtype != np.uint8:
            raise TypeError("calc_optical_flow_farneback_batch: frames must be uint8")
    if tuple(prev.shape) != tuple(next.shape) or prev.ndim != 3:
        raise ValueError(f"calc_optical_flow_farneback_batch: prev and next must be [n, H, W] of one shape, "
                         f"not {tuple(prev.shape)} and {tuple(next.shape)}")
    ctx.set_farneback(pyr_scale, levels, winsize, iterations, poly_n, poly_sigma, flags)
    n, h, w = prev.shape
    if n == 0:
        return torch.empty((0, h, w, 2), dtype=torch.float32, device=prev.device) if tensors[0] else np.empty((0, h, w, 2), np.float32)
    ctx.configure(w, h, _pairs_batch(w, h, n), n)
    if not tensors[0]:
        return ctx.farneback_pairs(prev, next)["flow"]
    prev, next = prev.contiguous(), next.contiguous()
    out = torch.empty((n, h, w, 2), dtype=torch.float32, device=prev.device)
    ctx.farneback_pairs_ptr(prev.data_ptr(), next.data_ptr(), n, w, h, w, w * h, out.data_ptr(), w * 8, w * h * 8,
                            torch.cuda.current_stream(prev.device).cuda_stream)
    return out


def calc_optical_flow_farneback_batch_bidirectional(prev, next, flow, pyr_scale: float, levels: int, winsize: int,
                                                    iterations: int, poly_n: int, poly_sigma: float, flags: int = 0, *,
                                                    alpha: float = 0.01, beta: float = 0.5,
                                                    ctx: Optional[_native.FlowContext] = None):
    """calc_optical_flow_farneback_batch plus the backward flow of every pair and the forward-backward consistency mask,
    in one call with each frame expanded once: returns (forward, backward, mask), float32 [n, H, W, 2] twice and bool
    [n, H, W].  forward[i] is the flow prev[i] -> next[i], backward[i] the flow next[i] -> prev[i]
    (calc_optical_flow_farneback(next[i], prev[i], ...) bit for bit), and mask[i] is
    calc_optical_flow_farneback_sequence_bidirectional's: True where the forward target lies in the frame and the
    backward flow there cancels the forward flow.  For the two eyes of a side-by-side frame it is the left-right check of
    stereo matching.  Inputs, refusals, the torch path (tensors on the frames' device, ordered on
    torch.cuda.current_stream(), no host round trip) and the context's batch are calc_optical_flow_farneback_batch's;
    strided NumPy views are copied to dense frames first.  There are no per-pair results, so max_pairs is not raised."""
    fn = "calc_optical_flow_farneback_batch_bidirectional"
    if flow is not None:
        raise ValueError(f"{fn}: flow must be None (an initial flow is not supported)")
    ctx = ctx or get_context()
    tensors = _is_torch_tensor(prev), _is_torch_tensor(next)
    if tensors[0] != tensors[1]:
        raise TypeError(f"{fn}: prev and next must both be NumPy arrays or both torch tensors")
    if tensors[0]:
        import torch
        if prev.dtype != torch.uint8 or next.dtype != torch.uint8 or not prev.is_cuda or not next.is_cuda:
            raise TypeError(f"{fn}: tensors must be torch.uint8 on a CUDA device")
        if prev.device != next.device or prev.device.index != ctx.device:
            raise ValueError(f"{fn}: tensors on {prev.device} / {next.device}, the context on cuda:{ctx.device}")
    else:
        prev, next = np.asarray(prev), np.asarray(next)
        if prev.dtype != np.uint8 or next.dtype != np.uint8:
            raise TypeError(f"{fn}: frames must be uint8")
        # the call reads dense frames: a strided view (one eye of side-by-side frames, every other frame) is copied first
        prev, next = np.ascontiguousarray(prev), np.ascontiguousarray(next)
    if tuple(prev.shape) != tuple(next.shape) or prev.ndim != 3:
        raise ValueError(f"{fn}: prev and next must be [n, H, W] of one shape, not {tuple(prev.shape)} and "
                         f"{tuple(next.shape)}")
    ctx.set_farneback(pyr_scale, levels, winsize, iterations, poly_n, poly_sigma, flags)
    n, h, w = prev.shape
    if tensors[0]:
        prev, next = prev.contiguous(), next.contiguous()
        fw = torch.empty((n, h, w, 2), dtype=torch.float32, device=prev.device)
        bw = torch.empty_like(fw)
        mask = torch.empty((n, h, w), dtype=torch.bool, device=prev.device)
    else:
        fw, bw, mask = np.empty((n, h, w, 2), np.float32), np.empty((n, h, w, 2), np.float32), np.empty((n, h, w), np.bool_)
    if n == 0:
        return fw, bw, mask
    ctx.configure(w, h, _pairs_batch(w, h, n), 1)
    if not tensors[0]:
        ctx.farneback_pairs_bidir_ptr(prev.ctypes.data, next.ctypes.data, n, w, h, w, w * h, fw, bw, mask=mask, alpha=alpha,
                                      beta=beta)
        return fw, bw, mask
    ctx.farneback_pairs_bidir_ptr(prev.data_ptr(), next.data_ptr(), n, w, h, w, w * h, fw.data_ptr(), bw.data_ptr(), w * 8,
                                  w * h * 8, mask.data_ptr(), w, w * h, torch.cuda.current_stream(prev.device).cuda_stream,
                                  alpha=alpha, beta=beta)
    return fw, bw, mask


def _sequence_batch(width: int, height: int, n_frames: int) -> int:
    """batch_frames for a sequence of n_frames frames: the runner's batch for the frame size, no more than the
    sequence needs (its first batch takes batch_frames + 1 frames)."""
    from .runner import default_batch_frames
    return max(1, min(default_batch_frames(width, height), n_frames - 1))


def calc_optical_flow_farneback_sequence(frames, flow, pyr_scale: float, levels: int, winsize: int, iterations: int,
                                         poly_n: int, poly_sigma: float, flags: int = 0, *,
                                         ctx: Optional[_native.FlowContext] = None):
    """calc_optical_flow_farneback for every pair of consecutive frames (frames[j], frames[j + 1]) in one call, cv2's
    order after a leading frame axis: uint8 [n, H, W] -> float32 [n - 1, H, W, 2].  Each frame is expanded once (a
    bracket), where the batch function would expand it twice.  NumPy arrays give a NumPy array.  A torch.uint8 CUDA
    tensor on the context's device gives a tensor on that device, ordered on torch.cuda.current_stream(): the frames and
    the flows never pass through host memory.  `flow` must be None and `flags` 0.  It (re)configures the context: this
    frame size and the runner's batch for it (at most n - 1 frames) become its limits."""
    if flow is not None:
        raise ValueError("calc_optical_flow_farneback_sequence: flow must be None (an initial flow is not supported)")
    ctx = ctx or get_context()
    tensor = _is_torch_tensor(frames)
    if tensor:
        import torch
        if frames.dtype != torch.uint8 or not frames.is_cuda:
            raise TypeError("calc_optical_flow_farneback_sequence: a tensor must be torch.uint8 on a CUDA device")
        if frames.device.index != ctx.device:
            raise ValueError(f"calc_optical_flow_farneback_sequence: frames on {frames.device}, the context on cuda:{ctx.device}")
    else:
        frames = np.asarray(frames)
        if frames.dtype != np.uint8:
            raise TypeError("calc_optical_flow_farneback_sequence: frames must be uint8")
    if frames.ndim != 3:
        raise ValueError(f"calc_optical_flow_farneback_sequence: frames must be [n, H, W], not {tuple(frames.shape)}")
    ctx.set_farneback(pyr_scale, levels, winsize, iterations, poly_n, poly_sigma, flags)
    n, h, w = frames.shape
    if n < 2:
        shape = (0, h, w, 2)
        return torch.empty(shape, dtype=torch.float32, device=frames.device) if tensor else np.empty(shape, np.float32)
    ctx.configure(w, h, _sequence_batch(w, h, n), 1)
    if not tensor:
        return ctx.farneback_sequence(frames)["flow"]
    frames = frames.contiguous()
    out = torch.empty((n - 1, h, w, 2), dtype=torch.float32, device=frames.device)
    ctx.farneback_sequence_ptr(frames.data_ptr(), n, w, h, w, w * h, out.data_ptr(), w * 8, w * h * 8,
                               torch.cuda.current_stream(frames.device).cuda_stream)
    return out


def calc_optical_flow_farneback_sequence_bidirectional(frames, flow, pyr_scale: float, levels: int, winsize: int,
                                                       iterations: int, poly_n: int, poly_sigma: float, flags: int = 0, *,
                                                       alpha: float = 0.01, beta: float = 0.5,
                                                       ctx: Optional[_native.FlowContext] = None):
    """calc_optical_flow_farneback_sequence plus the backward flow of every pair and the forward-backward consistency
    mask (Sundaram, Brox & Keutzer, ECCV 2010), in one call with each frame expanded once: returns (forward, backward,
    mask), float32 [n - 1, H, W, 2] twice and bool [n - 1, H, W].  forward[j] is the flow frames[j] -> frames[j + 1],
    backward[j] the flow frames[j + 1] -> frames[j] (calc_optical_flow_farneback(frames[j + 1], frames[j], ...) bit for
    bit), and mask[j] is True where the pixel's forward target lies in the frame and |w + w_b|^2 <= alpha (|w|^2 +
    |w_b|^2) + beta, w_b the backward flow sampled bilinearly at the target: False marks occlusions, disocclusions and
    unreliable motion.  Inputs, refusals, the context's configuration and the torch path (tensors on the frames'
    device, ordered on torch.cuda.current_stream(), no host round trip) are calc_optical_flow_farneback_sequence's."""
    if flow is not None:
        raise ValueError("calc_optical_flow_farneback_sequence_bidirectional: flow must be None (an initial flow is not supported)")
    ctx = ctx or get_context()
    tensor = _is_torch_tensor(frames)
    if tensor:
        import torch
        if frames.dtype != torch.uint8 or not frames.is_cuda:
            raise TypeError("calc_optical_flow_farneback_sequence_bidirectional: a tensor must be torch.uint8 on a CUDA device")
        if frames.device.index != ctx.device:
            raise ValueError(f"calc_optical_flow_farneback_sequence_bidirectional: frames on {frames.device}, the context on "
                             f"cuda:{ctx.device}")
    else:
        frames = np.asarray(frames)
        if frames.dtype != np.uint8:
            raise TypeError("calc_optical_flow_farneback_sequence_bidirectional: frames must be uint8")
        frames = np.ascontiguousarray(frames)   # the call reads dense frames: a strided view is copied first
    if frames.ndim != 3:
        raise ValueError(f"calc_optical_flow_farneback_sequence_bidirectional: frames must be [n, H, W], not {tuple(frames.shape)}")
    ctx.set_farneback(pyr_scale, levels, winsize, iterations, poly_n, poly_sigma, flags)
    n, h, w = frames.shape
    m = max(n - 1, 0)
    if tensor:
        frames = frames.contiguous()
        fw = torch.empty((m, h, w, 2), dtype=torch.float32, device=frames.device)
        bw = torch.empty_like(fw)
        mask = torch.empty((m, h, w), dtype=torch.bool, device=frames.device)
    else:
        fw, bw, mask = np.empty((m, h, w, 2), np.float32), np.empty((m, h, w, 2), np.float32), np.empty((m, h, w), np.bool_)
    if n < 2:
        return fw, bw, mask
    ctx.configure(w, h, _sequence_batch(w, h, n), 1)
    if not tensor:
        ctx.farneback_sequence_bidir_ptr(frames.ctypes.data, n, w, h, w, w * h, fw, bw, mask=mask, alpha=alpha, beta=beta)
        return fw, bw, mask
    ctx.farneback_sequence_bidir_ptr(frames.data_ptr(), n, w, h, w, w * h, fw.data_ptr(), bw.data_ptr(), w * 8, w * h * 8,
                                     mask.data_ptr(), w, w * h, torch.cuda.current_stream(frames.device).cuda_stream,
                                     alpha=alpha, beta=beta)
    return fw, bw, mask


def remap_by_flow(src, flow, border_mode: int = 0, border_value: int = 0, *, ctx: Optional[_native.FlowContext] = None):
    """Warp images by dense flows: cv2.remap(src, flow, None, cv2.INTER_LINEAR | cv2.WARP_RELATIVE_MAP, border_mode,
    (border_value,) * 3) bit for bit, so dst(x, y) samples src at (x + flow_x, y + flow_y).  src is uint8 [H, W],
    [H, W, 3], [n, H, W] or [n, H, W, 3], flow float32 [H, W, 2] or [n, H, W, 2]; flow.ndim tells one image from a
    batch.  border_mode 0 is cv2.BORDER_CONSTANT (value border_value, 0..255), 1 cv2.BORDER_REPLICATE.  The output has
    src's shape.  NumPy arrays give a NumPy array (strided views are copied to dense arrays first).  torch CUDA tensors
    (uint8 and float32) on the context's device give a tensor there, ordered on torch.cuda.current_stream(), with no
    host round trip.  remap_by_flow(frames[1:], calc_optical_flow_farneback_sequence(frames, ...)) warps each next frame
    onto its previous one.  The context's configuration is left as it is."""
    fn = "remap_by_flow"
    ctx = ctx or get_context()
    tensors = _is_torch_tensor(src), _is_torch_tensor(flow)
    if tensors[0] != tensors[1]:
        raise TypeError(f"{fn}: src and flow must both be NumPy arrays or both torch tensors")
    if not tensors[0]:
        return ctx.remap_flow(np.asarray(src), np.asarray(flow), border_mode, border_value)
    import torch
    if src.dtype != torch.uint8 or flow.dtype != torch.float32 or not src.is_cuda or not flow.is_cuda:
        raise TypeError(f"{fn}: tensors must be torch.uint8 (src) and torch.float32 (flow) on a CUDA device")
    if src.device != flow.device or src.device.index != ctx.device:
        raise ValueError(f"{fn}: tensors on {src.device} / {flow.device}, the context on cuda:{ctx.device}")
    single = flow.ndim == 3
    src_b, flow_b = (src[None], flow[None]) if single else (src, flow)
    if flow_b.ndim != 4 or flow_b.shape[3] != 2 or tuple(src_b.shape[:3]) != tuple(flow_b.shape[:3]) \
            or src_b.ndim not in (3, 4) or (src_b.ndim == 4 and src_b.shape[3] != 3):
        raise ValueError(f"{fn}: src {tuple(src.shape)} and flow {tuple(flow.shape)} are not [n,] H, W[, 3] and "
                         f"[n,] H, W, 2")
    src_b, flow_b = src_b.contiguous(), flow_b.contiguous()
    n, h, w = flow_b.shape[:3]
    ch = 3 if src_b.ndim == 4 else 1
    out = torch.empty_like(src_b)
    if n:
        ctx.remap_flow_ptr(src_b.data_ptr(), n, w, h, ch, w * ch, w * h * ch, flow_b.data_ptr(), w * 8, w * h * 8,
                           out.data_ptr(), w * ch, w * h * ch, border_mode, border_value,
                           torch.cuda.current_stream(src.device).cuda_stream)
    return out[0] if single else out


def process_sequence(frames, params: Optional[Dict] = None, *, ctx: Optional[_native.FlowContext] = None,
                     batch_frames: int = DEFAULT_BATCH_FRAMES) -> Dict:
    """process_bracket(frames, params) plus `flows` (f32 [N-1, H, W, 2]), the flow of every pair, in one pass: the same
    per-pair arrays bit for bit, each flow bit-identical to calc_optical_flow_farneback on that pair."""
    params = params or {}
    ctx = ctx or get_context()
    arr = _as_frames(frames)
    n, h, w = arr.shape
    apply_farneback(ctx, params)
    ctx.configure(w, h, max(1, min(batch_frames, n)), max(n - 1, 1))
    res = ctx.farneback_sequence(arr, stats=True, pov=bool(params.get("pov_mode", False)),
                                 cut_threshold=float(params.get("cut_threshold", DEFAULT_CUT_THRESHOLD)))
    res["flows"] = res.pop("flow")
    return res


def precompute_flow_info_batch(pairs, config: Dict) -> list:
    """[precompute_wrapper(p, config) for p in pairs] in one call: the same 8-key dicts (F:898-907) with the same types.
    Every pair must have the frame size of the first.  The shared context is configured as calc_optical_flow_farneback_batch
    configures it."""
    pairs = list(pairs)
    if not pairs:
        return []
    prev = np.stack([np.asarray(p[0], dtype=np.uint8) for p in pairs])
    nxt = np.stack([np.asarray(p[1], dtype=np.uint8) for p in pairs])
    if prev.shape != nxt.shape or prev.ndim != 3:
        raise ValueError("every pair must be two equal-sized 2-D uint8 arrays of one frame size")
    ctx = get_context()
    n, h, w = prev.shape
    pov = bool(config.get("pov_mode"))
    apply_farneback(ctx, config)
    ctx.configure(w, h, _pairs_batch(w, h, n), n)
    r = ctx.farneback_pairs(prev, nxt, pov=pov, cut_threshold=float(config.get("cut_threshold", DEFAULT_CUT_THRESHOLD)))
    out = []
    for i in range(n):
        if pov:   # F:882: plain Python ints and the int 0
            pos_center, val = (w // 2, h - 1), 0
        else:     # F:757-758: NumPy integer / float32 scalars
            pos_center, val = (np.int64(r["cx"][i]), np.int64(r["cy"][i])), np.float32(r["val"][i])
        out.append({
            "flow": r["flow"][i],
            "pos_center": pos_center,
            "neg_center": pos_center,
            "val_pos": val,
            "val_neg": val,
            "cut": bool(r["cut"][i]),
            "cut_center": pos_center[0],
            "mean_mag": np.float32(r["mean_mag"][i]),
        })
    return out


def precompute_flow_info_gpu(p0: np.ndarray, p1: np.ndarray, cut_threshold) -> Dict:
    """F:982-1017: same dict, threshold passed positionally, no config (hence no POV mode)."""
    return precompute_flow_info(p0, p1, {"cut_threshold": cut_threshold})


def precompute_wrapper(p, params):
    """F:1019-1021."""
    return precompute_flow_info(p[0], p[1], params)


def max_divergence(flow: np.ndarray):
    """F:748-758: (x, y, value) of the first maximum of |d flow[...,0]/d row + d flow[...,1]/d col|."""
    x, y, v = get_context().max_divergence(flow)
    return np.int64(x), np.int64(y), v


def radial_motion_weighted(flow: np.ndarray, center, is_cut, pov_mode: bool = False):
    """F:761-785."""
    if is_cut:
        return 0.0
    return np.float64(get_context().radial_motion(flow, center, False, bool(pov_mode)))


def smooth_centers(centers: Sequence, radius: int = 6) -> np.ndarray:
    """F:1201-1214 on the host (the runner does this on the device; kept for API parity)."""
    c = np.asarray(centers, dtype=np.int64).reshape(-1, 2)
    n = len(c)
    csum = np.concatenate([np.zeros((1, 2), np.int64), np.cumsum(c, axis=0)])
    j = np.arange(n)
    lo = np.maximum(j - radius, 0)
    hi = np.minimum(j + radius + 1, n)
    return (csum[hi] - csum[lo]) / (hi - lo)[:, None].astype(np.float64)
