"""GPU batch runner with the reference's orchestration contracts.

    process_video(video_path, params, log_func, progress_callback=None, cancel_flag=None,
                  preview_callback=None) -> error_occurred        (F:1094-1404)
    run_headless(input_path, settings)                              (F:2606-2638)
    process_frames(frames, fps, params, ...) -> actions             (same pipeline on in-memory frames)

Semantics kept from the reference: brackets of `batch_size` sampled frames are independent (no pair
spans two brackets, a trailing 1-frame bracket is dropped, the +-6 centre window is truncated at
bracket ends: F:1145-1153, 1188, 1203-1214); `step = ceil(fps/30)` sub-sampling (F:1127); skip when
the .funscript exists unless `overwrite` (F:1105-1109).  The reference's prefetch race (SURVEY
section 5.3) is *not* reproduced: every bracket is computed on its own frames.

Frame acquisition: decode stays on the host (cv2.VideoCapture); the resize to 256x256 (or the VR crop)
and RGB->gray of F:1051-1091 run on the GPU (SURVEY row N2, `ffb_bracket_push_bgr`, bit-exact with cv2's
8-bit fixed-point arithmetic), so the decoded BGR frames are the only thing that crosses PCIe.
"""
from __future__ import annotations

import math
import os
import time
from typing import Callable, Dict, List, Optional, Sequence

import numpy as np

from . import api, postproc

SUPPORTED_VIDEO_EXTENSIONS = {".mp4", ".avi", ".mov", ".mkv", ".webm", ".flv", ".wmv", ".m4v", ".mpg", ".mpeg", ".ts"}


def _brackets(n_frames: int, bracket: int):
    for a in range(0, n_frames, bracket):
        b = min(a + bracket, n_frames)
        if b - a >= 2:      # F:1152-1153
            yield a, b


def process_many(clips: Sequence, fps: float, params: Dict, ctx=None, return_series: bool = False,
                 progress_callback: Optional[Callable[[int], None]] = None, cancel_flag: Optional[Callable[[], bool]] = None):
    """The bracket loop (F:1145-1253) + post-processing (F:1266-1386) over several in-memory clips (each a sequence of
    sampled gray frames, or a (frames, frame_indices) tuple), with ALL their brackets pipelined over two contexts of the
    GPU (api.BracketPipeline): the frames of the next bracket -- of the same clip or of the next one -- upload while
    the current one computes.  Returns one entry per clip: actions, or (actions, series) with return_series.
    Per-bracket results are those of api.process_bracket, bit for bit."""
    bracket = int(params.get("batch_size", 3000.0))
    pipe = api.BracketPipeline(ctx, batch_frames=int(params.get("gpu_batch_frames", api.DEFAULT_BATCH_FRAMES)))
    items = []                      # per clip: frames, frame indices, list of bracket bounds
    for clip in clips:
        frames, idx = clip if isinstance(clip, tuple) else (clip, None)
        n = len(frames)
        items.append((frames, list(range(n)) if idx is None else list(idx), list(_brackets(n, bracket))))
    acc = [dict(values=[], cuts=[], stamps=[]) for _ in items]
    order = [(k, a, b) for k, (_, _, br) in enumerate(items) for a, b in br]
    total = max(1, len(order))

    def take(res, k, a, b):
        acc[k]["values"].extend(res["scalar"].tolist())
        acc[k]["cuts"].extend(res["cut"].tolist())
        acc[k]["stamps"].extend(items[k][1][a:b - 1])          # F:1151: frame index of the first frame of each pair
    prev = None
    for j, (k, a, b) in enumerate(order):
        if cancel_flag and cancel_flag():
            pipe.flush()
            return None
        done = pipe.submit(items[k][0][a:b], params)
        if prev is not None:
            take(done, *prev)
        prev = (k, a, b)
        if progress_callback:
            progress_callback(min(100, int(100 * (j + 1) / total)))
    if prev is not None:
        take(pipe.flush(), *prev)
    out = []
    for k in range(len(items)):
        v = acc[k]
        actions = postproc.scalars_to_actions(v["values"], v["cuts"], v["stamps"], fps, params) if v["values"] else []
        if return_series:
            out.append((actions, dict(values=np.asarray(v["values"]), cuts=np.asarray(v["cuts"], bool),
                                      frame_indices=np.asarray(v["stamps"]))))
        else:
            out.append(actions)
    return out


def process_frames(frames: Sequence[np.ndarray], fps: float, params: Dict, frame_indices: Optional[Sequence[int]] = None,
                   ctx=None, progress_callback: Optional[Callable[[int], None]] = None,
                   cancel_flag: Optional[Callable[[], bool]] = None, return_series: bool = False):
    """Bracket loop (F:1145-1253) + post-processing (F:1266-1386) over in-memory sampled frames (one clip of
    process_many: consecutive brackets are pipelined over two contexts of the GPU)."""
    res = process_many([(frames, frame_indices)], fps, params, ctx=ctx, return_series=return_series,
                       progress_callback=progress_callback, cancel_flag=cancel_flag)
    return None if res is None else res[0]


def _container_shape(cap):
    """(H, W, 3) of the frames a cv2.VideoCapture delivers, None when the container does not say."""
    import cv2
    w, h = int(cap.get(cv2.CAP_PROP_FRAME_WIDTH)), int(cap.get(cv2.CAP_PROP_FRAME_HEIGHT))
    return (h, w, 3) if w > 0 and h > 0 else None


def iter_sampled_bgr(video_path: str, indices: Sequence[int], shape_hint=None):
    """Decode the sampled frames (BGR, as cv2.VideoCapture returns them); undecodable frames are black at the
    container's frame size (F:239-245, F:274-280: a file that over-reports its frame count still yields a script).
    Sequential read + grab instead of the reference's per-frame seek."""
    import cv2
    cap = cv2.VideoCapture(video_path)
    if not cap.isOpened():
        raise IOError(f"cannot open {video_path}")
    want = set(int(i) for i in indices)
    last = max(want) if want else -1
    shape = shape_hint or _container_shape(cap)
    pos = 0
    while pos <= last:
        if pos in want:
            ok, frame = cap.read()
            if ok:
                shape = frame.shape
            else:
                if shape is None:
                    raise IOError(f"{video_path}: no frame could be decoded and the container reports no frame size")
                frame = np.zeros(shape, np.uint8)
            yield frame
        else:
            cap.grab()
        pos += 1
    cap.release()


def _decode_span(video_path: str, wanted: Sequence[int], shape_hint):
    """Frames `wanted` (increasing indices) from their own cv2.VideoCapture: seek to the first, then read / grab
    forward.  Returns (frames, seek_ok); seek_ok is False when the container did not land on the requested frame.
    Frames that cannot be read are black at the container's frame size (`shape_hint`, else what the handle reports)."""
    import cv2
    cap = cv2.VideoCapture(video_path)
    out = []
    ok_seek = True
    try:
        first = int(wanted[0])
        if first > 0:
            cap.set(cv2.CAP_PROP_POS_FRAMES, first)
            ok_seek = int(round(cap.get(cv2.CAP_PROP_POS_FRAMES))) == first
        want = set(int(i) for i in wanted)
        pos, last, shape = first, int(wanted[-1]), shape_hint or _container_shape(cap)
        while pos <= last:
            if pos in want:
                ok, frame = cap.read()
                if ok:
                    shape = frame.shape
                else:
                    if shape is None:
                        raise IOError(f"{video_path}: no frame could be decoded and the container reports no frame size")
                    frame = np.zeros(shape, np.uint8)       # F:274-280
                out.append(frame)
            else:
                cap.grab()
            pos += 1
    finally:
        cap.release()
    return out, ok_seek


def iter_sampled_bgr_parallel(video_path: str, indices: Sequence[int], workers: int = 4, span: int = 64, shape_hint=None):
    """iter_sampled_bgr with the decode spread over `workers` threads (the reference decodes on up to 4 handles,
    F:103-291): the sampled indices are cut into spans of `span` frames, each span is decoded on its own
    VideoCapture (cv2 releases the GIL while decoding) and the spans are handed out in order with a bounded
    look-ahead.  Containers on which a seek does not land on the requested frame fall back to the sequential
    reader for the rest of the file, so the frames are the same either way."""
    from concurrent.futures import ThreadPoolExecutor
    idx = [int(i) for i in indices]
    if workers <= 1 or len(idx) <= span:
        yield from iter_sampled_bgr(video_path, idx, shape_hint)
        return
    spans = [idx[a:a + span] for a in range(0, len(idx), span)]
    with ThreadPoolExecutor(max_workers=workers) as pool:
        pending = {}
        nxt = 0

        def fill():
            nonlocal nxt
            while nxt < len(spans) and len(pending) < workers + 1:
                pending[nxt] = pool.submit(_decode_span, video_path, spans[nxt], shape_hint)
                nxt += 1
        fill()
        for k in range(len(spans)):
            frames, ok_seek = pending.pop(k).result()
            if not ok_seek:      # inexact seek: decode the rest sequentially from the start of this span
                for fut in pending.values():
                    fut.cancel()
                rest = [i for sp in spans[k:] for i in sp]
                yield from iter_sampled_bgr(video_path, rest, shape_hint)
                return
            fill()
            yield from frames


def read_sampled_gray(video_path: str, indices: Sequence[int], params: Dict) -> List[np.ndarray]:
    """HOST version of the frame contract (F:1051-1091), kept for tests: BGR->RGB, resize to 256x256
    (VR: 512x512 then the bottom-left 256x256), RGB->gray with cv2.  process_video() does the same
    arithmetic on the GPU (ffb_bracket_push_bgr, bit-exact)."""
    import cv2
    out = []
    vr = bool(params.get("vr_mode"))
    for frame in iter_sampled_bgr(video_path, indices):
        rgb = cv2.cvtColor(frame, cv2.COLOR_BGR2RGB)
        rgb = cv2.resize(rgb, (512, 512))[256:, :256] if vr else cv2.resize(rgb, (256, 256))
        out.append(cv2.cvtColor(rgb, cv2.COLOR_RGB2GRAY))
    return out


def preprocess_plan(src_w: int, src_h: int, params: Dict, eye: Optional[str] = None):
    """(target, window, cut_scale) of the frame contract for `params`.

    Reference modes: resize to 256x256 (F:1057) or, with `vr_mode`, to 512x512 and keep the bottom-left
    quadrant (F:1076-1079).  Row N4 options the reference has no equivalent of:
      native_resolution  no resampling: the flow runs on the decoded frame (VR: on the lower half of
                         one eye of the side-by-side frame); `cut_threshold` (F:876, tuned for 256x256
                         frames) is multiplied by cut_scale = sqrt(w*h)/256 because flow magnitudes
                         are in pixels;
      vr_eye             "left" (the reference's choice), "right", or "both": process_video_series then runs
                         the two eyes as two independent series on two contexts of the same GPU (one decode,
                         every chunk pushed to both) and reports the mean scalar and the OR of the cut flags.
                         For "both" this function returns the left eye's plan; `eye` overrides params.
    """
    vr = bool(params.get("vr_mode"))
    eye = str(eye if eye is not None else params.get("vr_eye", "left")).lower()
    if eye not in ("left", "right", "both"):
        raise ValueError("vr_eye must be 'left', 'right' or 'both'")
    right = vr and eye == "right"
    if params.get("native_resolution"):
        if vr:
            w, h = src_w // 2, src_h // 2
            target, window = (src_w, src_h), (src_w - w if right else 0, src_h - h, w, h)
        else:
            target, window = (src_w, src_h), (0, 0, src_w, src_h)
        return target, window, math.sqrt(window[2] * window[3]) / 256.0
    if vr:
        return (512, 512), (256 if right else 0, 256, 256, 256), 1.0
    return (256, 256), (0, 0, 256, 256), 1.0


def default_batch_frames(width: int, height: int) -> int:
    """Frames per GPU batch.  Small frames need many pairs per launch to fill 148 SMs (the reference's 256x256
    product mode: 512), 720p / 1080p take 128, 4K runs at full rate from 64, and above 4K the batch shrinks so that the
    per-batch device buffers (about 64 bytes per pixel and frame) stay near 35 GB."""
    px = max(1, width * height)
    if px <= 256 * 256:
        return 1024       # the reference's product mode: +4 % over 512 (profiles/r2_sweep_flow_iter.txt), 4 GB of buffers
    if px <= 640 * 360:
        return 512
    if px <= 1920 * 1080:
        return 128        # 1080p: +1.4 % over 64 (profiles/r2_sweep_flow_iter.txt), 17 GB of device buffers
    return max(2, min(64, int(64 * (3840 * 2160) / px)))


def process_video_series(video_path: str, params: Dict, ctx=None, progress_callback=None, cancel_flag=None,
                         chunk_frames: int = 64):
    """Bracket loop over a video file with decode on the host and everything else on the GPU:
    decoded BGR frames are uploaded in chunks, resized + gray-converted (row N2), and run through the
    hot path.  Returns (values, cuts, frame_indices, fps) or None when cancelled."""
    import cv2
    ctx = ctx or api.get_context()
    both = bool(params.get("vr_mode")) and str(params.get("vr_eye", "left")).lower() == "both"
    cap = cv2.VideoCapture(video_path)
    if not cap.isOpened():
        raise IOError(f"cannot open {video_path}")
    total = int(cap.get(cv2.CAP_PROP_FRAME_COUNT))
    fps = float(cap.get(cv2.CAP_PROP_FPS))
    src_w, src_h = int(cap.get(cv2.CAP_PROP_FRAME_WIDTH)), int(cap.get(cv2.CAP_PROP_FRAME_HEIGHT))
    cap.release()
    if total < 2 or fps <= 0 or src_w < 2 or src_h < 2:
        raise IOError("unable to read video properties")
    target, window, cut_scale = preprocess_plan(src_w, src_h, params, "left" if both else None)
    out_w, out_h = window[2], window[3]
    ctx.preprocess_configure_window(src_w, src_h, target, window)
    ctxs = [ctx]
    if both:      # the other eye: same geometry, its own context (streams, rings) on the same device
        ctx_r = api.get_aux_context(ctx)
        ctx_r.preprocess_configure_window(src_w, src_h, *preprocess_plan(src_w, src_h, params, "right")[:2])
        ctxs.append(ctx_r)
    cut_threshold = float(params.get("cut_threshold", api.DEFAULT_CUT_THRESHOLD)) * cut_scale
    step = postproc.sampling_step(fps)
    indices = list(range(0, total, step))
    bracket = int(params.get("batch_size", 3000.0))
    batch = int(params.get("gpu_batch_frames", default_batch_frames(out_w, out_h)))
    chunk_frames = max(1, min(chunk_frames, (256 << 20) // (src_w * src_h * 3)))   # bound the host-side stack
    values: List[float] = []
    cuts: List[bool] = []
    stamps: List[int] = []
    # `threads` is the reference's pool size (F:2654); here it bounds the decode threads (the GPU needs none)
    frames = iter_sampled_bgr_parallel(video_path, indices, workers=max(1, min(4, int(params.get("threads", 4)))),
                                       shape_hint=(src_h, src_w, 3))
    # one configuration per video: batch size fixed, pair limit of the longest bracket (ffb_configure is incremental,
    # so the shorter last bracket re-allocates nothing)
    max_pairs = min(bracket, len(indices)) - 1
    for c in ctxs:
        api.apply_farneback(c, params)
        c.configure(out_w, out_h, max(1, min(batch, max_pairs + 1)), max(1, max_pairs))
    done = 0
    for a in range(0, len(indices), bracket):
        b = min(a + bracket, len(indices))
        nfr = b - a
        if cancel_flag and cancel_flag():
            return None
        if nfr < 2:          # F:1152-1153 (the frame is still consumed from the decoder)
            for _ in range(nfr):
                next(frames, None)
            continue
        for c in ctxs:
            c.bracket_begin(bool(params.get("pov_mode", False)), cut_threshold)
        try:
            got = 0
            while got < nfr:
                if cancel_flag and cancel_flag():      # F:1147-1149, checked per chunk instead of per bracket
                    for c in ctxs:
                        c.bracket_abort()
                    return None
                chunk = []
                while len(chunk) < chunk_frames and got + len(chunk) < nfr:
                    f = next(frames, None)
                    if f is None:
                        break
                    chunk.append(f)
                if not chunk:
                    break
                arr = np.ascontiguousarray(np.stack(chunk))
                if arr.shape[1:3] != (src_h, src_w):
                    raise IOError(f"decoded frame size {arr.shape[2]}x{arr.shape[1]} differs from the container's {src_w}x{src_h}")
                for c in ctxs:
                    c.bracket_push_bgr(arr)   # pageable input is copied into pinned staging before the call returns
                got += len(chunk)
                done += len(chunk)
                if progress_callback:
                    progress_callback(min(100, int(100 * done / len(indices))))
        except BaseException:
            for c in ctxs:      # leave the contexts usable for the next video
                c.bracket_abort()
            raise
        rs = [c.bracket_finish() for c in ctxs]
        r = rs[0]
        if both:
            values.extend((0.5 * (rs[0]["scalar"] + rs[1]["scalar"])).tolist())
            cuts.extend((rs[0]["cut"].astype(bool) | rs[1]["cut"].astype(bool)).tolist())
        else:
            values.extend(r["scalar"].tolist())
            cuts.extend(r["cut"].tolist())
        stamps.extend(indices[a:a + r["n_pairs"]])
    return values, cuts, stamps, fps


def process_video(video_path, params, log_func, progress_callback=None, cancel_flag=None, preview_callback=None):
    """Same contract as F:1094: writes <video>.funscript, returns error_occurred."""
    start = time.time()
    base, _ = os.path.splitext(video_path)
    output_path = base + ".funscript"
    if os.path.exists(output_path) and not params["overwrite"]:
        log_func(f"Skipping: output file exists ({output_path})")
        return False
    log_func(f"Processing video: {video_path}")
    try:      # F:1114-1131: properties first, so the two header lines precede the work as in the reference
        import cv2
        cap = cv2.VideoCapture(video_path)
        if not cap.isOpened():
            raise IOError("cannot open the container")
        total, fps0 = int(cap.get(cv2.CAP_PROP_FRAME_COUNT)), float(cap.get(cv2.CAP_PROP_FPS))
        cap.release()
        step0 = postproc.sampling_step(fps0)
        log_func(f"FPS: {fps0:.2f}; downsampled to ~{fps0 / step0:.2f} fps; {len(range(0, total, step0))} frames selected.")
    except Exception as exc:
        log_func(f"ERROR: Unable to open video at {video_path}: {exc}")
        return True
    log_func("Using backend: B200 (sm_100a)")
    try:
        res = process_video_series(video_path, params, progress_callback=progress_callback, cancel_flag=cancel_flag)
    except Exception as exc:   # surfaced, never swallowed into a CPU fallback
        log_func(f"ERROR: {exc}")
        return True
    if res is None:
        log_func("User bailed.")
        return False
    values, cuts, stamps, fps = res
    errors: List[str] = []
    actions = postproc.scalars_to_actions(values, cuts, stamps, fps, params, errors) if values else []
    for msg in errors:           # F:1383-1385: series shorter than the smoother (fewer than 6 sampled frames)
        log_func(msg)
    log_func(f"Keyframe reduction: {len(actions)} actions computed.")
    try:
        postproc.write_funscript(output_path, actions)
        log_func(f"Funscript saved: {output_path}")
    except Exception as exc:
        log_func(f"ERROR: {exc}")
        return True
    log_func(f"Processing time: {time.time() - start:.2f} seconds")
    return bool(errors)


def list_videos(input_path: str) -> List[str]:
    if os.path.isfile(input_path):
        return [input_path]
    found = []
    for root, _, files in os.walk(input_path):
        for f in sorted(files):
            if os.path.splitext(f)[1].lower() in SUPPORTED_VIDEO_EXTENSIONS:
                found.append(os.path.join(root, f))
    return found


def shard(items: Sequence, rank: int, world: int) -> List:
    """Whole-video sharding across GPUs (SURVEY 8(e)): video i goes to rank i % world."""
    return [it for i, it in enumerate(items) if i % world == rank]


def video_cost(path: str) -> float:
    """Work estimate of one video for the scheduler: its frame count (what the bracket loop iterates
    over, F:1113, F:1145); the file size when the container cannot be read."""
    try:
        import cv2
        cap = cv2.VideoCapture(path)
        n = float(cap.get(cv2.CAP_PROP_FRAME_COUNT)) if cap.isOpened() else 0.0
        cap.release()
        if n > 0:
            return n
    except Exception:
        pass
    try:
        return float(os.path.getsize(path)) * 1e-6
    except OSError:
        return 0.0


def schedule_longest_first(items: Sequence, costs: Sequence[float], world: int) -> List[List]:
    """Longest-processing-time-first assignment of whole videos to `world` GPUs (SURVEY row N3): visit
    the videos by decreasing cost and give each to the least-loaded rank.  Deterministic (ties: listing
    order, then lowest rank), so every rank derives the same plan without communicating; each rank's
    list keeps the listing order."""
    order = sorted(range(len(items)), key=lambda i: (-float(costs[i]), i))
    load = [0.0] * world
    owner = [0] * len(items)
    for i in order:
        r = min(range(world), key=lambda k: (load[k], k))
        owner[i] = r
        load[r] += float(costs[i])
    return [[items[i] for i in range(len(items)) if owner[i] == r] for r in range(world)]


def run_headless(input_path: str, settings: Dict, log_func: Optional[Callable[[str], None]] = None) -> int:
    """F:2606-2638: walk the folder, process every supported video, log to run.log and stdout.
    Under torchrun (one process per GPU) the videos are spread longest-first over the ranks
    (schedule_longest_first) and each rank writes run.<rank>.log.
    Returns the number of videos that reported an error."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    logf = None
    if log_func is None:
        logf = open("run.log" if world == 1 else f"run.{rank}.log", "w")

        def log_func(msg):
            logf.write(msg + "\n")
            logf.flush()
            print(msg)
    if world > 1:       # one process per GPU: keep the host side on the GPU's NUMA node
        from . import distributed
        distributed.bind_to_gpu_numa_node()
    vids = list_videos(input_path)
    if world > 1:
        vids = schedule_longest_first(vids, [video_cost(v) for v in vids], world)[rank]
    if not vids:
        log_func("No video files found.")
    else:
        log_func(f"Found {len(vids)} file(s)." + (f" (rank {rank} of {world})" if world > 1 else ""))      # F:376
    errors = 0
    for i, v in enumerate(vids):
        log_func(f"--- Processing file {i + 1}/{len(vids)}: {v} ---")                                       # F:377
        progress = (lambda prog: print(f"Video progress: {prog}%")) if logf else None      # F:2634
        errors += bool(process_video(v, settings, log_func, progress_callback=progress))
    log_func("Batch processing complete.")
    if logf:
        logf.close()
        print(f"Done. See {logf.name} for details.")                                         # F:2637
    return errors
