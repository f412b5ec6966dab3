"""Throughput of warping images by dense flows (ffb_remap_flow), next to the torch composition and to cv2.remap on the
host, in one process.

    python tools/bench_remap.py [--out FILE] [--rounds R] [--sizes 1920x1080,256x256]

Per frame size and channel count (gray, BGR), n images so that the flows alone take 256 MB or more (nothing stays in the
126 MB L2 between calls), uint8 sources and smooth float32 flows of tens of pixels, synthetic and seeded.  Arms,
alternated round by round (the median round of each is reported):
  device       FlowContext.remap_flow_ptr on torch CUDA tensors (device-resident), CUDA events on the current stream
  grid_sample  torch.nn.functional.grid_sample (bilinear, zero padding, align_corners=True) on the same images as
               float32 plus the conversions to and from uint8: what a torch user composes today.  It does not
               reproduce cv2's fixed-point arithmetic; it is here for scale.
  cv2          cv2.remap(..., INTER_LINEAR | WARP_RELATIVE_MAP) on host arrays, with cv2's default threads on the
               host's cores (the core count is recorded), host clock, a few images per round
Also: the kernel's own time from ffb_kernel_stats in a separate profiled pass, its algorithmic bytes
(8 + 2 * channels per pixel: flow, taps counted once, output) over that time as a share of the HBM copy rate measured in
the same run (a 2 GB device-to-device torch copy, read + write bytes), whether the device arm equals cv2.remap on the
first image, and the card's name and power limit, read in the same run.  Needs a CUDA device.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import numpy as np  # noqa: E402

from bench_bidir import card  # noqa: E402

FLOW_BYTES = 256 << 20


def smooth_flows(n, h, w, seed, amplitude=30.0):
    rng = np.random.default_rng(seed)
    ys, xs = np.mgrid[0:h, 0:w].astype(np.float32)
    base = np.empty((4, h, w, 2), np.float32)
    for i in range(4):
        for c in range(2):
            k = rng.uniform(0.5, 3.0, 4) * 2 * np.pi
            base[i, ..., c] = amplitude * (np.sin(k[0] * xs / w + k[1] * ys / h + rng.uniform(0, 6)) +
                                           0.5 * np.cos(k[2] * xs / w - k[3] * ys / h))
    return base[np.arange(n) % 4]


def copy_rate(torch):
    """Device-to-device copy rate of a 2 GB tensor (read + write bytes per second), median of 10."""
    a = torch.empty(1 << 31, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    ts = []
    for _ in range(12):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        b.copy_(a)
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1) / 1e3)
    del a, b
    return 2 * (1 << 31) / float(np.median(ts[2:])) / 1e9


def measure(W, H, ch, rounds, peak):
    import cv2
    import torch
    import torch.nn.functional as F
    from funscript_flow_b200 import _native
    n = -(-FLOW_BYTES // (W * H * 8))
    rng = np.random.default_rng(W + ch)
    shape = (n, H, W) if ch == 1 else (n, H, W, 3)
    src = rng.integers(0, 256, shape, dtype=np.uint8)
    flow = smooth_flows(n, H, W, seed=ch)
    ctx = _native.FlowContext(0)
    dev = torch.device("cuda", 0)
    s_t, f_t = torch.from_numpy(src).to(dev), torch.from_numpy(flow).to(dev)
    d_t = torch.empty_like(s_t)
    stream = torch.cuda.current_stream(dev)

    def device():
        ctx.remap_flow_ptr(s_t.data_ptr(), n, W, H, ch, W * ch, W * H * ch, f_t.data_ptr(), W * 8, W * H * 8,
                           d_t.data_ptr(), W * ch, W * H * ch, 0, 0, stream.cuda_stream)

    ys, xs = torch.meshgrid(torch.arange(H, device=dev, dtype=torch.float32),
                            torch.arange(W, device=dev, dtype=torch.float32), indexing="ij")
    scale = torch.tensor([2.0 / max(W - 1, 1), 2.0 / max(H - 1, 1)], device=dev)
    chunk = 16 if W * H > 1 << 20 else 256

    def grid_sample():
        for i0 in range(0, n, chunk):
            s = s_t[i0:i0 + chunk]
            img = (s[:, None] if ch == 1 else s.permute(0, 3, 1, 2)).float()
            grid = (torch.stack([xs, ys], -1) + f_t[i0:i0 + chunk]) * scale - 1.0
            out = F.grid_sample(img, grid, mode="bilinear", padding_mode="zeros", align_corners=True)
            out = out.round_().clamp_(0, 255).to(torch.uint8)
            d_t[i0:i0 + chunk] = out[:, 0] if ch == 1 else out.permute(0, 2, 3, 1)

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        fn()
        e1.record(stream)
        e1.synchronize()
        return e0.elapsed_time(e1) / 1e3

    n_cv = 4 if W * H > 1 << 20 else 64

    def cv():
        t = time.perf_counter()
        for i in range(n_cv):
            cv2.remap(src[i], flow[i], None, cv2.INTER_LINEAR | cv2.WARP_RELATIVE_MAP)
        return (time.perf_counter() - t) / n_cv

    device()
    exact = bool(np.array_equal(d_t[0].cpu().numpy(), cv2.remap(src[0], flow[0], None,
                                                                 cv2.INTER_LINEAR | cv2.WARP_RELATIVE_MAP)))
    grid_sample()
    gs_differ = float((d_t[0].cpu().numpy() != cv2.remap(src[0], flow[0], None,
                                                          cv2.INTER_LINEAR | cv2.WARP_RELATIVE_MAP)).mean())
    cv()
    t_dev, t_gs, t_cv = [], [], []
    for _ in range(rounds):
        t_dev.append(timed(device))
        t_gs.append(timed(grid_sample))
        t_cv.append(cv())
    ctx.profile(True)
    ctx.profile_reset()
    for _ in range(rounds):
        device()
    stream.synchronize()
    st = ctx.kernel_stats()["remap"]
    ctx.profile(False)
    ctx.close()
    k_ms = st["ms"] / st["launches"]
    alg = n * W * H * (8 + 2 * ch)
    med = lambda v: float(np.median(v))  # noqa: E731
    return dict(n=n, channels=ch, equals_cv2=exact, grid_sample_pixels_differing_from_cv2=round(gs_differ, 4),
                device_warps_per_s=round(n / med(t_dev), 1), device_call_ms=round(med(t_dev) * 1e3, 3),
                kernel_ms=round(k_ms, 3), kernel_alg_bytes_per_px=8 + 2 * ch,
                kernel_gbs=round(alg / (k_ms / 1e3) / 1e9, 1), kernel_share_of_copy_rate=round(alg / (k_ms / 1e3) / 1e9 / peak, 3),
                grid_sample_warps_per_s=round(n / med(t_gs), 1), cv2_host_warps_per_s=round(1.0 / med(t_cv), 1))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--sizes", default="1920x1080,256x256")
    args = ap.parse_args()
    import cv2
    import torch
    peak = copy_rate(torch)
    res = dict(card=card(), host_cores=os.cpu_count(), cv2_threads=cv2.getNumThreads(), cv2_version=cv2.__version__,
               hbm_copy_gbs=round(peak, 1), rounds=args.rounds, results={})
    print(f"{res['card']}; device-to-device copy {peak:.0f} GB/s", flush=True)
    for size in args.sizes.split(","):
        W, H = (int(v) for v in size.split("x"))
        for ch in (1, 3):
            r = measure(W, H, ch, args.rounds, peak)
            res["results"][f"{size}_{'gray' if ch == 1 else 'bgr'}"] = r
            print(size, ch, json.dumps(r), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
