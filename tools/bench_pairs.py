"""Throughput of Farneback flow for independent frame pairs (ffb_farneback_pairs), next to the bracket rate and the
per-pair drop-in, in one process.

    python tools/bench_pairs.py [--out FILE] [--steps K] [--sizes 256x256,1920x1080]

Per frame size, reference parameters, batch_frames = runner.default_batch_frames (the batch of the product's brackets
and of api.calc_optical_flow_farneback_batch), n = 3 chunks of (batch_frames + 1) / 2 pairs, the frames synthetic and
seeded, each pair two frames of one clip in a shuffled order:
  device      torch uint8 CUDA tensors in, a float32 CUDA tensor out (api.calc_optical_flow_farneback_batch), timed
              with CUDA events on the current torch stream
  pinned      page-locked host frames in, page-locked host flow out (the flow crosses PCIe: 8 bytes per pixel)
  stats       device frames in, no flow out, the per-pair centre / value / mean magnitude / cut to the host
  bracket     the n + 1 frames as one bracket already resident in HBM (bracket_push_ptr) at the same batch_frames, the
              streaming path's rate
  per_pair    api.calc_optical_flow_farneback on host arrays, one call per pair (a few pairs)
Host-clock arms end in a device synchronisation.  Algorithmic bytes per pixel of a pair (ffb_kernel_stats) for the
pairs path and the bracket, their ratio (the device arm's expected share of the bracket rate), the geometry each arm
ran with (ctx.geometry), and the card's name and power limit are read in the same run.  Needs a CUDA device; there is
no CPU path.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

REF = (0.5, 3, 15, 3, 5, 1.2)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power, smax = (s.strip() for s in q.stdout.strip().split(","))
    return dict(name=name, power_limit=power, sm_max_clock=smax)


def host_rate(fn, n, steps):
    fn()
    t0 = time.perf_counter()
    for _ in range(steps):
        fn()
    return n * steps / (time.perf_counter() - t0)


def alg_bytes_per_px(ctx, fn, n, W, H):
    ctx.profile_reset()
    fn()
    return sum(v["alg_bytes"] for v in ctx.kernel_stats().values()) / n / (W * H)


def measure(W, H, steps):
    import torch
    from funscript_flow_b200 import _native, api, runner
    from funscript_flow_b200.synth import make_clip
    batch = runner.default_batch_frames(W, H)
    n = 3 * ((batch + 1) // 2)
    clip = np.ascontiguousarray(np.stack(make_clip(W, H, 17, seed=11, period=9.0, amplitude=0.3)))
    rng = np.random.default_rng(3)
    prev = np.ascontiguousarray(clip[rng.integers(0, len(clip), n)])
    nxt = np.ascontiguousarray(clip[rng.integers(0, len(clip), n)])
    ctx = _native.FlowContext(0)
    ctx.configure(W, H, batch, n)
    dev = torch.device("cuda", 0)
    p_t, n_t = torch.from_numpy(prev).to(dev), torch.from_numpy(nxt).to(dev)
    out = {}

    # device tensors in, device flow out
    def device_call():
        return api.calc_optical_flow_farneback_batch(p_t, n_t, None, *REF, 0, ctx=ctx)
    device_call()
    torch.cuda.synchronize()
    geometry = dict(pairs=ctx.geometry)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        flow_t = device_call()
    e1.record()
    e1.synchronize()
    out["device_pairs_per_s"] = round(n * steps / (e0.elapsed_time(e1) / 1e3), 1)
    ref = flow_t.cpu().numpy()

    # pinned host in and out
    pin_p, pin_n = _native.PinnedBuffer(prev.shape), _native.PinnedBuffer(nxt.shape)
    pin_p.array[...] = prev
    pin_n.array[...] = nxt
    pin_f = _native.PinnedBuffer((n, H, W, 8))
    flow_h = pin_f.array.view(np.float32).reshape(n, H, W, 2)

    def pinned_call():
        ctx.farneback_pairs_ptr(pin_p.array.ctypes.data, pin_n.array.ctypes.data, n, W, H, W, W * H, flow_h.ctypes.data,
                                W * 8, W * H * 8)
    out["pinned_pairs_per_s"] = round(host_rate(pinned_call, n, steps), 1)
    same = bool(np.array_equal(flow_h, ref))

    # per-pair results only
    def stats_call():
        return ctx.farneback_pairs_ptr(p_t.data_ptr(), n_t.data_ptr(), n, W, H, W, W * H, stats=True)
    out["stats_pairs_per_s"] = round(host_rate(stats_call, n, steps), 1)
    pairs_bpp = alg_bytes_per_px(ctx, device_call, n, W, H)
    torch.cuda.synchronize()
    del flow_t

    # the bracket of the same number of pairs, frames resident in HBM
    frames = torch.from_numpy(np.concatenate([clip] * (n // len(clip) + 1))[:n + 1].copy()).to(dev)
    ctx.configure(W, H, batch, n)

    def bracket_call():
        ctx.bracket_begin(False, 7.0)
        ctx.bracket_push_ptr(frames.data_ptr(), n + 1, W, W * H)
        return ctx.bracket_finish()
    bracket_call()
    geometry["bracket"] = ctx.geometry
    ctx.timer_mark(0)
    for _ in range(steps):
        bracket_call()
    ctx.timer_mark(1)
    out["bracket_pairs_per_s"] = round(n * steps / (ctx.timer_elapsed_ms(0, 1) / 1e3), 1)
    bracket_bpp = alg_bytes_per_px(ctx, bracket_call, n, W, H)

    # the per-pair drop-in on a few pairs
    k = 8 if W * H > 640 * 360 else 32

    def per_pair_call():
        for i in range(k):
            api.calc_optical_flow_farneback(prev[i], nxt[i], None, *REF, 0, ctx=ctx)
    out["per_pair_pairs_per_s"] = round(host_rate(per_pair_call, k, max(1, steps // 2)), 1)

    for b in (pin_p, pin_n, pin_f):
        b.free()
    ctx.close()
    assert geometry["pairs"][2] == batch and geometry["bracket"][2] == batch, geometry
    out.update(batch_frames=batch, pairs_per_chunk=(batch + 1) // 2, n_pairs=n, steps=steps,
               geometry={k: dict(zip(("width", "height", "batch_frames", "max_pairs"), v)) for k, v in geometry.items()},
               pinned_flows_equal_device=same,
               alg_bytes_per_px=dict(pairs=round(pairs_bpp, 1), bracket=round(bracket_bpp, 1),
                                     bracket_over_pairs=round(bracket_bpp / pairs_bpp, 3)),
               device_over_bracket=round(out["device_pairs_per_s"] / out["bracket_pairs_per_s"], 3),
               pcie_bytes_per_pair_pinned=W * H * (2 + 8))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--sizes", default="256x256,1920x1080")
    args = ap.parse_args()
    res = dict(card=card(), params=dict(zip(("pyr_scale", "levels", "winsize", "iterations", "poly_n", "poly_sigma"), REF)),
               results={})
    for size in args.sizes.split(","):
        W, H = (int(v) for v in size.split("x"))
        r = measure(W, H, args.steps)
        res["results"][size] = r
        print(f"{size}: device {r['device_pairs_per_s']} pairs/s ({r['device_over_bracket']} of the bracket's "
              f"{r['bracket_pairs_per_s']}), pinned {r['pinned_pairs_per_s']}, stats {r['stats_pairs_per_s']}, "
              f"per-pair {r['per_pair_pairs_per_s']}; {r['alg_bytes_per_px']['pairs']} B/px vs "
              f"{r['alg_bytes_per_px']['bracket']}", flush=True)
    text = json.dumps(res, indent=1)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")
    else:
        print(text)


if __name__ == "__main__":
    main()
