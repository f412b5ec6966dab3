"""Throughput of Farneback flow along a sequence of frames (ffb_farneback_sequence), next to the bracket and the
independent-pairs path over the same pairs, in one process.

    python tools/bench_sequence.py [--out FILE] [--steps K] [--sizes 256x256,1920x1080]

Per frame size, reference parameters, batch_frames = runner.default_batch_frames (what
api.calc_optical_flow_farneback_sequence picks), a sequence of 4 * batch_frames + 1 synthetic, seeded frames
(4 * batch_frames pairs, several GB of flows at 1080p: nothing stays in the 126 MB L2 between steps):
  device      a torch uint8 CUDA tensor in, a float32 CUDA tensor out (api.calc_optical_flow_farneback_sequence), timed
              with CUDA events on the current torch stream
  pinned      page-locked host frames in, page-locked host flows out (the flows cross PCIe: 8 bytes per pixel)
  stats       device frames in, device flows out, and the bracket's per-pair results to the host
  bracket     the same frames as one bracket resident in HBM (bracket_push_ptr), flows not exported: the streaming rate
  pairs       the same pairs as independent pairs (api.calc_optical_flow_farneback_batch on frames[:-1], frames[1:]),
              tensors in and out, CUDA events
Host-clock arms end in a device synchronisation.  Algorithmic bytes per pixel of a pair (ffb_kernel_stats; the flow
copy-out of a sequence is a copy, not a kernel, and is listed apart) for each path, whether the flows of every arm are
bit-identical, the geometry each arm ran with, and the card's name and power limit are read in the same run.  Needs a
CUDA device; there is no CPU path.
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


def event_rate(torch, fn, n, steps):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    e1.synchronize()
    return n * steps / (e0.elapsed_time(e1) / 1e3)


def alg_bytes_per_px(torch, ctx, fn, n, W, H):
    torch.cuda.synchronize()
    ctx.profile_reset()
    fn()
    torch.cuda.synchronize()
    return sum(v["alg_bytes"] for v in ctx.kernel_stats().values()) / n / (W * H)


def measure(W, H, steps):
    import torch
    from funscript_flow_b200 import _native, api, runner
    from funscript_flow_b200.synth import make_clip
    batch = runner.default_batch_frames(W, H)
    n = 4 * batch                                      # pairs
    base = np.ascontiguousarray(make_clip(W, H, 33, seed=11, period=9.0, amplitude=0.3))
    frames = np.ascontiguousarray(np.concatenate([base, base[::-1][1:]] * (n // 64 + 1))[:n + 1])
    ctx = _native.FlowContext(0)
    dev = torch.device("cuda", 0)
    f_t = torch.from_numpy(frames).to(dev)
    out, geometry, same = {}, {}, {}

    def device_call():
        return api.calc_optical_flow_farneback_sequence(f_t, None, *REF, 0, ctx=ctx)
    flow_t = device_call()
    geometry["sequence"] = ctx.geometry
    out["device_pairs_per_s"] = round(event_rate(torch, device_call, n, steps), 1)
    seq_bpp = alg_bytes_per_px(torch, ctx, device_call, n, W, H)
    flow_t = device_call()
    torch.cuda.synchronize()

    pin_f = _native.PinnedBuffer(frames.shape)
    pin_f.array[...] = frames
    pin_o = _native.PinnedBuffer((n, H, W, 8))
    flow_h = pin_o.array.view(np.float32).reshape(n, H, W, 2)

    def pinned_call():
        ctx.farneback_sequence_ptr(pin_f.array.ctypes.data, n + 1, W, H, W, W * H, flow_h.ctypes.data, W * 8, W * H * 8)
    out["pinned_pairs_per_s"] = round(host_rate(pinned_call, n, steps), 1)
    same["pinned"] = bool(np.array_equal(flow_h, flow_t.cpu().numpy()))

    out_t = torch.empty_like(flow_t)

    def stats_call():
        return ctx.farneback_sequence_ptr(f_t.data_ptr(), n + 1, W, H, W, W * H, out_t.data_ptr(), W * 8, W * H * 8, stats=True)
    out["stats_pairs_per_s"] = round(host_rate(stats_call, n, steps), 1)
    stats_bpp = alg_bytes_per_px(torch, ctx, stats_call, n, W, H)
    same["stats"] = bool(torch.equal(out_t, flow_t))

    ctx.configure(W, H, batch, n)

    def bracket_call():
        ctx.bracket_begin(False, 7.0)
        ctx.bracket_push_ptr(f_t.data_ptr(), n + 1, W, W * H)
        return ctx.bracket_finish()
    bracket_call()
    geometry["bracket"] = ctx.geometry
    ctx.timer_mark(0)
    for _ in range(steps):
        bracket_call()
    ctx.timer_mark(1)
    out["bracket_pairs_per_s"] = round(n * steps / (ctx.timer_elapsed_ms(0, 1) / 1e3), 1)
    bracket_bpp = alg_bytes_per_px(torch, ctx, bracket_call, n, W, H)

    def pairs_call():
        return api.calc_optical_flow_farneback_batch(f_t[:-1], f_t[1:], None, *REF, 0, ctx=ctx)
    del out_t
    pairs_call()
    geometry["pairs"] = ctx.geometry
    out["pairs_pairs_per_s"] = round(event_rate(torch, pairs_call, n, steps), 1)
    pairs_bpp = alg_bytes_per_px(torch, ctx, pairs_call, n, W, H)
    same["pairs"] = bool(torch.equal(pairs_call(), flow_t))

    for b in (pin_f, pin_o):
        b.free()
    ctx.close()
    assert geometry["sequence"][2] == batch and geometry["bracket"][2] == batch, geometry
    out.update(batch_frames=batch, n_pairs=n, steps=steps,
               geometry={k: dict(zip(("width", "height", "batch_frames", "max_pairs"), v)) for k, v in geometry.items()},
               flows_equal_device=same,
               alg_bytes_per_px=dict(sequence_kernels=round(seq_bpp, 1), sequence_flow_copy=16.0,
                                     sequence_stats_kernels=round(stats_bpp, 1), bracket=round(bracket_bpp, 1),
                                     pairs=round(pairs_bpp, 1)),
               device_over_bracket=round(out["device_pairs_per_s"] / out["bracket_pairs_per_s"], 3),
               device_over_pairs=round(out["device_pairs_per_s"] / out["pairs_pairs_per_s"], 3),
               pcie_bytes_per_pair_pinned=W * H * (1 + 8))
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
              f"{r['bracket_pairs_per_s']}, {r['device_over_pairs']} x the pairs path's {r['pairs_pairs_per_s']}), "
              f"pinned {r['pinned_pairs_per_s']}, stats {r['stats_pairs_per_s']}; B/px {r['alg_bytes_per_px']}", flush=True)
    text = json.dumps(res, indent=1)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")
    else:
        print(text)


if __name__ == "__main__":
    main()
