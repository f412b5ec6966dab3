"""Throughput of backward flows and the forward-backward consistency mask for independent frame pairs
(ffb_farneback_pairs_bidir), next to the forward-only pairs call and to the composition it replaces, in one process.

    python tools/bench_pairs_bidir.py [--out FILE] [--rounds R] [--sizes 1920x1080,256x256]

Per frame size, reference parameters, batch_frames = api._pairs_batch (what the api functions pick), n = 3 chunks of
(batch_frames + 1) / 2 pairs, the frames synthetic and seeded, each pair two frames of one clip in a shuffled order
(several GB of flows at 1080p: nothing stays in the 126 MB L2 between calls).  Four arms, alternated round by round, each
timed with a host clock around the call and a device synchronisation (the median round of each arm is reported):
  forward      api.calc_optical_flow_farneback_batch on torch uint8 CUDA tensors: forward flows only
  bidir        api.calc_optical_flow_farneback_batch_bidirectional on the same tensors: both flows and the mask
  composition  the batch call, the batch call on the reversed pairs (every frame staged and expanded twice more), and
               the check as a bilinear gather in torch (bench_bidir.torch_check)
  pinned       FlowContext.farneback_pairs_bidir_ptr from page-locked host frames into page-locked host flows and masks
               (each pair crosses PCIe as 2 frames in, 2 flows and a mask out: 2 + 16 + 1 bytes per pixel)
Algorithmic bytes per pixel of a pair from ffb_kernel_stats for each arm (the composition's torch check and the flow
copy-outs are not kernels of the library and are not counted), whether the bidir arm's flows and masks equal the
composition's and the pinned arm's, and the card's name and power limit, read in the same run.  Needs a CUDA device.
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

from bench_bidir import ALPHA, BETA, REF, card, torch_check  # noqa: E402


def measure(W, H, rounds):
    import torch
    from funscript_flow_b200 import _native, api
    from funscript_flow_b200.synth import make_clip
    batch = api._pairs_batch(W, H, 1 << 20)
    n = 3 * ((batch + 1) // 2)
    clip = make_clip(W, H, 33, seed=11, period=9.0, amplitude=0.3)
    rng = np.random.default_rng(5)
    ia, ib = rng.integers(0, 33, n), rng.integers(0, 33, n)
    prev, nxt = np.ascontiguousarray(clip[ia]), np.ascontiguousarray(clip[ib])
    ctx = _native.FlowContext(0)
    dev = torch.device("cuda", 0)
    p_t, n_t = torch.from_numpy(prev).to(dev), torch.from_numpy(nxt).to(dev)
    pins = [_native.PinnedBuffer(prev.shape), _native.PinnedBuffer(nxt.shape), _native.PinnedBuffer((2, n, H, W, 8)),
            _native.PinnedBuffer((n, H, W))]
    pins[0].array[...] = prev
    pins[1].array[...] = nxt
    fw_h, bw_h = pins[2].array.view(np.float32).reshape(2, n, H, W, 2)
    mask_h = pins[3].array

    def composition():
        fw = api.calc_optical_flow_farneback_batch(p_t, n_t, None, *REF, 0, ctx=ctx)
        bw = api.calc_optical_flow_farneback_batch(n_t, p_t, None, *REF, 0, ctx=ctx)
        return fw, bw, torch_check(torch, fw, bw)

    def pinned():
        ctx.configure(W, H, batch, 1)
        ctx.farneback_pairs_bidir_ptr(pins[0].array.ctypes.data, pins[1].array.ctypes.data, n, W, H, W, W * H, fw_h, bw_h,
                                      mask=mask_h, alpha=ALPHA, beta=BETA)
        return fw_h, bw_h, mask_h

    arms = {
        "forward": lambda: (api.calc_optical_flow_farneback_batch(p_t, n_t, None, *REF, 0, ctx=ctx),),
        "bidir": lambda: api.calc_optical_flow_farneback_batch_bidirectional(p_t, n_t, None, *REF, 0, alpha=ALPHA,
                                                                              beta=BETA, ctx=ctx),
        "composition": composition,
        "pinned": pinned,
    }
    res, geometry, bpp = {}, {}, {}
    try:
        for name, fn in arms.items():        # warm-up, geometry, algorithmic bytes
            out = fn()
            torch.cuda.synchronize()
            geometry[name] = ctx.geometry
            del out
            ctx.profile_reset()
            out = fn()
            torch.cuda.synchronize()
            bpp[name] = round(sum(v["alg_bytes"] for v in ctx.kernel_stats().values()) / n / (W * H), 1)
            del out
        times = {k: [] for k in arms}
        for _ in range(rounds):
            for name, fn in arms.items():
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                out = fn()
                torch.cuda.synchronize()
                times[name].append(time.perf_counter() - t0)
                del out
        for name, t in times.items():
            res[f"{name}_pairs_per_s"] = round(n / float(np.median(t)), 1)
            res[f"{name}_pairs_per_s_rounds"] = [round(n / x, 1) for x in t]
        bfw, bbw, bmask = arms["bidir"]()
        cfw, cbw, cmask = composition()
        pinned()
        torch.cuda.synchronize()
        same = dict(forward_vs_composition=bool(torch.equal(bfw, cfw)), backward_vs_composition=bool(torch.equal(bbw, cbw)),
                    mask_vs_torch_check=bool(torch.equal(bmask, cmask)),
                    mask_pixels_differing_from_torch_check=int((bmask != cmask).sum()),
                    pinned_vs_bidir=bool(np.array_equal(fw_h, bfw.cpu().numpy()) and np.array_equal(bw_h, bbw.cpu().numpy())
                                         and np.array_equal(mask_h.view(np.bool_), bmask.cpu().numpy())),
                    consistent_fraction=round(float(bmask.float().mean()), 4))
        del bfw, bbw, bmask, cfw, cbw, cmask
    finally:
        for b in pins:
            b.free()
        ctx.close()
    res.update(batch_frames=batch, n_pairs=n, rounds=rounds,
               geometry={k: dict(zip(("width", "height", "batch_frames", "max_pairs"), v)) for k, v in geometry.items()},
               outputs_equal=same, alg_bytes_per_px=bpp,
               bidir_over_forward=round(res["bidir_pairs_per_s"] / res["forward_pairs_per_s"], 3),
               bidir_over_composition=round(res["bidir_pairs_per_s"] / res["composition_pairs_per_s"], 3),
               pinned_over_bidir=round(res["pinned_pairs_per_s"] / res["bidir_pairs_per_s"], 3))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--sizes", default="1920x1080,256x256")
    args = ap.parse_args()
    res = dict(card=card(), params=dict(zip(("pyr_scale", "levels", "winsize", "iterations", "poly_n", "poly_sigma"), REF)),
               check=dict(alpha=ALPHA, beta=BETA), results={})
    for size in args.sizes.split(","):
        W, H = (int(v) for v in size.split("x"))
        r = measure(W, H, args.rounds)
        res["results"][size] = r
        print(f"{size}: forward {r['forward_pairs_per_s']} pairs/s, bidir {r['bidir_pairs_per_s']} "
              f"({r['bidir_over_forward']} of forward), composition {r['composition_pairs_per_s']} "
              f"(bidir {r['bidir_over_composition']}x), pinned {r['pinned_pairs_per_s']}; B/px {r['alg_bytes_per_px']}; "
              f"{r['outputs_equal']}", flush=True)
    text = json.dumps(res, indent=1)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")
    else:
        print(text)


if __name__ == "__main__":
    main()
