"""Throughput of backward flows and the forward-backward consistency mask along a sequence of frames
(ffb_farneback_sequence_bidir), next to the forward-only sequence and to the composition it replaces, in one process.

    python tools/bench_bidir.py [--out FILE] [--rounds R] [--sizes 1920x1080,256x256]

Per frame size, reference parameters, batch_frames = runner.default_batch_frames (what the api functions pick), a
sequence of 4 * batch_frames + 1 synthetic, seeded frames as a torch uint8 CUDA tensor (several GB of flows at 1080p:
nothing stays in the 126 MB L2 between calls), outputs as CUDA tensors, three arms timed with CUDA events on the
current torch stream and alternated round by round (the median round of each arm is reported):
  forward      api.calc_optical_flow_farneback_sequence: forward flows only
  bidir        api.calc_optical_flow_farneback_sequence_bidirectional: forward and backward flows and the mask
  composition  the sequence call, api.calc_optical_flow_farneback_batch(frames[1:], frames[:-1]) for the backward flows
               (every frame staged and expanded twice more), and the check as a bilinear gather in torch
Algorithmic bytes per pixel of a pair from ffb_kernel_stats for each arm (the composition's torch check and the flow
copy-outs are not kernels of the library and are not counted), whether the bidir arm's flows equal the other arms' and
its masks the torch check's, and the card's name and power limit, read in the same run.  Needs a CUDA device.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

REF = (0.5, 3, 15, 3, 5, 1.2)
ALPHA, BETA = 0.01, 0.5


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power, smax = (s.strip() for s in q.stdout.strip().split(","))
    return dict(name=name, power_limit=power, sm_max_clock=smax)


def torch_check(torch, fw, bw, chunk=16):
    """The forward-backward check as a bilinear gather in torch (what a user composes today), chunk pairs at a time."""
    n, h, w = fw.shape[:3]
    ys, xs = torch.meshgrid(torch.arange(h, device=fw.device, dtype=torch.float32),
                            torch.arange(w, device=fw.device, dtype=torch.float32), indexing="ij")
    out = torch.empty((n, h, w), dtype=torch.bool, device=fw.device)
    for j0 in range(0, n, chunk):
        f, b = fw[j0:j0 + chunk], bw[j0:j0 + chunk]
        m = f.shape[0]
        tx, ty = xs + f[..., 0], ys + f[..., 1]
        inside = (tx >= 0) & (tx <= w - 1) & (ty >= 0) & (ty <= h - 1)
        tx, ty = torch.where(inside, tx, 0.0), torch.where(inside, ty, 0.0)
        x0f, y0f = torch.floor(tx), torch.floor(ty)
        x0, y0 = x0f.long(), y0f.long()
        x1, y1 = torch.clamp(x0 + 1, max=w - 1), torch.clamp(y0 + 1, max=h - 1)
        ax, ay = tx - x0f, ty - y0f
        rx, ry = 1.0 - ax, 1.0 - ay
        base = (torch.arange(m, device=fw.device) * (h * w)).view(m, 1, 1)
        flat = b.reshape(m * h * w, 2)

        def at(yy, xx):
            return flat[(base + yy * w + xx).reshape(-1)].reshape(m, h, w, 2)
        b00, b01, b10, b11 = at(y0, x0), at(y0, x1), at(y1, x0), at(y1, x1)
        bb = (b00 * rx[..., None] + b01 * ax[..., None]) * ry[..., None] + (b10 * rx[..., None] + b11 * ax[..., None]) * ay[..., None]
        e = ((f + bb) ** 2).sum(-1)
        out[j0:j0 + m] = inside & (e <= ALPHA * ((f ** 2).sum(-1) + (bb ** 2).sum(-1)) + BETA)
    return out


def measure(W, H, rounds):
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

    arms = {
        "forward": lambda: (api.calc_optical_flow_farneback_sequence(f_t, None, *REF, 0, ctx=ctx),),
        "bidir": lambda: api.calc_optical_flow_farneback_sequence_bidirectional(f_t, None, *REF, 0, ctx=ctx),
        "composition": lambda: _composition(),
    }

    def _composition():
        fw = api.calc_optical_flow_farneback_sequence(f_t, None, *REF, 0, ctx=ctx)
        bw = api.calc_optical_flow_farneback_batch(f_t[1:], f_t[:-1], None, *REF, 0, ctx=ctx)
        return fw, bw, torch_check(torch, fw, bw)

    res, geometry, bpp = {}, {}, {}
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
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = fn()
            e1.record()
            e1.synchronize()
            times[name].append(e0.elapsed_time(e1) / 1e3)
            del out
    for name, t in times.items():
        res[f"{name}_pairs_per_s"] = round(n / float(np.median(t)), 1)
        res[f"{name}_pairs_per_s_rounds"] = [round(n / x, 1) for x in t]
    fwd = arms["forward"]()[0]
    bfw, bbw, bmask = arms["bidir"]()
    cfw, cbw, cmask = _composition()
    torch.cuda.synchronize()
    same = dict(forward_vs_forward_arm=bool(torch.equal(bfw, fwd)), forward_vs_composition=bool(torch.equal(bfw, cfw)),
                backward_vs_composition=bool(torch.equal(bbw, cbw)), mask_vs_torch_check=bool(torch.equal(bmask, cmask)),
                mask_pixels_differing_from_torch_check=int((bmask != cmask).sum()),
                consistent_fraction=round(float(bmask.float().mean()), 4))
    del fwd, bfw, bbw, bmask, cfw, cbw, cmask
    ctx.close()
    res.update(batch_frames=batch, n_pairs=n, rounds=rounds,
               geometry={k: dict(zip(("width", "height", "batch_frames", "max_pairs"), v)) for k, v in geometry.items()},
               outputs_equal=same, alg_bytes_per_px=bpp,
               bidir_over_forward=round(res["bidir_pairs_per_s"] / res["forward_pairs_per_s"], 3),
               bidir_over_composition=round(res["bidir_pairs_per_s"] / res["composition_pairs_per_s"], 3))
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
              f"(bidir {r['bidir_over_composition']}x); B/px {r['alg_bytes_per_px']}; {r['outputs_equal']}", flush=True)
    text = json.dumps(res, indent=1)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")
    else:
        print(text)


if __name__ == "__main__":
    main()
