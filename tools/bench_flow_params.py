"""Device-resident throughput of the flow path for several Farneback parameter sets (bench.py measures the
reference's set only).

    python tools/bench_flow_params.py [--out FILE] [--steps K] [--sizes 256x256,1920x1080]

Per frame size and parameter set: one bracket of frames already resident in HBM (synthetic, seeded) through the whole
hot path, timed with CUDA events on the library's compute stream over --steps brackets after one warm-up bracket;
pairs/s, the algorithmic bytes of the step (ffb_kernel_stats, DESIGN.md section 4) and their share of the HBM data-sheet
bandwidth (7.7 TB/s for one B200), plus per-kernel device times and shares from one profiled bracket.  The card's name
and power limit are read in the same run.  Needs a CUDA device; there is no CPU path.
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

HBM_GBS = 7700.0    # NVIDIA HGX B200 data sheet, one GPU
SETS = {            # (pyr_scale, levels, winsize, iterations, poly_n, poly_sigma)
    "reference": (0.5, 3, 15, 3, 5, 1.2),
    "winsize21": (0.5, 3, 21, 3, 5, 1.2),
    "poly_n7": (0.5, 3, 15, 3, 7, 1.5),
    "levels5": (0.5, 5, 15, 3, 5, 1.2),
    "pyr_scale0.8": (0.8, 3, 15, 3, 5, 1.2),
}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power, smax = (s.strip() for s in q.stdout.strip().split(","))
    return dict(name=name, power_limit=power, sm_max_clock=smax)


def measure(W, H, prm, steps):
    import torch
    from funscript_flow_b200 import _native, runner
    from funscript_flow_b200.synth import make_clip
    batch = runner.default_batch_frames(W, H)
    nf = 2 * batch + 1
    frames = np.ascontiguousarray(np.stack(make_clip(W, H, 17, seed=11, period=9.0, amplitude=0.3)))
    frames = np.concatenate([frames] * (nf // len(frames) + 1))[:nf]
    d = torch.from_numpy(frames).cuda()
    ctx = _native.FlowContext(0)
    ctx.set_farneback(*prm)
    ctx.configure(W, H, batch, nf - 1)

    def step():
        ctx.bracket_begin(False, 7.0)
        ctx.bracket_push_ptr(d.data_ptr(), nf, W, W * H)
        return ctx.bracket_finish()
    step()
    torch.cuda.synchronize()
    ctx.profile_reset()
    ctx.timer_mark(0)
    for _ in range(steps):
        step()
    ctx.timer_mark(1)
    ms = ctx.timer_elapsed_ms(0, 1) / steps
    bytes_step = sum(v["alg_bytes"] for v in ctx.kernel_stats().values()) / steps
    ctx.profile(True)
    ctx.profile_reset()
    step()
    st = ctx.kernel_stats()
    ctx.profile(False)
    kernels = {k: dict(launches=v["launches"], ms=round(v["ms"], 4),
                       hbm_frac=round(v["alg_bytes"] / (v["ms"] / 1e3) / 1e9 / HBM_GBS, 4) if v["ms"] > 0 else None)
               for k, v in st.items() if v["launches"]}
    plan = _native.level_plan_ex(W, H, prm[0], prm[1])
    ctx.close()
    return dict(params=dict(zip(("pyr_scale", "levels", "winsize", "iterations", "poly_n", "poly_sigma"), prm)),
                levels_planned=len(plan), batch_frames=batch, pairs_per_step=nf - 1, ms_per_step=round(ms, 3),
                pairs_per_s=round((nf - 1) / (ms / 1e3), 1), alg_bytes_per_pair=round(bytes_step / (nf - 1)),
                hbm_frac=round(bytes_step / (ms / 1e3) / 1e9 / HBM_GBS, 4), kernels=kernels)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--sizes", default="256x256,1920x1080")
    args = ap.parse_args()
    from funscript_flow_b200 import build
    build.build()
    res = dict(card=card(), hbm_peak_gbs=HBM_GBS, steps=args.steps, results={})
    for size in args.sizes.split(","):
        W, H = (int(v) for v in size.split("x"))
        for name, prm in SETS.items():
            r = measure(W, H, prm, args.steps)
            res["results"][f"{size}/{name}"] = r
            print(f"{size} {name}: {r['pairs_per_s']} pairs/s, {r['hbm_frac']:.3f} of HBM peak", flush=True)
    text = json.dumps(res, indent=1)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")
    else:
        print(text)


if __name__ == "__main__":
    main()
