"""Command line with the reference's options (FunscriptFlow.pyw F:2641-2691), GPU backend only.

    python -m funscript_flow_b200 INPUT [--threads N] [--detrend_window S] [--norm_window S] [--batch_size N]
                                  [--overwrite] [--vr_mode] [--pov_mode] [--disable_keyframe_reduction]
                                  [--native_resolution] [--vr_eye left|right|both]      (extensions, SURVEY row N4)
                                  [--flow_pyr_scale S] [--flow_levels N] [--flow_winsize N] [--flow_iterations N]
                                  [--flow_poly_n 5|7] [--flow_poly_sigma S]             (Farneback parameters)

Under `torchrun --nproc-per-node N` every rank takes each N-th video of the folder on its own GPU.
The reference's quirk is kept (SURVEY Q4): `--disable_keyframe_reduction` is a store_false flag whose
value is negated again, so keyframe reduction is OFF by default and the flag turns it ON.
"""
from __future__ import annotations

import argparse
import os
import sys

from . import api, runner


def build_parser() -> argparse.ArgumentParser:
    p = argparse.ArgumentParser(prog="funscript_flow_b200", description="Optical-flow funscript generation on B200")
    p.add_argument("input", help="video file or folder")
    p.add_argument("--threads", type=int, default=8, help="accepted for compatibility; the GPU path does not use it")
    p.add_argument("--detrend_window", type=float, default=2.0)
    p.add_argument("--norm_window", type=float, default=3.0)
    p.add_argument("--batch_size", type=int, default=3000)
    p.add_argument("--overwrite", action="store_true")
    p.add_argument("--vr_mode", action="store_true")
    p.add_argument("--pov_mode", action="store_true")
    p.add_argument("--disable_keyframe_reduction", action="store_false")
    p.add_argument("--backend", default="CUDA", help="accepted for compatibility; there is one backend")
    # extensions the reference has no equivalent of (runner.preprocess_plan)
    p.add_argument("--native_resolution", action="store_true", help="run the flow on the decoded frame size instead of 256x256")
    p.add_argument("--vr_eye", choices=["left", "right", "both"], default="left",
                   help="which eye of a side-by-side VR frame (with --vr_mode); both = mean of the two eyes' scalars")
    # cv2.calcOpticalFlowFarneback's parameters; the defaults are the reference's call (F:878-879)
    ref = api.REFERENCE_FARNEBACK
    p.add_argument("--flow_pyr_scale", type=float, default=ref["pyr_scale"], help="pyramid scale between levels, 0 < s < 1")
    p.add_argument("--flow_levels", type=int, default=ref["levels"], help="pyramid levels above the frame (>= 0)")
    p.add_argument("--flow_winsize", type=int, default=ref["winsize"], help="averaging window, 3 .. 63")
    p.add_argument("--flow_iterations", type=int, default=ref["iterations"], help="iterations per level, 1 .. 20")
    p.add_argument("--flow_poly_n", type=int, choices=[5, 7], default=ref["poly_n"], help="polynomial expansion size")
    p.add_argument("--flow_poly_sigma", type=float, default=ref["poly_sigma"], help="polynomial expansion sigma (>= 0)")
    return p


def settings_from_args(args) -> dict:
    """The settings dict of F:2654-2664 (same keys; the extension keys appear only when used)."""
    settings = {
        "threads": args.threads,
        "detrend_window": args.detrend_window,
        "norm_window": args.norm_window,
        "batch_size": args.batch_size,
        "overwrite": args.overwrite,
        "vr_mode": args.vr_mode,
        "pov_mode": args.pov_mode,
        "keyframe_reduction": not args.disable_keyframe_reduction,
        "backend": "CUDA",
    }
    if getattr(args, "native_resolution", False):
        settings["native_resolution"] = True
    if getattr(args, "vr_eye", "left") != "left":
        settings["vr_eye"] = args.vr_eye
    for key, name in api.FARNEBACK_SETTINGS.items():
        value = getattr(args, key, None)
        if value is not None and value != api.REFERENCE_FARNEBACK[name]:
            settings[key] = value
    return settings


def main(argv=None) -> int:
    args = build_parser().parse_args(argv)
    if not os.path.exists(args.input):
        print(f"input not found: {args.input}", file=sys.stderr)
        return 2
    errors = runner.run_headless(args.input, settings_from_args(args))
    return 1 if errors else 0


if __name__ == "__main__":
    sys.exit(main())
