#!/usr/bin/env python
"""bench.py -- frame-pairs/sec of the hot path at 1080p (BASELINE.json metric), one process per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2|c2-strong|c5]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
           --master-port P bench.py --gpus N --steps K --warmup W

Workloads (BASELINE.json configs):
  c2         (default, the headline) a step = one bracket of (pairs_per_step + 1) synthetic 1080p frames
             ("synthetic 1920x1080 30 fps 10-minute clip on 1 B200", a window of it) through the whole hot path:
             pyramid + polynomial expansion per frame, 3 flow iterations on each of the 4 levels per pair,
             divergence argmax + magnitude mean, +-6 centre smoothing, radial reduction, D2H of the per-pair
             scalars.  With N GPUs every rank runs its own window: weak scaling, no data-path collective.
  c2-strong  ONE bracket of --strong-pairs pairs cut into N frame ranges with one frame of overlap
             (distributed.process_bracket_sharded: flows per shard, all-gather of the raw centres, radial pass,
             all-gather of the scalars): strong scaling of a single video over the GPUs.
  c5         64 in-memory synthetic 1080p clips of unequal length dealt longest-first to the ranks
             (runner.schedule_longest_first), every clip through runner.process_frames (brackets, post-processing),
             scalars gathered with all_gather_object: whole-library throughput, host frames, end to end.

`value` is measured with the frames already resident in HBM (CUDA events on the library's compute stream);
`e2e` through the public bracket API from pinned host frames (H2D inside the timed region, wall clock between
device synchronisations).  Rank 0 prints ONE JSON line.

--dump-outputs DIR: rank 0 writes what the timed path returned in its last timed step as DIR/<name>.npy (float32 or
float64; integer and boolean outputs as float64, which holds them exactly).  The inputs are generated from fixed
seeds, so two builds run with the same arguments can be compared output for output.

The benchmark writes nothing into the source tree, which may be read-only: a library older than its sources is
rebuilt in a temporary directory, and no bytecode is cached.
"""
from __future__ import annotations

import argparse
import atexit
import hashlib
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True
os.environ["PYTHONDONTWRITEBYTECODE"] = "1"      # for the spawned workers of the CPU baseline too

import numpy as np  # noqa: E402

METRIC = "frame_pairs_per_sec_1080p"
UNIT = "pairs/s"
WHOLE_PATH_B_PER_PX = 269.7     # SURVEY.md 8(d): streaming-mode algorithmic bytes per pixel and pair, 4 levels


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=["c2", "c2-strong", "c5"])
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--pairs-per-step", type=int, default=256,
                    help="pairs of one bracket = one step (the reference's brackets hold 3000 frames, F:2661)")
    ap.add_argument("--batch-frames", type=int, default=0, help="0 = runner.default_batch_frames(width, height)")
    ap.add_argument("--strong-pairs", type=int, default=1536, help="c2-strong: pairs of the one bracket that is split")
    ap.add_argument("--c5-videos", type=int, default=64)
    ap.add_argument("--c5-pageable", action="store_true", help="c5: clips in ordinary (pageable) NumPy memory instead of pinned buffers")
    ap.add_argument("--cpu-sample-pairs", type=int, default=0, help="0 = 2 x host cores (bounded to 8..64)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the pageable / drop-in / per-level side measurements")
    ap.add_argument("--no-numa-bind", action="store_true", help="do not pin the process to the GPU's NUMA node")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def dump_outputs(out_dir, arrays):
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        if a.dtype not in (np.float32, np.float64):
            a = a.astype(np.float64)
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def bench_config(args, world):
    """The `config` object of the JSON line: identical for the GPU arm and the reference arm."""
    W, H, P = args.width, args.height, args.pairs_per_step
    if args.workload == "c2":
        wl = f"C2: synthetic {W}x{H} 30 fps clip, window of {P + 1} frames per step per GPU"
        par = f"brackets x{world}"
    elif args.workload == "c2-strong":
        wl = f"C2 strong: ONE bracket of {args.strong_pairs + 1} synthetic {W}x{H} frames split into {world} frame ranges"
        par = f"frame ranges x{world} (one frame of overlap, all-gather of raw centres)"
    else:
        wl = f"C5: {args.c5_videos} in-memory synthetic {W}x{H} clips of 65..193 frames, longest-first over {world} GPU(s)"
        par = f"videos x{world}"
    return {"workload": wl, "pairs_per_step": P if args.workload == "c2" else None, "levels": 4, "iterations": 3,
            "l2": "inputs_exceed_l2 (per-step working set >> 126 MB)", "parallelism": par}


def workload_frames(width, height, n, rank, start=7):
    from funscript_flow_b200.synth import ClipGenerator, ClipSpec
    spec = ClipSpec(width, height, 18000, seed=0, amplitude=0.15, period=30.0)   # config C2 generator
    gen = ClipGenerator(spec)
    first = start + rank * n
    return gen.stack(first, first + n)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 50 ms while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


def kernels_sha():
    h = hashlib.sha256()
    for f in ("ffb_kernels.cuh", "ffb_api.cu", "ffb_common.h"):
        h.update(open(os.path.join(ROOT, "funscript_flow_b200", "csrc", f), "rb").read())
    return h.hexdigest()[:16]


def committed_traffic(W, H):
    """DRAM bytes of the dominant launch from the committed `ncu --set full` capture -- refused when the kernel
    sources have changed since it was taken (the record carries their hash)."""
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))
    except Exception:
        return None, "no committed capture"
    if (W, H) != (1920, 1080):
        return None, "the committed capture is of the 1920x1080 launch"
    if tj.get("kernels_sha") != kernels_sha():
        return None, f"stale: captured at kernel sources {tj.get('kernels_sha')}, now {kernels_sha()} -- re-run tools/profile_round.sh"
    note = (f"{tj['launch_shape']}: dram read+write {tj['traffic'] / 1e9:.3f} GB vs algorithmic "
            f"{tj['alg_bytes_per_launch'] / 1e9:.3f} GB per launch ({tj['source']})")
    return tj["traffic"], note


# ------------------------------------------------------------------------------------------- reference arm
def cpu_arm(frames, cores, sample_pairs):
    """The reference's CPU implementation of the path on `cores` host cores, on the first `sample_pairs` pairs of
    `frames`: the reference's own functions (oracle/ref_pipeline.py, FunscriptFlow.pyw staged in baseline/_ref/)
    when the file is present, else the port (oracle/cpu_pipeline.py: the same cv2 / NumPy calls).
    Returns (pairs/s, seconds, flow-phase pairs/s, kind)."""
    from oracle import ref_pipeline
    sub = list(frames[:sample_pairs + 1])
    if ref_pipeline.available():
        _, _, sec, sec_flow = ref_pipeline.run_bracket(sub, {}, cores)
        kind = "reference"
    else:
        from oracle import cpu_pipeline
        _, _, sec, sec_flow = cpu_pipeline.run_bracket(sub, {}, cores)
        kind = "port"
    return sample_pairs / sec, sec, sample_pairs / sec_flow, kind


def cpu_sample_text(kind, sample, cores, extra=""):
    import cv2
    what = ("the reference's own precompute_wrapper / radial_motion_weighted (FunscriptFlow.pyw, unmodified, staged in baseline/_ref/) "
            "driven as F:1190-1236" if kind == "reference" else "port of F:1190-1236 calling the same cv2 Farneback + NumPy")
    return f"{sample} pairs{extra}; {what}; Pool({cores}) + ProcessPoolExecutor({cores}), cv2 {cv2.__version__}"


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path, all host cores, rank 0 only."""
    if rank != 0:
        return
    from oracle import cpu_pipeline
    cores = cpu_pipeline.usable_cores()
    sample = args.cpu_sample_pairs or int(min(64, max(8, 2 * cores)))
    frames = workload_frames(args.width, args.height, sample + 1, 0)
    for _ in range(max(0, min(args.warmup, 1))):
        cpu_arm(frames, cores, min(sample, cores))
    t, kind = [], "port"
    for _ in range(args.steps):
        _, sec, _, kind = cpu_arm(frames, cores, sample)
        t.append(sec)
    total = sum(t)
    value = sample * args.steps / total
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1000 * total / args.steps, "higher_is_better": True,
            "scaling": "strong" if args.workload == "c2-strong" else "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": bench_config(args, world),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind,
                             "sample": cpu_sample_text(kind, sample, cores, f" per step x {args.steps} steps (each step a bounded "
                                                       f"sample of the GPU arm's step: its first {sample} pairs)")},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------- GPU arm
class Dist:
    """torch.distributed over NCCL for the barrier, the max-over-ranks reduction and the scalar gathers."""

    def __init__(self, rank, world, local):
        self.rank, self.world, self.dist = rank, world, None
        if world > 1:
            import torch
            import torch.distributed as dist
            # NCCL announces its version on stdout when the communicator is created; stdout carries the ONE JSON
            # line of the contract, so that chatter goes to stderr
            sys.stdout.flush()
            saved_stdout = os.dup(1)
            os.dup2(2, 1)
            try:
                dist.init_process_group(backend="nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local))
                dist.barrier()
            finally:
                sys.stdout.flush()
                os.dup2(saved_stdout, 1)
                os.close(saved_stdout)
            self.dist = dist

    def barrier(self):
        if self.dist is not None:
            import torch
            self.dist.barrier()
            torch.cuda.synchronize()

    def max(self, x):
        if self.dist is None:
            return x
        import torch
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def close(self):
        if self.dist is not None:
            self.dist.barrier()
            self.dist.destroy_process_group()


def per_level_pass(local, W, H, batch, d_frames, nf, peak):
    """roofline.by_level: one flow stream gives per-launch CUDA-event times (with two streams the launch chains
    overlap and only the phase can be timed), so a second context created with FFB_FLOW_STREAMS=1 runs two steps."""
    from funscript_flow_b200 import _native
    old = os.environ.get("FFB_FLOW_STREAMS")
    os.environ["FFB_FLOW_STREAMS"] = "1"
    try:
        ctx = _native.FlowContext(local)
    finally:
        if old is None:
            os.environ.pop("FFB_FLOW_STREAMS", None)
        else:
            os.environ["FFB_FLOW_STREAMS"] = old
    ctx.configure(W, H, batch, nf - 1)

    def step():
        ctx.bracket_begin(False, 7.0)
        ctx.bracket_push_ptr(d_frames.data_ptr(), nf, W, W * H)
        return ctx.bracket_finish()
    step()
    ctx.profile(True)
    ctx.profile_reset()
    for _ in range(2):
        step()
    lv = ctx.flow_iter_level_stats()
    st = ctx.kernel_stats()
    ctx.profile(False)
    ctx.close()
    by_level = {f"k{k}": {"launches": v["launches"], "ms_per_launch": v["ms"] / v["launches"],
                          "achieved": v["alg_bytes"] / (v["ms"] / 1000.0) / 1e9,
                          "frac": v["alg_bytes"] / (v["ms"] / 1000.0) / 1e9 / peak}
                for k, v in sorted(lv.items()) if v["ms"] > 0}
    kernels = {k: {"ms_per_launch": v["ms"] / v["launches"], "achieved": v["alg_bytes"] / (v["ms"] / 1000.0) / 1e9,
                   "frac": v["alg_bytes"] / (v["ms"] / 1000.0) / 1e9 / peak}
               for k, v in st.items() if v["launches"] and v["ms"] > 0 and v["alg_bytes"] > 0}
    return by_level, kernels


def run_c2(args, rank, world, local, dd, numa_node, all_cpus):
    import torch
    from funscript_flow_b200 import _native, api, runner
    W, H, P = args.width, args.height, args.pairs_per_step
    batch = args.batch_frames or runner.default_batch_frames(W, H)
    nf = P + 1
    frames = workload_frames(W, H, nf, rank)                     # uint8 [nf, H, W]; 257 x 2 MB >> L2
    ctx = _native.FlowContext(local)
    ctx.configure(W, H, batch, P)
    d_frames = torch.from_numpy(frames).cuda()
    pinned = _native.PinnedBuffer(frames.shape)
    pinned.array[...] = frames

    def step_resident():
        ctx.bracket_begin(False, 7.0)
        ctx.bracket_push_ptr(d_frames.data_ptr(), nf, W, W * H)
        return ctx.bracket_finish()

    def step_host(arr):
        ctx.bracket_begin(False, 7.0)
        ctx.bracket_push(arr)
        return ctx.bracket_finish()

    def fence():
        ctx.sync()
        torch.cuda.synchronize()
        dd.barrier()

    # ---- device-resident arm ("value") --------------------------------------------------------
    r0 = None
    for _ in range(args.warmup):
        r0 = step_resident()
    fence()
    allocs0 = ctx.alloc_counts()
    sampler = ClockSampler(local)
    sampler.start()
    ctx.profile(True)
    ctx.profile_reset()
    l0 = ctx.launch_count
    ctx.timer_mark(0)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        r = step_resident()
    ctx.timer_mark(1)
    fence()
    wall_res = time.perf_counter() - t0
    dev_ms = ctx.timer_elapsed_ms(0, 1)
    launches = ctx.launch_count - l0
    stats = ctx.kernel_stats()
    ctx.profile(False)
    # ---- end-to-end arm ("e2e"): pinned host frames, H2D + D2H of every step inside the timed region.  Consecutive
    # brackets go through the public api.BracketPipeline, as runner.process_frames sends the brackets of a video:
    # two contexts of the GPU alternate, so the upload of step i+1 overlaps the kernels of step i (each step still
    # uploads its 257 frames and fetches its 256 results).  `e2e_single_context` below is the same loop without it.
    pipe = api.BracketPipeline(ctx, batch_frames=batch)
    for _ in range(max(2, args.warmup // 2)):
        pipe.submit(pinned.array, {})
    pipe.flush()
    fence()
    allocs0 = ctx.alloc_counts()
    t0 = time.perf_counter()
    r_e = None
    for _ in range(args.steps):
        done = pipe.submit(pinned.array, {})
        r_e = done if done is not None else r_e
    r_e = pipe.flush()
    pipe.ctxs[1].sync()
    fence()
    wall_e2e = time.perf_counter() - t0
    for _ in range(2):
        step_host(pinned.array)
    fence()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_host(pinned.array)
    fence()
    wall_e2e_single = dd.max(time.perf_counter() - t0)
    clocks = sampler.stop()
    # the device-resident and the end-to-end arm (and the warm-up) computed the same numbers
    assert r["n_pairs"] == P and np.array_equal(r["scalar"], r_e["scalar"])
    assert r0 is None or np.array_equal(r["scalar"], r0["scalar"])
    assert ctx.alloc_counts() == allocs0, "the timed region allocated memory"
    extras = {"e2e_single_context": {"value": P * args.steps * world / wall_e2e_single, "unit": UNIT,
                                     "note": "the e2e loop on ONE context: every bracket's first upload and last kernels are exposed"}}

    dev_ms = dd.max(dev_ms)
    wall_e2e = dd.max(wall_e2e)
    total_pairs = P * args.steps * world
    value = total_pairs / (dev_ms / 1000.0)
    e2e = total_pairs / wall_e2e

    if not args.no_extras:
        # what callers actually hold: ordinary (pageable) NumPy frames, staged through the library's pinned buffers
        k = max(2, min(args.steps, 8))
        for _ in range(2):
            pipe.submit(frames, {})
        pipe.flush()
        fence()
        t0 = time.perf_counter()
        for _ in range(k):
            pipe.submit(frames, {})
        r_p = pipe.flush()
        pipe.ctxs[1].sync()
        fence()
        wall_p = dd.max(time.perf_counter() - t0)
        assert np.array_equal(r_p["scalar"], r["scalar"])
        extras["e2e_pageable"] = {"value": P * k * world / wall_p, "unit": UNIT, "steps": k,
                                  "note": "the e2e loop from pageable NumPy memory (4 host threads copy into the pinned double buffer, then DMA)"}
        # the per-pair drop-in (F:843 precompute_flow_info + F:761 radial_motion_weighted): two frames up, one flow field down
        if rank == 0:
            api.set_context(ctx, api.default_device())
            n_drop = 24
            api.precompute_flow_info(frames[0], frames[1], {})
            t0 = time.perf_counter()
            for j in range(n_drop):
                info = api.precompute_flow_info(frames[j], frames[j + 1], {})
                api.radial_motion_weighted(info["flow"], info["pos_center"], info["cut"])
            extras["dropin_per_pair"] = {"value": n_drop / (time.perf_counter() - t0), "unit": UNIT, "pairs": n_drop,
                                         "note": "precompute_flow_info + radial_motion_weighted per pair through the Python mirror "
                                                 "(16.6 MB flow field down and up again per pair, as the reference's dict contract requires)"}
        dd.barrier()

    line = None
    if rank == 0:
        peak, peak_kind = measured_peak()
        it = stats["flow_iter"]
        achieved = it["alg_bytes"] / (it["ms"] / 1000.0) / 1e9 if it["ms"] > 0 else 0.0
        kernel_ms = {k: round(v["ms"] / args.steps, 4) for k, v in stats.items()}
        traffic, traffic_note = committed_traffic(W, H)
        by_level, per_kernel = ({}, {})
        if not args.no_extras:
            by_level, per_kernel = per_level_pass(local, W, H, batch, d_frames, nf, peak)
        cfg = bench_config(args, world)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": cfg,
            "run": {"batch_frames": batch, "numa_node": numa_node, "flow_streams": int(os.environ.get("FFB_FLOW_STREAMS", "2")),
                    "kernels_sha": kernels_sha()},
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": int(nf * W * H), "d2h_bytes_per_step": int(P * 41),
                    "ms_per_step": 1000 * wall_e2e / args.steps,
                    "source": "pinned host frames, consecutive brackets through api.BracketPipeline (two contexts of the GPU alternate)"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": "k_flow_iter", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "traffic_note": traffic_note,
                         "peak_source": f"MEASURED_PEAKS.json ({peak_kind})",
                         "alg_bytes_per_launch": it["alg_bytes"] / max(1, it["launches"]),
                         "avg_launch_ms": it["ms"] / max(1, it["launches"]), "launches": it["launches"],
                         "timing": ("the launch chains of the half-batches overlap on two streams, so the time is the device time of "
                                    "the flow phases (CUDA events on the compute stream around fork..join) and achieved = bytes of all "
                                    "k_flow_iter launches / that time; by_level and per_kernel come from a one-stream pass of two steps "
                                    "in the same run (per-launch CUDA events)"),
                         "by_level": by_level, "per_kernel_one_stream": per_kernel,
                         "whole_path_bytes_per_pair": WHOLE_PATH_B_PER_PX * W * H,
                         "whole_path_frac": WHOLE_PATH_B_PER_PX * W * H * value / world / 1e9 / peak},
            "kernel_ms_per_step": kernel_ms,
            "kernel_ms_note": ("CUDA-event time per kernel class; with 2 flow streams k_flow_iter is the flow-phase time and "
                               "k_divmag (launched per slice, overlapping the other slice's flow tail) includes that overlap"),
            "wall_ms_per_step_resident": 1000 * wall_res / args.steps,
        }
        line.update(extras)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {k: v for k, v in r.items() if isinstance(v, np.ndarray)})
        if world == 1 and not args.no_cpu_baseline:
            from oracle import cpu_pipeline
            os.sched_setaffinity(0, all_cpus)      # the CPU baseline gets every host core again
            cores = cpu_pipeline.usable_cores()
            sample = args.cpu_sample_pairs or int(min(64, max(8, 2 * cores)))
            sample = min(sample, P)
            v, sec, vflow, kind = cpu_arm(frames, cores, sample)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": kind,
                                    "sample": cpu_sample_text(kind, sample, cores, f" (the first {sample} pairs of the same step), {sec:.1f} s"),
                                    "flow_phase_only": vflow}
    ctx.close()
    return line


def run_c2_strong(args, rank, world, local, dd, numa_node):
    """One bracket over all GPUs: rank r owns pairs [a_r, b_r), pushes frames a_r .. b_r, the raw centres are
    all-gathered between the phases and the scalars at the end (distributed.process_bracket_sharded)."""
    import torch
    from funscript_flow_b200 import _native, api, distributed, runner
    W, H, NP = args.width, args.height, args.strong_pairs
    batch = args.batch_frames or runner.default_batch_frames(W, H)
    a, b = api.shard_bounds(NP, world)[rank]
    frames = workload_frames(W, H, b - a + 1, 0, start=7 + a)     # this rank's frame range of the one clip
    ctx = _native.FlowContext(local)
    api.set_context(ctx, api.default_device())
    pinned = _native.PinnedBuffer(frames.shape)
    pinned.array[...] = frames
    d_frames = torch.from_numpy(frames).cuda()
    most = max(hi - lo for lo, hi in api.shard_bounds(NP, world))

    def step(src_ptr=None, host=None):
        ctx.configure(W, H, batch, b - a)
        ctx.bracket_begin_shard(b - a, False, 7.0)
        if host is not None:
            ctx.bracket_push(host)
        else:
            ctx.bracket_push_ptr(src_ptr, b - a + 1, W, W * H)
        p1 = ctx.bracket_phase1_finish()
        local_c = np.stack([p1["cx"], p1["cy"], p1["cut"].astype(np.int32)], axis=1).astype(np.int32)
        raw = np.concatenate(distributed.all_gather_padded(local_c, most))
        scalar, centers = api.shard_phase2(ctx, raw[:, 0], raw[:, 1], a, b)
        allv = np.concatenate(distributed.all_gather_padded(scalar[:, None], most))
        return allv[:, 0]

    def fence():
        ctx.sync()
        torch.cuda.synchronize()
        dd.barrier()

    steps = args.steps
    for _ in range(max(1, min(args.warmup, 2))):
        ref = step(src_ptr=d_frames.data_ptr())
    fence()
    sampler = ClockSampler(local)
    sampler.start()
    l0 = ctx.launch_count
    t0 = time.perf_counter()
    for _ in range(steps):
        got = step(src_ptr=d_frames.data_ptr())
    fence()
    wall_res = dd.max(time.perf_counter() - t0)
    launches = ctx.launch_count - l0
    step(host=pinned.array)
    fence()
    t0 = time.perf_counter()
    for _ in range(steps):
        got_e = step(host=pinned.array)
    fence()
    wall_e2e = dd.max(time.perf_counter() - t0)
    clocks = sampler.stop()
    assert len(got) == NP and np.array_equal(got, ref) and np.array_equal(got, got_e)
    line = None
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {"scalar": got})
    if rank == 0:
        peak, peak_kind = measured_peak()
        value = NP * steps / wall_res
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": args.warmup,
                "ms_per_step": 1000 * wall_res / steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": bench_config(args, world),
                "run": {"batch_frames": batch, "numa_node": numa_node, "pairs_per_rank": most, "kernels_sha": kernels_sha(),
                        "timing": "wall clock between device synchronisations + barriers, max over ranks (the step contains two host-side all-gathers)"},
                "e2e": {"value": NP * steps / wall_e2e, "unit": UNIT, "h2d_bytes_per_step": int((NP + world) * W * H),
                        "d2h_bytes_per_step": int(NP * 41), "ms_per_step": 1000 * wall_e2e / steps, "source": "pinned host frames"},
                "gpu_launches": int(launches), "clocks": clocks,
                "roofline": {"bound": "hbm", "kernel": "whole path", "achieved": WHOLE_PATH_B_PER_PX * W * H * value / world / 1e9,
                             "peak": peak, "unit": "GB/s", "frac": WHOLE_PATH_B_PER_PX * W * H * value / world / 1e9 / peak,
                             "traffic": None, "peak_source": f"MEASURED_PEAKS.json ({peak_kind})",
                             "note": "per-GPU whole-path algorithmic bytes (269.7 B/px/pair) over the wall time of the sharded step"},
                "scalar_checksum": float(np.sum(got))}
    ctx.close()
    return line


def run_c5(args, rank, world, local, dd, numa_node):
    """Whole-library throughput: videos dealt longest-first to the ranks, each through the runner's bracket loop and
    post-processing; scalars gathered as Python objects (the only exchange)."""
    import torch
    from funscript_flow_b200 import _native, api, distributed, runner
    from funscript_flow_b200.synth import ClipGenerator, ClipSpec
    W, H, NV = args.width, args.height, args.c5_videos
    lengths = [65 + 16 * ((7 * v) % 9) for v in range(NV)]                 # 65 .. 193 frames, deterministic, unequal
    plan = runner.schedule_longest_first(list(range(NV)), lengths, world)
    mine = plan[rank]
    # four base clips (seeds 0..3); video v is a window of base v % 4 (distinct start per video): generating 64 full
    # clips would take minutes of host time that is not part of the path
    need = {}
    for v in mine:
        need.setdefault(v % 4, 0)
        need[v % 4] = max(need[v % 4], (v // 4) * 3 + lengths[v])
    # the clips live in page-locked host memory, as a decoder that writes into buffers from ffb_host_alloc would leave
    # them (frames DMA straight out of them; --c5-pageable keeps them in ordinary NumPy memory instead, which adds the
    # library's staging memcpy -- the host-side limiter when 8 processes do it at once, profiles/r2_scaling.txt)
    bases, pins = {}, []
    for sd, n in need.items():
        arr = ClipGenerator(ClipSpec(W, H, 18000, seed=sd, amplitude=0.15, period=30.0)).stack(0, n)
        if not args.c5_pageable:
            pb = _native.PinnedBuffer(arr.shape)
            pb.array[...] = arr
            pins.append(pb)
            arr = pb.array
        bases[sd] = arr
    vids = {v: bases[v % 4][(v // 4) * 3:(v // 4) * 3 + lengths[v]] for v in mine}
    ctx = _native.FlowContext(local)
    api.set_context(ctx, api.default_device())
    prm = {"batch_size": 3000, "detrend_window": 2.0, "norm_window": 3.0, "keyframe_reduction": True,
           "gpu_batch_frames": args.batch_frames or runner.default_batch_frames(W, H)}

    last = {}

    def step():
        out = {}
        res = runner.process_many([vids[v] for v in mine], 30.0, prm, ctx=ctx, return_series=True)     # clips pipelined
        last["res"] = res
        for v, (actions, series) in zip(mine, res):
            out[v] = (len(actions), float(np.sum(series["values"])))
        merged = {}
        for part in distributed.gather_objects(out):
            merged.update(part)
        return merged

    def fence():
        ctx.sync()
        torch.cuda.synchronize()
        dd.barrier()

    steps = args.steps
    ref = step()
    fence()
    sampler = ClockSampler(local)
    sampler.start()
    l0 = ctx.launch_count
    t0 = time.perf_counter()
    for _ in range(steps):
        got = step()
    fence()
    wall = dd.max(time.perf_counter() - t0)
    clocks = sampler.stop()
    assert got == ref and len(got) == NV
    line = None
    if rank == 0 and args.dump_outputs:          # this rank's videos, in the order of plan[0], concatenated
        res = last["res"]
        dump_outputs(args.dump_outputs, {
            "videos": mine, "pairs_per_video": [len(series["values"]) for _, series in res],
            "actions_per_video": [len(actions) for actions, _ in res],
            "values": np.concatenate([series["values"] for _, series in res]),
            "cuts": np.concatenate([series["cuts"] for _, series in res]),
            "frame_indices": np.concatenate([series["frame_indices"] for _, series in res]),
            "actions_at": [a["at"] for actions, _ in res for a in actions],
            "actions_pos": [a["pos"] for actions, _ in res for a in actions]})
    if rank == 0:
        pairs = sum(n - 1 for n in lengths)
        peak, peak_kind = measured_peak()
        value = pairs * steps / wall
        loads = [sum(lengths[v] for v in p) for p in plan]
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": 1,
                "ms_per_step": 1000 * wall / steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": bench_config(args, world),
                "run": {"numa_node": numa_node, "videos": NV, "pairs_per_step": pairs, "frames_per_rank": loads,
                        "schedule": "longest-first", "kernels_sha": kernels_sha(),
                        "host_memory": "pageable" if args.c5_pageable else "pinned",
                        "timing": "wall clock, host frames through runner.process_frames (H2D, post-processing and the object gather inside)"},
                "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": int(sum(lengths) * W * H), "d2h_bytes_per_step": int(pairs * 41),
                        "ms_per_step": 1000 * wall / steps, "source": ("pageable" if args.c5_pageable else "pinned") + " host frames"},
                "gpu_launches": int(ctx.launch_count - l0), "clocks": clocks,
                "roofline": {"bound": "hbm", "kernel": "whole path", "achieved": WHOLE_PATH_B_PER_PX * W * H * value / world / 1e9,
                             "peak": peak, "unit": "GB/s", "frac": WHOLE_PATH_B_PER_PX * W * H * value / world / 1e9 / peak,
                             "traffic": None, "peak_source": f"MEASURED_PEAKS.json ({peak_kind})"},
                "actions_total": int(sum(v[0] for v in got.values()))}
    ctx.close()
    return line


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    from funscript_flow_b200 import _native, build
    if build.needs_build(build.LIB, build.DEPS):
        tmp = tempfile.mkdtemp(prefix="ffb_bench_")
        _native.DEFAULT_LIB = build.build(force=True, lib=os.path.join(tmp, "libffb.so"))
        atexit.register(shutil.rmtree, tmp, True)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local)
    # host side of the e2e path: staging buffers and upload calls on the NUMA node of the GPU's PCIe root
    all_cpus = os.sched_getaffinity(0)
    numa_node = None
    if not args.no_numa_bind:
        from funscript_flow_b200 import distributed as ffdist
        numa_node = ffdist.bind_to_gpu_numa_node(local)
    dd = Dist(rank, world, local)
    if args.workload == "c2":
        line = run_c2(args, rank, world, local, dd, numa_node, all_cpus)
    elif args.workload == "c2-strong":
        line = run_c2_strong(args, rank, world, local, dd, numa_node)
    else:
        line = run_c5(args, rank, world, local, dd, numa_node)
    if rank == 0:
        print(json.dumps(line), flush=True)
    dd.close()


if __name__ == "__main__":
    main()
