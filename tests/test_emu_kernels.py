"""CPU suite, part 3: the kernel SOURCES (csrc/*.cu), compiled with g++ against the test-only CUDA
emulation in tests/emu/, checked against the oracle on small inputs -- tiling, halos, ring buffers,
batching and reductions are exercised before any GPU time is spent.  The real parity tests are the
`-m gpu` ones; this file only proves the logic, not the sm_100a build."""
import os

import numpy as np
import pytest

import parity_checks as pc
from funscript_flow_b200 import api, runner
from funscript_flow_b200.synth import make_clip


@pytest.mark.parametrize("size", [(150, 101), (64, 48)])
def test_stages(emu_ctx, size):
    pc.check_stages(emu_ctx, *size)


@pytest.mark.parametrize("size", [(256, 256), (333, 217)])
def test_farneback_vs_cv2(emu_ctx, size):
    pc.check_farneback_vs_cv2(emu_ctx, *size)


def test_reduction_known_answers(emu_ctx, golden_dir):
    pc.check_reductions_kat(emu_ctx, golden_dir)


def test_reductions_random_fields(emu_ctx):
    pc.check_reductions_random(emu_ctx, n_cases=12, max_side=64)


def test_golden_pairs(emu_ctx, golden_dir):
    pc.check_golden_pairs(emu_ctx, golden_dir, names=("b", "c"))


def test_golden_bracket(emu_ctx, golden_dir):
    pc.check_golden_bracket(emu_ctx, golden_dir)


def test_batch_independence(emu_ctx):
    pc.check_batch_independence(emu_ctx, 120, 72, n_frames=12)


def test_edge_brackets(emu_ctx):
    pc.check_edge_brackets(emu_ctx)


def test_process_frames_brackets(emu_ctx):
    """Bracket semantics of F:1145-1153: no pair across brackets, trailing 1-frame bracket dropped."""
    api.set_context(emu_ctx)
    clip = make_clip(96, 64, 11, seed=6, period=7.0, amplitude=0.3)
    prm = {"batch_size": 5, "detrend_window": 2.0, "norm_window": 3.0, "keyframe_reduction": False}
    acts, series = runner.process_frames(clip, 30.0, prm, ctx=emu_ctx, return_series=True)
    # brackets [0,5) [5,10) [10,11) -> 4 + 4 + 0 pairs, stamped with the first frame of each pair
    assert series["frame_indices"].tolist() == [0, 1, 2, 3, 5, 6, 7, 8]
    assert len(acts) == 8
    one = api.process_bracket(clip[5:10], {}, ctx=emu_ctx)
    assert np.array_equal(series["values"][4:], one["scalar"])


def test_preprocess(emu_ctx):
    pc.check_preprocess(emu_ctx)
    pc.check_bgr_push_equals_gray_push(emu_ctx)


def test_preprocess_window_and_native_resolution(emu_ctx):
    """Row N4: windowed pre-processing and brackets at the decoded resolution (plain and VR eyes)."""
    pc.check_preprocess_window(emu_ctx)
    pc.check_native_resolution_bracket(emu_ctx, 96, 64, 4)
    pc.check_native_resolution_bracket(emu_ctx, 160, 128, 4, vr=True, eye="right")
    # configuring the flow for another size than the window is refused, with the expected size in the text
    emu_ctx.preprocess_configure_window(96, 64, (96, 64), (0, 0, 96, 64))
    emu_ctx.configure(256, 256, 2, 4)
    emu_ctx.bracket_begin(False, 7.0)
    with pytest.raises(Exception, match="96x64"):
        emu_ctx.bracket_push_bgr(np.zeros((2, 64, 96, 3), np.uint8))
    emu_ctx.bracket_finish()
    with pytest.raises(Exception):
        emu_ctx.preprocess_configure_window(96, 64, (96, 64), (50, 0, 96, 64))    # window leaves the target
    with pytest.raises(ValueError):
        runner.preprocess_plan(96, 64, {"vr_mode": True, "vr_eye": "up"})
    assert runner.preprocess_plan(96, 64, {"vr_mode": True, "vr_eye": "both"}) == runner.preprocess_plan(96, 64, {"vr_mode": True})
    assert runner.preprocess_plan(1920, 1080, {}) == ((256, 256), (0, 0, 256, 256), 1.0)
    assert runner.preprocess_plan(1920, 1080, {"vr_mode": True}) == ((512, 512), (0, 256, 256, 256), 1.0)
    assert runner.preprocess_plan(1920, 1080, {"vr_mode": True, "vr_eye": "right"})[1] == (256, 256, 256, 256)
    assert runner.preprocess_plan(3840, 1920, {"vr_mode": True, "native_resolution": True})[:2] == ((3840, 1920), (0, 960, 1920, 960))


def test_process_video_file(emu_ctx, tmp_path):
    """process_video() on a small lossless clip: decode on the host, resize / gray / flow / reductions in
    the kernels; equals the host pre-processing path and honours the skip-if-exists rule (F:1105-1109)."""
    import json
    import cv2
    api.set_context(emu_ctx)
    clip = make_clip(160, 120, 9, seed=6, period=7.0, amplitude=0.3)
    path = str(tmp_path / "tiny.avi")
    vw = cv2.VideoWriter(path, cv2.VideoWriter_fourcc(*"FFV1"), 30.0, (160, 120), True)
    if not vw.isOpened():
        pytest.skip("FFV1 writer unavailable")
    for f in clip:
        vw.write(cv2.cvtColor(f, cv2.COLOR_GRAY2BGR))
    vw.release()
    prm = {"batch_size": 3000, "detrend_window": 2.0, "norm_window": 3.0, "keyframe_reduction": False, "overwrite": True,
           "vr_mode": False, "pov_mode": False, "gpu_batch_frames": 4}
    logs = []
    assert runner.process_video(path, prm, logs.append) is False, logs
    acts = json.load(open(str(tmp_path / "tiny.funscript")))["actions"]
    gray = runner.read_sampled_gray(path, list(range(9)), prm)
    ref = runner.process_frames(gray, 30.0, prm, ctx=emu_ctx)
    assert acts == ref and len(acts) == 8
    logs.clear()
    assert runner.process_video(path, dict(prm, overwrite=False), logs.append) is False and any("Skipping" in l for l in logs)
    # row N4: the same file at its native 160x120 (FFV1 is lossless, so the decoded frames are the clip)
    res = runner.process_video_series(path, dict(prm, native_resolution=True), ctx=emu_ctx)
    direct = api.process_bracket(clip, {"cut_threshold": 7.0 * np.sqrt(160 * 120) / 256.0}, ctx=emu_ctx, batch_frames=4)
    assert res[0] == direct["scalar"].tolist() and res[1] == direct["cut"].tolist()
    # both eyes of a side-by-side frame = mean of the two single-eye series (two contexts, one decode)
    vr = dict(prm, vr_mode=True, native_resolution=True)
    left = runner.process_video_series(path, dict(vr, vr_eye="left"), ctx=emu_ctx)
    right = runner.process_video_series(path, dict(vr, vr_eye="right"), ctx=emu_ctx)
    both = runner.process_video_series(path, dict(vr, vr_eye="both"), ctx=emu_ctx)
    assert left[0] != right[0]
    assert both[0] == (0.5 * (np.asarray(left[0]) + np.asarray(right[0]))).tolist()
    assert both[1] == [a or b for a, b in zip(left[1], right[1])] and both[2] == left[2]


def test_headless_folder_sharded_over_ranks(emu_ctx, tmp_path, monkeypatch):
    """Config C5 in miniature (whole videos sharded over ranks): the union of what ranks 0 and 1 of a
    2-process job write equals what a single process writes (no collective: videos are independent)."""
    import json
    import cv2
    api.set_context(emu_ctx)
    monkeypatch.chdir(tmp_path)
    prm = {"batch_size": 3000, "detrend_window": 2.0, "norm_window": 3.0, "keyframe_reduction": True, "overwrite": True,
           "vr_mode": False, "pov_mode": False, "gpu_batch_frames": 4}
    for k in range(3):
        clip = make_clip(96, 64, 6, seed=20 + k, period=5.0, amplitude=0.3)
        vw = cv2.VideoWriter(str(tmp_path / f"v{k}.avi"), cv2.VideoWriter_fourcc(*"FFV1"), 30.0, (96, 64), True)
        if not vw.isOpened():
            pytest.skip("FFV1 writer unavailable")
        for f in clip:
            vw.write(cv2.cvtColor(f, cv2.COLOR_GRAY2BGR))
        vw.release()
    monkeypatch.delenv("RANK", raising=False)
    monkeypatch.delenv("WORLD_SIZE", raising=False)
    assert runner.run_headless(str(tmp_path), prm, log_func=lambda m: None) == 0
    single = {k: json.load(open(str(tmp_path / f"v{k}.funscript"))) for k in range(3)}
    for k in range(3):
        (tmp_path / f"v{k}.funscript").unlink()
    monkeypatch.setenv("WORLD_SIZE", "2")
    for rank in (0, 1):
        monkeypatch.setenv("RANK", str(rank))
        assert runner.run_headless(str(tmp_path), prm, log_func=lambda m: None) == 0
        present = [k for k in range(3) if (tmp_path / f"v{k}.funscript").exists()]
        assert present == ([0, 2] if rank == 0 else [0, 1, 2])
    assert {k: json.load(open(str(tmp_path / f"v{k}.funscript"))) for k in range(3)} == single


def test_large_frame_variant_in_subprocess(emu_lib, golden_dir):
    """Frames under 1280x720 run the 160-thread strips, so the small frames of this CPU suite would never reach the
    128-thread kernel that 1080p and 4K use: FFB_ITER_CFG=128x2x4 forces it (the GPU suite covers it at full size)."""
    import os
    import subprocess
    import sys
    code = (
        "import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
        "from funscript_flow_b200 import _native\n"
        "import parity_checks as pc\n"
        "ctx = _native.FlowContext(0, %r)\n"
        "print(pc.check_farneback_vs_cv2(ctx, 333, 217))\n"
        "pc.check_batch_independence(ctx, 300, 72, n_frames=6)\n"
        "pc.check_golden_bracket(ctx, %r)\n"
    ) % (os.path.dirname(os.path.dirname(os.path.abspath(__file__))), os.path.dirname(os.path.abspath(__file__)), emu_lib, golden_dir)
    env = dict(os.environ, FFB_ITER_CFG="128x2x4")
    res = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout + res.stderr


@pytest.mark.parametrize("cfg", ["160x2x4", "256x4x8"])
def test_strip_variants_in_subprocess(emu_lib, cfg):
    """k_flow_iter variants forced on any frame size with FFB_ITER_CFG=NTxUxHO (threads per strip x rows per step x
    outputs per horizontal task): 160x2x4 is the default for frames up to 320 columns; 256x4x8, the default for frames
    of 1280x720 and more, exercises the single row buffer with two barriers per step and the de-interleaved row layout
    of the 8-output tasks.  Frames narrower than a strip also exercise the idle-warp path."""
    import os
    import subprocess
    import sys
    code = (
        "import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
        "from funscript_flow_b200 import _native\n"
        "import parity_checks as pc\n"
        "ctx = _native.FlowContext(0, %r)\n"
        "print(pc.check_farneback_vs_cv2(ctx, 256, 256))\n"
        "pc.check_batch_independence(ctx, 300, 72, n_frames=6)\n"
    ) % (os.path.dirname(os.path.dirname(os.path.abspath(__file__))), os.path.dirname(os.path.abspath(__file__)), emu_lib)
    env = dict(os.environ, FFB_ITER_CFG=cfg)
    res = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout + res.stderr


def test_error_paths_and_strided_input(emu_ctx):
    """Host logic of the C ABI: calls out of sequence and out-of-range requests fail with the documented
    codes (no exceptions swallowed, no fallback); frames given as a strided view (pitch > width) are
    handled like contiguous ones."""
    from funscript_flow_b200 import _native
    clip = make_clip(96, 64, 6, seed=3)
    emu_ctx.configure(96, 64, 2, 3)
    with pytest.raises(_native.FFBError) as ei:
        emu_ctx.bracket_push(clip[:2])                       # no bracket open
    assert ei.value.code == -1
    emu_ctx.bracket_begin(False, 7.0)
    with pytest.raises(_native.FFBError) as ei:
        emu_ctx.bracket_push(clip)                           # 5 pairs > max_bracket_pairs = 3
    assert ei.value.code == -1 and "max_bracket_pairs" in str(ei.value)
    emu_ctx.bracket_finish()
    ref = api.process_bracket(clip, {}, ctx=emu_ctx, batch_frames=3, return_flows=True)
    with pytest.raises(_native.FFBError) as ei:
        emu_ctx.get_flow(99)
    assert ei.value.code == -5
    big = np.zeros((6, 80, 128), np.uint8)
    big[:, 8:72, 16:112] = clip
    view = big[:, 8:72, 16:112]                              # pitch 128, frame stride 80 * 128
    assert not view.flags["C_CONTIGUOUS"]
    emu_ctx.configure(96, 64, 3, 5)
    emu_ctx.bracket_begin(False, 7.0)
    emu_ctx.bracket_push(view)
    got = emu_ctx.bracket_finish()
    for k in ("scalar", "cx", "cy", "val", "mean_mag"):
        assert np.array_equal(ref[k], got[k]), k


def test_bracket_abort_and_cancel(emu_ctx, tmp_path):
    """ffb_bracket_abort drops an open bracket and leaves the context configurable; the runner uses it when the
    user cancels (F:1147-1149) or a chunk fails, so the next video is not refused with 'inside a bracket'."""
    import cv2
    clip = make_clip(96, 64, 7, seed=31)
    full = api.process_bracket(clip, {}, ctx=emu_ctx, batch_frames=3)
    emu_ctx.configure(96, 64, 3, 6)
    emu_ctx.bracket_begin(False, 7.0)
    emu_ctx.bracket_push(clip[:4])
    with pytest.raises(Exception, match="inside a bracket|in a bracket|bracket"):
        emu_ctx.preprocess_configure(96, 64, False)
    emu_ctx.bracket_abort()
    emu_ctx.bracket_abort()                                   # no-op outside a bracket
    emu_ctx.preprocess_configure(96, 64, False)               # accepted again
    again = api.process_bracket(clip, {}, ctx=emu_ctx, batch_frames=3)
    assert np.array_equal(full["scalar"], again["scalar"])    # nothing of the dropped bracket leaks into the next
    # runner: cancel in the middle of a bracket, then process the same file normally
    api.set_context(emu_ctx)
    path = str(tmp_path / "c.avi")
    vw = cv2.VideoWriter(path, cv2.VideoWriter_fourcc(*"FFV1"), 30.0, (96, 64), True)
    if not vw.isOpened():
        pytest.skip("FFV1 writer unavailable")
    for f in clip:
        vw.write(cv2.cvtColor(f, cv2.COLOR_GRAY2BGR))
    vw.release()
    prm = {"batch_size": 3000, "detrend_window": 2.0, "norm_window": 3.0, "keyframe_reduction": False, "overwrite": True,
           "vr_mode": False, "pov_mode": False, "gpu_batch_frames": 3}
    calls = {"n": 0}

    def cancel_after_first_chunk():
        calls["n"] += 1
        return calls["n"] > 2
    assert runner.process_video_series(path, prm, ctx=emu_ctx, cancel_flag=cancel_after_first_chunk, chunk_frames=3) is None
    logs = []
    assert runner.process_video(path, prm, logs.append) is False, logs


def test_integration_stub_from_the_docs_runs(emu_lib, emu_ctx):
    """The ctypes stub INTEGRATION.md tells a reference maintainer to paste (replacement body of
    precompute_flow_info_gpu, F:982-1017) is executed as written, against the emulated library, and returns
    the same 8-key dict as the shipped Python mirror."""
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    text = open(os.path.join(root, "INTEGRATION.md")).read()
    code = re.search(r"```python\n(# --- in FunscriptFlow\.pyw.*?)```", text, re.S).group(1)
    code = code.replace("/path/to/funscript_flow_b200/libffb.so", emu_lib)
    ns = {}
    exec(compile(code, "INTEGRATION.md", "exec"), ns)
    clip = make_clip(96, 64, 2, seed=77)
    got = ns["precompute_flow_info_gpu"](clip[0], clip[1], 7)
    api.set_context(emu_ctx)
    want = api.precompute_flow_info_gpu(clip[0], clip[1], 7)
    assert set(got) == set(want) == {"flow", "pos_center", "neg_center", "val_pos", "val_neg", "cut", "cut_center", "mean_mag"}
    assert np.array_equal(got["flow"], want["flow"]) and got["pos_center"] == want["pos_center"]
    assert got["val_pos"] == want["val_pos"] and got["cut"] == want["cut"] and got["mean_mag"] == want["mean_mag"]


def test_process_video_log_lines_follow_the_reference(emu_ctx, golden_dir, tmp_path):
    """Same log lines, in the same order, as the reference's process_video on the same file (backend name and the
    elapsed time excepted): the lines recorded in tests/golden/reference_records.json, and the
    AST-loaded reference is run as well when oracle/ref_loader.py finds FunscriptFlow.pyw."""
    import json
    from oracle import ref_loader
    api.set_context(emu_ctx)
    want = json.load(open(os.path.join(golden_dir, "reference_records.json")))["process_video_logs"]
    ours = pc.record_process_video_logs(runner.process_video, str(tmp_path))
    if ours is None:
        pytest.skip("FFV1 writer unavailable")
    assert ours == want
    if ref_loader.available():
        (tmp_path / "ref").mkdir()
        ref = ref_loader.load("ffref_logs", serial_pools=True)
        assert pc.record_process_video_logs(ref.process_video, str(tmp_path / "ref")) == want


def test_configure_is_incremental(emu_lib):
    """ffb_configure re-allocates only what a request outgrows: same or smaller limits touch nothing (no cudaMalloc,
    no cudaHostAlloc -- counted by the library), a refused call leaves the configuration usable, and results do not
    depend on the capacities a context happens to hold."""
    from funscript_flow_b200 import _native
    ctx = _native.FlowContext(0, emu_lib)
    assert ctx.geometry is None
    clip = make_clip(96, 64, 9, seed=12)
    ref = api.process_bracket(clip, {}, ctx=ctx, batch_frames=4)
    base = ctx.alloc_counts()
    assert base[0] > 0 and base[1] > 0 and ctx.geometry == (96, 64, 4, 8)
    for _ in range(3):                                        # bracket after bracket of one video: nothing is allocated
        again = api.process_bracket(clip, {}, ctx=ctx, batch_frames=4)
    assert ctx.alloc_counts() == base and np.array_equal(again["scalar"], ref["scalar"])
    short = api.process_bracket(clip[:5], {}, ctx=ctx, batch_frames=4)        # a shorter last bracket
    assert ctx.alloc_counts() == base and ctx.geometry == (96, 64, 4, 4)
    assert np.array_equal(short["cx"], ref["cx"][:4])
    # the per-pair drop-in functions reuse the configuration of the same frame size
    api.set_context(ctx)
    info = api.precompute_flow_info(clip[0], clip[1], {})
    api.radial_motion_weighted(info["flow"], (40.0, 30.0), False)
    api.max_divergence(info["flow"])
    assert ctx.alloc_counts() == base
    # a bad request is refused before anything is freed
    with pytest.raises(_native.FFBError) as ei:
        ctx.configure(8, 8, 4, 8)
    assert ei.value.code == -1 and ctx.alloc_counts() == base and ctx.geometry[:2] == (96, 64)
    assert np.array_equal(api.process_bracket(clip, {}, ctx=ctx, batch_frames=4)["scalar"], ref["scalar"])
    # growing one limit re-allocates that group only: more pairs -> the per-pair arrays, not the per-batch buffers
    ctx.configure(96, 64, 4, 100)
    grown = ctx.alloc_counts()
    assert 0 < grown[0] - base[0] < base[0] // 2 and grown[1] - base[1] == 1
    big = api.process_bracket(clip, {}, ctx=ctx, batch_frames=8)              # larger batch: per-batch buffers grow
    assert ctx.alloc_counts()[0] > grown[0] and np.array_equal(big["scalar"], ref["scalar"])
    ctx.close()


def test_shard_api_sequence_and_errors(emu_lib):
    """Two-phase shard brackets through the C ABI: call order is enforced, the external centre frame is validated, a whole
    bracket as a single shard equals ffb_bracket_finish, and an aborted shard leaves the context usable."""
    from funscript_flow_b200 import _native
    ctx = _native.FlowContext(0, emu_lib)
    clip = make_clip(96, 64, 11, seed=4, period=6.0, amplitude=0.3)
    ref = api.process_bracket(clip, {}, ctx=ctx, batch_frames=4)
    ctx.configure(96, 64, 4, 10)
    with pytest.raises(_native.FFBError):
        ctx.bracket_phase1_finish()                                      # no bracket
    ctx.bracket_begin(False, 7.0)
    with pytest.raises(_native.FFBError):
        ctx.bracket_phase1_finish()                                      # not a shard bracket
    with pytest.raises(_native.FFBError):
        ctx.bracket_begin_shard(4)                                       # a bracket is open
    ctx.bracket_abort()
    ctx.bracket_begin_shard(10)
    ctx.bracket_push(clip)
    with pytest.raises(_native.FFBError):
        ctx.bracket_finish()                                             # shard brackets end with bracket_radial
    with pytest.raises(_native.FFBError):
        ctx.bracket_radial(ref["cx"], ref["cy"], 0, 10)                  # phase 1 has not been read
    p1 = ctx.bracket_phase1_finish()
    assert p1["n_pairs"] == 10 and np.array_equal(p1["cx"], ref["cx"]) and np.array_equal(p1["cut"], ref["cut"])
    with pytest.raises(_native.FFBError):
        ctx.bracket_push(clip[:2])                                       # no frames after phase 1
    for bad in ((p1["cx"][:9], p1["cy"][:9], 0), (p1["cx"], p1["cy"], 7), (np.zeros(17, np.int32), np.zeros(17, np.int32), 0)):
        with pytest.raises(_native.FFBError):
            ctx.bracket_radial(bad[0], bad[1], bad[2], 10)
    scalar, centers = ctx.bracket_radial(p1["cx"], p1["cy"], 0, 10)
    assert np.array_equal(scalar, ref["scalar"]) and np.array_equal(centers, ref["centers"])
    # more pairs than announced are refused; abort recovers
    ctx.bracket_begin_shard(3)
    with pytest.raises(_native.FFBError):
        ctx.bracket_push(np.concatenate([clip] * 3))
    ctx.bracket_abort()
    assert np.array_equal(api.process_bracket(clip, {}, ctx=ctx, batch_frames=4)["scalar"], ref["scalar"])
    ctx.close()


def test_colour_pushes_gather_into_full_batches(emu_lib):
    """ffb_bracket_push_bgr accumulates pre-processed frames until a GPU batch is full, however the caller cuts its
    pushes (ADVICE round 1: 64-frame chunks never reached the 128 / 512-frame batches of small frames): pushing one
    frame at a time launches as many kernels as one push of the whole bracket, and gives the same numbers."""
    import cv2
    from funscript_flow_b200 import _native
    ctx = _native.FlowContext(0, emu_lib)
    gray = make_clip(96, 64, 13, seed=9)
    bgr = np.stack([cv2.cvtColor(f, cv2.COLOR_GRAY2BGR) for f in gray])
    ctx.preprocess_configure_window(96, 64, (96, 64), (0, 0, 96, 64))

    def run(step):
        ctx.configure(96, 64, 8, 12)
        ctx.bracket_begin(False, 7.0)
        l0 = ctx.launch_count
        for a in range(0, len(bgr), step):
            ctx.bracket_push_bgr(bgr[a:a + step])
        r = ctx.bracket_finish()
        return r, ctx.launch_count - l0
    whole, n_whole = run(len(bgr))
    single, n_single = run(1)
    threes, n_threes = run(3)
    assert np.array_equal(whole["scalar"], single["scalar"]) and np.array_equal(whole["scalar"], threes["scalar"])
    # only the per-chunk pre-processing launches differ (chunks of <= 8 colour frames): the flow batches are the same
    assert n_single - n_whole == len(bgr) - 3 and n_threes - n_whole <= 3
    ref = api.process_bracket(gray, {}, ctx=ctx, batch_frames=8)
    assert np.array_equal(ref["scalar"], whole["scalar"])
    ctx.close()


def test_bracket_pipeline_equals_single_brackets(emu_lib):
    """api.BracketPipeline (two contexts alternating, kernels chained with ffb_chain_after, uploads overlapping) returns
    for every bracket what api.process_bracket returns, bit for bit, in submission order -- brackets of different
    lengths and frame sizes, POV parameters per bracket, an empty tail; runner.process_many keeps the clips apart."""
    from funscript_flow_b200 import _native
    ctx = _native.FlowContext(0, emu_lib)
    single = _native.FlowContext(0, emu_lib)
    clips = [make_clip(96, 64, 9, seed=1), make_clip(96, 64, 4, seed=2), make_clip(80, 48, 6, seed=3), make_clip(96, 64, 2, seed=4)]
    prms = [{}, {"pov_mode": True}, {"cut_threshold": 0.01}, {}]
    pipe = api.BracketPipeline(ctx, batch_frames=4)
    got = []
    for c, p in zip(clips, prms):
        done = pipe.submit(c, p)
        if done is not None:
            got.append(done)
    got.append(pipe.flush())
    assert pipe.flush() is None and len(got) == len(clips)
    for c, p, g in zip(clips, prms, got):
        ref = api.process_bracket(c, p, ctx=single, batch_frames=4)
        for k in ("scalar", "cut", "cx", "cy", "val", "mean_mag", "centers"):
            assert np.array_equal(ref[k], g[k]), k
    prm = {"batch_size": 4, "detrend_window": 2.0, "norm_window": 3.0, "keyframe_reduction": False, "gpu_batch_frames": 3}
    many = runner.process_many([clips[0], clips[1]], 30.0, prm, ctx=ctx, return_series=True)
    for clip, (acts, series) in zip(clips[:2], many):
        a1, s1 = runner.process_frames(clip, 30.0, prm, ctx=single, return_series=True)
        assert acts == a1 and np.array_equal(series["values"], s1["values"]) and np.array_equal(series["frame_indices"], s1["frame_indices"])
    with pytest.raises(_native.FFBError):
        ctx.chain_after(ctx)
    ctx.close(); single.close()
