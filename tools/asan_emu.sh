#!/bin/bash
# Memory-safety pass over the kernel SOURCES on the CPU: the g++ emulation build (tests/emu) with AddressSanitizer,
# driven through the C ABI on awkward frame sizes (odd, non-multiple-of-4 widths, frames smaller than a tile), the
# randomized reductions, the pre-processing windows, the stage hooks and warping by flows.  Run here (no GPU): tools/asan_emu.sh [FFB_ITER_CFG]
# compute-sanitizer is not available on the GPU pool, so this is the out-of-bounds check of the tiling / halo / padding logic.
set -e
ROOT=$(cd "$(dirname "$0")/.." && pwd)
OUT=$(mktemp -d)
g++ -x c++ -std=c++17 -O1 -g -fPIC -shared -DFFB_EMU -mfma -ffp-contract=fast -fsanitize=address -fno-omit-frame-pointer \
    -Wno-unknown-pragmas -I "$ROOT/tests/emu" -I "$ROOT/funscript_flow_b200/csrc" -I "$ROOT/include" \
    -o "$OUT/libffb_emu_asan.so" "$ROOT/funscript_flow_b200/csrc/ffb_api.cu"
cat > "$OUT/run.py" <<PY
import sys
sys.path.insert(0, "$ROOT"); sys.path.insert(0, "$ROOT/tests")
import numpy as np
from funscript_flow_b200 import _native, api
from funscript_flow_b200.synth import make_clip
import parity_checks as pc
ctx = _native.FlowContext(0, lib_path="$OUT/libffb_emu_asan.so")
for (w, h) in [(256, 256), (150, 101), (33, 20), (264, 72), (97, 131)]:
    r = api.process_bracket(make_clip(w, h, 4, seed=w), {}, ctx=ctx, batch_frames=2)
    print(w, h, "ok", float(np.sum(r["scalar"])))
for (w, h, b) in [(97, 70, 3), (33, 20, 16)]:   # sequences that wrap the final-flow ring; b = 16: host-input ramp
    seq = make_clip(w, h, 41, seed=b)
    ctx.configure(w, h, b, 8)
    r = ctx.farneback_sequence(seq, stats=True)
    flow = np.zeros((40, h + 1, w + 3, 2), np.float32)
    ctx.farneback_sequence_ptr(seq.ctypes.data, 41, w, h, w, w * h, flow.ctypes.data, (w + 3) * 8, (h + 1) * (w + 3) * 8)
    assert np.array_equal(flow[:, :h, :w], r["flow"])
    print(w, h, "sequence ok", float(np.sum(r["scalar"])))
    # backward flows, masks and counts through the same wrapping rings, into pitched buffers
    b = ctx.farneback_sequence_bidir(seq)
    assert np.array_equal(b["flow"], r["flow"])
    bw = np.zeros((40, h + 1, w + 3, 2), np.float32)
    mask = np.zeros((40, h + 2, w + 5), np.uint8)
    cnt = ctx.farneback_sequence_bidir_ptr(seq.ctypes.data, 41, w, h, w, w * h, 0, bw.ctypes.data, (w + 3) * 8,
                                           (h + 1) * (w + 3) * 8, mask.ctypes.data, w + 5, (h + 2) * (w + 5), counts=True)
    assert np.array_equal(bw[:, :h, :w], b["flow_bw"]) and np.array_equal(mask[:, :h, :w], b["mask"].view(np.uint8))
    assert np.array_equal(cnt, b["n_consistent"]) and np.array_equal(cnt, b["mask"].sum(axis=(1, 2)))
    m, k = ctx.stage_fb_check(b["flow"][3], b["flow_bw"][3])
    assert np.array_equal(m, b["mask"][3]) and k == cnt[3]
    print(w, h, "bidirectional ok", int(cnt.sum()))
    # independent pairs with backward flows, masks and counts: chunks alternate ring halves, into pitched buffers
    prev, nxt = np.ascontiguousarray(seq[0:40:2]), np.ascontiguousarray(seq[40:0:-2])
    p = ctx.farneback_pairs_bidir(prev, nxt)
    assert np.array_equal(p["flow"], ctx.farneback_pairs(prev, nxt)["flow"])
    assert np.array_equal(p["flow_bw"][5], ctx.farneback(nxt[5], prev[5]))
    fw = np.zeros((20, h + 1, w + 3, 2), np.float32)
    bw = np.zeros((20, h + 1, w + 3, 2), np.float32)
    mask = np.zeros((20, h + 2, w + 5), np.uint8)
    cnt = ctx.farneback_pairs_bidir_ptr(prev.ctypes.data, nxt.ctypes.data, 20, w, h, w, w * h, fw.ctypes.data, bw.ctypes.data,
                                        (w + 3) * 8, (h + 1) * (w + 3) * 8, mask.ctypes.data, w + 5, (h + 2) * (w + 5),
                                        counts=True)
    assert np.array_equal(fw[:, :h, :w], p["flow"]) and np.array_equal(bw[:, :h, :w], p["flow_bw"])
    assert np.array_equal(mask[:, :h, :w], p["mask"].view(np.uint8)) and np.array_equal(cnt, p["n_consistent"])
    assert np.array_equal(cnt, p["mask"].sum(axis=(1, 2)))
    print(w, h, "pairs bidirectional ok", int(cnt.sum()))
# warping by flows at awkward sizes, gray and BGR, both borders, flows far outside the image, pitched buffers; the
# 300 x 300 gray batch takes two staging chunks
for (w, h, c, n) in [(1, 1, 1, 3), (37, 1, 3, 3), (1, 29, 1, 3), (97, 70, 3, 3), (131, 5, 1, 4), (300, 300, 1, 12)]:
    rng = np.random.default_rng(w * h)
    src = rng.integers(0, 256, (n, h, w) if c == 1 else (n, h, w, 3), dtype=np.uint8)
    fl = rng.uniform(-2 * max(w, h), 2 * max(w, h), (n, h, w, 2)).astype(np.float32)
    fl[:, ::3, ::2, 0] = np.nan
    out = [ctx.remap_flow(src, fl, b, 7) for b in (0, 1)]
    s_wide = np.zeros((n, h + 1, (w + 3) * c), np.uint8)
    s_wide[:, :h, :w * c] = src.reshape(n, h, w * c)
    f_wide = np.zeros((n, h + 1, w + 1, 2), np.float32)
    f_wide[:, :h, :w] = fl
    d_wide = np.zeros((n, h + 2, (w + 5) * c), np.uint8)
    ctx.remap_flow_ptr(s_wide.ctypes.data, n, w, h, c, (w + 3) * c, (h + 1) * (w + 3) * c, f_wide.ctypes.data, (w + 1) * 8,
                       (h + 1) * (w + 1) * 8, d_wide.ctypes.data, (w + 5) * c, (h + 2) * (w + 5) * c, 1, 7)
    assert np.array_equal(d_wide[:, :h, :w * c], out[1].reshape(n, h, w * c))
    print(w, h, c, "remap ok", int(out[0].sum()), int(out[1].sum()))
pc.check_reductions_random(ctx, n_cases=8, max_side=70)
pc.check_preprocess(ctx, sizes=((97, 131), (64, 48)))
pc.check_preprocess_window(ctx)
pc.check_native_resolution_bracket(ctx, 96, 64, 4)
pc.check_stages(ctx, 150, 101)
print("asan run complete")
PY
[ -n "$1" ] && export FFB_ITER_CFG=$1
ASAN_OPTIONS=detect_leaks=0:halt_on_error=1 LD_PRELOAD=$(gcc -print-file-name=libasan.so) python "$OUT/run.py"
rm -rf "$OUT"
