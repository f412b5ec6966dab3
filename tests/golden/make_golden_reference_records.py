"""Regenerates tests/golden/reference_records.json: what the reference comparisons of tests/test_oracle.py and
tests/test_emu_kernels.py compare, recorded so that they run without the reference (FunscriptFlow.pyw), which is
not part of the repository.  Run:  python tests/golden/make_golden_reference_records.py

The records are computed with the oracle restatement (oracle/motion_np.py) and, for the log lines, with the
product's process_video on the g++ emulation of the kernels (tests/emu/).  Those tests had asserted both equal,
value for value, to the reference's own functions; when oracle/ref_loader.py finds the reference, this script runs
it on the same inputs and refuses to write unless every record is identical.
"""
from __future__ import annotations

import json
import os
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import cv2  # noqa: E402
import numpy as np  # noqa: E402

import parity_checks as pc  # noqa: E402
from oracle import motion_np as mo  # noqa: E402
from oracle import ref_loader  # noqa: E402


def product_logs():
    from emu import build_emu
    from funscript_flow_b200 import _native, api, runner
    ctx = _native.FlowContext(0, build_emu.build())
    api.set_context(ctx)
    with tempfile.TemporaryDirectory() as td:
        rec = pc.record_process_video_logs(runner.process_video, td)
    ctx.close()
    return rec


def main():
    out = {"pairs_and_postprocess": pc.record_pairs_and_postprocess(mo, pc.oracle_postprocess),
           "random_fields": pc.record_random_fields(mo),
           "random_postprocess": pc.record_random_postprocess(pc.oracle_postprocess),
           "process_video_logs": product_logs()}
    assert out["process_video_logs"] is not None, "cv2 has no FFV1 writer"
    checked = ref_loader.available()
    if checked:
        ref = ref_loader.load("ffref_records", serial_pools=True)
        with tempfile.TemporaryDirectory() as td:
            theirs = {"pairs_and_postprocess": pc.record_pairs_and_postprocess(ref, pc.reference_postprocess(ref)),
                      "random_fields": pc.record_random_fields(ref),
                      "random_postprocess": pc.record_random_postprocess(pc.reference_postprocess(ref)),
                      "process_video_logs": pc.record_process_video_logs(ref.process_video, td)}
        for key in out:
            assert theirs[key] == out[key], f"the reference and the restatement differ on {key}"
    out["meta"] = {"cv2": cv2.__version__, "numpy": np.__version__,
                   "source": "oracle restatement and product on the emulated kernels" +
                             ("; identical to the reference's own functions on every record" if checked else "")}
    json.dump(out, open(os.path.join(HERE, "reference_records.json"), "w"), separators=(",", ":"))
    print("written", os.path.join(HERE, "reference_records.json"), "checked against the reference:", checked)


if __name__ == "__main__":
    main()
