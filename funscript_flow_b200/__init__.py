"""funscript_flow_b200 -- B200-native (sm_100a) implementation of Funscript-Flow's per-frame-pair
motion hot path: dense Farneback flow -> max-|"divergence"| centre -> balanced radial projection
mean + scene-cut test, behind the reference's processing-function API.

The arithmetic runs only in hand-written CUDA kernels (csrc/) reached through the C ABI in
include/ffb.h; importing this package does not need a GPU, calling any processing function does.
"""
from .api import (BracketPipeline, calc_optical_flow_farneback_batch, calc_optical_flow_farneback_sequence,  # noqa: F401
                  calc_optical_flow_farneback_batch_bidirectional, calc_optical_flow_farneback_sequence_bidirectional,
                  get_available_backends, get_context, get_gpu_info, max_divergence, precompute_flow_info,
                  precompute_flow_info_batch, precompute_flow_info_gpu, precompute_wrapper, process_bracket,
                  process_bracket_on_contexts, process_sequence, radial_motion_weighted, remap_by_flow, set_context,
                  smooth_centers)
from .runner import process_frames, process_many, process_video, run_headless  # noqa: F401

__version__ = "0.2.0"
