/*
 * ffb.h -- C ABI of the B200-native Funscript-Flow motion hot path
 *          (grayscale frame pair -> per-pair radial expansion scalar).
 *
 * The reference (ConwayBeyond/Funscript-Flow, FunscriptFlow.pyw; "F:n" = line n of that file) has
 * no FFI of its own: its seam is Python-level (config["backend"], F:854-873) and the arithmetic
 * lives in cv2 / NumPy calls.  Each entry point below names the reference interface it replaces,
 * so a maintainer can bind it with ctypes (see INTEGRATION.md for the stub).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no C++ / torch types.
 *   - every function returns 0 on success or a negative FFB_E_* code; ffb_last_error() gives text.
 *   - a context is bound to one CUDA device and is NOT thread-safe (one per host thread / GPU).
 *   - host buffers are borrowed, never retained past the documented point, never written unless
 *     they are outputs.  All device memory, streams and pinned staging belong to the context.
 *   - there is no CPU fallback: without a usable CUDA device ffb_create() fails.
 *   - image layout: uint8 gray, row-major, `pitch` bytes per row, `frame_stride` bytes per frame.
 *   - flow layout: float32 [H][W][2] interleaved, channel 0 = x displacement, 1 = y displacement
 *     (exactly cv2.calcOpticalFlowFarneback's output, F:878-879).
 */
#ifndef FFB_H_
#define FFB_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FFB_VERSION 200

#define FFB_OK             0
#define FFB_E_INVALID     -1   /* bad argument / call out of sequence                     */
#define FFB_E_CUDA        -2   /* CUDA runtime error (text in ffb_last_error)              */
#define FFB_E_NOMEM       -3   /* host or device allocation failed                         */
#define FFB_E_NODEVICE    -4   /* no CUDA device: there is no CPU fallback                 */
#define FFB_E_RANGE       -5   /* index outside what is resident (e.g. evicted flow field) */

typedef struct ffb_ctx ffb_ctx;

/* ---- library / device ------------------------------------------------------------------ */
int  ffb_version(void);
/* replaces get_available_backends()["CUDA"] (F:32-63): number of usable CUDA devices. */
int  ffb_device_count(int* n_devices);
/* PCI bus id ("0000:1b:00.0") of a device, for placing the host process (and so its pinned staging
 * buffers) on the NUMA node the GPU hangs off; no context needed. */
int  ffb_device_pci_bus_id(int device, char* buf, int buf_len);
/* Marketing name of a device ("NVIDIA B200"), what the reference shows through cv2.cuda.getDeviceName (F:77). */
int  ffb_device_name(int device, char* buf, int buf_len);
const char* ffb_last_error(const ffb_ctx* ctx /* NULL = last error of ffb_create */);

int  ffb_create(int device, ffb_ctx** out_ctx);
void ffb_destroy(ffb_ctx* ctx);

/* Pinned host memory for frame buffers (so ffb_bracket_push can DMA straight out of them). */
int  ffb_host_alloc(void** ptr, size_t bytes);
int  ffb_host_free(void* ptr);

/* ---- geometry ---------------------------------------------------------------------------
 * (Re)allocate device buffers for width x height frames.
 *   batch_frames       frames expanded per launch group (>= 1); pairs of a batch share launches
 *   max_bracket_pairs  upper bound on pairs between bracket_begin and bracket_finish
 * The Farneback parameters are the context's (ffb_set_farneback below); a new context holds the reference's call
 * (F:878-879): pyr_scale 0.5, levels 3, winsize 15, iterations 3, poly_n 5, poly_sigma 1.2, flags 0. */
int  ffb_configure(ffb_ctx* ctx, int width, int height, int batch_frames, int max_bracket_pairs);
/* ffb_configure is incremental: a call with the frame size already configured and limits that fit the
 * allocated capacities changes nothing on the device (no cudaMalloc, no cudaHostAlloc, no synchronisation);
 * a larger batch or pair limit re-allocates only the buffers that depend on it; invalid arguments leave the
 * existing configuration untouched.  Results never depend on the capacities (DESIGN.md section 4).
 * ffb_get_geometry returns the frame size and limits of the last successful ffb_configure (0s before it);
 * ffb_alloc_counts the cudaMalloc / cudaHostAlloc calls this context has made so far (a runner that
 * configures once per video must see them stand still after the first bracket). */
int  ffb_get_geometry(const ffb_ctx* ctx, int* width, int* height, int* batch_frames, int* max_bracket_pairs);
int  ffb_alloc_counts(const ffb_ctx* ctx, int64_t* device_allocs, int64_t* host_allocs);

/* ---- Farneback parameters (cv2.calcOpticalFlowFarneback's arguments after the flow) ---------------------------
 * ffb_set_farneback sets the parameters every flow of the context uses: ffb_farneback, the bracket and shard APIs and
 * the stage hooks.  Accepted (anything else is FFB_E_INVALID with a message, and changes nothing):
 *   0 < pyr_scale < 1;  levels >= 0 (levels stop where the coarsest one would be under 32 px, as in OpenCV; a plan of
 *   more than 16 levels is refused);  3 <= winsize <= 63 (an even size sums 2 * (winsize / 2) + 1 taps with mean
 *   scale 1 / winsize^2, as OpenCV does);  1 <= iterations <= 20;  poly_n 5 or 7;  poly_sigma >= 0 (below FLT_EPSILON
 *   it becomes poly_n * 0.3);  flags 0 (OPTFLOW_USE_INITIAL_FLOW = 4 and OPTFLOW_FARNEBACK_GAUSSIAN = 256 are refused).
 * Parameters equal to the current ones change nothing (no allocation, no synchronisation); others re-plan the
 * configured geometry as a new frame size does.  Refused inside a bracket.
 * ffb_level_plan_ex: the level geometry of a frame size for (pyr_scale, levels), coarsest level first; fills at most
 * max_n entries and returns the level count in *n_levels. */
int  ffb_set_farneback(ffb_ctx* ctx, double pyr_scale, int levels, int winsize, int iterations,
                       int poly_n, double poly_sigma, int flags);
int  ffb_get_farneback(const ffb_ctx* ctx, double* pyr_scale, int* levels, int* winsize, int* iterations,
                       int* poly_n, double* poly_sigma, int* flags);
int  ffb_level_plan_ex(int width, int height, double pyr_scale, int levels, int max_n,
                       int* n_levels, int* w, int* h, int* ksize, double* sigma);

/* ---- streaming bracket API (replaces the bracket loop body F:1188-1242) ------------------
 * A bracket is a run of consecutive sampled frames; pairs never span brackets (F:1150-1153,
 * 1188) and the +-6 centre window is truncated at bracket ends (F:1203-1214).
 *
 *   ffb_bracket_begin(ctx, pov_mode, cut_threshold)
 *   ffb_bracket_push(ctx, frames, n, pitch, frame_stride)      any number of times
 *   ffb_bracket_finish(ctx, &n_pairs, outputs...)
 *
 * push: `frames` may be pageable host memory (copied through the context's pinned double
 * buffer), pinned host memory (DMA'd directly; keep it valid until ffb_bracket_finish or
 * ffb_sync) or device memory (used in place; same lifetime rule).  Uploads run with
 * cudaMemcpyAsync on a side stream, double-buffered against compute.
 *
 * finish outputs (each may be NULL), one entry per pair j = (frame j, frame j+1):
 *   scalar[j]    radial_motion_weighted(flow_j, smoothed_centre_j, cut_j, pov_mode)  F:761-785
 *   cut[j]       mean(|flow_j|) > cut_threshold                                        F:889-894
 *   cx, cy, val  max_divergence(flow_j) (or the POV shortcut F:880-882)               F:748-758
 *   mean_mag[j]  float32 mean flow magnitude                                           F:890
 *   centers[2j], centers[2j+1]   the +-6 smoothed centre (x, y) as float64            F:1201-1214 */
int  ffb_bracket_begin(ffb_ctx* ctx, int pov_mode, double cut_threshold);
int  ffb_bracket_push(ffb_ctx* ctx, const uint8_t* frames, int n_frames, size_t pitch, size_t frame_stride);
int  ffb_bracket_finish(ffb_ctx* ctx, int* n_pairs, double* scalar, uint8_t* cut, int32_t* cx, int32_t* cy,
                        float* val, float* mean_mag, double* centers);
/* ---- frame-range shards of one bracket (SURVEY.md 8(e); reference semantics F:1188, F:1203-1214) ----
 * A GPU that owns pairs [a, b) of a bracket pushes frames a .. b (one frame of overlap with the next
 * shard) and needs, for the +-6 centre window, the raw centres of pairs [a-6, b+6) clipped to the bracket;
 * those of its neighbours come from the GPUs that computed them.  The bracket is therefore run in two phases:
 *
 *   ffb_bracket_begin_shard(ctx, pov_mode, cut_threshold, shard_pairs)   final flows of all shard_pairs stay resident
 *   ffb_bracket_push / ffb_bracket_push_bgr ...                          flow, centre, cut test per pair (A1-A4)
 *   ffb_bracket_phase1_finish(ctx, &n, cx, cy, val, mean_mag, cut)       raw per-pair results of the shard
 *       ... the host exchanges (cx, cy) with the neighbouring shards (an all_gather of int32[2] per pair) ...
 *   ffb_bracket_radial(ctx, cx_ext, cy_ext, n_ext, first, scalar, centers)
 *
 * cx_ext / cy_ext: raw centres of the n_ext consecutive pairs [a - first, a - first + n_ext) of the bracket,
 * 0 <= first <= 6 and at most 6 pairs beyond the shard's last one, already clipped to the bracket (so the
 * window truncation at bracket ends falls out of the array bounds, exactly as F:1203-1214 truncates).
 * Outputs: scalar[j], centers[2j..2j+1] for the shard's pairs; this call ends the bracket.  A whole bracket
 * pushed as one shard (first = 0, n_ext = n) returns what ffb_bracket_finish returns, bit for bit. */
int  ffb_bracket_begin_shard(ffb_ctx* ctx, int pov_mode, double cut_threshold, int shard_pairs);
int  ffb_bracket_phase1_finish(ffb_ctx* ctx, int* n_pairs, int32_t* cx, int32_t* cy, float* val, float* mean_mag,
                               uint8_t* cut);
int  ffb_bracket_radial(ffb_ctx* ctx, const int32_t* cx_ext, const int32_t* cy_ext, int n_ext, int first,
                        double* scalar, double* centers);
/* Drop the open bracket without results (after an error, or on user cancel: F:1147-1149 "User bailed"):
 * waits for the device work already queued, then leaves the context ready for ffb_bracket_begin /
 * ffb_configure.  A no-op outside a bracket. */
int  ffb_bracket_abort(ffb_ctx* ctx);
/* Two contexts on one device used alternately pipeline consecutive brackets: the frames of bracket i+1 are pushed
 * (uploaded on its context's copy stream) while bracket i still computes, and the results of bracket i are fetched
 * afterwards.  ffb_chain_after(later, earlier) orders the KERNELS `later` queues from now on behind everything
 * `earlier` has queued so far (the two contexts' kernels would otherwise run side by side and compete for the SMs);
 * uploads are not delayed.  Results do not depend on it. */
int  ffb_chain_after(ffb_ctx* later, ffb_ctx* earlier);
/* Block until all uploads issued so far have left the caller's buffers. */
int  ffb_sync(ffb_ctx* ctx);
/* Copy the final flow field of pair `pair` of the current / last bracket to host (test hook and
 * the "flow" entry of the drop-in dict, F:899).  Only the most recent ring of pairs is resident
 * (FFB_E_RANGE otherwise); ffb_flow_ring_size() tells how many. */
int  ffb_bracket_get_flow(ffb_ctx* ctx, int pair, float* flow_hw2);
int  ffb_flow_ring_size(const ffb_ctx* ctx);

/* ---- per-call functions on host arrays (drop-ins for the module-level functions) ----------
 * ffb_farneback   == cv2.calcOpticalFlowFarneback(p0, p1, None, <the context's parameters>)  F:878
 *                    (a new context: .5, 3, 15, 3, 5, 1.2, 0)
 * ffb_max_divergence     == max_divergence(flow)                                         F:748
 * ffb_mean_magnitude     == np.mean(cv2.cartToPolar(u, v)[0])                            F:889-890
 * ffb_radial_motion      == radial_motion_weighted(flow, (cx, cy), is_cut, pov_mode)     F:761 */
int  ffb_farneback(ffb_ctx* ctx, const uint8_t* prev, const uint8_t* next, int width, int height,
                   size_t pitch, float* flow_hw2);
int  ffb_max_divergence(ffb_ctx* ctx, const float* flow_hw2, int width, int height,
                        int32_t* x, int32_t* y, float* val);
int  ffb_mean_magnitude(ffb_ctx* ctx, const float* flow_hw2, int width, int height, float* mean_mag);
int  ffb_radial_motion(ffb_ctx* ctx, const float* flow_hw2, int width, int height,
                       double cx, double cy, int is_cut, int pov_mode, double* out);

/* ---- independent pairs: ffb_farneback for n pairs in one call, through the batched launch chains of a bracket ----
 * Independent pairs (prev + i*frame_stride, next + i*frame_stride), i < n_pairs, uint8 width x height, the context's
 * Farneback parameters.  Outputs may be NULL: flow [n][height][width][2] at flow + i*flow_stride (rows flow_pitch bytes
 * apart); cx, cy, val (max_divergence or the POV shortcut), mean_mag, cut (mean |flow| > cut_threshold) per pair.
 *
 * prev, next and flow may each be pageable host, pinned host or device memory (of the context's device); the per-pair
 * outputs are host arrays.  Every pair's flow is bit-identical to ffb_farneback on that pair.  Pairs run in chunks of
 * (batch_frames + 1) / 2; the call configures the frame size incrementally (the current batch_frames, 2 on a new
 * context; max_pairs grows to n_pairs when a per-pair output is requested).  There is no +-6 centre smoothing and no
 * radial scalar: those are defined along a bracket only.  The flows of an earlier bracket are no longer resident.
 * stream: a cudaStream_t or NULL.  Non-NULL: the work starts after what is queued on `stream`, and `stream` waits
 * until the inputs have been read and the flow written; with every buffer on the device and no per-pair output the
 * call returns without waiting for the device.  NULL, or any host buffer: the call returns when the outputs are
 * complete.  FFB_E_INVALID inside a bracket, for n_pairs < 0, pitch < width, flow_pitch < 8 * width, strides shorter
 * than a frame, and a device pointer on another device; n_pairs == 0 does nothing. */
int  ffb_farneback_pairs(ffb_ctx* ctx, const uint8_t* prev, const uint8_t* next, int n_pairs, int width, int height,
                         size_t pitch, size_t frame_stride, float* flow, size_t flow_pitch, size_t flow_stride,
                         int pov_mode, double cut_threshold, int32_t* cx, int32_t* cy, float* val, float* mean_mag,
                         uint8_t* cut, void* stream);

/* ---- sequences: the flows of every pair of consecutive frames, each frame expanded once (a bracket) -----------------
 * Pair j = (frame j, frame j+1), j < n_frames - 1, frames uint8 width x height at frames + j*frame_stride, the context's
 * Farneback parameters.  Outputs may be NULL: flow of pair j at flow + j*flow_stride (rows flow_pitch bytes apart, the
 * layout of ffb_farneback_pairs); scalar, cut, cx, cy, val, mean_mag, centers as ffb_bracket_finish returns them.
 *
 * The call is a bracket: ffb_bracket_begin(pov_mode, cut_threshold) + ffb_bracket_push(frames) + ffb_bracket_finish,
 * whose final flows are also copied out, one batch behind the kernels.  Every flow is bit-identical to ffb_farneback
 * on that pair, and the per-pair outputs (the +-6 smoothed centres and the radial scalar included) to that bracket's.
 * With no per-pair output only the flows are computed.  frames and flow may each be pageable host, pinned host or
 * device memory (of the context's device); the per-pair outputs are host arrays.  The call configures the frame size
 * incrementally like ffb_farneback_pairs (the current batch_frames, 2 on a new context; max_pairs grows to
 * n_frames - 1 when a per-pair output is requested; with a flow, a final-flow ring of 2*batch_frames + 8 pairs).  The
 * flows of an earlier bracket are no longer resident.  stream: as in ffb_farneback_pairs.  FFB_E_INVALID inside a
 * bracket, for n_frames < 0, pitch < width, flow_pitch < 8 * width, strides shorter than a frame or a flow, and a device
 * pointer on another device; n_frames of 0 or 1 does nothing. */
int  ffb_farneback_sequence(ffb_ctx* ctx, const uint8_t* frames, int n_frames, int width, int height, size_t pitch,
                            size_t frame_stride, float* flow, size_t flow_pitch, size_t flow_stride, int pov_mode,
                            double cut_threshold, double* scalar, uint8_t* cut, int32_t* cx, int32_t* cy, float* val,
                            float* mean_mag, double* centers, void* stream);

/* ---- sequences with backward flows and a forward-backward consistency mask --------------------------------------
 * ffb_farneback_sequence for pair j = (frame j, frame j+1), plus its backward flow (frame j+1 -> frame j) and the
 * forward-backward check (Sundaram, Brox & Keutzer, ECCV 2010).  Outputs may be NULL:
 *   flow_fw      pair j's flow at flow_fw + j*flow_stride (rows flow_pitch bytes apart): ffb_farneback_sequence's flow
 *   flow_bw      the backward flow, same layout: bit-identical to ffb_farneback(frame j+1, frame j)
 *   mask         uint8 [height][width] per pair at mask + j*mask_stride (rows mask_pitch bytes apart): 1 where the
 *                pixel is consistent, 0 otherwise
 *   n_consistent int64 per pair (host array): the number of mask bytes that are 1
 * A pixel (x, y) with forward flow f is consistent when its target t = (x + fx, y + fy) lies in [0, width-1] x
 * [0, height-1] and the backward flow b sampled there bilinearly satisfies |f + b|^2 <= alpha (|f|^2 + |b|^2) + beta
 * (alpha and beta rounded to float32; every operation one float32 rounding, no contraction; the reference values are
 * alpha 0.01, beta 0.5).  Each frame is expanded once: the backward flows re-use the expansions of the forward pass.
 * frames, the flows and the mask may each be pageable host, pinned host or device memory (of the context's device).
 * Configuration and the stream contract are ffb_farneback_sequence's (a ring of 2*batch_frames + 8 pairs with a flow or
 * mask output); the backward ring, the mask ring and the counts are allocated by the first call that needs them and
 * only grow.  There are no per-pair bracket results.  The flows of an earlier bracket are no longer resident.
 * FFB_E_INVALID for everything ffb_farneback_sequence refuses, mask_pitch < width, mask_stride shorter than a mask, and
 * alpha or beta negative or not finite; n_frames of 0 or 1 does nothing. */
int  ffb_farneback_sequence_bidir(ffb_ctx* ctx, const uint8_t* frames, int n_frames, int width, int height,
                                  size_t pitch, size_t frame_stride,
                                  float* flow_fw, float* flow_bw, size_t flow_pitch, size_t flow_stride,
                                  uint8_t* mask, size_t mask_pitch, size_t mask_stride,
                                  double alpha, double beta, int64_t* n_consistent, void* stream);

/* ---- independent pairs with backward flows and a forward-backward consistency mask ------------------------------
 * ffb_farneback_pairs for pair i = (prev + i*frame_stride, next + i*frame_stride), plus its backward flow (next[i] ->
 * prev[i]) and the forward-backward check; for the two eyes of a side-by-side frame it is the left-right check of
 * stereo matching.  Outputs may be NULL:
 *   flow_fw      pair i's flow at flow_fw + i*flow_stride (rows flow_pitch bytes apart): bit-identical to
 *                ffb_farneback(prev[i], next[i])
 *   flow_bw      the backward flow, same layout: bit-identical to ffb_farneback(next[i], prev[i])
 *   mask         uint8 [height][width] per pair at mask + i*mask_stride (rows mask_pitch bytes apart), and
 *   n_consistent int64 per pair (host array): as in ffb_farneback_sequence_bidir
 * Each frame is expanded once: the backward flows re-use the expansions of the forward pass.  prev, next, the flows and
 * the mask may each be pageable host, pinned host or device memory (of the context's device).  Configuration, chunks
 * and the stream contract are ffb_farneback_pairs'; the backward ring, the mask ring and the counts are allocated by
 * the first call that needs them and only grow.  There are no per-pair bracket results, and max_pairs does not grow.
 * The flows of an earlier bracket are no longer resident.  FFB_E_INVALID for everything ffb_farneback_pairs refuses,
 * mask_pitch < width, mask_stride shorter than a mask, and alpha or beta negative or not finite; n_pairs == 0 does
 * nothing. */
int  ffb_farneback_pairs_bidir(ffb_ctx* ctx, const uint8_t* prev, const uint8_t* next, int n_pairs, int width,
                               int height, size_t pitch, size_t frame_stride,
                               float* flow_fw, float* flow_bw, size_t flow_pitch, size_t flow_stride,
                               uint8_t* mask, size_t mask_pitch, size_t mask_stride,
                               double alpha, double beta, int64_t* n_consistent, void* stream);

/* ---- warping by a flow: cv2.remap(src, flow, None, INTER_LINEAR | WARP_RELATIVE_MAP, border, (v, v, v)) -------------
 * For i < n: dst[i] = cv2.remap(src[i], flow[i], None, cv2.INTER_LINEAR | cv2.WARP_RELATIVE_MAP, border_mode,
 * (border_value,) * 3), bit for bit.  src[i] at src + i*src_stride and dst[i] at dst + i*dst_stride are uint8 width x
 * height images of `channels` (1 or 3) bytes per pixel, rows src_pitch / dst_pitch bytes apart; flow[i] at
 * flow + i*flow_stride is float32 [height][width][2] (rows flow_pitch bytes apart), the displacement of each output
 * pixel: dst(x, y) samples src at (x + fx, y + fy).  The arithmetic is cv2's 8-bit one (DESIGN.md "Warping by flow"):
 * positions quantised to 1/32 px, 15-bit bilinear weights, non-finite and huge flows as cv2 takes them.  border_mode 0
 * is cv2.BORDER_CONSTANT (taps outside the image read border_value), 1 cv2.BORDER_REPLICATE.
 * src, flow and dst may each be pageable host, pinned host or device memory (of the context's device); host buffers
 * move through the context's own grow-only staging in chunks of images, with uploads and downloads overlapping the
 * previous chunk's kernel.  The call does not configure the context: its geometry, Farneback parameters and the flows
 * of the last bracket (ffb_bracket_get_flow) stay as they were.  stream: as in ffb_farneback_pairs -- with a stream
 * and every buffer on the device the call returns without waiting for the device, otherwise when dst is complete.
 * FFB_E_INVALID inside a bracket, for n < 0, no buffer, a size of 0 or of 32767 and more (cv2's limit), channels other
 * than 1 or 3, border_mode other than 0 or 1, border_value outside 0..255, src_pitch or dst_pitch < width*channels,
 * flow_pitch < 8*width, strides shorter than an image or a flow, and a device pointer on another device; n == 0 does
 * nothing. */
int  ffb_remap_flow(ffb_ctx* ctx, const uint8_t* src, int n, int width, int height, int channels,
                    size_t src_pitch, size_t src_stride,
                    const float* flow, size_t flow_pitch, size_t flow_stride,
                    uint8_t* dst, size_t dst_pitch, size_t dst_stride,
                    int border_mode, int border_value, void* stream);

/* ---- per-stage hooks (each runs exactly the production kernel of that stage, for the context's parameters) -----
 * Level geometry of the Farneback pyramid for a frame size with the reference's pyr_scale 0.5, levels 3 (coarsest
 * level first): fills up to 4 entries of w[], h[], ksize[], sigma[]; returns the level count in *n_levels. */
int  ffb_level_plan(int width, int height, int* n_levels, int* w, int* h, int* ksize, double* sigma);
/* A1a: u8 frame -> float32 level image (GaussianBlur REFLECT_101 at full res + bilinear resize). */
int  ffb_stage_pyramid(ffb_ctx* ctx, const uint8_t* img, int width, int height, size_t pitch,
                       int level_k, float* out_hw);
/* A1b: float32 image -> float32 [5][h][w] planes (d/dy, d/dx, yy, xx, xy), with the context's poly_n / poly_sigma. */
int  ffb_stage_polyexp(ffb_ctx* ctx, const float* img, int w, int h, float* out_5hw);
/* A1c: R0, R1 ([5][h][w] planes), flow [h][w][2] -> M [5][h][w] planes (G11,G12,G22,h1,h2). */
int  ffb_stage_update_matrices(ffb_ctx* ctx, const float* R0, const float* R1, const float* flow,
                               int w, int h, float* out_5hw);
/* A1c+A1d (the production flow iteration for the context's winsize: fused for 15, matrices + box solve otherwise):
 * R0, R1, flow_in -> flow_out [h][w][2].  flow_in may be NULL (zero initial flow). */
int  ffb_stage_flow_iter(ffb_ctx* ctx, const float* R0, const float* R1, const float* flow_in,
                         int w, int h, float* flow_out);
/* A1e: coarse flow [hc][wc][2] -> [h][w][2], bilinear, x (1 / the context's pyr_scale). */
int  ffb_stage_upsample_flow(ffb_ctx* ctx, const float* flow_c, int wc, int hc, int w, int h, float* out);
/* Forward-backward check of one pair (ffb_farneback_sequence_bidir's k_fb_check): forward and backward flows
 * [h][w][2] -> mask [h][w] (1 consistent, 0 not) and its count; mask and n_consistent may be NULL. */
int  ffb_stage_fb_check(ffb_ctx* ctx, const float* flow_fw, const float* flow_bw, int w, int h, double alpha,
                        double beta, uint8_t* mask, int64_t* n_consistent);

/* ---- frame pre-processing on the device (SURVEY row N2; replaces F:173-189 + F:1074-1082) ------
 * Decoded BGR frames (3 bytes per pixel, as cv2.VideoCapture returns them) are resized to 256 x 256
 * with cv2.resize's 8-bit fixed-point INTER_LINEAR arithmetic (VR mode: 512 x 512, bottom-left
 * quadrant) and converted with cv2's RGB2GRAY formula -- bit-exact with the reference's host path.
 * ffb_preprocess_configure sets the source geometry; the context must be configured for 256 x 256
 * frames (ffb_configure(ctx, 256, 256, ...)) before ffb_bracket_push_bgr is used. */
int  ffb_preprocess_configure(ffb_ctx* ctx, int src_width, int src_height, int vr_mode);
int  ffb_bracket_push_bgr(ffb_ctx* ctx, const uint8_t* bgr, int n_frames, size_t pitch, size_t frame_stride);
/* Stage hook: one BGR frame -> gray[256][256] on the host. */
int  ffb_stage_preprocess(ffb_ctx* ctx, const uint8_t* bgr, int width, int height, size_t pitch, int vr_mode,
                          uint8_t* gray_256x256);

/* Row N4 (SURVEY.md 8(f)): the same arithmetic with the geometry opened up.  The frame is resized to
 * target_w x target_h (equal to the source size = no resampling: cv2.resize returns the frame
 * unchanged and so does the fixed-point formula with weights 2048/0), the window
 * [win_y, win_y+win_h) x [win_x, win_x+win_w) of the resized frame is kept and converted to gray;
 * the context must then be configured for win_w x win_h frames.  The reference's two modes are
 * (256,256, 0,0,256,256) (F:1057) and (512,512, 0,256,256,256) (F:1076-1079); native-resolution
 * processing is (W,H, 0,0,W,H); one eye's lower half of a side-by-side VR frame at native resolution is
 * (W,H, 0 or W/2, H/2, W/2, H/2). */
int  ffb_preprocess_configure_window(ffb_ctx* ctx, int src_width, int src_height, int target_w, int target_h,
                                     int win_x, int win_y, int win_w, int win_h);
int  ffb_stage_preprocess_window(ffb_ctx* ctx, const uint8_t* bgr, int width, int height, size_t pitch,
                                 int target_w, int target_h, int win_x, int win_y, int win_w, int win_h, uint8_t* gray);

/* ---- instrumentation ----------------------------------------------------------------------
 * Kernel ids for ffb_kernel_stats. */
#define FFB_K_PYRAMID   0
#define FFB_K_POLYEXP   1
#define FFB_K_UPSAMPLE  2
#define FFB_K_FLOW_ITER 3
#define FFB_K_DIVMAG    4
#define FFB_K_RADIAL    5
#define FFB_K_SMALL     6   /* finish / centre-smoothing kernels */
#define FFB_K_PREPROC   7
#define FFB_K_FB_CHECK  8   /* forward-backward consistency check */
#define FFB_K_REMAP     9   /* ffb_remap_flow's warp */
#define FFB_K_COUNT     10
/* When enabled, every launch of the kernels above is bracketed by CUDA events on the compute
 * stream; ffb_kernel_stats returns launches, summed device milliseconds and the algorithmic
 * bytes those launches moved (DESIGN.md section "bytes per unit") since the last reset. */
int  ffb_profile(ffb_ctx* ctx, int enable);
int  ffb_profile_reset(ffb_ctx* ctx);
int  ffb_kernel_stats(ffb_ctx* ctx, int kernel_id, int64_t* launches, double* ms, double* alg_bytes);
/* The same three figures for the flow iteration alone, split by pyramid level k (0 = full resolution, up to 15). */
int  ffb_flow_iter_level_stats(ffb_ctx* ctx, int level_k, int64_t* launches, double* ms, double* alg_bytes);
int64_t ffb_launch_count(const ffb_ctx* ctx);   /* kernels launched by this context so far */
/* Device-side stopwatch on the compute stream (the stream every kernel is launched on):
 * ffb_timer_mark(ctx, slot) records CUDA event `slot` (0..7); ffb_timer_elapsed waits for both
 * events and returns the milliseconds between them. */
int  ffb_timer_mark(ffb_ctx* ctx, int slot);
int  ffb_timer_elapsed(ffb_ctx* ctx, int slot_from, int slot_to, double* ms);
const char* ffb_kernel_name(int kernel_id);

#ifdef __cplusplus
}
#endif
#endif /* FFB_H_ */
