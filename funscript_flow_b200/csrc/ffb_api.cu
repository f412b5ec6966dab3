// ffb_api.cu -- context, stream plumbing and the extern "C" ABI declared in include/ffb.h.
//
// One context = one GPU = one host thread.  Frames flow
//   host (pageable | pinned) --cudaMemcpyAsync on s_copy, double-buffered--> device u8 staging
//   --k_pyramid_pow2 | k_pyramid_level / k_polyexp--> per-frame expansion slots (ring of S = B+2 frames; each frame
//     is expanded once and used as `next` of pair j-1 and `prev` of pair j: streaming mode; ffb_farneback_pairs stages
//     independent pairs as prev_0, next_0, prev_1, ... and reads them with pair stride 2)
//   --k_flow_iter x iterations per level (flow up-sampling fused, k_upsample_flow otherwise; winsize != 15:
//     k_flow_matrices + k_box_solve)--> final-flow ring (>= B+8 pairs; ffb_farneback_pairs and ffb_farneback_sequence
//     copy the flows out of it on s_out, the sequence with a ring of >= 2B+8 pairs; ffb_farneback_sequence_bidir and
//     ffb_farneback_pairs_bidir also run the reversed pairs into a backward final-flow ring and k_fb_check into a mask
//     ring of the same slots)
//   --k_divmag / k_phase1_finish--> per-pair centre, value, mean magnitude, cut flag (device arrays)
//   --k_smooth_centers / k_radial / k_radial_finish (lagging 6 pairs)--> per-pair scalar
// and only the 1-D per-pair results are copied back at ffb_bracket_finish.
#include "../../include/ffb.h"
#include "ffb_kernels.cuh"

#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <limits>
#include <set>
#include <string>
#include <thread>
#include <vector>

namespace {

thread_local std::string g_create_error;

const char* const kKernelNames[FFB_K_COUNT] = {"k_pyramid_level", "k_polyexp",  "k_upsample_flow", "k_flow_iter",
                                               "k_divmag",        "k_radial",   "small",           "k_preprocess",
                                               "k_fb_check",      "k_remap_flow"};

// ------------------------------------------------------------------ host-side constant builders
int cv_round(double v) { return (int)nearbyint(v); }   // round-half-even in the default FP mode

// calcOpticalFlowFarneback's parameters (flags is always 0: the two flags are refused).  A new context holds the
// reference's call (F:878-879).
struct FarnebackParams {
    double pyr_scale = 0.5;
    int levels = 3, winsize = 15, iterations = 3, poly_n = 5;
    double poly_sigma = 1.2;
    bool operator==(const FarnebackParams& o) const {
        return pyr_scale == o.pyr_scale && levels == o.levels && winsize == o.winsize && iterations == o.iterations &&
               poly_n == o.poly_n && poly_sigma == o.poly_sigma;
    }
};

struct LevelPlan {
    int n;                  // may exceed FFB_PLAN_LEVELS: then only the first FFB_PLAN_LEVELS entries are filled
    double pyr_scale;
    int k[FFB_PLAN_LEVELS], w[FFB_PLAN_LEVELS], h[FFB_PLAN_LEVELS], ksize[FFB_PLAN_LEVELS];
    double sigma[FFB_PLAN_LEVELS];
};

// calcOpticalFlowFarneback level geometry (SURVEY.md 3.4 steps 1-2): levels stop where the coarsest one would be
// narrower or lower than 32 px.
LevelPlan make_plan(int W, int H, double pyr_scale, int levels) {
    LevelPlan p;
    p.pyr_scale = pyr_scale;
    int k = 0;
    double scale = 1.0;
    while (k < levels) {
        scale *= pyr_scale;
        if (W * scale < 32 || H * scale < 32) break;
        ++k;
    }
    p.n = k + 1;
    for (int i = 0; i < p.n && i < FFB_PLAN_LEVELS; ++i) {
        const int kk = k - i;   // coarsest first
        double s = 1.0;
        for (int j = 0; j < kk; ++j) s *= pyr_scale;
        const double sigma = (1.0 / s - 1.0) * 0.5;
        int ks = cv_round(sigma * 5) | 1;
        if (ks < 3) ks = 3;
        p.k[i] = kk;
        p.w[i] = cv_round(W * s);
        p.h[i] = cv_round(H * s);
        p.ksize[i] = ks;
        p.sigma[i] = sigma;
    }
    return p;
}
LevelPlan make_plan(int W, int H, const FarnebackParams& fp) { return make_plan(W, H, fp.pyr_scale, fp.levels); }

// cv::getGaussianKernel(ksize, sigma, CV_32F), half kernel (ksize / 2 + 1 taps).
std::vector<float> gaussian_half(int ksize, double sigma) {
    const int r = ksize / 2;
    if (sigma <= 0 && ksize == 3) return {0.5f, 0.25f};
    if (sigma <= 0) sigma = ((ksize - 1) * 0.5 - 1) * 0.3 + 0.8;
    std::vector<double> v(ksize);
    double sum = 0;
    for (int i = 0; i < ksize; ++i) {
        const double x = i - (ksize - 1) * 0.5;
        v[i] = exp(-0.5 / (sigma * sigma) * x * x);
        sum += v[i];
    }
    std::vector<float> k(r + 1);
    for (int i = 0; i <= r; ++i) k[i] = (float)(v[r + i] / sum);
    return k;
}

// The same half kernel in the fixed-size form the shared-memory pyramid kernels take (radius <= 9).
FfbTaps make_taps(int ksize, double sigma) {
    FfbTaps t;
    memset(&t, 0, sizeof(t));
    t.r = ksize / 2;
    const std::vector<float> k = gaussian_half(ksize, sigma);
    for (int i = 0; i <= t.r && i < 10; ++i) t.k[i] = k[i];
    return t;
}
constexpr int kTapsMaxR = 9;

// cv::resize INTER_LINEAR per-axis table.
void make_linear_table(int dst_n, int src_n, std::vector<int>& idx, std::vector<float>& alpha) {
    idx.resize(dst_n);
    alpha.resize(dst_n);
    const double scale = (double)src_n / dst_n;
    for (int d = 0; d < dst_n; ++d) {
        float f = (float)((d + 0.5) * scale - 0.5);
        int i0 = (int)floorf(f);
        f -= (float)i0;
        if (i0 < 0) { i0 = 0; f = 0.f; }
        if (i0 >= src_n - 1) { i0 = src_n - 1; f = 0.f; }
        idx[d] = i0;
        alpha[d] = f;
    }
}

// FarnebackPrepareGaussian(n, sigma): taps in float32, inverse moments in double.
void invert6(double G[6][6], double inv[6][6]) {
    double a[6][12];
    for (int i = 0; i < 6; ++i)
        for (int j = 0; j < 6; ++j) { a[i][j] = G[i][j]; a[i][j + 6] = i == j ? 1.0 : 0.0; }
    for (int c = 0; c < 6; ++c) {
        int piv = c;
        for (int r = c + 1; r < 6; ++r) if (fabs(a[r][c]) > fabs(a[piv][c])) piv = r;
        for (int j = 0; j < 12; ++j) { double t = a[c][j]; a[c][j] = a[piv][j]; a[piv][j] = t; }
        const double d = a[c][c];
        for (int j = 0; j < 12; ++j) a[c][j] /= d;
        for (int r = 0; r < 6; ++r) {
            if (r == c) continue;
            const double f = a[r][c];
            for (int j = 0; j < 12; ++j) a[r][j] -= f * a[c][j];
        }
    }
    for (int i = 0; i < 6; ++i)
        for (int j = 0; j < 6; ++j) inv[i][j] = a[i][j + 6];
}

template <int N>
FfbPolyConsts<N> make_poly_consts(double sigma) {
    const int n = N;
    if (sigma < std::numeric_limits<float>::epsilon()) sigma = n * 0.3;
    float g[2 * N + 1], xg[2 * N + 1], xxg[2 * N + 1];
    double s = 0;
    for (int x = -n; x <= n; ++x) { g[x + n] = (float)exp(-x * x / (2 * sigma * sigma)); s += g[x + n]; }
    s = 1.0 / s;
    for (int x = -n; x <= n; ++x) {
        g[x + n] = (float)(g[x + n] * s);
        xg[x + n] = (float)(x * g[x + n]);
        xxg[x + n] = (float)(x * x * g[x + n]);
    }
    double G[6][6];
    memset(G, 0, sizeof(G));
    for (int y = -n; y <= n; ++y)
        for (int x = -n; x <= n; ++x) {
            const float gg = g[y + n] * g[x + n];
            G[0][0] += gg;
            G[1][1] += gg * (float)(x * x);
            G[3][3] += gg * (float)(x * x * x * x);
            G[5][5] += gg * (float)(x * x * y * y);
        }
    G[2][2] = G[0][3] = G[0][4] = G[3][0] = G[4][0] = G[1][1];
    G[4][4] = G[3][3];
    G[3][4] = G[4][3] = G[5][5];
    double inv[6][6];
    invert6(G, inv);
    FfbPolyConsts<N> c;
    for (int i = 0; i <= n; ++i) { c.g[i] = g[n + i]; c.xg[i] = xg[n + i]; c.xxg[i] = xxg[n + i]; }
    c.ig11 = (float)inv[1][1];
    c.ig03 = (float)inv[0][3];
    c.ig33 = (float)inv[3][3];
    c.ig55 = (float)inv[5][5];
    return c;
}

// ------------------------------------------------------------------ context
// k_flow_iter launch of one pyramid level: variant (threads per CTA = matrix columns per strip x rows per step x
// outputs per horizontal task), strip width and rows per march segment.  nt = 0: no variant forced.
struct FlowIterPlan { int nt = 0, u = 0, ho = 0, sw = 0, sh = 0; };

struct Level {
    int k = 0, w = 0, h = 0, ksize = 3;
    double sigma = 0;
    int rp = 0;            // R / I row pitch (floats)
    size_t plane = 0;      // rp * h
    int fp = 0;            // flow row pitch (float2)
    size_t r_off = 0;      // float offset of this level inside a frame's expansion slot
    FfbTaps taps;
    int RW = 0, RH = 0;    // source window bound of one 32x8 output tile
    bool wide = false;     // blur radius or tile window beyond k_pyramid_level: k_pyramid_wide_rows / _cols
    int *xi = nullptr, *yi = nullptr, *uxi = nullptr, *uyi = nullptr;
    float *xa = nullptr, *ya = nullptr, *uxa = nullptr, *uya = nullptr;
    float* wk = nullptr;   // half kernel of a wide level (device)
    float* I = nullptr;    // [B][h][rp]
    float2 *fA = nullptr, *fB = nullptr;   // [B][h][fp]
    FlowIterPlan iter;
    bool up2x = false;     // exact 2x refinement of the coarser level: its first iteration up-samples the flow itself
};

struct ProfRec { int kid; int level; double bytes; cudaEvent_t e0, e1; };
struct ProfMark { cudaEvent_t e1 = nullptr; cudaStream_t stream = nullptr; };   // end event of an open record

}  // namespace

struct ffb_ctx {
    int device = 0;
    std::string err;
    cudaStream_t s_comp = nullptr, s_copy = nullptr;
    cudaStream_t s_aux = nullptr;                      // second slice of the sliced flow phase
    cudaStream_t s_time = nullptr;                     // only carries the end-of-flow-phase timing event
    cudaEvent_t ev_flow_end[2] = {nullptr, nullptr};
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    cudaEvent_t ev_chain = nullptr;                    // "everything queued on s_comp so far": ffb_chain_after
    cudaEvent_t ev_h2d[2] = {nullptr, nullptr}, ev_expand[2] = {nullptr, nullptr};
    // ffb_farneback_pairs / _sequence: final flows leave the final-flow ring on s_out.  ev_fin[h] / ev_out[h]: the flows
    // of the chunk in ring half h (of the sequence batch of parity h) are complete / have been copied out; ev_user /
    // ev_done order the call after / before the caller's stream; ev_h2d_next[b]: the upload of a chunk's `next` frames
    // through staging buffer b is done (the `prev` frames use ev_h2d[b]), so that the host stages them without waiting
    // for the `prev` frames' DMA.
    cudaStream_t s_out = nullptr;
    cudaEvent_t ev_fin[2] = {nullptr, nullptr}, ev_out[2] = {nullptr, nullptr}, ev_user = nullptr, ev_done = nullptr;
    cudaEvent_t ev_h2d_next[2] = {nullptr, nullptr};
    FarnebackParams fb;
    FfbPolyConsts<5> poly5;
    FfbPolyConsts<7> poly7;
    // geometry
    int W = 0, H = 0, B = 0, maxPairs = 0, nlev = 0, S = 0, ring_n = 0, fp0 = 0;
    int Bcap = 0, pairsCap = 0;                 // allocated capacities (B / maxPairs are the limits of the last ffb_configure)
    int64_t n_dev_alloc = 0, n_host_alloc = 0;  // cudaMalloc / cudaHostAlloc calls made for this context so far
    bool pyr_fast = false;
    Level lev[FFB_PLAN_LEVELS];
    int wide_w = 0;                 // widest level that takes the large-radius pyramid (0: none)
    float* pyr_tmp = nullptr;       // its scratch image, (Bcap + 1) x H x wide_w floats
    float* M = nullptr;             // matrices of the unfused flow iteration (winsize != 15), Bcap pairs at level 0
    float* R = nullptr;
    size_t r_slot_floats = 0;
    float2* ring = nullptr;
    size_t ring_stride = 0;   // float2 per ring element
    // ffb_farneback_sequence_bidir / _pairs_bidir, allocated by the first call that needs them (alloc_backward): backward
    // final flows and consistency masks in the slots of the final-flow ring (bw_n / mask_n slots, 0 or ring_n),
    // consistent-pixel counts per pair of the call
    float2* ring_bw = nullptr;
    uint8_t* mask_ring = nullptr;
    int bw_n = 0, mask_n = 0;
    unsigned* d_ncons = nullptr;
    int ncons_cap = 0;
    uint8_t* d_u8[2] = {nullptr, nullptr};
    uint8_t* h_pin[2] = {nullptr, nullptr};
    // per-bracket results (device) + partials
    int *d_cx = nullptr, *d_cy = nullptr;
    int *d_cx_ext = nullptr, *d_cy_ext = nullptr;   // raw centres handed in by ffb_bracket_radial (shard + 6 each side)
    float *d_val = nullptr, *d_mm = nullptr;
    unsigned char* d_cut = nullptr;
    double *d_centers = nullptr, *d_scalar = nullptr;
    unsigned long long* d_pkey = nullptr;
    double *d_psum = nullptr, *d_rpart = nullptr;
    int div_nblk = 0, div_rpb = 0, rad_gx = 0, rad_gy = 0, rad_rpb = 0;
    char* h_res = nullptr;    // pinned result staging
    // frame pre-processing (row N2): source geometry, tables, chunked colour staging
    // source size -> resize target (TW x TH) -> kept window [y0, y0+OH) x [x0, x0+OW) of the target
    struct PrePlan { int W = 0, H = 0, TW = 0, TH = 0, x0 = 0, y0 = 0, OW = 0, OH = 0;
                     bool operator==(const PrePlan& o) const {
                         return W == o.W && H == o.H && TW == o.TW && TH == o.TH && x0 == o.x0 && y0 == o.y0 && OW == o.OW && OH == o.OH; } } pre;
    int *pre_xt = nullptr, *pre_yt = nullptr;
    uint8_t* d_color[2] = {nullptr, nullptr};
    uint8_t* h_color[2] = {nullptr, nullptr};
    cudaEvent_t ev_ch2d[2] = {nullptr, nullptr}, ev_pre[2] = {nullptr, nullptr};
    int color_no = 0;
    // ffb_remap_flow's staging, grow-only and independent of the geometry: per buffer b of a chunk, the device images
    // of host (or misaligned) inputs and of a host output, and the pinned copies of pageable inputs
    uint8_t *rm_src[2] = {nullptr, nullptr}, *rm_flow[2] = {nullptr, nullptr}, *rm_dst[2] = {nullptr, nullptr};
    uint8_t *rm_hsrc[2] = {nullptr, nullptr}, *rm_hflow[2] = {nullptr, nullptr};
    size_t rm_src_cap = 0, rm_flow_cap = 0, rm_dst_cap = 0, rm_hsrc_cap = 0, rm_hflow_cap = 0;
    // bracket state
    bool in_bracket = false;
    int pov = 0;
    float thr = 7.f;
    int frames_seen = 0, pairs_done = 0, radial_done = 0, batch_no = 0;
    bool deferred = false;      // shard mode: the radial pass waits for ffb_bracket_radial (external raw centres)
    bool phase1_read = false;   // ffb_bracket_phase1_finish has been called for the open bracket
    int pend = 0;               // pre-processed gray frames waiting in d_u8[batch_no & 1] for a full batch
    // instrumentation
    bool prof = false;
    std::vector<ProfRec> recs;
    std::vector<cudaEvent_t> ev_pool;
    int64_t k_launches[FFB_K_COUNT] = {0};
    double k_ms[FFB_K_COUNT] = {0}, k_bytes[FFB_K_COUNT] = {0};
    int64_t it_launches[FFB_PLAN_LEVELS] = {0};         // k_flow_iter (or k_flow_matrices + k_box_solve) split by level k
    double it_ms[FFB_PLAN_LEVELS] = {0}, it_bytes[FFB_PLAN_LEVELS] = {0};
    // cudaFuncSetAttribute is per device: remember per context which kernels already had their
    // dynamic shared-memory limit raised (a process may own contexts on several GPUs)
    size_t pyr_smem_max = 48 * 1024;
    bool attr_poly = false, attr_poly7 = false, attr_pyr2 = false;
    std::set<const void*> attr_iter;                     // k_flow_iter instantiations already configured
    FlowIterPlan iter_cfg;                               // variant forced by FFB_ITER_CFG for every level
    int flow_streams = 2;
    int64_t launches = 0;
    cudaEvent_t timers[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
};

namespace {

int fail(ffb_ctx* c, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (c) c->err = buf; else g_create_error = buf;
    return code;
}

#define CK(c, call)                                                                                   \
    do {                                                                                              \
        cudaError_t e_ = (call);                                                                      \
        if (e_ != cudaSuccess)                                                                        \
            return fail((c), FFB_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)
#define CKL(c)                                                                                        \
    do {                                                                                              \
        cudaError_t e_ = cudaGetLastError();                                                          \
        if (e_ != cudaSuccess)                                                                        \
            return fail((c), FFB_E_CUDA, "kernel launch failed: %s (%s:%d)", cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)
#define TRY(expr)                   \
    do {                            \
        int rc_ = (expr);           \
        if (rc_ != FFB_OK) return rc_; \
    } while (0)

template <class T>
int dev_alloc(ffb_ctx* c, T** p, size_t count) {
    void* v = nullptr;
    cudaError_t e = cudaMalloc(&v, count * sizeof(T) + 256);   // +256: vector loads may touch a row's tail
    if (e != cudaSuccess) return fail(c, FFB_E_NOMEM, "cudaMalloc(%zu bytes) failed: %s", count * sizeof(T), cudaGetErrorString(e));
    if (c) c->n_dev_alloc++;
    *p = (T*)v;
    return FFB_OK;
}
template <class T>
void dev_free(T*& p) {
    if (p) cudaFree(p);
    p = nullptr;
}
template <class T>
int upload_vec(ffb_ctx* c, T** dptr, const std::vector<T>& v) {
    TRY(dev_alloc(c, dptr, v.size()));
    CK(c, cudaMemcpy(*dptr, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
    return FFB_OK;
}

// ---- profiling helpers
// Opens a timed record of kernel `kid`: its start event is recorded on `stream` now, its end event by prof_end.
ProfMark prof_record(ffb_ctx* c, int kid, int level, double bytes, cudaStream_t stream) {
    ProfRec r{kid, level, bytes, nullptr, nullptr};
    for (cudaEvent_t* e : {&r.e0, &r.e1}) {
        if (!c->ev_pool.empty()) { *e = c->ev_pool.back(); c->ev_pool.pop_back(); }
        else cudaEventCreate(e);
    }
    cudaEventRecord(r.e0, stream);
    c->recs.push_back(r);
    return ProfMark{r.e1, stream};
}
// Counts a launch of `kid` on `stream` (a k_flow_iter launch also under its pyramid level; -1: no level) and, when
// profiling is on and the launch is timed on its own, brackets it with events on that stream.
ProfMark prof_begin(ffb_ctx* c, int kid, int level, double bytes, cudaStream_t stream, bool timed = true) {
    c->launches++;
    c->k_launches[kid]++;
    c->k_bytes[kid] += bytes;
    if (level >= 0) { c->it_launches[level]++; c->it_bytes[level] += bytes; }
    return c->prof && timed ? prof_record(c, kid, level, bytes, stream) : ProfMark{};
}
void prof_end(const ProfMark& m) {
    if (m.e1) cudaEventRecord(m.e1, m.stream);
}
// Sliced flow phase: the launch chains of the slices overlap, so per-launch event times would count
// the same device time several times.  The phase is timed as a whole on s_comp instead
// (fork ... join) and attributed to k_flow_iter.
ProfMark prof_phase_begin(ffb_ctx* c) {
    return c->prof ? prof_record(c, FFB_K_FLOW_ITER, -1, 0, c->s_comp) : ProfMark{};
}
// the phase ends when the last slice's last flow iteration does: a side stream waits for every slice's
// end-of-flow event and records the timing event, so that the per-slice reductions that follow on the
// slice streams are not counted
void prof_phase_end(ffb_ctx* c, const ProfMark& phase, int nslice) {
    if (!phase.e1) return;
    for (int i = 0; i < nslice; ++i) cudaStreamWaitEvent(c->s_time, c->ev_flow_end[i], 0);
    cudaEventRecord(phase.e1, c->s_time);
}

void prof_collect(ffb_ctx* c) {
    for (ProfRec& r : c->recs) {
        float ms = 0.f;
        cudaEventSynchronize(r.e1);
        cudaEventElapsedTime(&ms, r.e0, r.e1);
        c->k_ms[r.kid] += ms;
        if (r.level >= 0) c->it_ms[r.level] += ms;
        c->ev_pool.push_back(r.e0);
        c->ev_pool.push_back(r.e1);
    }
    c->recs.clear();
}

// ------------------------------------------------------------------ kernel launchers
constexpr int PYR_TW = 32, PYR_TH = 8;

// Upper bound of the source window (in source pixels) any 32x8 output tile of a level needs.
void pyramid_window(const std::vector<int>& idx, int dst_n, int src_n, int tile, int r, int* bound) {
    int best = 0;
    for (int t0 = 0; t0 < dst_n; t0 += tile) {
        const int t1 = (t0 + tile < dst_n ? t0 + tile : dst_n) - 1;
        int hi = idx[t1] + 1;
        if (hi > src_n - 1) hi = src_n - 1;
        const int ext = (hi + r) - (idx[t0] - r) + 1;
        if (ext > best) best = ext;
    }
    *bound = best;
}

// k_pyramid_level's dynamic shared memory for a source window bound RW x RH (the staged window + the row-pass plane)
size_t pyramid_smem(int RW, int RH) {
    return ((size_t)ffb_round_up((RW | 1) * RH, 4) + (size_t)RH * PYR_TW) * sizeof(float);
}
// A level takes the large-radius kernels when its radius exceeds FfbTaps or its tile window exceeds the 227 KB of
// shared memory a B200 block may use.
bool pyramid_wide(int r, int RW, int RH) { return r > kTapsMaxR || pyramid_smem(RW, RH) > 227u * 1024u; }

int launch_pyramid(ffb_ctx* c, const uint8_t* src, size_t src_stride, int src_pitch, int W, int H, float* dst,
                   size_t dst_stride, int dp, int w, int h, const int* xi, const float* xa, const int* yi,
                   const float* ya, const FfbTaps& taps, int RW, int RH, int nframes) {
    FfbPyrArgs a;
    a.src = src; a.src_frame_stride = src_stride; a.src_pitch = src_pitch; a.W = W; a.H = H;
    a.dst = dst; a.dst_frame_stride = dst_stride; a.dp = dp; a.w = w; a.h = h;
    a.xi = xi; a.xa = xa; a.yi = yi; a.ya = ya; a.taps = taps;
    a.RWp = RW | 1;                       // odd pitch: column walks of pass 1 stay conflict-free
    a.p_off = ffb_round_up(a.RWp * RH, 4);
    const size_t smem = pyramid_smem(RW, RH);
    if (taps.r >= W || taps.r >= H) return fail(c, FFB_E_INVALID, "frame smaller than the blur radius");
    auto kfn = k_pyramid_level<PYR_TW, PYR_TH>;
    if (smem > c->pyr_smem_max) {
        CK(c, cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        c->pyr_smem_max = smem;
    }
    dim3 grid((w + PYR_TW - 1) / PYR_TW, (h + PYR_TH - 1) / PYR_TH, nframes);
    const ProfMark pm = prof_begin(c, FFB_K_PYRAMID, -1, (double)nframes * ((double)W * H + 4.0 * w * h), c->s_comp);
    FFB_LAUNCH(kfn, grid, dim3(PYR_TW * PYR_TH), smem, c->s_comp, a);
    prof_end(pm);
    CKL(c);
    return FFB_OK;
}

// Large-radius pyramid level (Level::wide): row pass into `tmp` (H x w per frame), column pass into dst.
int launch_pyramid_wide(ffb_ctx* c, const uint8_t* src, size_t src_stride, int src_pitch, int W, int H, float* tmp, float* dst,
                        size_t dst_stride, int dp, int w, int h, const int* xi, const float* xa, const int* yi, const float* ya,
                        const float* k, int r, int nframes) {
    if (r >= W || r >= H) return fail(c, FFB_E_INVALID, "frame smaller than the blur radius");
    FfbPyrWideArgs a;
    a.src = src; a.src_frame_stride = src_stride; a.src_pitch = src_pitch; a.W = W; a.H = H;
    a.tmp = tmp; a.tmp_frame_stride = (size_t)H * w;
    a.dst = dst; a.dst_frame_stride = dst_stride; a.dp = dp; a.w = w; a.h = h;
    a.xi = xi; a.xa = xa; a.yi = yi; a.ya = ya; a.k = k; a.r = r;
    const ProfMark pr = prof_begin(c, FFB_K_PYRAMID, -1, (double)nframes * ((double)W * H + 4.0 * H * w), c->s_comp);
    FFB_LAUNCH(k_pyramid_wide_rows, dim3((w + 31) / 32, (H + 7) / 8, nframes), dim3(256), 0, c->s_comp, a);
    prof_end(pr);
    CKL(c);
    const ProfMark pc = prof_begin(c, FFB_K_PYRAMID, -1, (double)nframes * (4.0 * H * w + 4.0 * w * h), c->s_comp);
    FFB_LAUNCH(k_pyramid_wide_cols, dim3((w + 31) / 32, (h + 7) / 8, nframes), dim3(256), 0, c->s_comp, a);
    prof_end(pc);
    CKL(c);
    return FFB_OK;
}

template <int N>
int launch_polyexp_t(ffb_ctx* c, FfbPolyArgs<N>& a, const FfbPolyConsts<N>& consts, bool& attr, int nframes) {
    a.c = consts;
    // the kernel stores two pixels (32 bytes) of the float4 image per instruction
    if (a.rp % 4 != 0 || ((uintptr_t)a.dst.base | (uintptr_t)a.dst.stride) % 32 != 0)
        return fail(c, FFB_E_INVALID, "expansion output is not 32-byte aligned (pitch %d, stride %zu)", a.rp, a.dst.stride);
    if (!attr) {
        CK(c, cudaFuncSetAttribute(k_polyexp<N>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)POLY_SMEM));
        attr = true;
    }
    // (a variant with packed fp32 arithmetic -- FFMA2 / FADD2 / FMUL2 on row pairs -- was measured in round 2: 4.60 ms
    // against 3.92 ms per 257 1080p frames for this scalar kernel; the packed instructions issue at half rate and the
    // 114 registers they need halve the occupancy.  profiles/r2_other_kernels.txt)
    dim3 grid((a.w + POLY_OW - 1) / POLY_OW, (a.h + POLY_ROWS - 1) / POLY_ROWS, nframes);
    const ProfMark pm = prof_begin(c, FFB_K_POLYEXP, -1, (double)nframes * 24.0 * a.w * a.h, c->s_comp);
    FFB_LAUNCH(k_polyexp<N>, grid, dim3(256), POLY_SMEM, c->s_comp, a);
    prof_end(pm);
    CKL(c);
    return FFB_OK;
}

// the context's poly_n selects the instantiation (5 or 7)
int launch_polyexp(ffb_ctx* c, const float* src, size_t src_stride, int sp, int w, int h, FfbRing dst, size_t plane,
                   int rp, int nframes) {
    auto fill = [&](auto& a) {
        a.src = src; a.src_frame_stride = src_stride; a.sp = sp; a.w = w; a.h = h;
        a.dst = dst; a.plane = plane; a.rp = rp;
    };
    if (c->fb.poly_n == 7) {
        FfbPolyArgs<7> a;
        fill(a);
        return launch_polyexp_t(c, a, c->poly7, c->attr_poly7, nframes);
    }
    FfbPolyArgs<5> a;
    fill(a);
    return launch_polyexp_t(c, a, c->poly5, c->attr_poly, nframes);
}

// k_upsample_flow: the flow is doubled with pyr_scale 0.5, multiplied by 1 / pyr_scale otherwise
int launch_upsample(ffb_ctx* c, const float2* src, size_t src_stride, int sp, int wc, int hc, float2* dst,
                    size_t dst_stride, int dp, int w, int h, const int* xi, const float* xa, const int* yi,
                    const float* ya, int npairs) {
    FfbUpArgs a;
    a.src = src; a.src_stride = src_stride; a.sp = sp; a.wc = wc; a.hc = hc;
    a.dst = dst; a.dst_stride = dst_stride; a.dp = dp; a.w = w; a.h = h;
    a.xi = xi; a.xa = xa; a.yi = yi; a.ya = ya;
    a.scale = (float)(1.0 / c->fb.pyr_scale);
    dim3 grid((w + 31) / 32, (h + 7) / 8, npairs);
    const ProfMark pm = prof_begin(c, FFB_K_UPSAMPLE, -1, (double)npairs * (8.0 * wc * hc + 8.0 * w * h), c->s_comp);
    if (c->fb.pyr_scale == 0.5) FFB_LAUNCH(k_upsample_flow<false>, grid, dim3(256), 0, c->s_comp, a);
    else FFB_LAUNCH(k_upsample_flow<true>, grid, dim3(256), 0, c->s_comp, a);
    prof_end(pm);
    CKL(c);
    return FFB_OK;
}

// Launch plan of k_flow_iter on a w x h level of frame_w x frame_h frames (the frame the context is configured for;
// a stage hook passes the level itself).  It depends on this geometry alone, never on the batch, so a pair's result is
// bit-identical however frames are batched or sharded.  `forced`: a variant forced for every level (FFB_ITER_CFG).
FlowIterPlan flow_iter_plan(int frame_w, int frame_h, int w, int h, const FlowIterPlan& forced) {
    const bool large = (long long)frame_w * frame_h >= 1280LL * 720;
    FlowIterPlan p = forced;
    if (p.nt == 0) {
        // Defaults from the round-2 sweeps on a B200 (profiles/r2_sweep_flow_iter.txt):
        //   1280x720 and larger   256 threads, 4 rows per step, 8 outputs per horizontal task: 242-column strips carry
        //                         5.5 % halo columns instead of 10.9 %, and the 120 horizontal tasks of a step fill 4 of
        //                         the 8 warps (1080p: +8.4 % over 128x2x4, 4K: +7 %, 720p: +1 %)
        //   up to 320 columns     160 threads x 2 rows x 4 outputs (the reference's 256x256 product mode: 2 strips); its
        //                         64- and 32-column levels take 96- and 64-thread strips (5 / 8 CTAs per SM instead of
        //                         mostly idle 160-thread ones) and a single row segment per level: +3 % together
        //   in between            128 threads x 2 rows x 4 outputs (640x360: +8 % over 160x2x4)
        if (large) { p.nt = 256; p.u = 4; p.ho = 8; }
        else if (frame_w <= 320) { p.nt = w <= 48 ? 64 : (w <= 80 ? 96 : 160); p.u = 2; p.ho = 4; }     // by LEVEL width
        else { p.nt = 128; p.u = 2; p.ho = 4; }
    }
    if (p.u < 1 || p.ho < 1) return p;      // no such variant: launch_flow_iter refuses it
    // full-width strips; the last one is narrower and its idle warps skip the gather (k_flow_iter `live`)
    p.sw = (p.nt - 2 * FFB_WIN_R) / p.ho * p.ho;
    // at most 270 rows per segment, at least min_seg segments per level (coarse levels would otherwise be a handful of
    // long, latency-bound marches), never under 32 rows.  Frames of 1280x720 and more: at least 3 segments on every
    // level (parallelism for their 64-pair batches; 2 .. 4 measure the same at 1080p, 5 and more lose); smaller frames
    // come in batches of hundreds, and every segment pays 14 halo rows: 2 (+7 % at 256x256, +3.5 % at 640x360) --
    // profiles/r1_sweep_segments.txt, r2_sweep_flow_iter.txt.
    const int min_seg = large ? 3 : (frame_w <= 320 ? 1 : 2);
    int nseg = (h + 269) / 270;
    if (nseg < min_seg) nseg = min_seg;
    if (nseg > (h + 31) / 32) nseg = (h + 31) / 32;
    if (nseg < 1) nseg = 1;
    p.sh = ffb_round_up((h + nseg - 1) / nseg, p.u);     // even: see the fused up-sampling in k_flow_iter
    return p;
}

template <int NT, int U, int MINB, int HO, int PS, bool REV>
int launch_flow_iter_t(ffb_ctx* c, const FfbIterArgs& a, int npairs, int level, double bytes, cudaStream_t stream, bool timed) {
    auto kfn = a.up_src ? k_flow_iter<NT, U, MINB, true, HO, PS, REV> : k_flow_iter<NT, U, MINB, false, HO, PS, REV>;
    const size_t smem = ffb_flow_iter_smem<NT, U, HO>();
    if (!c->attr_iter.count((const void*)kfn)) {
        CK(c, cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        c->attr_iter.insert((const void*)kfn);
    }
    const ProfMark pm = prof_begin(c, FFB_K_FLOW_ITER, level, bytes, stream, timed);
    // pair index varies fastest in launch order: the CTAs working on one spatial tile of consecutive
    // pairs are co-resident, so frame j+1's expansion (R1 of pair j, R0 of pair j+1) is read from
    // HBM once and hit in L2 the second time.
    FFB_LAUNCH(kfn, dim3(npairs, (a.w + a.SW - 1) / a.SW, (a.h + a.SH - 1) / a.SH), dim3(NT), smem, stream, a);
    prof_end(pm);
    CKL(c);
    return FFB_OK;
}

struct UpSrc {   // coarser-level flow to be up-sampled inside the iteration kernel (A1e fused)
    const float2* src = nullptr; size_t stride = 0; int sp = 0, wc = 0, hc = 0;
};

// the k_flow_iter variant of plan `p` with pair stride PS and slot order REV
template <int PS, bool REV>
int launch_flow_iter_ps(ffb_ctx* c, const FlowIterPlan& p, const FfbIterArgs& a, int npairs, int level, double bytes,
                        cudaStream_t stream, bool timed) {
    // compiled in: 256x4x8, 128x2x4, 160x2x4, 96x2x4, 64x2x4 (the round-2 sweeps measured and dropped 192 / 512-thread
    // strips, 8-output tasks on 2-row steps, 4-output tasks on 4-row steps, non-allocating loads, bulk L2 prefetch, early
    // issue of the second row pair, and a barrier-free variant in which neighbouring warps synchronise through
    // shared-memory flags: profiles/r2_sweep_flow_iter.txt)
    switch (p.nt * 100 + p.u * 10 + p.ho) {
        case 25648: return launch_flow_iter_t<256, 4, 2, 8, PS, REV>(c, a, npairs, level, bytes, stream, timed);
        case 12824: return launch_flow_iter_t<128, 2, 4, 4, PS, REV>(c, a, npairs, level, bytes, stream, timed);
        case 16024: return launch_flow_iter_t<160, 2, 3, 4, PS, REV>(c, a, npairs, level, bytes, stream, timed);
        case 9624:  return launch_flow_iter_t<96, 2, 5, 4, PS, REV>(c, a, npairs, level, bytes, stream, timed);
        case 6424:  return launch_flow_iter_t<64, 2, 8, 4, PS, REV>(c, a, npairs, level, bytes, stream, timed);
        default: break;
    }
    return fail(c, FFB_E_INVALID, "FFB_ITER_CFG: no k_flow_iter variant %dx%dx%d (compiled in: 256x4x8, 128x2x4, 160x2x4, 96x2x4, 64x2x4)",
                p.nt, p.u, p.ho);
}

// One k_flow_iter launch of plan `p` on `stream`, counted under pyramid level `level` (-1: none).  timed = false inside
// the sliced flow phase, which is timed as a whole.  pair_stride: 1 (bracket) or 2 (independent pairs); rev: the backward
// flows of the pairs, see k_flow_iter.
int launch_flow_iter(ffb_ctx* c, const FlowIterPlan& p, int level, cudaStream_t stream, bool timed, FfbRing R, size_t plane,
                     int rp, int w, int h, const float2* fin, size_t fin_stride, int fip, FfbRing fout, int fop, int npairs,
                     const UpSrc* up = nullptr, int pair_stride = 1, bool rev = false) {
    FfbIterArgs a;
    a.R = R; a.plane = (int)plane; a.rp = rp; a.w = w; a.h = h;
    a.fin = fin; a.fin_stride = fin_stride; a.fip = fip; a.fout = fout; a.fop = fop;
    a.SW = p.sw; a.SH = p.sh;
    a.up_src = nullptr; a.up_stride = 0; a.usp = a.wc = a.hc = 0;
    double bpp = fin ? 56.0 : 48.0;
    if (up && up->src) {
        a.up_src = up->src; a.up_stride = up->stride; a.usp = up->sp; a.wc = up->wc; a.hc = up->hc;
        a.fin = nullptr;
        bpp = 48.0 + 8.0 * ((double)up->wc * up->hc) / ((double)w * h);
    }
    const double bytes = (double)npairs * bpp * w * h;
    // the kernel stores four flow vectors with one 32-byte instruction
    if (fop % 4 != 0 || ((uintptr_t)fout.base | (uintptr_t)fout.stride) % 32 != 0)
        return fail(c, FFB_E_INVALID, "flow output is not 32-byte aligned (pitch %d, stride %zu)", fop, fout.stride);
    if (pair_stride == 2)
        return rev ? launch_flow_iter_ps<2, true>(c, p, a, npairs, level, bytes, stream, timed)
                   : launch_flow_iter_ps<2, false>(c, p, a, npairs, level, bytes, stream, timed);
    return rev ? launch_flow_iter_ps<1, true>(c, p, a, npairs, level, bytes, stream, timed)
               : launch_flow_iter_ps<1, false>(c, p, a, npairs, level, bytes, stream, timed);
}

// One flow iteration with the context's winsize != 15: k_flow_matrices into the scratch M (npairs x 5 planes), then
// k_box_solve into fout.  Same arguments, counters and output layout as launch_flow_iter.
int launch_flow_unfused(ffb_ctx* c, int level, float* M, FfbRing R, size_t plane, int rp, int w, int h, const float2* fin,
                        size_t fin_stride, int fip, FfbRing fout, int fop, int npairs, int pair_stride = 1, bool rev = false) {
    const int win = c->fb.winsize, r = win / 2;
    if (BOX_NT - 2 * r < 1) return fail(c, FFB_E_INVALID, "winsize %d too large for k_box_solve", win);
    FfbMatrixArgs m;
    m.R = R; m.plane = (int)plane; m.rp = rp; m.w = w; m.h = h;
    m.fin = fin; m.fin_stride = fin_stride; m.fip = fip;
    m.M = M; m.m_stride = 5 * plane;
    // algorithmic bytes: the fused kernel's reads (expansions + incoming flow) plus the matrices written (20 B/px) ...
    const double px = (double)npairs * w * h;
    const ProfMark pm = prof_begin(c, FFB_K_FLOW_ITER, level, px * ((fin ? 48.0 : 40.0) + 20.0), c->s_comp);
    const dim3 mgrid((w + 31) / 32, (h + 7) / 8, npairs);
    auto kfn = pair_stride == 2 ? (rev ? k_flow_matrices<2, true> : k_flow_matrices<2, false>)
                                : (rev ? k_flow_matrices<1, true> : k_flow_matrices<1, false>);
    FFB_LAUNCH(kfn, mgrid, dim3(256), 0, c->s_comp, m);
    prof_end(pm);
    CKL(c);
    FfbBoxArgs b;
    b.M = M; b.m_stride = 5 * plane; b.plane = (int)plane; b.rp = rp; b.w = w; b.h = h;
    b.r = r; b.scale = (float)(1.0 / ((double)win * win));
    b.fout = fout; b.fop = fop;
    b.SW = BOX_NT - 2 * r;
    b.SH = 64;     // 2r rows of every segment are re-read to start its sums
    // ... read back (20 B/px) and the flow written (8 B/px)
    const ProfMark pb = prof_begin(c, FFB_K_FLOW_ITER, level, px * 28.0, c->s_comp);
    FFB_LAUNCH(k_box_solve, dim3(npairs, (w + b.SW - 1) / b.SW, (h + b.SH - 1) / b.SH), dim3(BOX_NT), 0, c->s_comp, b);
    prof_end(pb);
    CKL(c);
    return FFB_OK;
}

// ------------------------------------------------------------------ geometry
// Device / pinned memory comes in four groups with their own lifetimes, so that ffb_configure only
// re-allocates what a request outgrows:
//   frame size   level tables (freed when width or height change, together with everything below)
//   batch        level images, flow ping-pong, expansion ring, frame staging     capacity Bcap frames
//   flow ring    final-flow ring and the reduction partials indexed by ring slot  capacity ring_n pairs
//   pairs        per-pair results and their pinned staging                        capacity pairsCap pairs
void free_batch_group(ffb_ctx* c) {
    for (int l = 0; l < FFB_PLAN_LEVELS; ++l) {
        Level& L = c->lev[l];
        dev_free(L.I); dev_free(L.fA); dev_free(L.fB);
    }
    dev_free(c->R);
    dev_free(c->M);
    dev_free(c->pyr_tmp);
    for (int b = 0; b < 2; ++b) {
        dev_free(c->d_u8[b]);
        if (c->h_pin[b]) cudaFreeHost(c->h_pin[b]);
        c->h_pin[b] = nullptr;
    }
    c->Bcap = 0;
    c->S = 0;
}
void free_ring_group(ffb_ctx* c) {
    dev_free(c->ring); dev_free(c->d_pkey); dev_free(c->d_psum); dev_free(c->d_rpart);
    dev_free(c->ring_bw); dev_free(c->mask_ring);
    c->ring_n = c->bw_n = c->mask_n = 0;
}
void free_pairs_group(ffb_ctx* c) {
    dev_free(c->d_cx); dev_free(c->d_cy); dev_free(c->d_val); dev_free(c->d_mm); dev_free(c->d_cut);
    dev_free(c->d_centers); dev_free(c->d_scalar); dev_free(c->d_cx_ext); dev_free(c->d_cy_ext);
    if (c->h_res) cudaFreeHost(c->h_res);
    c->h_res = nullptr;
    c->pairsCap = 0;
}
void free_geometry(ffb_ctx* c) {
    free_batch_group(c);
    free_ring_group(c);
    free_pairs_group(c);
    dev_free(c->d_ncons);
    c->ncons_cap = 0;
    for (int l = 0; l < FFB_PLAN_LEVELS; ++l) {
        Level& L = c->lev[l];
        dev_free(L.xi); dev_free(L.yi); dev_free(L.uxi); dev_free(L.uyi);
        dev_free(L.xa); dev_free(L.ya); dev_free(L.uxa); dev_free(L.uya);
        dev_free(L.wk);
        L = Level();
    }
    c->W = c->H = c->B = c->maxPairs = c->nlev = c->wide_w = 0;
}

int host_alloc(ffb_ctx* c, void** p, size_t bytes) {
    if (cudaHostAlloc(p, bytes, cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError();
        return fail(c, FFB_E_NOMEM, "cudaHostAlloc(%zu) failed", bytes);
    }
    c->n_host_alloc++;
    return FFB_OK;
}

int build_level_tables(ffb_ctx* c, Level& L, int W, int H, int wc, int hc) {
    std::vector<int> xi, yi;
    std::vector<float> xa, ya;
    make_linear_table(L.w, W, xi, xa);
    make_linear_table(L.h, H, yi, ya);
    pyramid_window(xi, L.w, W, PYR_TW, L.taps.r, &L.RW);
    pyramid_window(yi, L.h, H, PYR_TH, L.taps.r, &L.RH);
    L.wide = pyramid_wide(L.taps.r, L.RW, L.RH);
    if (L.wide) TRY(upload_vec(c, &L.wk, gaussian_half(L.ksize, L.sigma)));
    TRY(upload_vec(c, &L.xi, xi)); TRY(upload_vec(c, &L.xa, xa));
    TRY(upload_vec(c, &L.yi, yi)); TRY(upload_vec(c, &L.ya, ya));
    if (wc > 0) {
        make_linear_table(L.w, wc, xi, xa);
        make_linear_table(L.h, hc, yi, ya);
        TRY(upload_vec(c, &L.uxi, xi)); TRY(upload_vec(c, &L.uxa, xa));
        TRY(upload_vec(c, &L.uyi, yi)); TRY(upload_vec(c, &L.uya, ya));
    }
    return FFB_OK;
}

bool pyramid_fast_ok(int W, int H, const LevelPlan& p);

int quiesce(ffb_ctx* c) {
    CK(c, cudaStreamSynchronize(c->s_comp));
    CK(c, cudaStreamSynchronize(c->s_copy));
    CK(c, cudaStreamSynchronize(c->s_aux));
    CK(c, cudaStreamSynchronize(c->s_out));
    return FFB_OK;
}

// ring_pairs: final flows that must stay resident at once (0 = the streaming minimum, batch + 8)
int configure(ffb_ctx* c, int W, int H, int B, int maxPairs, int ring_pairs = 0) {
    // arguments are checked before anything is touched: a refused call leaves the configuration as it was
    if (W < 16 || H < 16 || B < 1 || maxPairs < 1 || ring_pairs < 0 || (double)W * H >= 4294967295.0)
        return fail(c, FFB_E_INVALID, "ffb_configure: bad geometry %dx%d batch %d pairs %d", W, H, B, maxPairs);
    if (c->in_bracket) return fail(c, FFB_E_INVALID, "ffb_configure inside a bracket");
    const int need_ring = ring_pairs > B + 8 ? ring_pairs : B + 8;
    const bool new_frame = W != c->W || H != c->H;
    if (!new_frame && B <= c->Bcap && need_ring <= c->ring_n && maxPairs <= c->pairsCap) {
        c->B = B;                 // logical limits; the capacities stay
        c->maxPairs = maxPairs;
        return FFB_OK;
    }
    const LevelPlan p = make_plan(W, H, c->fb);
    if (p.n > FFB_PLAN_LEVELS)
        return fail(c, FFB_E_INVALID, "ffb_configure: %dx%d with pyr_scale %g, levels %d plans %d pyramid levels (at most %d)",
                    W, H, c->fb.pyr_scale, c->fb.levels, p.n, FFB_PLAN_LEVELS);
    TRY(quiesce(c));
    if (new_frame) {
        free_geometry(c);
        c->W = W; c->H = H; c->nlev = p.n;
        c->pyr_fast = pyramid_fast_ok(W, H, p);
        size_t off = 0;
        for (int l = 0; l < p.n; ++l) {
            Level& L = c->lev[l];
            L.k = p.k[l]; L.w = p.w[l]; L.h = p.h[l]; L.ksize = p.ksize[l]; L.sigma = p.sigma[l];
            L.rp = ffb_round_up(L.w, 4);
            L.plane = (size_t)L.rp * L.h;
            L.fp = ffb_round_up(L.w, 4);
            L.r_off = off;
            off += 5 * L.plane;
            off = (off + 63) / 64 * 64;
            L.taps = make_taps(L.ksize, L.sigma);
            L.iter = flow_iter_plan(W, H, L.w, L.h, c->iter_cfg);
            // the fused up-sampling doubles the flow: pyr_scale 0.5 only
            L.up2x = l > 0 && c->fb.pyr_scale == 0.5 && L.w == 2 * c->lev[l - 1].w && L.h == 2 * c->lev[l - 1].h;
            TRY(build_level_tables(c, L, W, H, l > 0 ? c->lev[l - 1].w : 0, l > 0 ? c->lev[l - 1].h : 0));
            if (L.wide && L.w > c->wide_w) c->wide_w = L.w;
        }
        c->r_slot_floats = (off + 127) / 128 * 128;      // 512-byte multiples
        c->fp0 = c->lev[p.n - 1].fp;
        c->ring_stride = (size_t)c->fp0 * H;
        // reduction geometry: fixed per frame size so results do not depend on batch composition
        c->div_rpb = 8;       // whole rows per block: long contiguous reads (a column-marching variant measured slower)
        c->div_nblk = (H + c->div_rpb - 1) / c->div_rpb;
        c->rad_gx = (W + 255) / 256;
        c->rad_rpb = 32;
        c->rad_gy = (H + c->rad_rpb - 1) / c->rad_rpb;
    }
    if (B > c->Bcap) {
        free_batch_group(c);
        for (int l = 0; l < c->nlev; ++l) {
            Level& L = c->lev[l];
            TRY(dev_alloc(c, &L.I, (size_t)(B + 1) * L.plane));
            TRY(dev_alloc(c, &L.fA, (size_t)B * L.fp * L.h));
            TRY(dev_alloc(c, &L.fB, (size_t)B * L.fp * L.h));
        }
        c->S = B + 2;      // the first batch of a bracket may carry B + 1 frames (= B pairs)
        TRY(dev_alloc(c, &c->R, (size_t)c->S * c->r_slot_floats));
        if (c->fb.winsize != FFB_WIN) TRY(dev_alloc(c, &c->M, (size_t)B * 5 * c->lev[c->nlev - 1].plane));
        if (c->wide_w > 0) TRY(dev_alloc(c, &c->pyr_tmp, (size_t)(B + 1) * H * c->wide_w));
        const size_t fbytes = (size_t)W * H;
        for (int b = 0; b < 2; ++b) {
            TRY(dev_alloc(c, &c->d_u8[b], (size_t)(B + 1) * fbytes));
            void* hp = nullptr;
            TRY(host_alloc(c, &hp, (size_t)(B + 1) * fbytes));
            c->h_pin[b] = (uint8_t*)hp;
        }
        c->Bcap = B;
    }
    if (need_ring > c->ring_n) {
        free_ring_group(c);
        TRY(dev_alloc(c, &c->ring, (size_t)need_ring * c->ring_stride));
        TRY(dev_alloc(c, &c->d_pkey, (size_t)need_ring * c->div_nblk));
        TRY(dev_alloc(c, &c->d_psum, (size_t)need_ring * c->div_nblk));
        TRY(dev_alloc(c, &c->d_rpart, (size_t)need_ring * c->rad_gx * c->rad_gy));
        c->ring_n = need_ring;
    }
    if (maxPairs > c->pairsCap) {
        free_pairs_group(c);
        const size_t m = (size_t)maxPairs;
        TRY(dev_alloc(c, &c->d_cx, m)); TRY(dev_alloc(c, &c->d_cy, m));
        TRY(dev_alloc(c, &c->d_val, m)); TRY(dev_alloc(c, &c->d_mm, m));
        TRY(dev_alloc(c, &c->d_cut, m));
        TRY(dev_alloc(c, &c->d_centers, 2 * m)); TRY(dev_alloc(c, &c->d_scalar, m));
        TRY(dev_alloc(c, &c->d_cx_ext, m + 12)); TRY(dev_alloc(c, &c->d_cy_ext, m + 12));
        void* hr = nullptr;
        TRY(host_alloc(c, &hr, m * 48 + 256));
        c->h_res = (char*)hr;
        c->pairsCap = maxPairs;
    }
    c->B = B;
    c->maxPairs = maxPairs;
    return FFB_OK;
}

// ------------------------------------------------------------------ the per-batch pipeline
// All levels in one pass when every level is an exact 2^k decimation (W, H multiples of 8).
bool pyramid_fast_ok(int W, int H, const LevelPlan& p) {
    if (W % 8 || H % 8 || W < 64 || H < 64) return false;
    if (p.pyr_scale != 0.5 || p.n > FFB_MAX_LEVELS) return false;
    static const int want[FFB_MAX_LEVELS] = {3, 3, 9, 19};
    for (int l = 0; l < p.n; ++l)
        if (p.ksize[l] != want[p.k[l]] || p.w[l] != (W >> p.k[l]) || p.h[l] != (H >> p.k[l])) return false;
    return true;
}

// dst / dstride / dp are indexed by level k (0 = full resolution)
int launch_pyramid_pow2(ffb_ctx* c, const uint8_t* src, size_t stride, int pitch, int W, int H, int nlev,
                        float* const* dst, const size_t* dstride, const int* dp, int nb) {
    FfbPyr2Args a;
    memset(&a, 0, sizeof(a));
    a.src = src; a.src_frame_stride = stride; a.src_pitch = pitch; a.W = W; a.H = H;
    a.nlev = nlev;
    a.aligned = (pitch % 4 == 0) && (stride % 4 == 0) && (((uintptr_t)src) % 4 == 0);
    static const int ks[FFB_MAX_LEVELS] = {3, 3, 9, 19};
    double px = 0;
    for (int k = 0; k < nlev; ++k) {
        a.dst[k] = dst[k]; a.dstride[k] = dstride[k]; a.dp[k] = dp[k];
        a.taps[k] = make_taps(ks[k], k == 0 ? 0.0 : ((double)(1 << k) - 1.0) * 0.5);
        px += (double)(W >> k) * (H >> k);
    }
    if (!c->attr_pyr2) {
        CK(c, cudaFuncSetAttribute(k_pyramid_pow2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PYR2_SMEM));
        c->attr_pyr2 = true;
    }
    dim3 grid((W + PYR2_TX - 1) / PYR2_TX, (H + PYR2_TY - 1) / PYR2_TY, nb);
    const ProfMark pm = prof_begin(c, FFB_K_PYRAMID, -1, (double)nb * ((double)W * H + 4.0 * px), c->s_comp);
    FFB_LAUNCH(k_pyramid_pow2, grid, dim3(256), PYR2_SMEM, c->s_comp, a);
    prof_end(pm);
    CKL(c);
    return FFB_OK;
}

int expand_frames(ffb_ctx* c, const uint8_t* src, size_t stride, int pitch, int nb, int first_frame) {
    const bool fast = c->pyr_fast;
    if (fast) {
        float* dst[FFB_MAX_LEVELS] = {nullptr, nullptr, nullptr, nullptr};
        size_t dstride[FFB_MAX_LEVELS] = {0, 0, 0, 0};
        int dp[FFB_MAX_LEVELS] = {0, 0, 0, 0};
        for (int l = 0; l < c->nlev; ++l) {
            Level& L = c->lev[l];
            dst[L.k] = L.I; dstride[L.k] = L.plane; dp[L.k] = L.rp;
        }
        TRY(launch_pyramid_pow2(c, src, stride, pitch, c->W, c->H, c->nlev, dst, dstride, dp, nb));
    }
    for (int l = 0; l < c->nlev; ++l) {
        Level& L = c->lev[l];
        if (!fast && L.wide)
            TRY(launch_pyramid_wide(c, src, stride, pitch, c->W, c->H, c->pyr_tmp, L.I, L.plane, L.rp, L.w, L.h, L.xi, L.xa,
                                    L.yi, L.ya, L.wk, L.taps.r, nb));
        else if (!fast)
            TRY(launch_pyramid(c, src, stride, pitch, c->W, c->H, L.I, L.plane, L.rp, L.w, L.h, L.xi, L.xa, L.yi, L.ya,
                               L.taps, L.RW, L.RH, nb));
        FfbRing dst;
        dst.base = (char*)(c->R + L.r_off);
        dst.stride = c->r_slot_floats * sizeof(float);
        dst.first = first_frame % c->S;
        dst.mod = c->S;
        TRY(launch_polyexp(c, L.I, L.plane, L.rp, L.w, L.h, dst, L.plane, L.rp, nb));
    }
    return FFB_OK;
}

// divergence / magnitude partials of `cnt` pairs starting at pair p0 + off of the bracket, on `stream`
int launch_divmag(ffb_ctx* c, int p0, int off, int cnt, cudaStream_t stream) {
    FfbDivArgs d;
    d.flow = FfbRing{(char*)c->ring, c->ring_stride * sizeof(float2), (p0 + off) % c->ring_n, c->ring_n};
    d.fp = c->fp0; d.w = c->W; d.h = c->H; d.rows_per_block = c->div_rpb;
    d.pkey = c->d_pkey + (size_t)off * c->div_nblk;
    d.psum = c->d_psum + (size_t)off * c->div_nblk;
    const ProfMark pm = prof_begin(c, FFB_K_DIVMAG, -1, (double)cnt * 8.0 * c->W * c->H, stream);
    FFB_LAUNCH(k_divmag, dim3(c->div_nblk, 1, cnt), dim3(256), 0, stream, d);
    prof_end(pm);
    CKL(c);
    return FFB_OK;
}

// Final flows of np pairs into final-flow ring slots f0 .. (mod ring_n), and their divergence / magnitude partials
// (divmag = false: flows only).  Pair j reads the expansions in slots r0 + pair_stride * j and the one after it
// (mod S): bracket pairs [p0, p0 + np) are r0 = f0 = p0 with stride 1, a chunk of independent pairs r0 = 0 with
// stride 2.  backward (divmag = false): the flows of the reversed pairs (R0 = the later frame of a bracket pair, `next`
// of an independent pair) into the same slots of the backward final-flow ring.
int flow_pairs(ffb_ctx* c, int r0, int pair_stride, int f0, int np, bool divmag = true, bool backward = false) {
    // The pairs of a batch are split in two slices whose launch chains run on two streams, so that the short
    // coarse-level launches (and the tail of every launch) of one slice overlap the other slice's work (+4 %; 3-4 slices
    // measured no better).  Every buffer is indexed by pair; the slices share nothing that is written.
    // FFB_FLOW_STREAMS=1 keeps one chain, whose launches can be timed one by one.
    // winsize 15: the fused k_flow_iter; any other: k_flow_matrices + k_box_solve through the scratch c->M, whose pairs
    // are those of one launch chain (so the unfused path keeps one chain)
    const bool fused = c->fb.winsize == FFB_WIN;
    bool all_fused = fused;
    for (int l = 1; l < c->nlev; ++l) all_fused = all_fused && c->lev[l].up2x;
    const int nslice = c->flow_streams > 1 && all_fused && np >= 8 ? 2 : 1;
    const bool sliced = nslice > 1;
    const int soff[3] = {0, np / nslice, np};
    const cudaStream_t streams[2] = {c->s_comp, c->s_aux};
    ProfMark phase;
    if (sliced) {
        phase = prof_phase_begin(c);
        CK(c, cudaEventRecord(c->ev_fork, c->s_comp));
        CK(c, cudaStreamWaitEvent(c->s_aux, c->ev_fork, 0));
    }
    // iteration it writes fB (it even) or fA (it odd), the last one of level 0 the final-flow ring instead
    const int iters = c->fb.iterations;
    auto level_out = [&](const Level& X) { return (iters - 1) % 2 == 0 ? X.fB : X.fA; };
    for (int l = 0; l < c->nlev; ++l) {
        Level& L = c->lev[l];
        const size_t fstride = (size_t)L.fp * L.h;
        const bool last = l == c->nlev - 1;
        const bool fuse_up = fused && L.up2x;
        const float2* fin0 = nullptr;
        if (l > 0 && !fuse_up) {
            Level& C = c->lev[l - 1];
            TRY(launch_upsample(c, level_out(C), (size_t)C.fp * C.h, C.fp, C.w, C.h, L.fA, fstride, L.fp, L.w, L.h, L.uxi,
                                L.uxa, L.uyi, L.uya, np));
            fin0 = L.fA;
        }
        for (int it = 0; it < iters; ++it) {
            for (int sl = 0; sl < nslice; ++sl) {
                const int off = soff[sl], cnt = soff[sl + 1] - soff[sl];
                FfbRing R;
                R.base = (char*)(c->R + L.r_off);
                R.stride = c->r_slot_floats * sizeof(float);
                R.first = (r0 + pair_stride * off) % c->S;
                R.mod = c->S;
                FfbRing toB{(char*)(L.fB + (size_t)off * fstride), fstride * sizeof(float2), 0, 1 << 30};
                FfbRing toA{(char*)(L.fA + (size_t)off * fstride), fstride * sizeof(float2), 0, 1 << 30};
                FfbRing toRing{(char*)(backward ? c->ring_bw : c->ring), c->ring_stride * sizeof(float2), (f0 + off) % c->ring_n,
                               c->ring_n};
                UpSrc up;
                if (l > 0 && fuse_up) {
                    Level& C = c->lev[l - 1];
                    up.stride = (size_t)C.fp * C.h;
                    up.src = level_out(C) + (size_t)off * up.stride; up.sp = C.fp; up.wc = C.w; up.hc = C.h;
                }
                // iteration 0 starts from the up-sampled coarser flow (or zero); with the reference's 3 iterations:
                // fB, fB -> fA, fA -> ring | fB
                const float2* fin = it == 0 ? (fin0 ? fin0 + (size_t)off * fstride : nullptr)
                                            : ((it - 1) % 2 == 0 ? L.fB : L.fA) + (size_t)off * fstride;
                const FfbRing& fout = it == iters - 1 && last ? toRing : (it % 2 == 0 ? toB : toA);
                if (fused)
                    TRY(launch_flow_iter(c, L.iter, L.k, streams[sl], !sliced, R, L.plane, L.rp, L.w, L.h, fin, fstride, L.fp,
                                         fout, L.fp, cnt, it == 0 ? &up : nullptr, pair_stride, backward));
                else
                    TRY(launch_flow_unfused(c, L.k, c->M, R, L.plane, L.rp, L.w, L.h, fin, fstride, L.fp, fout, L.fp, cnt,
                                            pair_stride, backward));
            }
        }
    }
    if (sliced) {
        for (int sl = 0; sl < nslice; ++sl) CK(c, cudaEventRecord(c->ev_flow_end[sl], streams[sl]));
        prof_phase_end(c, phase, nslice);
    }
    // each slice reduces its own pairs as soon as its chain is done (overlaps the other slice's tail)
    if (divmag)
        for (int sl = 0; sl < nslice; ++sl) TRY(launch_divmag(c, f0, soff[sl], soff[sl + 1] - soff[sl], streams[sl]));
    if (sliced) {
        CK(c, cudaEventRecord(c->ev_join, c->s_aux));
        CK(c, cudaStreamWaitEvent(c->s_comp, c->ev_join, 0));
    }
    return FFB_OK;
}

// per-pair centre, value, mean magnitude and cut flag of the np pairs in final-flow ring slots f0 .. from their
// divergence / magnitude partials, into the per-pair arrays at out0 ..
int launch_phase1_finish(ffb_ctx* c, int f0, int out0, int np, int pov, float cut_threshold) {
    FfbP1Args f;
    f.flow = FfbRing{(char*)c->ring, c->ring_stride * sizeof(float2), f0 % c->ring_n, c->ring_n};
    f.fp = c->fp0; f.w = c->W; f.h = c->H;
    f.pkey = c->d_pkey; f.psum = c->d_psum; f.nblk = c->div_nblk;
    f.pov = pov; f.cut_threshold = cut_threshold; f.out0 = out0;
    f.cx = c->d_cx; f.cy = c->d_cy; f.val = c->d_val; f.mean_mag = c->d_mm; f.cut = c->d_cut;
    const ProfMark pm = prof_begin(c, FFB_K_SMALL, -1, 0, c->s_comp);
    FFB_LAUNCH(k_phase1_finish, dim3(np), dim3(32), 0, c->s_comp, f);
    prof_end(pm);
    CKL(c);
    return FFB_OK;
}

// k_fb_check of np pairs: forward / backward flows in rings fw / bw (rows fp float2 apart), masks into `mask` (rows mp
// bytes apart; base NULL: no mask), consistent-pixel counts added to count[0 .. np) (NULL: not counted)
int launch_fb_check(ffb_ctx* c, FfbRing fw, FfbRing bw, int fp, int w, int h, FfbRing mask, int mp, unsigned* count,
                    float alpha, float beta, int np) {
    FfbCheckArgs a;
    a.fw = fw; a.bw = bw; a.fp = fp; a.w = w; a.h = h;
    a.mask = mask; a.mp = mp; a.count = count; a.alpha = alpha; a.beta = beta;
    // algorithmic bytes: the forward flow and, per pixel, one backward vector (the 2x2 footprints of neighbouring
    // targets overlap), 8 + 8 B/px, plus the mask byte
    const ProfMark pm = prof_begin(c, FFB_K_FB_CHECK, -1, (double)np * w * h * (mask.base ? 17.0 : 16.0), c->s_comp);
    FFB_LAUNCH(k_fb_check, dim3((w + 31) / 32, (h + 7) / 8, np), dim3(256), 0, c->s_comp, a);
    prof_end(pm);
    CKL(c);
    return FFB_OK;
}

// k_remap_flow of n images (n <= 65535) of w x h pixels of ch bytes: sources at src + i * ss (rows sp bytes apart),
// flows in ring `flow` (rows fp bytes apart), outputs at dst + i * ds (rows dp bytes apart); border 0 constant (value
// bval), 1 replicate
int launch_remap(ffb_ctx* c, const uint8_t* src, size_t ss, size_t sp, FfbRing flow, size_t fp, uint8_t* dst, size_t ds,
                 size_t dp, int w, int h, int ch, int border, int bval, int n) {
    FfbRemapArgs a;
    a.src = src; a.src_stride = ss; a.src_pitch = sp;
    a.flow = flow; a.fp = fp;
    a.dst = dst; a.dst_stride = ds; a.dst_pitch = dp;
    a.w = w; a.h = h; a.border_value = bval;
    a.flow_v8 = ((uintptr_t)flow.base | (n > 1 ? flow.stride : 0) | fp) % 32 == 0;
    a.dst_v4 = ((uintptr_t)dst | dp | (n > 1 ? ds : 0)) % 4 == 0;
    // algorithmic bytes: the flow, the taps counted once (neighbouring outputs share their footprints), the output
    const ProfMark pm = prof_begin(c, FFB_K_REMAP, -1, (double)n * w * h * (8.0 + 2.0 * ch), c->s_comp);
    auto kfn = ch == 1 ? (border ? k_remap_flow<1, true> : k_remap_flow<1, false>)
                       : (border ? k_remap_flow<3, true> : k_remap_flow<3, false>);
    FFB_LAUNCH(kfn, dim3((w + 127) / 128, (h + 7) / 8, n), dim3(256), 0, c->s_comp, a);
    prof_end(pm);
    CKL(c);
    return FFB_OK;
}

// k_radial + k_radial_finish of ring pairs [j0, j0 + cnt) (cnt <= ring_n): d_scalar[j0 ..] from d_centers and d_cut
int launch_radial(ffb_ctx* c, int j0, int cnt, int pov) {
    FfbRadArgs r;
    r.flow = FfbRing{(char*)c->ring, c->ring_stride * sizeof(float2), j0 % c->ring_n, c->ring_n};
    r.fp = c->fp0; r.w = c->W; r.h = c->H; r.rows_per_block = c->rad_rpb;
    r.centers = c->d_centers; r.cut = c->d_cut; r.out0 = j0; r.pov = pov; r.partial = c->d_rpart;
    const ProfMark pm = prof_begin(c, FFB_K_RADIAL, -1, (double)cnt * 8.0 * c->W * c->H, c->s_comp);
    FFB_LAUNCH(k_radial, dim3(c->rad_gx, c->rad_gy, cnt), dim3(256), 0, c->s_comp, r);
    prof_end(pm);
    CKL(c);
    const ProfMark pf = prof_begin(c, FFB_K_SMALL, -1, 0, c->s_comp);
    FFB_LAUNCH(k_radial_finish, dim3(cnt), dim3(32), 0, c->s_comp, (const double*)c->d_rpart, c->rad_gx * c->rad_gy, c->W,
               c->H, j0, c->d_scalar);
    prof_end(pf);
    CKL(c);
    return FFB_OK;
}

// radial pass for bracket pairs [j0, j1); n = number of pairs known so far (window truncation).
// smooth = false: d_centers already holds the centres of these pairs (ffb_bracket_radial)
int radial_range(ffb_ctx* c, int j0, int j1, int n, bool smooth = true) {
    while (j0 < j1) {
        const int cnt = (j1 - j0 < c->ring_n) ? j1 - j0 : c->ring_n;
        if (smooth) {
            const ProfMark pm = prof_begin(c, FFB_K_SMALL, -1, 0, c->s_comp);
            FFB_LAUNCH(k_smooth_centers, dim3((cnt + 127) / 128), dim3(128), 0, c->s_comp, c->d_cx, c->d_cy, n, j0,
                       j0 + cnt, 0, c->d_centers);
            prof_end(pm);
            CKL(c);
        }
        TRY(launch_radial(c, j0, cnt, c->pov));
        j0 += cnt;
    }
    return FFB_OK;
}

// Pageable frames reach the pinned staging buffer through host memcpy: one thread moves ~7 GB/s, less than the
// GPU consumes at 1080p (a 257-frame bracket is 533 MB every 36 ms), so large copies are cut into row ranges and
// moved by kCopyThreads threads (they inherit the caller's CPU affinity, i.e. the NUMA node of the GPU when the
// process was bound to it; one thread: 3 700 pairs/s at 1080p, four: 5 990 -- profiles/r2_host_paths.txt).
// n frames of `rows` rows of `row` bytes each.
constexpr int kCopyThreads = 4;
void copy_frames(uint8_t* dst, size_t dst_frame, const uint8_t* src, size_t src_frame, size_t src_pitch, int n, int rows,
                 size_t row) {
    const long long total_rows = (long long)n * rows;
    auto work = [=](long long r0, long long r1) {
        while (r0 < r1) {
            const int f = (int)(r0 / rows), a = (int)(r0 % rows);
            const int b = (int)((r1 - (long long)f * rows) < rows ? (r1 - (long long)f * rows) : rows);
            const uint8_t* s0 = src + (size_t)f * src_frame + (size_t)a * src_pitch;
            uint8_t* d0 = dst + (size_t)f * dst_frame + (size_t)a * row;
            if (src_pitch == row) memcpy(d0, s0, (size_t)(b - a) * row);
            else for (int y = 0; y < b - a; ++y) memcpy(d0 + (size_t)y * row, s0 + (size_t)y * src_pitch, row);
            r0 += b - a;
        }
    };
    int t = (int)(((size_t)total_rows * row) >> 21);          // at least 2 MB per thread
    if (t > kCopyThreads) t = kCopyThreads;
    if (t <= 1) { work(0, total_rows); return; }
    std::vector<std::thread> pool;
    for (int i = 1; i < t; ++i) pool.emplace_back(work, total_rows * i / t, total_rows * (i + 1) / t);
    work(0, total_rows / t);
    for (std::thread& th : pool) th.join();
}

enum PtrKind { PTR_PAGEABLE, PTR_PINNED, PTR_DEVICE };
// `device`: where a device pointer lives
PtrKind classify(const void* p, int* device = nullptr) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return PTR_PAGEABLE;
    }
    if (device) *device = at.device;
    if (at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged) return PTR_DEVICE;
    if (at.type == cudaMemoryTypeHost) return PTR_PINNED;
    return PTR_PAGEABLE;
}

// Copy on s_copy of n frames (`rows` rows of `row` bytes, `pitch` bytes apart; frames `stride` bytes apart) into the
// device buffer `dst` (frames dst_frame bytes apart; 0: dense), which the kernels before `ev_consumer` read.  Pinned
// and device input is copied directly, pageable input through the pinned staging buffer `pin` (same layout as dst).
// `ev_dma` marks the end of the copy (and so the end of the last DMA out of `pin`); s_comp waits for it.
int upload_frames(ffb_ctx* c, uint8_t* dst, uint8_t* pin, cudaEvent_t ev_dma, cudaEvent_t ev_consumer, const uint8_t* src,
                  PtrKind kind, int n, int rows, size_t row, size_t pitch, size_t stride, size_t dst_frame = 0) {
    const size_t fbytes = row * rows;
    if (dst_frame == 0) dst_frame = fbytes;
    const cudaMemcpyKind dir = kind == PTR_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    CK(c, cudaStreamWaitEvent(c->s_copy, ev_consumer, 0));
    if (kind == PTR_PAGEABLE) {
        CK(c, cudaEventSynchronize(ev_dma));
        copy_frames(pin, dst_frame, src, stride, pitch, n, rows, row);
        if (dst_frame == fbytes) CK(c, cudaMemcpyAsync(dst, pin, (size_t)n * fbytes, cudaMemcpyHostToDevice, c->s_copy));
        else CK(c, cudaMemcpy2DAsync(dst, dst_frame, pin, dst_frame, fbytes, n, cudaMemcpyHostToDevice, c->s_copy));
    } else if (pitch == row && stride == fbytes && dst_frame == fbytes) {
        CK(c, cudaMemcpyAsync(dst, src, (size_t)n * fbytes, dir, c->s_copy));
    } else if (pitch == row && stride >= fbytes) {     // whole frames as the rows of one 2-D copy
        CK(c, cudaMemcpy2DAsync(dst, dst_frame, src, stride, fbytes, n, dir, c->s_copy));
    } else {
        for (int f = 0; f < n; ++f)
            CK(c, cudaMemcpy2DAsync(dst + (size_t)f * dst_frame, row, src + (size_t)f * stride, pitch, row, rows, dir, c->s_copy));
    }
    CK(c, cudaEventRecord(ev_dma, c->s_copy));
    CK(c, cudaStreamWaitEvent(c->s_comp, ev_dma, 0));
    return FFB_OK;
}

// Backward pass of a bidirectional call (ffb_farneback_sequence_bidir, ffb_farneback_pairs_bidir): after the forward
// flows of a batch or chunk, the backward flows into the backward final-flow ring and, with a mask or counts,
// k_fb_check into the mask ring / the per-pair counts.
struct Backward {
    bool mask = false, count = false;
    float alpha = 0.f, beta = 0.f;
};

// The backward pass of np pairs whose forward flows are in final-flow ring slots f0 .. (flow_pairs' r0 / pair_stride /
// f0): their counts go to d_ncons[n0 .. n0 + np).
int backward_pass(ffb_ctx* c, const Backward& bw, int r0, int pair_stride, int f0, int np, int n0) {
    TRY(flow_pairs(c, r0, pair_stride, f0, np, false, true));
    if (!bw.mask && !bw.count) return FFB_OK;
    const size_t fs = c->ring_stride * sizeof(float2), ms = (size_t)c->W * c->H;
    const int s0 = f0 % c->ring_n;
    return launch_fb_check(c, FfbRing{(char*)c->ring, fs, s0, c->ring_n}, FfbRing{(char*)c->ring_bw, fs, s0, c->ring_n},
                           c->fp0, c->W, c->H, FfbRing{bw.mask ? (char*)c->mask_ring : nullptr, ms, s0, c->ring_n}, c->W,
                           bw.count ? c->d_ncons + n0 : nullptr, bw.alpha, bw.beta, np);
}

// One batch of the open bracket (or sequence): upload, expansion, final flows and, with stats, the per-pair results
// and the radial pass lagging 6 pairs.  stats = false computes the flows only (ffb_farneback_sequence without per-pair
// outputs): no k_divmag, phase-1 finish, centre smoothing or radial pass, and max_pairs does not bound the pairs.
// bw: the backward pass of the batch's pairs (stats = false).
int process_batch(ffb_ctx* c, const uint8_t* frames, int nb, size_t pitch, size_t stride, PtrKind kind, bool stats = true,
                  const Backward* bw = nullptr) {
    const int b = c->batch_no & 1;
    const size_t fbytes = (size_t)c->W * c->H;
    const uint8_t* src = frames;
    size_t s_stride = stride;
    int s_pitch = (int)pitch;
    if (kind != PTR_DEVICE) {
        // staging buffer b was last read by the expansion kernels two batches ago
        TRY(upload_frames(c, c->d_u8[b], c->h_pin[b], c->ev_h2d[b], c->ev_expand[b], frames, kind, nb, c->H, (size_t)c->W,
                          pitch, stride));
        src = c->d_u8[b];
        s_stride = fbytes;
        s_pitch = c->W;
    }
    const int g0 = c->frames_seen;
    TRY(expand_frames(c, src, s_stride, s_pitch, nb, g0));
    CK(c, cudaEventRecord(c->ev_expand[b], c->s_comp));
    const int np = nb - (g0 == 0 ? 1 : 0);
    if (np > 0) {
        const int p0 = c->pairs_done;
        if (stats && p0 + np > c->maxPairs) return fail(c, FFB_E_INVALID, "bracket exceeds max_bracket_pairs=%d", c->maxPairs);
        if (c->deferred && p0 + np > c->ring_n)
            return fail(c, FFB_E_INVALID, "shard exceeds the %d pairs announced to ffb_bracket_begin_shard", c->ring_n);
        TRY(flow_pairs(c, p0, 1, p0, np, stats));
        if (stats) TRY(launch_phase1_finish(c, p0, p0, np, c->pov, c->thr));
        if (bw) TRY(backward_pass(c, *bw, p0, 1, p0, np, p0));
        c->pairs_done += np;
        const int r1 = c->pairs_done - 6;
        if (stats && !c->deferred && r1 > c->radial_done) {
            TRY(radial_range(c, c->radial_done, r1, c->pairs_done));
            c->radial_done = r1;
        }
    }
    c->frames_seen += nb;
    c->batch_no++;
    return FFB_OK;
}

int ensure_config(ffb_ctx* c, int w, int h) {
    if (c->W == w && c->H == h && c->B >= 2) return FFB_OK;
    return configure(c, w, h, 2, 64);
}

}  // namespace

namespace {
struct Scratch {   // frees everything it allocated when the hook returns
    std::vector<void*> ptrs;
    ~Scratch() { for (void* p : ptrs) cudaFree(p); }
    template <class T> int alloc(ffb_ctx* c, T** p, size_t n) {
        TRY(dev_alloc(c, p, n));
        ptrs.push_back(*p);
        return FFB_OK;
    }
    template <class T> int upload(ffb_ctx* c, T** p, const T* h, size_t n) {
        TRY(alloc(c, p, n));
        CK(c, cudaMemcpy(*p, h, n * sizeof(T), cudaMemcpyHostToDevice));
        return FFB_OK;
    }
};
}  // namespace

// ------------------------------------------------------------------ frame pre-processing (row N2)
constexpr int PRE_CHUNK = 8;      // colour frames per staging chunk
constexpr int PRE_OUT = 256;

// cv::resize INTER_LINEAR uint8 tables: [x0 | x1 | a0 | a1] (x: weights reset where the footprint
// leaves the image; y: only the indices are clipped) -- see oracle/preproc_np.py.
std::vector<int> make_u8_resize_table(int dst_n, int src_n, bool reset_at_borders) {
    std::vector<int> t(4 * (size_t)dst_n);
    const double scale = (double)src_n / dst_n;
    for (int d = 0; d < dst_n; ++d) {
        float f = (float)((d + 0.5) * scale - 0.5);
        int s0 = (int)floorf(f);
        f -= (float)s0;
        if (reset_at_borders) {
            if (s0 < 0) { s0 = 0; f = 0.f; }
            if (s0 >= src_n - 1) { s0 = src_n - 1; f = 0.f; }
        }
        const int a1 = (int)nearbyintf(f * 2048.f);
        const int a0 = (int)nearbyintf((1.f - f) * 2048.f);
        auto clip = [&](int v) { return v < 0 ? 0 : (v > src_n - 1 ? src_n - 1 : v); };
        t[d] = clip(s0);
        t[dst_n + d] = clip(s0 + 1);
        t[2 * dst_n + d] = a0;
        t[3 * dst_n + d] = a1;
    }
    return t;
}

void free_preprocess(ffb_ctx* c) {
    dev_free(c->pre_xt); dev_free(c->pre_yt);
    for (int b = 0; b < 2; ++b) {
        dev_free(c->d_color[b]);
        if (c->h_color[b]) cudaFreeHost(c->h_color[b]);
        c->h_color[b] = nullptr;
    }
    c->pre = ffb_ctx::PrePlan();
}

// Grow-only pair of ffb_remap_flow staging buffers of at least `bytes` each, on the device or pinned on the host.
static int grow_staging(ffb_ctx* c, uint8_t* (&buf)[2], size_t& cap, size_t bytes, bool pinned) {
    if (bytes <= cap) return FFB_OK;
    for (uint8_t*& p : buf) {
        if (!pinned) dev_free(p);
        else if (p) cudaFreeHost(p);
        p = nullptr;
    }
    cap = 0;
    for (uint8_t*& p : buf) {
        if (pinned) {
            void* hp = nullptr;
            TRY(host_alloc(c, &hp, bytes));
            p = (uint8_t*)hp;
        } else {
            TRY(dev_alloc(c, &p, bytes));
        }
    }
    cap = bytes;
    return FFB_OK;
}

static void free_remap_staging(ffb_ctx* c) {
    for (int b = 0; b < 2; ++b) {
        dev_free(c->rm_src[b]); dev_free(c->rm_flow[b]); dev_free(c->rm_dst[b]);
        if (c->rm_hsrc[b]) cudaFreeHost(c->rm_hsrc[b]);
        if (c->rm_hflow[b]) cudaFreeHost(c->rm_hflow[b]);
        c->rm_hsrc[b] = c->rm_hflow[b] = nullptr;
    }
    c->rm_src_cap = c->rm_flow_cap = c->rm_dst_cap = c->rm_hsrc_cap = c->rm_hflow_cap = 0;
}

int launch_preprocess(ffb_ctx* c, const uint8_t* src, size_t stride, int pitch, uint8_t* dst, const ffb_ctx::PrePlan& p,
                      const int* xt, const int* yt, int n) {
    FfbPreArgs a;
    a.src = src; a.src_frame_stride = stride; a.src_pitch = pitch;
    a.dst = dst; a.dst_frame_stride = (size_t)p.OW * p.OH; a.dst_pitch = p.OW;
    a.xt = xt; a.yt = yt; a.TW = p.TW; a.TH = p.TH; a.x_off = p.x0; a.y_off = p.y0; a.OW = p.OW; a.OH = p.OH;
    // algorithmic bytes: the 2x2 footprint of every output pixel (3 bytes each) + the gray output
    const ProfMark pm = prof_begin(c, FFB_K_PREPROC, -1, (double)n * ((double)p.OW * p.OH * 13.0), c->s_comp);
    FFB_LAUNCH(k_preprocess, dim3((p.OW + 31) / 32, (p.OH + 7) / 8, n), dim3(256), 0, c->s_comp, a);
    prof_end(pm);
    CKL(c);
    return FFB_OK;
}

// the reference's two modes (F:1057, F:1076-1079) as plans
ffb_ctx::PrePlan reference_plan(int W, int H, int vr) {
    ffb_ctx::PrePlan p;
    p.W = W; p.H = H; p.OW = p.OH = PRE_OUT;
    p.TW = p.TH = vr ? 2 * PRE_OUT : PRE_OUT;
    p.x0 = 0; p.y0 = vr ? PRE_OUT : 0;
    return p;
}
bool plan_ok(const ffb_ctx::PrePlan& p) {
    return p.W >= 2 && p.H >= 2 && p.TW >= 1 && p.TH >= 1 && p.OW >= 1 && p.OH >= 1 && p.x0 >= 0 && p.y0 >= 0 &&
           p.x0 + p.OW <= p.TW && p.y0 + p.OH <= p.TH;
}

// ======================================================================================
// extern "C" ABI
// ======================================================================================
extern "C" {

int ffb_version(void) { return FFB_VERSION; }

const char* ffb_kernel_name(int kid) { return kid >= 0 && kid < FFB_K_COUNT ? kKernelNames[kid] : "?"; }

int ffb_device_count(int* n) {
    if (!n) return FFB_E_INVALID;
    int k = 0;
    if (cudaGetDeviceCount(&k) != cudaSuccess) { cudaGetLastError(); k = 0; }
    *n = k;
    return FFB_OK;
}

int ffb_device_pci_bus_id(int device, char* buf, int buf_len) {
    if (!buf || buf_len < 16) return FFB_E_INVALID;
    if (cudaDeviceGetPCIBusId(buf, buf_len, device) != cudaSuccess) { cudaGetLastError(); buf[0] = 0; return FFB_E_NODEVICE; }
    return FFB_OK;
}

int ffb_device_name(int device, char* buf, int buf_len) {
    if (!buf || buf_len < 2) return FFB_E_INVALID;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { cudaGetLastError(); buf[0] = 0; return FFB_E_NODEVICE; }
    snprintf(buf, (size_t)buf_len, "%s", prop.name);
    return FFB_OK;
}

const char* ffb_last_error(const ffb_ctx* c) { return c ? c->err.c_str() : g_create_error.c_str(); }

int ffb_create(int device, ffb_ctx** out) {
    if (!out) return FFB_E_INVALID;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) {
        cudaGetLastError();
        return fail(nullptr, FFB_E_NODEVICE, "no CUDA device available (this library has no CPU fallback)");
    }
    if (device < 0 || device >= n) return fail(nullptr, FFB_E_INVALID, "device %d out of range (0..%d)", device, n - 1);
    ffb_ctx* c = new ffb_ctx();
    c->device = device;
    if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&c->s_comp, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&c->s_copy, cudaStreamNonBlocking) != cudaSuccess) {
        const int rc = fail(nullptr, FFB_E_CUDA, "stream creation failed: %s", cudaGetErrorString(cudaGetLastError()));
        delete c;
        return rc;
    }
    cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&c->ev_chain, cudaEventDisableTiming);
    cudaStreamCreateWithFlags(&c->s_time, cudaStreamNonBlocking);
    for (int i = 0; i < 2; ++i) cudaEventCreateWithFlags(&c->ev_flow_end[i], cudaEventDisableTiming);
    cudaStreamCreateWithFlags(&c->s_aux, cudaStreamNonBlocking);
    cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming);
    cudaStreamCreateWithFlags(&c->s_out, cudaStreamNonBlocking);
    for (cudaEvent_t* e : {&c->ev_fin[0], &c->ev_fin[1], &c->ev_out[0], &c->ev_out[1], &c->ev_user, &c->ev_done,
                           &c->ev_h2d_next[0], &c->ev_h2d_next[1]})
        cudaEventCreateWithFlags(e, cudaEventDisableTiming);
    // FFB_FLOW_STREAMS=1: one launch chain for the flow phase, so that bench.py can time its launches one by one
    if (const char* e = getenv("FFB_FLOW_STREAMS")) c->flow_streams = atoi(e);
    // FFB_ITER_CFG=NTxUxHO forces one k_flow_iter variant on every level (the CPU tests run each variant on small frames)
    if (const char* e = getenv("FFB_ITER_CFG")) {
        int nt = 0, u = 0, ho = 0;
        if (sscanf(e, "%dx%dx%d", &nt, &u, &ho) == 3) { c->iter_cfg.nt = nt; c->iter_cfg.u = u; c->iter_cfg.ho = ho; }
    }
    for (int b = 0; b < 2; ++b) {
        cudaEventCreateWithFlags(&c->ev_h2d[b], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&c->ev_expand[b], cudaEventDisableTiming);
        cudaEventRecord(c->ev_h2d[b], c->s_copy);
        cudaEventRecord(c->ev_expand[b], c->s_comp);
        cudaEventCreateWithFlags(&c->ev_ch2d[b], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&c->ev_pre[b], cudaEventDisableTiming);
        cudaEventRecord(c->ev_ch2d[b], c->s_copy);
        cudaEventRecord(c->ev_pre[b], c->s_comp);
    }
    c->poly5 = make_poly_consts<5>(c->fb.poly_sigma);
    c->poly7 = make_poly_consts<7>(c->fb.poly_sigma);
    *out = c;
    return FFB_OK;
}

void ffb_destroy(ffb_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->s_comp);
    cudaStreamSynchronize(c->s_copy);
    cudaStreamSynchronize(c->s_out);
    prof_collect(c);
    for (cudaEvent_t e : c->ev_pool) cudaEventDestroy(e);
    for (cudaEvent_t e : c->timers) if (e) cudaEventDestroy(e);
    free_geometry(c);
    free_preprocess(c);
    free_remap_staging(c);
    for (int b = 0; b < 2; ++b) {
        cudaEventDestroy(c->ev_h2d[b]); cudaEventDestroy(c->ev_expand[b]);
        cudaEventDestroy(c->ev_ch2d[b]); cudaEventDestroy(c->ev_pre[b]);
    }
    cudaEventDestroy(c->ev_fork);
    cudaEventDestroy(c->ev_chain);
    for (int i = 0; i < 2; ++i) cudaEventDestroy(c->ev_flow_end[i]);
    cudaStreamDestroy(c->s_time);
    cudaEventDestroy(c->ev_join);
    cudaStreamDestroy(c->s_aux);
    for (cudaEvent_t e : {c->ev_fin[0], c->ev_fin[1], c->ev_out[0], c->ev_out[1], c->ev_user, c->ev_done, c->ev_h2d_next[0],
                          c->ev_h2d_next[1]})
        cudaEventDestroy(e);
    cudaStreamDestroy(c->s_out);
    cudaStreamDestroy(c->s_comp);
    cudaStreamDestroy(c->s_copy);
    delete c;
}

int ffb_host_alloc(void** p, size_t bytes) {
    if (!p) return FFB_E_INVALID;
    return cudaHostAlloc(p, bytes, cudaHostAllocDefault) == cudaSuccess ? FFB_OK : FFB_E_NOMEM;
}
int ffb_host_free(void* p) { return cudaFreeHost(p) == cudaSuccess ? FFB_OK : FFB_E_CUDA; }

static int configure_checked(ffb_ctx* c, int w, int h, int batch_frames, int max_pairs, int ring_pairs) {
    if (!c) return FFB_E_INVALID;
    CK(c, cudaSetDevice(c->device));
    const int rc = configure(c, w, h, batch_frames, max_pairs, ring_pairs);
    // an allocation that failed half-way leaves no half-built geometry behind (argument errors change nothing)
    if (rc != FFB_OK && rc != FFB_E_INVALID && !c->in_bracket) {
        const std::string msg = c->err;
        free_geometry(c);
        c->err = msg;
    }
    return rc;
}

int ffb_configure(ffb_ctx* c, int w, int h, int batch_frames, int max_pairs) {
    return configure_checked(c, w, h, batch_frames, max_pairs, 0);
}

// Parameter domain of ffb_set_farneback (include/ffb.h); nothing is touched when a value is outside it.
static int check_farneback(ffb_ctx* c, const FarnebackParams& p, int flags) {
    if (flags & 4) return fail(c, FFB_E_INVALID, "ffb_set_farneback: OPTFLOW_USE_INITIAL_FLOW (4) is not supported");
    if (flags & 256) return fail(c, FFB_E_INVALID, "ffb_set_farneback: OPTFLOW_FARNEBACK_GAUSSIAN (256) is not supported");
    if (flags != 0) return fail(c, FFB_E_INVALID, "ffb_set_farneback: unknown flags %d", flags);
    if (!(p.pyr_scale > 0.0 && p.pyr_scale < 1.0))
        return fail(c, FFB_E_INVALID, "ffb_set_farneback: pyr_scale %g outside (0, 1)", p.pyr_scale);
    if (p.levels < 0) return fail(c, FFB_E_INVALID, "ffb_set_farneback: levels %d < 0", p.levels);
    if (p.winsize < 3 || p.winsize > 63) return fail(c, FFB_E_INVALID, "ffb_set_farneback: winsize %d outside 3 .. 63", p.winsize);
    if (p.iterations < 1 || p.iterations > 20)
        return fail(c, FFB_E_INVALID, "ffb_set_farneback: iterations %d outside 1 .. 20", p.iterations);
    if (p.poly_n != 5 && p.poly_n != 7) return fail(c, FFB_E_INVALID, "ffb_set_farneback: poly_n %d is not 5 or 7", p.poly_n);
    if (!(p.poly_sigma >= 0.0 && isfinite(p.poly_sigma)))
        return fail(c, FFB_E_INVALID, "ffb_set_farneback: poly_sigma %g is not a finite value >= 0", p.poly_sigma);
    return FFB_OK;
}

int ffb_set_farneback(ffb_ctx* c, double pyr_scale, int levels, int winsize, int iterations, int poly_n, double poly_sigma,
                      int flags) {
    if (!c) return FFB_E_INVALID;
    FarnebackParams p;
    p.pyr_scale = pyr_scale; p.levels = levels; p.winsize = winsize; p.iterations = iterations;
    p.poly_n = poly_n; p.poly_sigma = poly_sigma;
    TRY(check_farneback(c, p, flags));
    if (c->in_bracket) return fail(c, FFB_E_INVALID, "ffb_set_farneback inside a bracket");
    if (p == c->fb) return FFB_OK;
    if (c->W > 0) {
        const LevelPlan lp = make_plan(c->W, c->H, p);
        if (lp.n > FFB_PLAN_LEVELS)
            return fail(c, FFB_E_INVALID, "ffb_set_farneback: %dx%d with pyr_scale %g, levels %d plans %d pyramid levels (at most %d)",
                        c->W, c->H, pyr_scale, levels, lp.n, FFB_PLAN_LEVELS);
    }
    CK(c, cudaSetDevice(c->device));
    // re-plan the configured geometry with the same capacities, as a new frame size would
    const int W = c->W, H = c->H, B = c->B, maxPairs = c->maxPairs, Bcap = c->Bcap, pairsCap = c->pairsCap, ring = c->ring_n;
    if (W > 0) {
        TRY(quiesce(c));
        free_geometry(c);
    }
    c->fb = p;
    c->poly5 = make_poly_consts<5>(p.poly_sigma);
    c->poly7 = make_poly_consts<7>(p.poly_sigma);
    if (W > 0) {
        TRY(configure_checked(c, W, H, Bcap, pairsCap, ring));
        c->B = B;
        c->maxPairs = maxPairs;
    }
    return FFB_OK;
}

int ffb_get_farneback(const ffb_ctx* c, double* pyr_scale, int* levels, int* winsize, int* iterations, int* poly_n,
                      double* poly_sigma, int* flags) {
    if (!c) return FFB_E_INVALID;
    if (pyr_scale) *pyr_scale = c->fb.pyr_scale;
    if (levels) *levels = c->fb.levels;
    if (winsize) *winsize = c->fb.winsize;
    if (iterations) *iterations = c->fb.iterations;
    if (poly_n) *poly_n = c->fb.poly_n;
    if (poly_sigma) *poly_sigma = c->fb.poly_sigma;
    if (flags) *flags = 0;
    return FFB_OK;
}

int ffb_get_geometry(const ffb_ctx* c, int* w, int* h, int* batch_frames, int* max_pairs) {
    if (!c) return FFB_E_INVALID;
    if (w) *w = c->W;
    if (h) *h = c->H;
    if (batch_frames) *batch_frames = c->B;
    if (max_pairs) *max_pairs = c->maxPairs;
    return FFB_OK;
}

int ffb_alloc_counts(const ffb_ctx* c, int64_t* device_allocs, int64_t* host_allocs) {
    if (!c) return FFB_E_INVALID;
    if (device_allocs) *device_allocs = c->n_dev_alloc;
    if (host_allocs) *host_allocs = c->n_host_alloc;
    return FFB_OK;
}

int ffb_bracket_begin(ffb_ctx* c, int pov, double thr) {
    if (!c || c->W == 0) return fail(c, FFB_E_INVALID, "ffb_bracket_begin before ffb_configure");
    if (c->in_bracket) return fail(c, FFB_E_INVALID, "ffb_bracket_begin inside a bracket (finish or abort it first)");
    CK(c, cudaSetDevice(c->device));
    c->in_bracket = true;
    c->deferred = false;
    c->phase1_read = false;
    c->pend = 0;
    c->pov = pov ? 1 : 0;
    c->thr = (float)thr;
    c->frames_seen = c->pairs_done = c->radial_done = 0;
    return FFB_OK;
}

int ffb_bracket_begin_shard(ffb_ctx* c, int pov, double thr, int shard_pairs) {
    if (!c || c->W == 0) return fail(c, FFB_E_INVALID, "ffb_bracket_begin_shard before ffb_configure");
    if (c->in_bracket) return fail(c, FFB_E_INVALID, "ffb_bracket_begin_shard inside a bracket (finish or abort it first)");
    if (shard_pairs < 1) return fail(c, FFB_E_INVALID, "ffb_bracket_begin_shard: shard_pairs must be >= 1");
    // every final flow of the shard stays resident until the centres of its neighbours are known
    const int pairs = c->maxPairs > shard_pairs ? c->maxPairs : shard_pairs;
    TRY(configure_checked(c, c->W, c->H, c->B, pairs, shard_pairs));
    TRY(ffb_bracket_begin(c, pov, thr));
    c->deferred = true;
    return FFB_OK;
}

// Frames the next batch of the bracket may take.
static int batch_cap(const ffb_ctx* c, PtrKind kind) {
    // a bracket of k*B pairs has k*B + 1 frames: let its first batch take one frame more
    // so that no degenerate one-frame batch is left over
    if (kind == PTR_DEVICE || c->B < 16) return c->frames_seen == 0 ? c->B + 1 : c->B;
    // Host input: the upload of batch i+1 hides behind the kernels of batch i only while it is not longer than
    // them.  A GPU consumes 1080p frames at ~15 GB/s and receives them at 25 .. 55 GB/s (eight GPUs uploading at
    // once share the host's memory and PCIe roots), so batches may grow by a factor of two, not more: B/4 + 1, B/2,
    // B, B, ...  (with a jump from B/4 + 1 straight to B = 128 the second upload took ~10 ms against 4.4 ms of
    // kernels on an 8-GPU box: end-to-end 0.84 of device-resident; a ramp from B/8 + 1 costs 1.4 % on one GPU because
    // of its small batches -- profiles/r2_scaling.txt).  A 3000-frame bracket pays this ramp once.
    if (c->frames_seen == 0) return c->B / 4 + 1;
    return c->frames_seen <= c->B / 4 + 1 ? c->B / 2 : c->B;
}

// ffb_bracket_push_bgr gathers pre-processed gray frames in the device staging buffer until a batch is full;
// whatever is waiting there runs as a (short) batch before results are read or gray frames are pushed directly
static int flush_pending(ffb_ctx* c) {
    if (c->pend <= 0) return FFB_OK;
    const int nb = c->pend;
    c->pend = 0;
    return process_batch(c, c->d_u8[c->batch_no & 1], nb, (size_t)c->W, (size_t)c->W * c->H, PTR_DEVICE);
}

int ffb_bracket_push(ffb_ctx* c, const uint8_t* frames, int n, size_t pitch, size_t stride) {
    if (!c || !c->in_bracket) return fail(c, FFB_E_INVALID, "ffb_bracket_push outside a bracket");
    CK(c, cudaSetDevice(c->device));      // several contexts (GPUs) may be driven by one host thread
    if (c->phase1_read) return fail(c, FFB_E_INVALID, "ffb_bracket_push after ffb_bracket_phase1_finish");
    if (!frames || n < 0 || pitch < (size_t)c->W || stride < pitch * (size_t)(c->H - 1) + c->W)
        return fail(c, FFB_E_INVALID, "ffb_bracket_push: bad arguments");
    TRY(flush_pending(c));
    const PtrKind kind = classify(frames);
    for (int i = 0; i < n;) {
        const int cap = batch_cap(c, kind);
        const int nb = n - i < cap ? n - i : cap;
        TRY(process_batch(c, frames + (size_t)i * stride, nb, pitch, stride, kind));
        i += nb;
    }
    return FFB_OK;
}

int ffb_bracket_abort(ffb_ctx* c) {
    if (!c) return FFB_E_INVALID;
    if (!c->in_bracket) return FFB_OK;
    cudaSetDevice(c->device);
    // queued work reads the caller's buffers and the staging rings: let it drain (errors are already recorded)
    cudaStreamSynchronize(c->s_copy);
    cudaStreamSynchronize(c->s_comp);
    cudaStreamSynchronize(c->s_aux);
    cudaGetLastError();
    c->in_bracket = false;
    c->deferred = c->phase1_read = false;
    c->pend = 0;
    c->frames_seen = c->pairs_done = c->radial_done = 0;
    return FFB_OK;
}

int ffb_chain_after(ffb_ctx* later, ffb_ctx* earlier) {
    if (!later || !earlier || later == earlier) return FFB_E_INVALID;
    if (later->device != earlier->device) return fail(later, FFB_E_INVALID, "ffb_chain_after: contexts on different devices");
    CK(later, cudaSetDevice(later->device));
    // the kernels `later` queues from now on start after everything `earlier` has queued so far; uploads (s_copy) do not wait
    CK(later, cudaEventRecord(earlier->ev_chain, earlier->s_comp));
    CK(later, cudaStreamWaitEvent(later->s_comp, earlier->ev_chain, 0));
    return FFB_OK;
}

int ffb_sync(ffb_ctx* c) {
    if (!c) return FFB_E_INVALID;
    CK(c, cudaSetDevice(c->device));      // several contexts (GPUs) may be driven by one host thread
    CK(c, cudaStreamSynchronize(c->s_copy));
    CK(c, cudaStreamSynchronize(c->s_comp));
    return FFB_OK;
}

// D2H of the per-pair results of the open bracket (each output may be NULL) through the pinned staging
// buffer, then a wait for both streams.  with_radial: scalar and centers are valid.
static int fetch_results(ffb_ctx* c, int n, bool with_radial, double* scalar, uint8_t* cut, int32_t* cx, int32_t* cy, float* val,
                         float* mean_mag, double* centers) {
    if (n > 0) {
        char* h = c->h_res;
        size_t o = 0;
        double* h_scalar = (double*)(h + o); o += (size_t)n * 8;
        double* h_centers = (double*)(h + o); o += (size_t)n * 16;
        int* h_cx = (int*)(h + o); o += (size_t)n * 4;
        int* h_cy = (int*)(h + o); o += (size_t)n * 4;
        float* h_val = (float*)(h + o); o += (size_t)n * 4;
        float* h_mm = (float*)(h + o); o += (size_t)n * 4;
        unsigned char* h_cut = (unsigned char*)(h + o);
        if (with_radial) {
            CK(c, cudaMemcpyAsync(h_scalar, c->d_scalar, (size_t)n * 8, cudaMemcpyDeviceToHost, c->s_comp));
            CK(c, cudaMemcpyAsync(h_centers, c->d_centers, (size_t)n * 16, cudaMemcpyDeviceToHost, c->s_comp));
        }
        CK(c, cudaMemcpyAsync(h_cx, c->d_cx, (size_t)n * 4, cudaMemcpyDeviceToHost, c->s_comp));
        CK(c, cudaMemcpyAsync(h_cy, c->d_cy, (size_t)n * 4, cudaMemcpyDeviceToHost, c->s_comp));
        CK(c, cudaMemcpyAsync(h_val, c->d_val, (size_t)n * 4, cudaMemcpyDeviceToHost, c->s_comp));
        CK(c, cudaMemcpyAsync(h_mm, c->d_mm, (size_t)n * 4, cudaMemcpyDeviceToHost, c->s_comp));
        CK(c, cudaMemcpyAsync(h_cut, c->d_cut, (size_t)n, cudaMemcpyDeviceToHost, c->s_comp));
        CK(c, cudaStreamSynchronize(c->s_comp));
        if (with_radial && scalar) memcpy(scalar, h_scalar, (size_t)n * 8);
        if (with_radial && centers) memcpy(centers, h_centers, (size_t)n * 16);
        if (cx) memcpy(cx, h_cx, (size_t)n * 4);
        if (cy) memcpy(cy, h_cy, (size_t)n * 4);
        if (val) memcpy(val, h_val, (size_t)n * 4);
        if (mean_mag) memcpy(mean_mag, h_mm, (size_t)n * 4);
        if (cut) memcpy(cut, h_cut, (size_t)n);
    } else {
        CK(c, cudaStreamSynchronize(c->s_comp));
    }
    CK(c, cudaStreamSynchronize(c->s_copy));
    return FFB_OK;
}

int ffb_bracket_finish(ffb_ctx* c, int* n_pairs, double* scalar, uint8_t* cut, int32_t* cx, int32_t* cy, float* val,
                       float* mean_mag, double* centers) {
    if (!c || !c->in_bracket) return fail(c, FFB_E_INVALID, "ffb_bracket_finish outside a bracket");
    CK(c, cudaSetDevice(c->device));      // several contexts (GPUs) may be driven by one host thread
    if (c->deferred) return fail(c, FFB_E_INVALID, "shard bracket: use ffb_bracket_phase1_finish + ffb_bracket_radial");
    TRY(flush_pending(c));
    const int n = c->pairs_done;
    if (n > c->radial_done) {
        TRY(radial_range(c, c->radial_done, n, n));
        c->radial_done = n;
    }
    c->in_bracket = false;
    if (n_pairs) *n_pairs = n;
    return fetch_results(c, n, true, scalar, cut, cx, cy, val, mean_mag, centers);
}

int ffb_bracket_phase1_finish(ffb_ctx* c, int* n_pairs, int32_t* cx, int32_t* cy, float* val, float* mean_mag, uint8_t* cut) {
    if (!c || !c->in_bracket || !c->deferred)
        return fail(c, FFB_E_INVALID, "ffb_bracket_phase1_finish outside a bracket opened with ffb_bracket_begin_shard");
    CK(c, cudaSetDevice(c->device));      // several contexts (GPUs) may be driven by one host thread
    TRY(flush_pending(c));
    c->phase1_read = true;
    if (n_pairs) *n_pairs = c->pairs_done;
    return fetch_results(c, c->pairs_done, false, nullptr, cut, cx, cy, val, mean_mag, nullptr);
}

int ffb_bracket_radial(ffb_ctx* c, const int32_t* cx_ext, const int32_t* cy_ext, int n_ext, int first, double* scalar,
                       double* centers) {
    if (!c || !c->in_bracket || !c->deferred || !c->phase1_read)
        return fail(c, FFB_E_INVALID, "ffb_bracket_radial before ffb_bracket_phase1_finish");
    CK(c, cudaSetDevice(c->device));      // several contexts (GPUs) may be driven by one host thread
    const int n = c->pairs_done;
    if (n > 0 && (!cx_ext || !cy_ext || first < 0 || first > 6 || n_ext < first + n || n_ext > first + n + 6))
        return fail(c, FFB_E_INVALID, "ffb_bracket_radial: %d external centres with the shard's first pair at %d do not frame %d pairs",
                    n_ext, first, n);
    if (n > 0) {
        // the raw centres of the shard and of up to 6 neighbours on each side, as the neighbours computed them
        CK(c, cudaMemcpyAsync(c->d_cx_ext, cx_ext, (size_t)n_ext * 4, cudaMemcpyHostToDevice, c->s_comp));
        CK(c, cudaMemcpyAsync(c->d_cy_ext, cy_ext, (size_t)n_ext * 4, cudaMemcpyHostToDevice, c->s_comp));
        const ProfMark pm = prof_begin(c, FFB_K_SMALL, -1, 0, c->s_comp);
        FFB_LAUNCH(k_smooth_centers, dim3((n + 127) / 128), dim3(128), 0, c->s_comp, c->d_cx_ext, c->d_cy_ext, n_ext, first,
                   first + n, first, c->d_centers);
        prof_end(pm);
        CKL(c);
        TRY(radial_range(c, 0, n, n, false));
        c->radial_done = n;
    }
    c->in_bracket = false;
    c->deferred = c->phase1_read = false;
    return fetch_results(c, n, true, scalar, nullptr, nullptr, nullptr, nullptr, nullptr, centers);
}

int ffb_flow_ring_size(const ffb_ctx* c) { return c ? c->ring_n : 0; }

int ffb_bracket_get_flow(ffb_ctx* c, int pair, float* out) {
    if (!c || !out || c->W == 0) return FFB_E_INVALID;
    CK(c, cudaSetDevice(c->device));      // several contexts (GPUs) may be driven by one host thread
    if (pair < 0 || pair >= c->pairs_done || pair < c->pairs_done - c->ring_n)
        return fail(c, FFB_E_RANGE, "flow of pair %d is not resident (pairs %d, ring %d)", pair, c->pairs_done, c->ring_n);
    CK(c, cudaStreamSynchronize(c->s_comp));
    const float2* src = c->ring + (size_t)(pair % c->ring_n) * c->ring_stride;
    CK(c, cudaMemcpy2D(out, (size_t)c->W * 8, src, (size_t)c->fp0 * 8, (size_t)c->W * 8, c->H, cudaMemcpyDeviceToHost));
    return FFB_OK;
}

// ---- per-call functions ------------------------------------------------------------------
int ffb_farneback(ffb_ctx* c, const uint8_t* prev, const uint8_t* next, int w, int h, size_t pitch, float* flow) {
    if (!c || !prev || !next || !flow) return FFB_E_INVALID;
    CK(c, cudaSetDevice(c->device));
    TRY(ensure_config(c, w, h));
    TRY(ffb_bracket_begin(c, 0, std::numeric_limits<float>::infinity()));
    TRY(ffb_bracket_push(c, prev, 1, pitch, pitch * h));
    TRY(ffb_bracket_push(c, next, 1, pitch, pitch * h));
    int n = 0;
    TRY(ffb_bracket_finish(c, &n, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr));
    return ffb_bracket_get_flow(c, 0, flow);
}

// Per-pair images in the slots of a ring (the final-flow rings, the mask ring, ffb_remap_flow's output staging): slot s
// at base + s * slot bytes, `rows` rows of `row` bytes, pitch bytes apart, with slot == rows * pitch.
struct SlotImages { const char* base; size_t slot, pitch, row; int rows; };
static SlotImages flow_slots(const ffb_ctx* c, const float2* ring) {
    return SlotImages{(const char*)ring, c->ring_stride * sizeof(float2), (size_t)c->fp0 * 8, (size_t)c->W * 8, c->H};
}
static SlotImages mask_slots(const ffb_ctx* c) {
    return SlotImages{(const char*)c->mask_ring, (size_t)c->W * c->H, (size_t)c->W, (size_t)c->W, c->H};
}

// Copy on s_out of the images in ring slots s0 .. s0 + np - 1 (no wrap) to `dst`: images `stride` bytes apart, rows
// `pitch` bytes apart, in host memory or on the device (`kind`).
static int copy_slots_out(ffb_ctx* c, const SlotImages& r, int s0, int np, char* dst, size_t pitch, size_t stride,
                          PtrKind kind) {
    const cudaMemcpyKind dir = kind == PTR_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
    const char* src = r.base + (size_t)s0 * r.slot;
    if (stride == pitch * r.rows)     // the pairs' rows are evenly spaced on both sides
        CK(c, cudaMemcpy2DAsync(dst, pitch, src, r.pitch, r.row, (size_t)np * r.rows, dir, c->s_out));
    else
        for (int j = 0; j < np; ++j)
            CK(c, cudaMemcpy2DAsync(dst + (size_t)j * stride, pitch, src + (size_t)j * r.slot, r.pitch, r.row, r.rows, dir,
                                    c->s_out));
    return FFB_OK;
}

// Kind of memory of a caller's buffer (PTR_DEVICE for NULL); device memory must be on the context's device.  `what`
// names the buffer with its verb ("frames are", "flow is") for the message.
static int buffer_kind(ffb_ctx* c, const char* fn, const char* what, const void* p, PtrKind* kind) {
    int dev = c->device;
    *kind = p ? classify(p, &dev) : PTR_DEVICE;
    if (*kind == PTR_DEVICE && dev != c->device)
        return fail(c, FFB_E_INVALID, "%s: %s on device %d, the context on device %d", fn, what, dev, c->device);
    return FFB_OK;
}

// Outputs of a pairs or sequence call that leave the final-flow rings (each may be NULL) and the memory each is in.
struct RingOut {
    float *flow = nullptr, *flow_bw = nullptr;
    size_t flow_pitch = 0, flow_stride = 0;
    uint8_t* mask = nullptr;
    size_t mask_pitch = 0, mask_stride = 0;
    PtrKind kf = PTR_DEVICE, kb = PTR_DEVICE, km = PTR_DEVICE;
    bool any() const { return flow || flow_bw || mask; }
};

// Copy on s_out of ring slots s .. s + m - 1 (no wrap) of every output of `o` to pairs i .. i + m - 1 of its buffer.
static int copy_outputs(ffb_ctx* c, const RingOut& o, int s, int m, int i) {
    if (o.flow)
        TRY(copy_slots_out(c, flow_slots(c, c->ring), s, m, (char*)o.flow + (size_t)i * o.flow_stride, o.flow_pitch,
                           o.flow_stride, o.kf));
    if (o.flow_bw)
        TRY(copy_slots_out(c, flow_slots(c, c->ring_bw), s, m, (char*)o.flow_bw + (size_t)i * o.flow_stride, o.flow_pitch,
                           o.flow_stride, o.kb));
    if (o.mask)
        TRY(copy_slots_out(c, mask_slots(c), s, m, (char*)o.mask + (size_t)i * o.mask_stride, o.mask_pitch, o.mask_stride,
                           o.km));
    return FFB_OK;
}

// The mask and check arguments of a bidirectional call (fn: its name in the messages) of n_pairs >= 1 pairs.
static int check_bidir_args(ffb_ctx* c, const char* fn, int n_pairs, int width, int height, const uint8_t* mask,
                            size_t mask_pitch, size_t mask_stride, double alpha, double beta) {
    if (mask && mask_pitch < (size_t)width)
        return fail(c, FFB_E_INVALID, "%s: mask_pitch %zu below the width %d", fn, mask_pitch, width);
    if (mask && n_pairs > 1 && mask_stride < mask_pitch * (size_t)(height - 1) + width)
        return fail(c, FFB_E_INVALID, "%s: mask_stride %zu shorter than a mask", fn, mask_stride);
    if (!(alpha >= 0.0 && isfinite(alpha)) || !(beta >= 0.0 && isfinite(beta)))
        return fail(c, FFB_E_INVALID, "%s: alpha %g and beta %g must be finite and >= 0", fn, alpha, beta);
    return FFB_OK;
}

// The backward ring (flows), the mask ring (mask) and n_counts per-pair counts of a bidirectional call: grow-only,
// allocated by the first call that needs them (a new frame size or a larger final-flow ring frees the rings).
static int alloc_backward(ffb_ctx* c, bool flows, bool mask, int n_counts) {
    if (flows && c->bw_n < c->ring_n) {
        dev_free(c->ring_bw);
        c->bw_n = 0;
        TRY(dev_alloc(c, &c->ring_bw, (size_t)c->ring_n * c->ring_stride));
        c->bw_n = c->ring_n;
    }
    if (mask && c->mask_n < c->ring_n) {
        dev_free(c->mask_ring);
        c->mask_n = 0;
        TRY(dev_alloc(c, &c->mask_ring, (size_t)c->ring_n * c->W * c->H));
        c->mask_n = c->ring_n;
    }
    if (c->ncons_cap < n_counts) {
        dev_free(c->d_ncons);
        c->ncons_cap = 0;
        TRY(dev_alloc(c, &c->d_ncons, (size_t)n_counts));
        c->ncons_cap = n_counts;
    }
    return FFB_OK;
}

// End of a bidirectional call of n_pairs pairs (host_in: frames in host memory): with a caller stream and every buffer
// on the device it returns at once, otherwise when the outputs are complete, with the counts copied out.
static int finish_bidir(ffb_ctx* c, const RingOut& o, bool host_in, int n_pairs, int64_t* n_consistent, void* stream) {
    const bool host_io = host_in || o.kf != PTR_DEVICE || o.kb != PTR_DEVICE || o.km != PTR_DEVICE || n_consistent;
    if (stream && !host_io) return FFB_OK;
    CK(c, cudaStreamSynchronize(c->s_comp));
    if (n_consistent) {
        std::vector<unsigned> h((size_t)n_pairs);
        CK(c, cudaMemcpy(h.data(), c->d_ncons, (size_t)n_pairs * sizeof(unsigned), cudaMemcpyDeviceToHost));
        for (int j = 0; j < n_pairs; ++j) n_consistent[j] = h[j];
    }
    return FFB_OK;
}

// The frame and flow arguments of an independent-pairs call (fn: its name in the messages), n_pairs >= 1.
static int check_pairs_args(ffb_ctx* c, const char* fn, const uint8_t* prev, const uint8_t* next, int n_pairs, int width,
                            int height, size_t pitch, size_t frame_stride, bool flow, size_t flow_pitch, size_t flow_stride) {
    if (!prev || !next || width < 1 || height < 1) return fail(c, FFB_E_INVALID, "%s: bad frames (%dx%d)", fn, width, height);
    if (pitch < (size_t)width) return fail(c, FFB_E_INVALID, "%s: pitch %zu below the width %d", fn, pitch, width);
    if (n_pairs > 1 && frame_stride < pitch * (size_t)(height - 1) + width)
        return fail(c, FFB_E_INVALID, "%s: frame_stride %zu shorter than a frame", fn, frame_stride);
    if (flow && flow_pitch < (size_t)width * 8)
        return fail(c, FFB_E_INVALID, "%s: flow_pitch %zu below 8 * width (%d)", fn, flow_pitch, 8 * width);
    if (flow && n_pairs > 1 && flow_stride < flow_pitch * (size_t)(height - 1) + (size_t)width * 8)
        return fail(c, FFB_E_INVALID, "%s: flow_stride %zu shorter than a flow", fn, flow_stride);
    return FFB_OK;
}

// Independent pairs: chunks of P = (B + 1) / 2 pairs.  A chunk stages its 2P frames as prev_0, next_0, prev_1, ... in
// the frame staging buffer and expands them into expansion slots 0 .. 2P-1; the flow phase reads them with pair stride
// 2, and with `bw` the backward pass reads them again in reverse slot order.  Consecutive chunks alternate between the
// slots [0, P) and [P, 2P) of the final-flow ring (ring_n >= B + 8 > 2P) and of the backward and mask rings, so the
// copy-out of one chunk on s_out overlaps the next chunk's kernels.  divmag: k_divmag after the forward flows; stats:
// also the per-pair results (pov, thr) into the per-pair arrays.  The geometry is configured by the caller; at the end
// the caller's stream waits for the call.
static int pairs_loop(ffb_ctx* c, const uint8_t* prev, const uint8_t* next, int n_pairs, size_t pitch, size_t frame_stride,
                      PtrKind kp, PtrKind kn, const RingOut& o, bool divmag, bool stats, int pov, float thr,
                      const Backward* bw, void* stream) {
    const int P = (c->B + 1) / 2;
    const int width = c->W, height = c->H;
    const size_t fbytes = (size_t)width * height;
    const bool copy = o.any();
    const cudaStream_t us = (cudaStream_t)stream;
    c->pairs_done = 0;   // the final-flow ring no longer holds a bracket's flows
    CK(c, cudaEventRecord(c->ev_user, us));
    CK(c, cudaStreamWaitEvent(c->s_copy, c->ev_user, 0));
    CK(c, cudaStreamWaitEvent(c->s_comp, c->ev_user, 0));
    if (bw && bw->count) CK(c, cudaMemsetAsync(c->d_ncons, 0, (size_t)n_pairs * sizeof(unsigned), c->s_comp));
    // outputs of pairs [i0, i0 + np) from ring half `half` to the caller's buffers
    auto copy_out = [&](int i0, int np, int half) -> int {
        CK(c, cudaStreamWaitEvent(c->s_out, c->ev_fin[half], 0));
        TRY(copy_outputs(c, o, half * P, np, i0));
        CK(c, cudaEventRecord(c->ev_out[half], c->s_out));
        return FFB_OK;
    };
    int pend_i0 = -1, pend_np = 0, pend_half = 0;   // chunk whose copy-out has not been issued yet
    for (int i0 = 0, k = 0; i0 < n_pairs; i0 += P, ++k) {
        const int np = n_pairs - i0 < P ? n_pairs - i0 : P, half = k & 1, b = c->batch_no & 1;
        const size_t off = (size_t)i0 * frame_stride;
        TRY(upload_frames(c, c->d_u8[b], c->h_pin[b], c->ev_h2d[b], c->ev_expand[b], prev + off, kp, np, height,
                          (size_t)width, pitch, frame_stride, 2 * fbytes));
        TRY(upload_frames(c, c->d_u8[b] + fbytes, c->h_pin[b] + fbytes, c->ev_h2d_next[b], c->ev_expand[b], next + off, kn, np,
                          height, (size_t)width, pitch, frame_stride, 2 * fbytes));
        TRY(expand_frames(c, c->d_u8[b], fbytes, width, 2 * np, 0));
        CK(c, cudaEventRecord(c->ev_expand[b], c->s_comp));
        c->batch_no++;
        // ring half `half` is free once the copy-out of chunk k - 2 (or of an earlier call) has read it
        CK(c, cudaStreamWaitEvent(c->s_comp, c->ev_out[half], 0));
        TRY(flow_pairs(c, 0, 2, half * P, np, divmag));
        if (stats) TRY(launch_phase1_finish(c, half * P, i0, np, pov, thr));
        if (bw) TRY(backward_pass(c, *bw, 0, 2, half * P, np, i0));
        if (!copy) continue;
        CK(c, cudaEventRecord(c->ev_fin[half], c->s_comp));
        // issued one chunk late: a copy into pageable memory returns only when it is done
        if (pend_i0 >= 0) TRY(copy_out(pend_i0, pend_np, pend_half));
        pend_i0 = i0; pend_np = np; pend_half = half;
    }
    if (pend_i0 >= 0) TRY(copy_out(pend_i0, pend_np, pend_half));
    if (copy) {   // later work of the context (a bracket, the next call) overwrites the rings after the copy-out
        CK(c, cudaEventRecord(c->ev_done, c->s_out));
        CK(c, cudaStreamWaitEvent(c->s_comp, c->ev_done, 0));
    }
    // s_comp has waited for every upload and copy-out: the caller's stream continues when the inputs have been read
    // and the outputs written
    CK(c, cudaEventRecord(c->ev_done, c->s_comp));
    CK(c, cudaStreamWaitEvent(us, c->ev_done, 0));
    return FFB_OK;
}

int ffb_farneback_pairs(ffb_ctx* c, const uint8_t* prev, const uint8_t* next, int n_pairs, int width, int height,
                        size_t pitch, size_t frame_stride, float* flow, size_t flow_pitch, size_t flow_stride,
                        int pov_mode, double cut_threshold, int32_t* cx, int32_t* cy, float* val, float* mean_mag,
                        uint8_t* cut, void* stream) {
    static const char* fn = "ffb_farneback_pairs";
    if (!c) return FFB_E_INVALID;
    if (c->in_bracket) return fail(c, FFB_E_INVALID, "ffb_farneback_pairs inside a bracket");
    if (n_pairs < 0) return fail(c, FFB_E_INVALID, "ffb_farneback_pairs: n_pairs %d < 0", n_pairs);
    if (n_pairs == 0) return FFB_OK;
    TRY(check_pairs_args(c, fn, prev, next, n_pairs, width, height, pitch, frame_stride, flow, flow_pitch, flow_stride));
    CK(c, cudaSetDevice(c->device));
    PtrKind kp, kn;
    RingOut o;
    o.flow = flow; o.flow_pitch = flow_pitch; o.flow_stride = flow_stride;
    TRY(buffer_kind(c, fn, "prev is", prev, &kp));
    TRY(buffer_kind(c, fn, "next is", next, &kn));
    TRY(buffer_kind(c, fn, "flow is", flow, &o.kf));
    const bool stats = cx || cy || val || mean_mag || cut;
    // the per-pair results of the whole call stay on the device until the end: max_pairs covers n_pairs
    const int maxPairs = stats && n_pairs > c->maxPairs ? n_pairs : (c->maxPairs > 0 ? c->maxPairs : 1);
    TRY(configure_checked(c, width, height, c->B > 0 ? c->B : 2, maxPairs, 0));
    TRY(pairs_loop(c, prev, next, n_pairs, pitch, frame_stride, kp, kn, o, true, stats, pov_mode ? 1 : 0,
                   (float)cut_threshold, nullptr, stream));
    const bool host_io = kp != PTR_DEVICE || kn != PTR_DEVICE || o.kf != PTR_DEVICE || stats;
    if (stream && !host_io) return FFB_OK;
    if (stats) return fetch_results(c, n_pairs, false, nullptr, cut, cx, cy, val, mean_mag, nullptr);
    CK(c, cudaStreamSynchronize(c->s_comp));
    return FFB_OK;
}

// Independent pairs with the backward flow of every pair as well: after the forward flows of a chunk (no k_divmag: there
// are no per-pair results), a second flow_pairs with the slot order reversed (R0 = next_i, R1 = prev_i, the chunk's
// expansions still in their slots) into the backward final-flow ring, then k_fb_check of the chunk into the mask ring
// and the per-pair counts.  The three rings share their slots, and the fences of ffb_farneback_pairs cover the three
// copy-outs of a chunk.
int ffb_farneback_pairs_bidir(ffb_ctx* c, const uint8_t* prev, const uint8_t* next, int n_pairs, int width, int height,
                              size_t pitch, size_t frame_stride, float* flow_fw, float* flow_bw, size_t flow_pitch,
                              size_t flow_stride, uint8_t* mask, size_t mask_pitch, size_t mask_stride, double alpha,
                              double beta, int64_t* n_consistent, void* stream) {
    static const char* fn = "ffb_farneback_pairs_bidir";
    if (!c) return FFB_E_INVALID;
    if (c->in_bracket) return fail(c, FFB_E_INVALID, "ffb_farneback_pairs_bidir inside a bracket");
    if (n_pairs < 0) return fail(c, FFB_E_INVALID, "ffb_farneback_pairs_bidir: n_pairs %d < 0", n_pairs);
    if (n_pairs == 0) return FFB_OK;
    TRY(check_pairs_args(c, fn, prev, next, n_pairs, width, height, pitch, frame_stride, flow_fw || flow_bw, flow_pitch,
                         flow_stride));
    TRY(check_bidir_args(c, fn, n_pairs, width, height, mask, mask_pitch, mask_stride, alpha, beta));
    CK(c, cudaSetDevice(c->device));
    PtrKind kp, kn;
    RingOut o;
    o.flow = flow_fw; o.flow_bw = flow_bw; o.flow_pitch = flow_pitch; o.flow_stride = flow_stride;
    o.mask = mask; o.mask_pitch = mask_pitch; o.mask_stride = mask_stride;
    TRY(buffer_kind(c, fn, "prev is", prev, &kp));
    TRY(buffer_kind(c, fn, "next is", next, &kn));
    TRY(buffer_kind(c, fn, "flow_fw is", flow_fw, &o.kf));
    TRY(buffer_kind(c, fn, "flow_bw is", flow_bw, &o.kb));
    TRY(buffer_kind(c, fn, "mask is", mask, &o.km));
    TRY(configure_checked(c, width, height, c->B > 0 ? c->B : 2, c->maxPairs > 0 ? c->maxPairs : 1, 0));
    const bool backward = flow_bw || mask || n_consistent;
    TRY(alloc_backward(c, backward, mask != nullptr, n_consistent ? n_pairs : 0));
    Backward bw;
    bw.mask = mask != nullptr;
    bw.count = n_consistent != nullptr;
    bw.alpha = (float)alpha;
    bw.beta = (float)beta;
    TRY(pairs_loop(c, prev, next, n_pairs, pitch, frame_stride, kp, kn, o, false, false, 0, 0.f, backward ? &bw : nullptr,
                   stream));
    return finish_bidir(c, o, kp != PTR_DEVICE || kn != PTR_DEVICE, n_pairs, n_consistent, stream);
}

// The frame and flow arguments of a sequence call (fn: its name in the messages), n_frames >= 2.
static int check_sequence_args(ffb_ctx* c, const char* fn, const uint8_t* frames, int n_frames, int width, int height,
                               size_t pitch, size_t frame_stride, bool flow, size_t flow_pitch, size_t flow_stride) {
    if (!frames || width < 1 || height < 1) return fail(c, FFB_E_INVALID, "%s: bad frames (%dx%d)", fn, width, height);
    if (pitch < (size_t)width) return fail(c, FFB_E_INVALID, "%s: pitch %zu below the width %d", fn, pitch, width);
    if (frame_stride < pitch * (size_t)(height - 1) + width)
        return fail(c, FFB_E_INVALID, "%s: frame_stride %zu shorter than a frame", fn, frame_stride);
    if (flow && flow_pitch < (size_t)width * 8)
        return fail(c, FFB_E_INVALID, "%s: flow_pitch %zu below 8 * width (%d)", fn, flow_pitch, 8 * width);
    if (flow && n_frames > 2 && flow_stride < flow_pitch * (size_t)(height - 1) + (size_t)width * 8)
        return fail(c, FFB_E_INVALID, "%s: flow_stride %zu shorter than a flow", fn, flow_stride);
    return FFB_OK;
}

// Consecutive pairs of a sequence: one bracket over the n_frames frames (the batches of ffb_bracket_push, with the
// ramp for host input; every frame expanded once; flow_pairs with pair stride 1), whose final flows -- and with `bw` the
// backward flows and masks in the same slots of their rings -- are also copied out.  Pair p sits in ring slot
// p mod ring_n, and the copy-out of batch k on s_out is issued after batch k + 1 has been queued, so it overlaps that
// batch's kernels.  With ring_n >= 2B + 8, batch k + 1 (at most B pairs) writes no slot of batch k (at most B) nor of
// the 6 pairs before it that its radial pass still reads; the slots it does overwrite held batch k - 1 or earlier, so
// it waits for the copy-out of batch k - 1 (ev_out[(k + 1) & 1]).  The radial pass runs on s_comp, in order with every
// later write.  The geometry is configured by the caller; at the end the caller's stream waits for the call.
static int sequence_loop(ffb_ctx* c, const uint8_t* frames, int n_frames, size_t pitch, size_t frame_stride, PtrKind kfr,
                         const RingOut& o, bool stats, const Backward* bw, void* stream) {
    const int n_pairs = n_frames - 1;
    const bool copy = o.any();
    const cudaStream_t us = (cudaStream_t)stream;
    // ffb_bracket_begin's state; the final-flow ring no longer holds an earlier bracket's flows
    c->deferred = c->phase1_read = false;
    c->pend = 0;
    c->frames_seen = c->pairs_done = c->radial_done = 0;
    CK(c, cudaEventRecord(c->ev_user, us));
    CK(c, cudaStreamWaitEvent(c->s_copy, c->ev_user, 0));
    CK(c, cudaStreamWaitEvent(c->s_comp, c->ev_user, 0));
    if (bw && bw->count) CK(c, cudaMemsetAsync(c->d_ncons, 0, (size_t)n_pairs * sizeof(unsigned), c->s_comp));
    // outputs of pairs [p0, p0 + np) of batch parity `par` to the caller's buffers: one or two runs of ring slots each
    auto copy_out = [&](int p0, int np, int par) -> int {
        CK(c, cudaStreamWaitEvent(c->s_out, c->ev_fin[par], 0));
        for (int p = p0; p < p0 + np;) {
            const int s = p % c->ring_n, m = p0 + np - p < c->ring_n - s ? p0 + np - p : c->ring_n - s;
            TRY(copy_outputs(c, o, s, m, p));
            p += m;
        }
        CK(c, cudaEventRecord(c->ev_out[par], c->s_out));
        return FFB_OK;
    };
    int k = 0, pend_p0 = 0, pend_np = 0;   // batch k - 1, whose copy-out has not been issued yet
    for (int i = 0; i < n_frames; ++k) {
        const int cap = batch_cap(c, kfr);
        const int nb = n_frames - i < cap ? n_frames - i : cap;
        const int p0 = c->pairs_done;
        if (copy) CK(c, cudaStreamWaitEvent(c->s_comp, c->ev_out[k & 1], 0));   // copy-out of batch k - 2 done
        TRY(process_batch(c, frames + (size_t)i * frame_stride, nb, pitch, frame_stride, kfr, stats, bw));
        i += nb;
        if (!copy) continue;
        CK(c, cudaEventRecord(c->ev_fin[k & 1], c->s_comp));
        // issued one batch late: a copy into pageable memory returns only when it is done
        if (pend_np > 0) TRY(copy_out(pend_p0, pend_np, (k - 1) & 1));
        pend_p0 = p0;
        pend_np = c->pairs_done - p0;
    }
    if (stats && n_pairs > c->radial_done) TRY(radial_range(c, c->radial_done, n_pairs, n_pairs));
    if (pend_np > 0) TRY(copy_out(pend_p0, pend_np, (k - 1) & 1));
    c->frames_seen = c->pairs_done = c->radial_done = 0;
    if (copy) {   // later work of the context (a bracket, the next call) overwrites the rings after the copy-out
        CK(c, cudaEventRecord(c->ev_done, c->s_out));
        CK(c, cudaStreamWaitEvent(c->s_comp, c->ev_done, 0));
    }
    // s_comp has waited for every upload and copy-out: the caller's stream continues when the inputs have been read
    // and the outputs written
    CK(c, cudaEventRecord(c->ev_done, c->s_comp));
    CK(c, cudaStreamWaitEvent(us, c->ev_done, 0));
    return FFB_OK;
}

int ffb_farneback_sequence(ffb_ctx* c, const uint8_t* frames, int n_frames, int width, int height, size_t pitch,
                           size_t frame_stride, float* flow, size_t flow_pitch, size_t flow_stride, int pov_mode,
                           double cut_threshold, double* scalar, uint8_t* cut, int32_t* cx, int32_t* cy, float* val,
                           float* mean_mag, double* centers, void* stream) {
    static const char* fn = "ffb_farneback_sequence";
    if (!c) return FFB_E_INVALID;
    if (c->in_bracket) return fail(c, FFB_E_INVALID, "ffb_farneback_sequence inside a bracket");
    if (n_frames < 0) return fail(c, FFB_E_INVALID, "ffb_farneback_sequence: n_frames %d < 0", n_frames);
    if (n_frames < 2) return FFB_OK;
    const int n_pairs = n_frames - 1;
    TRY(check_sequence_args(c, fn, frames, n_frames, width, height, pitch, frame_stride, flow, flow_pitch, flow_stride));
    CK(c, cudaSetDevice(c->device));
    PtrKind kfr;
    RingOut o;
    o.flow = flow; o.flow_pitch = flow_pitch; o.flow_stride = flow_stride;
    TRY(buffer_kind(c, fn, "frames are", frames, &kfr));
    TRY(buffer_kind(c, fn, "flow is", flow, &o.kf));
    const bool stats = scalar || cut || cx || cy || val || mean_mag || centers;
    // the per-pair results of the whole call stay on the device until the end: max_pairs covers n_pairs
    const int maxPairs = stats && n_pairs > c->maxPairs ? n_pairs : (c->maxPairs > 0 ? c->maxPairs : 1);
    const int B = c->B > 0 ? c->B : 2;
    TRY(configure_checked(c, width, height, B, maxPairs, flow ? 2 * B + 8 : 0));
    c->pov = pov_mode ? 1 : 0;
    c->thr = (float)cut_threshold;
    TRY(sequence_loop(c, frames, n_frames, pitch, frame_stride, kfr, o, stats, nullptr, stream));
    const bool host_io = kfr != PTR_DEVICE || o.kf != PTR_DEVICE || stats;
    if (stream && !host_io) return FFB_OK;
    if (stats) return fetch_results(c, n_pairs, true, scalar, cut, cx, cy, val, mean_mag, centers);
    CK(c, cudaStreamSynchronize(c->s_comp));
    return FFB_OK;
}

// The sequence with the backward flow of every pair as well: a second flow_pairs per batch with the slot order reversed
// (R0 = frame j + 1, R1 = frame j, the expansions already in the ring) into the backward final-flow ring, then
// k_fb_check of the batch into the mask ring and the per-pair counts.  The three rings share their slots, and the
// fences of ffb_farneback_sequence cover the three copy-outs of a batch.
int ffb_farneback_sequence_bidir(ffb_ctx* c, const uint8_t* frames, int n_frames, int width, int height, size_t pitch,
                                 size_t frame_stride, float* flow_fw, float* flow_bw, size_t flow_pitch, size_t flow_stride,
                                 uint8_t* mask, size_t mask_pitch, size_t mask_stride, double alpha, double beta,
                                 int64_t* n_consistent, void* stream) {
    static const char* fn = "ffb_farneback_sequence_bidir";
    if (!c) return FFB_E_INVALID;
    if (c->in_bracket) return fail(c, FFB_E_INVALID, "ffb_farneback_sequence_bidir inside a bracket");
    if (n_frames < 0) return fail(c, FFB_E_INVALID, "ffb_farneback_sequence_bidir: n_frames %d < 0", n_frames);
    if (n_frames < 2) return FFB_OK;
    const int n_pairs = n_frames - 1;
    TRY(check_sequence_args(c, fn, frames, n_frames, width, height, pitch, frame_stride, flow_fw || flow_bw, flow_pitch,
                            flow_stride));
    TRY(check_bidir_args(c, fn, n_pairs, width, height, mask, mask_pitch, mask_stride, alpha, beta));
    CK(c, cudaSetDevice(c->device));
    PtrKind kfr;
    RingOut o;
    o.flow = flow_fw; o.flow_bw = flow_bw; o.flow_pitch = flow_pitch; o.flow_stride = flow_stride;
    o.mask = mask; o.mask_pitch = mask_pitch; o.mask_stride = mask_stride;
    TRY(buffer_kind(c, fn, "frames are", frames, &kfr));
    TRY(buffer_kind(c, fn, "flow_fw is", flow_fw, &o.kf));
    TRY(buffer_kind(c, fn, "flow_bw is", flow_bw, &o.kb));
    TRY(buffer_kind(c, fn, "mask is", mask, &o.km));
    const int B = c->B > 0 ? c->B : 2;
    TRY(configure_checked(c, width, height, B, c->maxPairs > 0 ? c->maxPairs : 1, o.any() ? 2 * B + 8 : 0));
    const bool backward = flow_bw || mask || n_consistent;
    TRY(alloc_backward(c, backward, mask != nullptr, n_consistent ? n_pairs : 0));
    Backward bw;
    bw.mask = mask != nullptr;
    bw.count = n_consistent != nullptr;
    bw.alpha = (float)alpha;
    bw.beta = (float)beta;
    TRY(sequence_loop(c, frames, n_frames, pitch, frame_stride, kfr, o, false, backward ? &bw : nullptr, stream));
    return finish_bidir(c, o, kfr != PTR_DEVICE, n_pairs, n_consistent, stream);
}

// ---- warping by a flow ---------------------------------------------------------------------------------------------
// Host buffers move in chunks of images whose source, flow and output take at most kRemapChunkBytes together (at least
// one image): large enough for full-rate copies, small enough that the copies of one chunk overlap the kernel of the
// previous one.  All-device calls launch once per 65535 images (the grid's z limit).
constexpr size_t kRemapChunkBytes = 8u << 20;
constexpr int kRemapMaxLaunch = 65535;

// cv2.remap(src[i], flow[i], None, INTER_LINEAR | WARP_RELATIVE_MAP, border_mode, (v, v, v)) of n uint8 images
// (k_remap_flow).  Device buffers are used in place (a device flow whose rows are not 4-byte aligned is copied to the
// staging first); host inputs are uploaded chunk by chunk on s_copy through staging buffer b = chunk & 1 (pageable ones
// through its pinned copy), a host output leaves the staging on s_out one chunk late, as in pairs_loop.  The fences are
// the pairs call's: ev_h2d[b] / ev_h2d_next[b] end the upload of the source / flow into buffer b, ev_expand[b] the
// kernel that read it, ev_fin[b] / ev_out[b] the kernel that wrote the output staging b and its copy-out.  The call
// touches neither the geometry, nor the Farneback parameters, nor the final-flow ring.
int ffb_remap_flow(ffb_ctx* c, const uint8_t* src, int n, int width, int height, int channels, size_t src_pitch,
                   size_t src_stride, const float* flow, size_t flow_pitch, size_t flow_stride, uint8_t* dst,
                   size_t dst_pitch, size_t dst_stride, int border_mode, int border_value, void* stream) {
    static const char* fn = "ffb_remap_flow";
    if (!c) return FFB_E_INVALID;
    if (c->in_bracket) return fail(c, FFB_E_INVALID, "ffb_remap_flow inside a bracket");
    if (n < 0) return fail(c, FFB_E_INVALID, "ffb_remap_flow: n %d < 0", n);
    if (n == 0) return FFB_OK;
    if (!src || !flow || !dst || width < 1 || height < 1 || width >= 32767 || height >= 32767)
        return fail(c, FFB_E_INVALID, "%s: bad images (%dx%d; cv2.remap takes sizes below 32767)", fn, width, height);
    if (channels != 1 && channels != 3) return fail(c, FFB_E_INVALID, "%s: %d channels (1 or 3)", fn, channels);
    if (border_mode != 0 && border_mode != 1)
        return fail(c, FFB_E_INVALID, "%s: border mode %d (0 constant, 1 replicate)", fn, border_mode);
    if (border_value < 0 || border_value > 255) return fail(c, FFB_E_INVALID, "%s: border value %d outside 0..255", fn, border_value);
    const size_t row = (size_t)width * channels, frow = (size_t)width * 8;
    if (src_pitch < row) return fail(c, FFB_E_INVALID, "%s: src_pitch %zu below width * channels (%zu)", fn, src_pitch, row);
    if (n > 1 && src_stride < src_pitch * (size_t)(height - 1) + row)
        return fail(c, FFB_E_INVALID, "%s: src_stride %zu shorter than an image", fn, src_stride);
    if (flow_pitch < frow) return fail(c, FFB_E_INVALID, "%s: flow_pitch %zu below 8 * width (%zu)", fn, flow_pitch, frow);
    if (n > 1 && flow_stride < flow_pitch * (size_t)(height - 1) + frow)
        return fail(c, FFB_E_INVALID, "%s: flow_stride %zu shorter than a flow", fn, flow_stride);
    if (dst_pitch < row) return fail(c, FFB_E_INVALID, "%s: dst_pitch %zu below width * channels (%zu)", fn, dst_pitch, row);
    if (n > 1 && dst_stride < dst_pitch * (size_t)(height - 1) + row)
        return fail(c, FFB_E_INVALID, "%s: dst_stride %zu shorter than an image", fn, dst_stride);
    CK(c, cudaSetDevice(c->device));
    PtrKind ks, kf, kd;
    TRY(buffer_kind(c, fn, "src is", src, &ks));
    TRY(buffer_kind(c, fn, "flow is", flow, &kf));
    TRY(buffer_kind(c, fn, "dst is", dst, &kd));
    const size_t img = row * height, fimg = frow * height;
    const bool flow_aligned = ((uintptr_t)flow | flow_pitch | (n > 1 ? flow_stride : 0)) % 4 == 0;
    const bool up_src = ks != PTR_DEVICE, up_flow = kf != PTR_DEVICE || !flow_aligned, down = kd != PTR_DEVICE;
    const bool staged = up_src || up_flow || down;
    const size_t per = (up_src ? img : 0) + (up_flow ? fimg : 0) + (down ? img : 0);
    const size_t fit = staged ? kRemapChunkBytes / per : 0;
    const int K = !staged || fit > (size_t)kRemapMaxLaunch ? kRemapMaxLaunch : (fit < 1 ? 1 : (int)fit);
    const int k_imgs = K < n ? K : n;
    if (up_src) TRY(grow_staging(c, c->rm_src, c->rm_src_cap, k_imgs * img, false));
    if (ks == PTR_PAGEABLE) TRY(grow_staging(c, c->rm_hsrc, c->rm_hsrc_cap, k_imgs * img, true));
    if (up_flow) TRY(grow_staging(c, c->rm_flow, c->rm_flow_cap, k_imgs * fimg, false));
    if (up_flow && kf == PTR_PAGEABLE) TRY(grow_staging(c, c->rm_hflow, c->rm_hflow_cap, k_imgs * fimg, true));
    if (down) TRY(grow_staging(c, c->rm_dst, c->rm_dst_cap, k_imgs * img, false));
    const cudaStream_t us = (cudaStream_t)stream;
    CK(c, cudaEventRecord(c->ev_user, us));
    CK(c, cudaStreamWaitEvent(c->s_copy, c->ev_user, 0));
    CK(c, cudaStreamWaitEvent(c->s_comp, c->ev_user, 0));
    // output of images [i0, i0 + m) from output staging b to dst
    auto copy_out = [&](int i0, int m, int b) -> int {
        CK(c, cudaStreamWaitEvent(c->s_out, c->ev_fin[b], 0));
        TRY(copy_slots_out(c, SlotImages{(const char*)c->rm_dst[b], img, row, row, height}, 0, m,
                           (char*)dst + (size_t)i0 * dst_stride, dst_pitch, dst_stride, kd));
        CK(c, cudaEventRecord(c->ev_out[b], c->s_out));
        return FFB_OK;
    };
    int pend_i0 = -1, pend_m = 0, pend_b = 0;   // chunk whose copy-out has not been issued yet
    for (int i0 = 0, k = 0; i0 < n; i0 += K, ++k) {
        const int m = n - i0 < K ? n - i0 : K, b = k & 1;
        const uint8_t* s = src + (size_t)i0 * src_stride;
        size_t ss = src_stride, sp = src_pitch;
        if (up_src) {
            TRY(upload_frames(c, c->rm_src[b], c->rm_hsrc[b], c->ev_h2d[b], c->ev_expand[b], s, ks, m, height, row, src_pitch,
                              src_stride));
            s = c->rm_src[b]; ss = img; sp = row;
        }
        FfbRing fr{(char*)flow + (size_t)i0 * flow_stride, flow_stride, 0, m};
        size_t fp = flow_pitch;
        if (up_flow) {
            TRY(upload_frames(c, c->rm_flow[b], c->rm_hflow[b], c->ev_h2d_next[b], c->ev_expand[b], (const uint8_t*)fr.base,
                              kf, m, height, frow, flow_pitch, flow_stride));
            fr = FfbRing{(char*)c->rm_flow[b], fimg, 0, m};
            fp = frow;
        }
        uint8_t* d = dst + (size_t)i0 * dst_stride;
        size_t ds = dst_stride, dp = dst_pitch;
        if (down) {
            CK(c, cudaStreamWaitEvent(c->s_comp, c->ev_out[b], 0));   // the copy-out of chunk k - 2 has read buffer b
            d = c->rm_dst[b]; ds = img; dp = row;
        }
        TRY(launch_remap(c, s, ss, sp, fr, fp, d, ds, dp, width, height, channels, border_mode, border_value, m));
        if (up_src || up_flow) CK(c, cudaEventRecord(c->ev_expand[b], c->s_comp));
        if (!down) continue;
        CK(c, cudaEventRecord(c->ev_fin[b], c->s_comp));
        // issued one chunk late: a copy into pageable memory returns only when it is done
        if (pend_i0 >= 0) TRY(copy_out(pend_i0, pend_m, pend_b));
        pend_i0 = i0; pend_m = m; pend_b = b;
    }
    if (pend_i0 >= 0) TRY(copy_out(pend_i0, pend_m, pend_b));
    if (down) {
        CK(c, cudaEventRecord(c->ev_done, c->s_out));
        CK(c, cudaStreamWaitEvent(c->s_comp, c->ev_done, 0));
    }
    // s_comp has waited for every upload and copy-out: the caller's stream continues when the inputs have been read
    // and the outputs written
    CK(c, cudaEventRecord(c->ev_done, c->s_comp));
    CK(c, cudaStreamWaitEvent(us, c->ev_done, 0));
    if (stream && ks == PTR_DEVICE && kf == PTR_DEVICE && kd == PTR_DEVICE) return FFB_OK;
    CK(c, cudaStreamSynchronize(c->s_comp));
    return FFB_OK;
}

static int upload_flow(ffb_ctx* c, const float* flow, int w, int h) {
    TRY(ensure_config(c, w, h));
    if (c->in_bracket) return fail(c, FFB_E_INVALID, "per-call function inside a bracket");
    CK(c, cudaMemcpy2DAsync(c->ring, (size_t)c->fp0 * 8, flow, (size_t)w * 8, (size_t)w * 8, h, cudaMemcpyHostToDevice, c->s_comp));
    c->pairs_done = 0;   // ring contents no longer belong to a bracket
    return FFB_OK;
}

static int flow_stats(ffb_ctx* c, const float* flow, int w, int h, int32_t* x, int32_t* y, float* val, float* mm) {
    if (!c || !flow) return FFB_E_INVALID;
    CK(c, cudaSetDevice(c->device));
    TRY(upload_flow(c, flow, w, h));
    TRY(launch_divmag(c, 0, 0, 1, c->s_comp));
    TRY(launch_phase1_finish(c, 0, 0, 1, 0, std::numeric_limits<float>::infinity()));
    int hx = 0, hy = 0;
    float hv = 0, hm = 0;
    CK(c, cudaMemcpyAsync(&hx, c->d_cx, 4, cudaMemcpyDeviceToHost, c->s_comp));
    CK(c, cudaMemcpyAsync(&hy, c->d_cy, 4, cudaMemcpyDeviceToHost, c->s_comp));
    CK(c, cudaMemcpyAsync(&hv, c->d_val, 4, cudaMemcpyDeviceToHost, c->s_comp));
    CK(c, cudaMemcpyAsync(&hm, c->d_mm, 4, cudaMemcpyDeviceToHost, c->s_comp));
    CK(c, cudaStreamSynchronize(c->s_comp));
    if (x) *x = hx;
    if (y) *y = hy;
    if (val) *val = hv;
    if (mm) *mm = hm;
    return FFB_OK;
}

int ffb_max_divergence(ffb_ctx* c, const float* flow, int w, int h, int32_t* x, int32_t* y, float* val) {
    return flow_stats(c, flow, w, h, x, y, val, nullptr);
}
int ffb_mean_magnitude(ffb_ctx* c, const float* flow, int w, int h, float* mm) {
    return flow_stats(c, flow, w, h, nullptr, nullptr, nullptr, mm);
}

int ffb_radial_motion(ffb_ctx* c, const float* flow, int w, int h, double cx, double cy, int is_cut, int pov, double* out) {
    if (!c || !flow || !out) return FFB_E_INVALID;
    CK(c, cudaSetDevice(c->device));
    if (is_cut) { *out = 0.0; return FFB_OK; }   // F:766-767
    TRY(upload_flow(c, flow, w, h));
    const double cen[2] = {cx, cy};
    const unsigned char zero = 0;
    CK(c, cudaMemcpyAsync(c->d_centers, cen, 16, cudaMemcpyHostToDevice, c->s_comp));
    CK(c, cudaMemcpyAsync(c->d_cut, &zero, 1, cudaMemcpyHostToDevice, c->s_comp));
    TRY(launch_radial(c, 0, 1, pov ? 1 : 0));
    CK(c, cudaMemcpyAsync(out, c->d_scalar, 8, cudaMemcpyDeviceToHost, c->s_comp));
    CK(c, cudaStreamSynchronize(c->s_comp));
    return FFB_OK;
}

// ---- stage hooks ---------------------------------------------------------------------------
static int level_plan_fill(const LevelPlan& p, int max_n, int* n, int* w, int* h, int* ksize, double* sigma) {
    *n = p.n;
    for (int i = 0; i < p.n && i < max_n; ++i) {
        if (w) w[i] = p.w[i];
        if (h) h[i] = p.h[i];
        if (ksize) ksize[i] = p.ksize[i];
        if (sigma) sigma[i] = p.sigma[i];
    }
    return FFB_OK;
}

int ffb_level_plan(int W, int H, int* n, int* w, int* h, int* ksize, double* sigma) {
    if (!n || W < 1 || H < 1) return FFB_E_INVALID;
    return level_plan_fill(make_plan(W, H, FarnebackParams()), FFB_MAX_LEVELS, n, w, h, ksize, sigma);
}

int ffb_level_plan_ex(int W, int H, double pyr_scale, int levels, int max_n, int* n, int* w, int* h, int* ksize, double* sigma) {
    if (!n || W < 1 || H < 1 || !(pyr_scale > 0.0 && pyr_scale < 1.0) || levels < 0 || max_n < 0) return FFB_E_INVALID;
    const LevelPlan p = make_plan(W, H, pyr_scale, levels);
    if (p.n > FFB_PLAN_LEVELS) return FFB_E_INVALID;
    return level_plan_fill(p, max_n, n, w, h, ksize, sigma);
}

int ffb_stage_pyramid(ffb_ctx* c, const uint8_t* img, int W, int H, size_t pitch, int level_k, float* out) {
    if (!c || !img || !out) return FFB_E_INVALID;
    CK(c, cudaSetDevice(c->device));
    const LevelPlan p = make_plan(W, H, c->fb);
    if (p.n > FFB_PLAN_LEVELS) return fail(c, FFB_E_INVALID, "%dx%d plans more than %d pyramid levels", W, H, FFB_PLAN_LEVELS);
    int li = -1;
    for (int i = 0; i < p.n; ++i) if (p.k[i] == level_k) li = i;
    if (li < 0) return fail(c, FFB_E_INVALID, "level %d does not exist for %dx%d", level_k, W, H);
    const int w = p.w[li], h = p.h[li];
    const FfbTaps taps = make_taps(p.ksize[li], p.sigma[li]);
    std::vector<int> xi, yi;
    std::vector<float> xa, ya;
    make_linear_table(w, W, xi, xa);
    make_linear_table(h, H, yi, ya);
    int RW, RH;
    pyramid_window(xi, w, W, PYR_TW, taps.r, &RW);
    pyramid_window(yi, h, H, PYR_TH, taps.r, &RH);
    Scratch s;
    uint8_t* d_img = nullptr; float* d_out = nullptr; int *dxi = nullptr, *dyi = nullptr; float *dxa = nullptr, *dya = nullptr;
    TRY(s.alloc(c, &d_img, (size_t)W * H));
    CK(c, cudaMemcpy2D(d_img, W, img, pitch, W, H, cudaMemcpyHostToDevice));
    if (pyramid_fast_ok(W, H, p)) {   // the production path for this geometry: all levels in one pass
        float* dst[FFB_MAX_LEVELS] = {nullptr, nullptr, nullptr, nullptr};
        size_t dstride[FFB_MAX_LEVELS] = {0, 0, 0, 0};
        int dp[FFB_MAX_LEVELS] = {0, 0, 0, 0};
        for (int k = 0; k < p.n; ++k) {
            TRY(s.alloc(c, &dst[k], (size_t)(W >> k) * (H >> k)));
            dp[k] = W >> k;
        }
        TRY(launch_pyramid_pow2(c, d_img, (size_t)W * H, W, W, H, p.n, dst, dstride, dp, 1));
        CK(c, cudaStreamSynchronize(c->s_comp));
        CK(c, cudaMemcpy(out, dst[level_k], (size_t)w * h * 4, cudaMemcpyDeviceToHost));
        return FFB_OK;
    }
    TRY(s.alloc(c, &d_out, (size_t)w * h));
    TRY(s.upload(c, &dxi, xi.data(), xi.size())); TRY(s.upload(c, &dxa, xa.data(), xa.size()));
    TRY(s.upload(c, &dyi, yi.data(), yi.size())); TRY(s.upload(c, &dya, ya.data(), ya.size()));
    if (pyramid_wide(taps.r, RW, RH)) {
        const std::vector<float> k = gaussian_half(p.ksize[li], p.sigma[li]);
        float *dk = nullptr, *dtmp = nullptr;
        TRY(s.upload(c, &dk, k.data(), k.size()));
        TRY(s.alloc(c, &dtmp, (size_t)H * w));
        TRY(launch_pyramid_wide(c, d_img, (size_t)W * H, W, W, H, dtmp, d_out, (size_t)w * h, w, w, h, dxi, dxa, dyi, dya, dk,
                                taps.r, 1));
    } else {
        TRY(launch_pyramid(c, d_img, (size_t)W * H, W, W, H, d_out, (size_t)w * h, w, w, h, dxi, dxa, dyi, dya, taps, RW, RH, 1));
    }
    CK(c, cudaStreamSynchronize(c->s_comp));
    CK(c, cudaMemcpy(out, d_out, (size_t)w * h * 4, cudaMemcpyDeviceToHost));
    return FFB_OK;
}

// Host-side conversion between the [5][h][w] planes of the hooks' interface and the device layout of
// an expansion (float4 [h][rp] = channels 0..3, then float [h][rp] = channel 4).
static void planes_to_expansion(const float* planes, int w, int h, int rp, std::vector<float>& dev) {
    const size_t plane = (size_t)rp * h;
    dev.assign(5 * plane, 0.f);
    for (int y = 0; y < h; ++y)
        for (int x = 0; x < w; ++x) {
            const size_t pix = (size_t)y * rp + x, src = (size_t)y * w + x;
            for (int ch = 0; ch < 4; ++ch) dev[4 * pix + ch] = planes[(size_t)ch * w * h + src];
            dev[4 * plane + pix] = planes[(size_t)4 * w * h + src];
        }
}
static void expansion_to_planes(const std::vector<float>& dev, int w, int h, int rp, float* planes) {
    const size_t plane = (size_t)rp * h;
    for (int y = 0; y < h; ++y)
        for (int x = 0; x < w; ++x) {
            const size_t pix = (size_t)y * rp + x, dst = (size_t)y * w + x;
            for (int ch = 0; ch < 4; ++ch) planes[(size_t)ch * w * h + dst] = dev[4 * pix + ch];
            planes[(size_t)4 * w * h + dst] = dev[4 * plane + pix];
        }
}

int ffb_stage_polyexp(ffb_ctx* c, const float* img, int w, int h, float* out) {
    if (!c || !img || !out) return FFB_E_INVALID;
    CK(c, cudaSetDevice(c->device));
    Scratch s;
    const int rp = ffb_round_up(w, 4);            // the kernel stores 16-byte vectors
    const size_t plane = (size_t)rp * h;
    float *d_in = nullptr, *d_out = nullptr;
    TRY(s.upload(c, &d_in, img, (size_t)w * h));
    TRY(s.alloc(c, &d_out, 5 * plane));
    FfbRing dst{(char*)d_out, 0, 0, 1};
    TRY(launch_polyexp(c, d_in, (size_t)w * h, w, w, h, dst, plane, rp, 1));
    CK(c, cudaStreamSynchronize(c->s_comp));
    std::vector<float> host(5 * plane);
    CK(c, cudaMemcpy(host.data(), d_out, 5 * plane * sizeof(float), cudaMemcpyDeviceToHost));
    expansion_to_planes(host, w, h, rp, out);
    return FFB_OK;
}

int ffb_stage_update_matrices(ffb_ctx* c, const float* R0, const float* R1, const float* flow, int w, int h, float* out) {
    if (!c || !R0 || !R1 || !out) return FFB_E_INVALID;
    CK(c, cudaSetDevice(c->device));
    Scratch s;
    float *d0 = nullptr, *d1 = nullptr, *dM = nullptr; float2* df = nullptr;
    TRY(s.upload(c, &d0, R0, (size_t)5 * w * h));
    TRY(s.upload(c, &d1, R1, (size_t)5 * w * h));
    if (flow) TRY(s.upload(c, &df, (const float2*)flow, (size_t)w * h));
    TRY(s.alloc(c, &dM, (size_t)5 * w * h));
    FfbMatArgs a{d0, d1, (size_t)w * h, w, w, h, df, w, dM};
    const ProfMark pm = prof_begin(c, FFB_K_SMALL, -1, 0, c->s_comp);
    FFB_LAUNCH(k_update_matrices, dim3((w + 31) / 32, (h + 7) / 8), dim3(256), 0, c->s_comp, a);
    prof_end(pm);
    CKL(c);
    CK(c, cudaStreamSynchronize(c->s_comp));
    CK(c, cudaMemcpy(out, dM, (size_t)5 * w * h * 4, cudaMemcpyDeviceToHost));
    return FFB_OK;
}

int ffb_stage_flow_iter(ffb_ctx* c, const float* R0, const float* R1, const float* flow_in, int w, int h, float* flow_out) {
    if (!c || !R0 || !R1 || !flow_out) return FFB_E_INVALID;
    CK(c, cudaSetDevice(c->device));
    Scratch s;
    const int rp = ffb_round_up(w, 4);
    const size_t plane = (size_t)rp * h;
    float* dR = nullptr; float2 *dfi = nullptr, *dfo = nullptr;
    TRY(s.alloc(c, &dR, 10 * plane));
    for (int f = 0; f < 2; ++f) {
        std::vector<float> host;
        planes_to_expansion(f ? R1 : R0, w, h, rp, host);
        CK(c, cudaMemcpy(dR + (size_t)f * 5 * plane, host.data(), 5 * plane * sizeof(float), cudaMemcpyHostToDevice));
    }
    if (flow_in) {
        TRY(s.alloc(c, &dfi, plane));
        CK(c, cudaMemcpy2D(dfi, (size_t)rp * 8, flow_in, (size_t)w * 8, (size_t)w * 8, h, cudaMemcpyHostToDevice));
    }
    TRY(s.alloc(c, &dfo, plane));
    FfbRing R{(char*)dR, 5 * plane * sizeof(float), 0, 2};
    FfbRing fo{(char*)dfo, 0, 0, 1};
    if (c->fb.winsize == FFB_WIN) {
        TRY(launch_flow_iter(c, flow_iter_plan(w, h, w, h, c->iter_cfg), -1, c->s_comp, true, R, plane, rp, w, h, dfi, 0, rp, fo,
                             rp, 1));
    } else {
        float* dM = nullptr;
        TRY(s.alloc(c, &dM, 5 * plane));
        TRY(launch_flow_unfused(c, -1, dM, R, plane, rp, w, h, dfi, 0, rp, fo, rp, 1));
    }
    CK(c, cudaStreamSynchronize(c->s_comp));
    CK(c, cudaMemcpy2D(flow_out, (size_t)w * 8, dfo, (size_t)rp * 8, (size_t)w * 8, h, cudaMemcpyDeviceToHost));
    return FFB_OK;
}

int ffb_stage_upsample_flow(ffb_ctx* c, const float* flow_c, int wc, int hc, int w, int h, float* out) {
    if (!c || !flow_c || !out) return FFB_E_INVALID;
    CK(c, cudaSetDevice(c->device));
    std::vector<int> xi, yi;
    std::vector<float> xa, ya;
    make_linear_table(w, wc, xi, xa);
    make_linear_table(h, hc, yi, ya);
    Scratch s;
    float2 *dsrc = nullptr, *ddst = nullptr; int *dxi = nullptr, *dyi = nullptr; float *dxa = nullptr, *dya = nullptr;
    TRY(s.upload(c, &dsrc, (const float2*)flow_c, (size_t)wc * hc));
    TRY(s.alloc(c, &ddst, (size_t)w * h));
    TRY(s.upload(c, &dxi, xi.data(), xi.size())); TRY(s.upload(c, &dxa, xa.data(), xa.size()));
    TRY(s.upload(c, &dyi, yi.data(), yi.size())); TRY(s.upload(c, &dya, ya.data(), ya.size()));
    TRY(launch_upsample(c, dsrc, 0, wc, wc, hc, ddst, 0, w, w, h, dxi, dxa, dyi, dya, 1));
    CK(c, cudaStreamSynchronize(c->s_comp));
    CK(c, cudaMemcpy(out, ddst, (size_t)w * h * 8, cudaMemcpyDeviceToHost));
    return FFB_OK;
}

int ffb_stage_fb_check(ffb_ctx* c, const float* flow_fw, const float* flow_bw, int w, int h, double alpha, double beta,
                       uint8_t* mask, int64_t* n_consistent) {
    if (!c || !flow_fw || !flow_bw || w < 1 || h < 1 || (double)w * h >= 4294967295.0) return FFB_E_INVALID;
    if (!(alpha >= 0.0 && isfinite(alpha)) || !(beta >= 0.0 && isfinite(beta)))
        return fail(c, FFB_E_INVALID, "ffb_stage_fb_check: alpha %g and beta %g must be finite and >= 0", alpha, beta);
    CK(c, cudaSetDevice(c->device));
    Scratch s;
    float2 *dfw = nullptr, *dbw = nullptr;
    uint8_t* dm = nullptr;
    unsigned* dn = nullptr;
    const size_t px = (size_t)w * h;
    TRY(s.upload(c, &dfw, (const float2*)flow_fw, px));
    TRY(s.upload(c, &dbw, (const float2*)flow_bw, px));
    TRY(s.alloc(c, &dm, px));
    TRY(s.alloc(c, &dn, 1));
    CK(c, cudaMemsetAsync(dn, 0, sizeof(unsigned), c->s_comp));
    TRY(launch_fb_check(c, FfbRing{(char*)dfw, 0, 0, 1}, FfbRing{(char*)dbw, 0, 0, 1}, w, w, h, FfbRing{(char*)dm, 0, 0, 1}, w,
                        dn, (float)alpha, (float)beta, 1));
    CK(c, cudaStreamSynchronize(c->s_comp));
    unsigned n = 0;
    CK(c, cudaMemcpy(&n, dn, sizeof(unsigned), cudaMemcpyDeviceToHost));
    if (mask) CK(c, cudaMemcpy(mask, dm, px, cudaMemcpyDeviceToHost));
    if (n_consistent) *n_consistent = n;
    return FFB_OK;
}

// ---- frame pre-processing (row N2) --------------------------------------------------------
static int preprocess_configure_plan(ffb_ctx* c, const ffb_ctx::PrePlan& p) {
    if (!c || !plan_ok(p)) return fail(c, FFB_E_INVALID, "ffb_preprocess_configure: bad geometry");
    CK(c, cudaSetDevice(c->device));
    if (c->in_bracket) return fail(c, FFB_E_INVALID, "ffb_preprocess_configure inside a bracket");
    if (c->pre == p) return FFB_OK;
    CK(c, cudaStreamSynchronize(c->s_comp));
    CK(c, cudaStreamSynchronize(c->s_copy));
    free_preprocess(c);
    TRY(upload_vec(c, &c->pre_xt, make_u8_resize_table(p.TW, p.W, true)));
    TRY(upload_vec(c, &c->pre_yt, make_u8_resize_table(p.TH, p.H, false)));
    const size_t cbytes = (size_t)PRE_CHUNK * p.W * p.H * 3;
    for (int b = 0; b < 2; ++b) {
        TRY(dev_alloc(c, &c->d_color[b], cbytes));
        void* hp = nullptr;
        TRY(host_alloc(c, &hp, cbytes));
        c->h_color[b] = (uint8_t*)hp;
    }
    c->pre = p;
    return FFB_OK;
}
int ffb_preprocess_configure(ffb_ctx* c, int W, int H, int vr) {
    return preprocess_configure_plan(c, reference_plan(W, H, vr));
}
int ffb_preprocess_configure_window(ffb_ctx* c, int W, int H, int target_w, int target_h, int win_x, int win_y, int win_w,
                                    int win_h) {
    ffb_ctx::PrePlan p;
    p.W = W; p.H = H; p.TW = target_w; p.TH = target_h; p.x0 = win_x; p.y0 = win_y; p.OW = win_w; p.OH = win_h;
    return preprocess_configure_plan(c, p);
}

int ffb_bracket_push_bgr(ffb_ctx* c, const uint8_t* bgr, int n, size_t pitch, size_t stride) {
    if (!c || !c->in_bracket) return fail(c, FFB_E_INVALID, "ffb_bracket_push_bgr outside a bracket");
    CK(c, cudaSetDevice(c->device));      // several contexts (GPUs) may be driven by one host thread
    if (c->phase1_read) return fail(c, FFB_E_INVALID, "ffb_bracket_push_bgr after ffb_bracket_phase1_finish");
    const ffb_ctx::PrePlan& pp = c->pre;
    if (pp.W == 0) return fail(c, FFB_E_INVALID, "ffb_bracket_push_bgr before ffb_preprocess_configure");
    if (c->W != pp.OW || c->H != pp.OH)
        return fail(c, FFB_E_INVALID, "pre-processed frames are %dx%d: ffb_configure(ctx, %d, %d, ...)", pp.OW, pp.OH, pp.OW, pp.OH);
    const size_t row = (size_t)pp.W * 3;
    const size_t obytes = (size_t)pp.OW * pp.OH;
    if (!bgr || n < 0 || pitch < row || stride < pitch * (size_t)(pp.H - 1) + row)
        return fail(c, FFB_E_INVALID, "ffb_bracket_push_bgr: bad arguments");
    const PtrKind kind = classify(bgr);
    const size_t fbytes = row * pp.H;
    // The gray frames gather in the device staging buffer of the next batch and run through the hot path once the
    // batch is full, however the caller cuts its pushes (a decoder hands over chunks much smaller than the batches
    // that fill the GPU at 256x256); ffb_bracket_finish runs what is left.
    for (int i = 0; i < n;) {
        const int cap = batch_cap(c, kind);
        const int b = c->batch_no & 1;
        int m = n - i;
        if (m > PRE_CHUNK) m = PRE_CHUNK;
        if (m > cap - c->pend) m = cap - c->pend;
        const uint8_t* src = bgr + (size_t)i * stride;
        uint8_t* dst = c->d_u8[b] + (size_t)c->pend * obytes;
        if (kind != PTR_DEVICE) {
            const int cb = c->color_no & 1;
            c->color_no++;
            TRY(upload_frames(c, c->d_color[cb], c->h_color[cb], c->ev_ch2d[cb], c->ev_pre[cb], src, kind, m, pp.H, row,
                              pitch, stride));
            TRY(launch_preprocess(c, c->d_color[cb], fbytes, (int)row, dst, pp, c->pre_xt, c->pre_yt, m));
            CK(c, cudaEventRecord(c->ev_pre[cb], c->s_comp));
        } else {
            TRY(launch_preprocess(c, src, stride, (int)pitch, dst, pp, c->pre_xt, c->pre_yt, m));
        }
        c->pend += m;
        i += m;
        // the gray frames now sit in the device staging buffer: continue as for device input
        if (c->pend >= cap) TRY(flush_pending(c));
    }
    return FFB_OK;
}

static int stage_preprocess_plan(ffb_ctx* c, const uint8_t* bgr, size_t pitch, const ffb_ctx::PrePlan& p, uint8_t* gray) {
    if (!c || !bgr || !gray || !plan_ok(p) || pitch < (size_t)p.W * 3) return fail(c, FFB_E_INVALID, "ffb_stage_preprocess: bad arguments");
    CK(c, cudaSetDevice(c->device));
    Scratch s;
    uint8_t *d_src = nullptr, *d_dst = nullptr;
    int *dxt = nullptr, *dyt = nullptr;
    const std::vector<int> xt = make_u8_resize_table(p.TW, p.W, true), yt = make_u8_resize_table(p.TH, p.H, false);
    TRY(s.alloc(c, &d_src, (size_t)p.W * p.H * 3));
    CK(c, cudaMemcpy2D(d_src, (size_t)p.W * 3, bgr, pitch, (size_t)p.W * 3, p.H, cudaMemcpyHostToDevice));
    TRY(s.alloc(c, &d_dst, (size_t)p.OW * p.OH));
    TRY(s.upload(c, &dxt, xt.data(), xt.size()));
    TRY(s.upload(c, &dyt, yt.data(), yt.size()));
    TRY(launch_preprocess(c, d_src, (size_t)p.W * p.H * 3, p.W * 3, d_dst, p, dxt, dyt, 1));
    CK(c, cudaStreamSynchronize(c->s_comp));
    CK(c, cudaMemcpy(gray, d_dst, (size_t)p.OW * p.OH, cudaMemcpyDeviceToHost));
    return FFB_OK;
}
int ffb_stage_preprocess(ffb_ctx* c, const uint8_t* bgr, int W, int H, size_t pitch, int vr, uint8_t* gray) {
    return stage_preprocess_plan(c, bgr, pitch, reference_plan(W, H, vr), gray);
}
int ffb_stage_preprocess_window(ffb_ctx* c, const uint8_t* bgr, int W, int H, size_t pitch, int target_w, int target_h, int win_x,
                                int win_y, int win_w, int win_h, uint8_t* gray) {
    ffb_ctx::PrePlan p;
    p.W = W; p.H = H; p.TW = target_w; p.TH = target_h; p.x0 = win_x; p.y0 = win_y; p.OW = win_w; p.OH = win_h;
    return stage_preprocess_plan(c, bgr, pitch, p, gray);
}

// ---- instrumentation ---------------------------------------------------------------------
int ffb_profile(ffb_ctx* c, int enable) {
    if (!c) return FFB_E_INVALID;
    CK(c, cudaStreamSynchronize(c->s_comp));
    prof_collect(c);
    c->prof = enable != 0;
    return FFB_OK;
}
int ffb_profile_reset(ffb_ctx* c) {
    if (!c) return FFB_E_INVALID;
    CK(c, cudaStreamSynchronize(c->s_comp));
    prof_collect(c);
    for (int i = 0; i < FFB_K_COUNT; ++i) { c->k_launches[i] = 0; c->k_ms[i] = 0; c->k_bytes[i] = 0; }
    for (int i = 0; i < FFB_PLAN_LEVELS; ++i) { c->it_launches[i] = 0; c->it_ms[i] = 0; c->it_bytes[i] = 0; }
    return FFB_OK;
}
int ffb_kernel_stats(ffb_ctx* c, int kid, int64_t* launches, double* ms, double* bytes) {
    if (!c || kid < 0 || kid >= FFB_K_COUNT) return FFB_E_INVALID;
    CK(c, cudaStreamSynchronize(c->s_comp));
    prof_collect(c);
    if (launches) *launches = c->k_launches[kid];
    if (ms) *ms = c->k_ms[kid];
    if (bytes) *bytes = c->k_bytes[kid];
    return FFB_OK;
}
int ffb_flow_iter_level_stats(ffb_ctx* c, int k, int64_t* launches, double* ms, double* bytes) {
    if (!c || k < 0 || k >= FFB_PLAN_LEVELS) return FFB_E_INVALID;
    CK(c, cudaStreamSynchronize(c->s_comp));
    prof_collect(c);
    if (launches) *launches = c->it_launches[k];
    if (ms) *ms = c->it_ms[k];
    if (bytes) *bytes = c->it_bytes[k];
    return FFB_OK;
}
int64_t ffb_launch_count(const ffb_ctx* c) { return c ? c->launches : 0; }

int ffb_timer_mark(ffb_ctx* c, int slot) {
    if (!c || slot < 0 || slot >= 8) return FFB_E_INVALID;
    if (!c->timers[slot]) CK(c, cudaEventCreate(&c->timers[slot]));
    CK(c, cudaEventRecord(c->timers[slot], c->s_comp));
    return FFB_OK;
}
int ffb_timer_elapsed(ffb_ctx* c, int a, int b, double* ms) {
    if (!c || !ms || a < 0 || a >= 8 || b < 0 || b >= 8 || !c->timers[a] || !c->timers[b]) return FFB_E_INVALID;
    CK(c, cudaEventSynchronize(c->timers[b]));
    float f = 0.f;
    CK(c, cudaEventElapsedTime(&f, c->timers[a], c->timers[b]));
    *ms = f;
    return FFB_OK;
}

}  // extern "C"
