// ffb_kernels.cuh -- hand-written sm_100a kernels of the frame-pair -> radial-scalar hot path.
//
// All kernels are HBM-bound stencils / gathers / reductions in fp32 (fp64 only in reductions);
// there is no GEMM-shaped work, so no tensor-core path.  Every kernel takes the batch index
// (frame or pair) in blockIdx.z so that small frames still fill the 148 SMs.
//
// Reference stages (F:n = FunscriptFlow.pyw line n; OpenCV = the un-vendored cv2 dependency):
//   k_pyramid_level   A1a  convertTo + GaussianBlur(REFLECT_101) + resize(INTER_LINEAR)   (inside F:878)
//   k_polyexp         A1b  FarnebackPolyExp                                                 (inside F:878)
//   k_upsample_flow   A1e  resize(prevFlow) * 2                                             (inside F:878)
//   k_flow_iter       A1c+A1d  FarnebackUpdateMatrices + 15x15 box mean + 2x2 solve, fused  (inside F:878)
//   k_divmag          A3+A4 np.gradient "divergence" argmax + magnitude sum                 F:754-757, F:889-890
//   k_phase1_finish   A2/A3/A4 finish: centre, value, mean magnitude, cut flag              F:880-894
//   k_smooth_centers  A5   +-6 centre mean                                                  F:1203-1214
//   k_radial(+finish) A6   balanced weighted radial projection mean                         F:761-785
// and, outside the reference's path, k_remap_flow (X9): cv2.remap of uint8 frames by dense flows, bit-exact.
#pragma once
#include "ffb_common.h"

// ======================================================================================
// small device helpers
// ======================================================================================
__device__ __forceinline__ int ffb_clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

template <class T>
__device__ __forceinline__ T ffb_warp_sum(T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ unsigned long long ffb_warp_max_u64(unsigned long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        unsigned long long t = __shfl_xor_sync(0xffffffffu, v, o);
        v = t > v ? t : v;
    }
    return v;
}

// ======================================================================================
// K1  pyramid level: u8 frame -> f32 level image
// ======================================================================================
// out(dx,dy) = lerp_y( blur_y( lerp_x( blur_x(src) ) ) ): the Gaussian is evaluated only at the two
// source columns / rows each bilinear output tap needs.  One CTA = one TW x TH output tile; its
// source window is staged once in shared memory as float (border: REFLECT_101, single bounce --
// the host guarantees radius < min(W, H)).
struct FfbPyrArgs {
    const uint8_t* src; size_t src_frame_stride; int src_pitch; int W, H;
    float* dst; size_t dst_frame_stride; int dp; int w, h;        // strides in floats
    const int* xi; const float* xa; const int* yi; const float* ya;  // resize tables (device)
    FfbTaps taps;
    int RWp;        // smem window row pitch (floats)
    int p_off;      // float offset of the plane P inside dynamic smem
};

__device__ __forceinline__ int ffb_reflect1(int i, int n) {   // BORDER_REFLECT_101, |overshoot| < n
    i = i < 0 ? -i : i;
    return i >= n ? 2 * n - 2 - i : i;
}

__device__ __forceinline__ float ffb_blur_row(const float* row, int c, const FfbTaps& t) {
    float s = t.k[0] * row[c];
    for (int i = 1; i <= t.r; ++i) s += t.k[i] * (row[c - i] + row[c + i]);
    return s;
}

template <int TW, int TH>
__global__ void __launch_bounds__(TW* TH) k_pyramid_level(FfbPyrArgs a) {
    FFB_DYN_SMEM(float, smem);
    float* reg = smem;
    float* P = smem + a.p_off;
    const int tid = threadIdx.x;
    const int tx = tid % TW, ty = tid / TW;
    const int x0 = blockIdx.x * TW, y0 = blockIdx.y * TH, f = blockIdx.z;
    const int x_last = min(x0 + TW, a.w) - 1, y_last = min(y0 + TH, a.h) - 1;
    const int r = a.taps.r;
    const int sx_lo = a.xi[x0] - r;
    const int sx_hi = min(a.xi[x_last] + 1, a.W - 1) + r;
    const int sy_lo = a.yi[y0] - r;
    const int sy_hi = min(a.yi[y_last] + 1, a.H - 1) + r;
    const int rw = sx_hi - sx_lo + 1, rh = sy_hi - sy_lo + 1;
    const uint8_t* src = a.src + (size_t)f * a.src_frame_stride;
    for (int ry = ty; ry < rh; ry += TH) {
        const uint8_t* srow = src + (size_t)ffb_reflect1(sy_lo + ry, a.H) * a.src_pitch;
        float* drow = reg + ry * a.RWp;
        for (int rx = tx; rx < rw; rx += TW) drow[rx] = (float)__ldg(srow + ffb_reflect1(sx_lo + rx, a.W));
    }
    __syncthreads();
    // pass 1: horizontal blur evaluated only at the two resize taps of each output column, lerped
    {
        const int dx = x0 + tx;
        const bool ok = dx < a.w;
        const int s0 = ok ? a.xi[dx] : 0;
        const float al = ok ? a.xa[dx] : 0.f;
        const int c0 = s0 - sx_lo, c1 = min(s0 + 1, a.W - 1) - sx_lo;
        for (int ry = ty; ry < rh; ry += TH) {
            float v = 0.f;
            if (ok) {
                const float* row = reg + ry * a.RWp;
                v = ffb_blur_row(row, c0, a.taps);
                if (al != 0.f) v = v * (1.f - al) + ffb_blur_row(row, c1, a.taps) * al;
            }
            P[ry * TW + tx] = v;
        }
    }
    __syncthreads();
    // pass 2: vertical blur at the two resize rows, lerped
    const int dx = x0 + tx, dy = y0 + ty;
    if (dx < a.w && dy < a.h) {
        const int s0 = a.yi[dy];
        const float be = a.ya[dy];
        const float* col = P + tx;
        int c = s0 - sy_lo;
        float b0 = a.taps.k[0] * col[c * TW];
        for (int i = 1; i <= r; ++i) b0 += a.taps.k[i] * (col[(c - i) * TW] + col[(c + i) * TW]);
        float v = b0;
        if (be != 0.f) {
            c = min(s0 + 1, a.H - 1) - sy_lo;
            float b1 = a.taps.k[0] * col[c * TW];
            for (int i = 1; i <= r; ++i) b1 += a.taps.k[i] * (col[(c - i) * TW] + col[(c + i) * TW]);
            v = b0 * (1.f - be) + b1 * be;
        }
        a.dst[(size_t)f * a.dst_frame_stride + (size_t)dy * a.dp + dx] = v;
    }
}

// ======================================================================================
// K1'  all pyramid levels in one pass (frames whose width and height are multiples of 8)
// ======================================================================================
// With W, H divisible by 8 every level is an exact 2^k decimation: output (dx, dy) of level k lerps
// (weights 1/2, 1/2) the blurred image at source columns 2^k dx + 2^(k-1) - 1, +1 (same for rows),
// so a 128 x 32 source tile with an 8-pixel halo yields the 128x32, 64x16, 32x8 and 16x4 output
// tiles of levels 0..3.  The source tile is read from HBM once (32-bit loads, converted to float in
// shared memory) instead of once per level; the arithmetic per output is the same expression, in
// the same order, as k_pyramid_level (the two paths agree to FMA-contraction rounding, <= 2 ulp).
constexpr int PYR2_TX = 128, PYR2_TY = 32, PYR2_HL = 8;
constexpr int PYR2_RW = PYR2_TX + 2 * PYR2_HL, PYR2_RH = PYR2_TY + 2 * PYR2_HL;
// Shared-memory pitches are chosen for the 16-byte loads of the row passes: a quarter-warp (the unit a
// 128-bit shared access is served in) reads chunks that are 32 or 64 bytes apart, so it is spread
// over 2 or 4 window rows, and 148 = 20 (mod 32) puts those rows on disjoint banks.
constexpr int PYR2_RWP = PYR2_RW + 4;
constexpr int PYR2_PMAX = 80;                           // largest pitch of the row-pass result (level 1)
constexpr size_t PYR2_SMEM = sizeof(float) * (PYR2_RWP * PYR2_RH + PYR2_RH * PYR2_PMAX);

struct FfbPyr2Args {
    const uint8_t* src; size_t src_frame_stride; int src_pitch; int W, H;
    float* dst[FFB_MAX_LEVELS]; size_t dstride[FFB_MAX_LEVELS]; int dp[FFB_MAX_LEVELS];   // index = level k
    FfbTaps taps[FFB_MAX_LEVELS];
    int nlev;
    int aligned;     // source rows are 4-byte aligned (pitch % 4 == 0 and base % 4 == 0)
};

template <int R>
__device__ __forceinline__ float ffb_blur_row_t(const float* row, const FfbTaps& t) {
    float s = t.k[0] * row[0];
#pragma unroll
    for (int i = 1; i <= R; ++i) s += t.k[i] * (row[-i] + row[i]);
    return s;
}
template <int R>
__device__ __forceinline__ float ffb_blur_col_t(const float* col, int pitch, const FfbTaps& t) {
    float s = t.k[0] * col[0];
#pragma unroll
    for (int i = 1; i <= R; ++i) s += t.k[i] * (col[-i * pitch] + col[i * pitch]);
    return s;
}

// Per-level shape of the row pass: one task = NOUT adjacent outputs of one window row, computed from
// NF4 aligned 16-byte loads held in registers; a quarter-warp covers 2^JB tasks along the row times
// 2^RB rows; PP = pitch of the row-pass result (padded so its vector stores do not collide either).
template <int K> struct FfbPyr2Shape;
template <> struct FfbPyr2Shape<1> { static constexpr int R = 1, NOUT = 4, NF4 = 4, JB = 2, RB = 1, PP = 80; };
template <> struct FfbPyr2Shape<2> { static constexpr int R = 4, NOUT = 2, NF4 = 4, JB = 2, RB = 1, PP = 48; };
template <> struct FfbPyr2Shape<3> { static constexpr int R = 9, NOUT = 2, NF4 = 8, JB = 1, RB = 2, PP = 24; };

template <int K>
__device__ __forceinline__ void ffb_pyr2_level(const FfbPyr2Args& a, const float* reg, float* P, int X0, int Y0, int f,
                                               int tid) {
    using SH = FfbPyr2Shape<K>;
    constexpr int R = SH::R, NOUT = SH::NOUT, NF4 = SH::NF4, JB = SH::JB, RB = SH::RB, PP = SH::PP;
    constexpr int S = 1 << K, OW = PYR2_TX >> K, OH = PYR2_TY >> K, NJ = OW / NOUT;
    constexpr int OFF = (1 << (K - 1)) - 1;                 // first bilinear tap inside a 2^K cell
    constexpr int BASE0 = (OFF + PYR2_HL - R) & ~3;          // aligned start of the first task's footprint
    constexpr int C0 = OFF + PYR2_HL - BASE0;                // register index of output 0's first tap centre
    static_assert(C0 - R >= 0 && C0 + (NOUT - 1) * S + 1 + R < 4 * NF4, "row-pass footprint");
    static_assert(BASE0 + (NJ - 1) * NOUT * S + 4 * NF4 <= PYR2_RWP, "row-pass footprint leaves the window");
    static_assert(PYR2_RH % (1 << RB) == 0 && NJ % (1 << JB) == 0 && PP >= OW && PP <= PYR2_PMAX, "task shape");
    const FfbTaps& t = a.taps[K];
    // pass 1: rows of the window -> P[ry][ox]
    for (int i = tid; i < PYR2_RH * NJ; i += 256) {
        const int jl = i & ((1 << JB) - 1), rl = (i >> JB) & ((1 << RB) - 1), rest = i >> (JB + RB);
        const int rh = rest / (NJ >> JB), jh = rest - rh * (NJ >> JB);
        const int j = (jh << JB) | jl, ry = (rh << RB) | rl;
        float w[4 * NF4];
        const float4* src4 = reinterpret_cast<const float4*>(reg + ry * PYR2_RWP + j * (NOUT * S) + BASE0);
#pragma unroll
        for (int q = 0; q < NF4; ++q) {
            const float4 v = src4[q];
            w[4 * q] = v.x; w[4 * q + 1] = v.y; w[4 * q + 2] = v.z; w[4 * q + 3] = v.w;
        }
        float o[NOUT];
#pragma unroll
        for (int n = 0; n < NOUT; ++n) {
            const float* row = w + C0 + n * S;
            float v = ffb_blur_row_t<R>(row, t);
            v = v * (1.f - 0.5f) + ffb_blur_row_t<R>(row + 1, t) * 0.5f;
            o[n] = v;
        }
        float* d = P + ry * PP + j * NOUT;
        if (NOUT == 4) *reinterpret_cast<float4*>(d) = make_float4(o[0], o[1], o[NOUT > 2 ? 2 : 0], o[NOUT > 3 ? 3 : 0]);
        else *reinterpret_cast<float2*>(d) = make_float2(o[0], o[1]);
    }
    __syncthreads();
    // pass 2
    const int wk = a.W >> K, hk = a.H >> K;
    float* dst = a.dst[K] + (size_t)f * a.dstride[K];
    for (int i = tid; i < OH * OW; i += 256) {
        const int oy = i / OW, ox = i - oy * OW;
        const int x = (X0 >> K) + ox, y = (Y0 >> K) + oy;
        if (x < wk && y < hk) {
            const float* col = P + ((oy << K) + OFF + PYR2_HL) * PP + ox;
            float v = ffb_blur_col_t<R>(col, PP, t);
            v = v * (1.f - 0.5f) + ffb_blur_col_t<R>(col + PP, PP, t) * 0.5f;
            dst[(size_t)y * a.dp[K] + x] = v;
        }
    }
    __syncthreads();
}

// Level 0 (3 x 3 taps, no decimation) straight from the staged window: one task = a 4 x 4 block of
// outputs from eighteen 16-byte shared loads (six window rows), both passes in registers, four 16-byte
// stores.  Same expressions as ffb_blur_row_t<1> / ffb_blur_col_t<1>.
__device__ __forceinline__ void ffb_pyr2_level0(const FfbPyr2Args& a, const float* reg, int X0, int Y0, int f, int tid) {
    const float k0 = a.taps[0].k[0], k1 = a.taps[0].k[1];
    float* dst = a.dst[0] + (size_t)f * a.dstride[0];
    for (int t = tid; t < (PYR2_TY / 4) * (PYR2_TX / 4); t += 256) {
        const int og = t / (PYR2_TX / 4), oy = 4 * og, ox = 4 * (t - og * (PYR2_TX / 4));
        const int x = X0 + ox, y = Y0 + oy;
        if (x >= a.W || y >= a.H) continue;
        float hrow[6][4];
#pragma unroll
        for (int r = 0; r < 6; ++r) {
            const float4* p = reinterpret_cast<const float4*>(reg + (oy + PYR2_HL - 1 + r) * PYR2_RWP + ox + PYR2_HL - 4);
            const float4 q0 = p[0], q1 = p[1], q2 = p[2];          // window columns ox-4 .. ox+7
            const float v[6] = {q0.w, q1.x, q1.y, q1.z, q1.w, q2.x};   // columns ox-1 .. ox+4
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                float s = k0 * v[1 + j];
                s += k1 * (v[j] + v[2 + j]);
                hrow[r][j] = s;
            }
        }
#pragma unroll
        for (int rr = 0; rr < 4; ++rr) {
            if (y + rr >= a.H) break;
            float o[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                float s = k0 * hrow[rr + 1][j];
                s += k1 * (hrow[rr][j] + hrow[rr + 2][j]);
                o[j] = s;
            }
            float* d = dst + (size_t)(y + rr) * a.dp[0] + x;
            if (x + 3 < a.W) {
                *reinterpret_cast<float4*>(d) = make_float4(o[0], o[1], o[2], o[3]);
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (x + j < a.W) d[j] = o[j];
            }
        }
    }
}

__global__ void __launch_bounds__(256) k_pyramid_pow2(FfbPyr2Args a) {
    FFB_DYN_SMEM(float, smem);
    float* reg = smem;                                  // [PYR2_RH][PYR2_RWP]
    float* P = smem + PYR2_RWP * PYR2_RH;               // [PYR2_RH][pitch of the level]
    const int tid = threadIdx.x;
    const int X0 = blockIdx.x * PYR2_TX, Y0 = blockIdx.y * PYR2_TY, f = blockIdx.z;
    const uint8_t* src = a.src + (size_t)f * a.src_frame_stride;
    const int W = a.W, H = a.H;
    // stage the window: one 4-pixel word per thread-iteration
    constexpr int WORDS = PYR2_RW / 4;
    for (int i = tid; i < PYR2_RH * WORDS; i += 256) {
        const int ry = i / WORDS, wx = i - ry * WORDS;
        const int sy = ffb_reflect1(Y0 - PYR2_HL + ry, H);
        const int sx = X0 - PYR2_HL + 4 * wx;
        const uint8_t* srow = src + (size_t)sy * a.src_pitch;
        float4 v;
        if (a.aligned && sx >= 0 && sx + 3 < W) {
            const unsigned u = __ldg(reinterpret_cast<const unsigned*>(srow + sx));
            v = make_float4((float)(u & 255u), (float)((u >> 8) & 255u), (float)((u >> 16) & 255u), (float)(u >> 24));
        } else {   // image border (REFLECT_101); far outside (only on partial tiles) is never used
            const int n2 = 2 * W - 2;
            int c0 = ffb_reflect1(min(sx, n2), W), c1 = ffb_reflect1(min(sx + 1, n2), W);
            int c2 = ffb_reflect1(min(sx + 2, n2), W), c3 = ffb_reflect1(min(sx + 3, n2), W);
            v = make_float4((float)__ldg(srow + c0), (float)__ldg(srow + c1), (float)__ldg(srow + c2), (float)__ldg(srow + c3));
        }
        *reinterpret_cast<float4*>(reg + ry * PYR2_RWP + 4 * wx) = v;
    }
    if (tid < PYR2_RH) *reinterpret_cast<float4*>(reg + tid * PYR2_RWP + PYR2_RW) = make_float4(0.f, 0.f, 0.f, 0.f);   // pitch padding
    __syncthreads();
    ffb_pyr2_level0(a, reg, X0, Y0, f, tid);
    if (a.nlev > 1) ffb_pyr2_level<1>(a, reg, P, X0, Y0, f, tid);
    if (a.nlev > 2) ffb_pyr2_level<2>(a, reg, P, X0, Y0, f, tid);
    if (a.nlev > 3) ffb_pyr2_level<3>(a, reg, P, X0, Y0, f, tid);
}

// ======================================================================================
// K1'' pyramid level with a large blur radius (deep levels: r > 9, or a tile window beyond shared memory)
// ======================================================================================
// The two passes of k_pyramid_level as two launches through a scratch image T[H][w]: the row pass evaluates the
// horizontal blur at the two resize taps of every output column on every source row and lerps them; the column pass
// evaluates the vertical blur of T at the two resize rows of every output row and lerps them.  Same taps, pairing and
// order as k_pyramid_level; the half kernel lives in device memory (any radius < min(W, H), REFLECT_101).
struct FfbPyrWideArgs {
    const uint8_t* src; size_t src_frame_stride; int src_pitch; int W, H;
    float* tmp; size_t tmp_frame_stride;                          // T[H][w] per frame (floats)
    float* dst; size_t dst_frame_stride; int dp; int w, h;        // strides in floats
    const int* xi; const float* xa; const int* yi; const float* ya;
    const float* k; int r;
};

__global__ void __launch_bounds__(256) k_pyramid_wide_rows(FfbPyrWideArgs a) {
    const int dx = blockIdx.x * 32 + (threadIdx.x & 31);
    const int y = blockIdx.y * 8 + (threadIdx.x >> 5);
    if (dx >= a.w || y >= a.H) return;
    const uint8_t* row = a.src + (size_t)blockIdx.z * a.src_frame_stride + (size_t)y * a.src_pitch;
    auto blur = [&](int c) {
        float s = __ldg(a.k) * (float)__ldg(row + c);
        for (int i = 1; i <= a.r; ++i)
            s += __ldg(a.k + i) * ((float)__ldg(row + ffb_reflect1(c - i, a.W)) + (float)__ldg(row + ffb_reflect1(c + i, a.W)));
        return s;
    };
    const int s0 = a.xi[dx];
    const float al = a.xa[dx];
    float v = blur(s0);
    if (al != 0.f) v = v * (1.f - al) + blur(min(s0 + 1, a.W - 1)) * al;
    a.tmp[(size_t)blockIdx.z * a.tmp_frame_stride + (size_t)y * a.w + dx] = v;
}

__global__ void __launch_bounds__(256) k_pyramid_wide_cols(FfbPyrWideArgs a) {
    const int dx = blockIdx.x * 32 + (threadIdx.x & 31);
    const int dy = blockIdx.y * 8 + (threadIdx.x >> 5);
    if (dx >= a.w || dy >= a.h) return;
    const float* col = a.tmp + (size_t)blockIdx.z * a.tmp_frame_stride + dx;
    auto blur = [&](int c) {
        float s = __ldg(a.k) * __ldg(col + (size_t)c * a.w);
        for (int i = 1; i <= a.r; ++i)
            s += __ldg(a.k + i) * (__ldg(col + (size_t)ffb_reflect1(c - i, a.H) * a.w) + __ldg(col + (size_t)ffb_reflect1(c + i, a.H) * a.w));
        return s;
    };
    const int s0 = a.yi[dy];
    const float be = a.ya[dy];
    float v = blur(s0);
    if (be != 0.f) v = v * (1.f - be) + blur(min(s0 + 1, a.H - 1)) * be;
    a.dst[(size_t)blockIdx.z * a.dst_frame_stride + (size_t)dy * a.dp + dx] = v;
}

// ======================================================================================
// K2  polynomial expansion: f32 image -> 5 planes (d/dy, d/dx, yy, xx, xy)
// ======================================================================================
// CTA = 256 threads = 128 columns x 2 row halves; it produces POLY_OW = 112 output columns (the
// other 10 + 6 columns are the replicate-border halo / padding) x POLY_ROWS rows.
//   phase V: each thread owns one column of one row half, loads its POLY_ROWS/2 + 10 input values
//            (all loads issued up front) and forms the three vertical sums (g, xg, xxg along y) of
//            every row of its half from registers -> shared rows vrow[3][POLY_ROWS][132]
//   phase H: each task = 4 adjacent outputs of one row: 4 aligned 16-byte shared loads per vertical
//            sum, six horizontal sums with the CPU code's symmetric pairing, 5 x 16-byte stores.
// N = poly_n: 5 (the reference's) or 7; the 112 output columns plus 2N halo columns fit the 128 loaded ones for both.
template <int N>
struct FfbPolyArgs {
    const float* src; size_t src_frame_stride; int sp; int w, h;  // strides in floats
    FfbRing dst;            // per frame-level: float4 [h][rp] (c0..c3) then float [h][rp] (c4); plane = rp * h
    size_t plane; int rp;
    FfbPolyConsts<N> c;
};

constexpr int POLY_OW = 112;
constexpr int POLY_ROWS = 32;
constexpr int POLY_VP = 132;    // shared row pitch (floats)
constexpr size_t POLY_SMEM = sizeof(float) * 3 * POLY_ROWS * POLY_VP;

template <int N>
__global__ void __launch_bounds__(256) k_polyexp(FfbPolyArgs<N> a) {
    static_assert(POLY_OW + 2 * N <= 128, "halo of the expansion");
    constexpr int NQ = (2 * N + 7) / 4;        // 16-byte loads per vertical sum in phase H (4 outputs + 2N halo)
    constexpr int HR = POLY_ROWS / 2;          // rows per half
    FFB_DYN_SMEM(float, vrow);                 // [3][POLY_ROWS][POLY_VP]
    const int tid = threadIdx.x;
    const int col = tid & 127, half = tid >> 7;
    const int x0 = blockIdx.x * POLY_OW, y0 = blockIdx.y * POLY_ROWS, f = blockIdx.z;
    const float* src = a.src + (size_t)f * a.src_frame_stride;
    const int w = a.w, h = a.h;
    // ---- phase V
    {
        const int x = ffb_clampi(x0 - N + col, 0, w - 1);      // replicate border
        const int yb = y0 + half * HR;
        float win[HR + 2 * N];
#pragma unroll
        for (int i = 0; i < HR + 2 * N; ++i) win[i] = __ldg(src + (size_t)ffb_clampi(yb - N + i, 0, h - 1) * a.sp + x);
#pragma unroll
        for (int r = 0; r < HR; ++r) {
            float t0 = win[r + N] * a.c.g[0], t1 = 0.f, t2 = 0.f;
#pragma unroll
            for (int k = 1; k <= N; ++k) {
                const float up = win[r + N - k], dn = win[r + N + k];
                const float p = up + dn;
                t0 += a.c.g[k] * p;
                t1 += a.c.xg[k] * (dn - up);
                t2 += a.c.xxg[k] * p;
            }
            const int row = half * HR + r;
            vrow[(0 * POLY_ROWS + row) * POLY_VP + col] = t0;
            vrow[(1 * POLY_ROWS + row) * POLY_VP + col] = t1;
            vrow[(2 * POLY_ROWS + row) * POLY_VP + col] = t2;
        }
        if (col < 4) {   // pad columns 128..131 are read (not used) by the last quad's 16-byte loads
#pragma unroll
            for (int r = 0; r < HR; ++r)
#pragma unroll
                for (int k = 0; k < 3; ++k) vrow[(k * POLY_ROWS + half * HR + r) * POLY_VP + 128 + col] = 0.f;
        }
    }
    __syncthreads();
    // ---- phase H
    constexpr int QUADS = POLY_OW / 4;
    float* dst0 = reinterpret_cast<float*>(ffb_ring_at(a.dst, f));
    for (int t = tid; t < QUADS * POLY_ROWS; t += 256) {
        const int r = t / QUADS, q = t - r * QUADS;
        const int x = x0 + 4 * q, y = y0 + r;
        if (x >= w || y >= h) continue;
        float v[3][4 * NQ];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const float4* p4 = reinterpret_cast<const float4*>(vrow + (k * POLY_ROWS + r) * POLY_VP + 4 * q);
#pragma unroll
            for (int j = 0; j < NQ; ++j) {
                const float4 t4 = p4[j];
                v[k][4 * j] = t4.x; v[k][4 * j + 1] = t4.y; v[k][4 * j + 2] = t4.z; v[k][4 * j + 3] = t4.w;
            }
        }
        float o[5][4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float* r0 = &v[0][j + N];
            const float* r1 = &v[1][j + N];
            const float* r2 = &v[2][j + N];
            float b1 = r0[0] * a.c.g[0], b2 = 0.f, b3 = r1[0] * a.c.g[0], b4 = 0.f, b5 = r2[0] * a.c.g[0], b6 = 0.f;
#pragma unroll
            for (int k = 1; k <= N; ++k) {
                const float pp = r0[k], mm = r0[-k];
                const float tg = pp + mm;
                b1 += tg * a.c.g[k];
                b4 += tg * a.c.xxg[k];
                b2 += (pp - mm) * a.c.xg[k];
                b3 += (r1[k] + r1[-k]) * a.c.g[k];
                b6 += (r1[k] - r1[-k]) * a.c.xg[k];
                b5 += (r2[k] + r2[-k]) * a.c.g[k];
            }
            o[0][j] = b3 * a.c.ig11;
            o[1][j] = b2 * a.c.ig11;
            o[2][j] = b1 * a.c.ig03 + b5 * a.c.ig33;
            o[3][j] = b1 * a.c.ig03 + b4 * a.c.ig33;
            o[4][j] = b6 * a.c.ig55;
        }
        // expansion layout: float4 (d/dy, d/dx, yy, xx) per pixel, then a separate float plane for xy
        const size_t pix = (size_t)y * a.rp + x;
        float4* dA = reinterpret_cast<float4*>(dst0) + pix;
        float* dB = dst0 + 4 * a.plane + pix;
        if (x + 3 < w) {   // x % 4 == 0 and rows are 64-byte aligned: the four pixels are two aligned 32-byte halves
            ffb_store_f8(reinterpret_cast<float*>(dA), make_float4(o[0][0], o[1][0], o[2][0], o[3][0]),
                         make_float4(o[0][1], o[1][1], o[2][1], o[3][1]));
            ffb_store_f8(reinterpret_cast<float*>(dA + 2), make_float4(o[0][2], o[1][2], o[2][2], o[3][2]),
                         make_float4(o[0][3], o[1][3], o[2][3], o[3][3]));
            *reinterpret_cast<float4*>(dB) = make_float4(o[4][0], o[4][1], o[4][2], o[4][3]);
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (x + j < w) {
                    dA[j] = make_float4(o[0][j], o[1][j], o[2][j], o[3][j]);
                    dB[j] = o[4][j];
                }
        }
    }
}

// ======================================================================================
// A1e  flow up-sampling between levels (bilinear, x2)
// ======================================================================================
struct FfbUpArgs {
    const float2* src; size_t src_stride; int sp; int wc, hc;     // strides in float2
    float2* dst; size_t dst_stride; int dp; int w, h;
    const int* xi; const float* xa; const int* yi; const float* ya;
    float scale;      // 1 / pyr_scale (SCALED only; otherwise the flow is doubled)
};

template <bool SCALED>
__global__ void __launch_bounds__(256) k_upsample_flow(FfbUpArgs a) {
    const int x = blockIdx.x * 32 + (threadIdx.x & 31);
    const int y = blockIdx.y * 8 + (threadIdx.x >> 5);
    if (x >= a.w || y >= a.h) return;
    const float2* src = a.src + (size_t)blockIdx.z * a.src_stride;
    const int x0 = a.xi[x], x1 = min(x0 + 1, a.wc - 1);
    const int y0 = a.yi[y], y1 = min(y0 + 1, a.hc - 1);
    const float al = a.xa[x], be = a.ya[y];
    const float2 p00 = src[(size_t)y0 * a.sp + x0], p01 = src[(size_t)y0 * a.sp + x1];
    const float2 p10 = src[(size_t)y1 * a.sp + x0], p11 = src[(size_t)y1 * a.sp + x1];
    const float tx = p00.x * (1.f - al) + p01.x * al, ty = p00.y * (1.f - al) + p01.y * al;
    const float bx = p10.x * (1.f - al) + p11.x * al, by = p10.y * (1.f - al) + p11.y * al;
    const float s = SCALED ? a.scale : 2.f;
    float2 o;
    o.x = (tx * (1.f - be) + bx * be) * s;
    o.y = (ty * (1.f - be) + by * be) * s;
    a.dst[(size_t)blockIdx.z * a.dst_stride + (size_t)y * a.dp + x] = o;
}

// ======================================================================================
// A1c  per-pixel matrix update (shared by the fused kernel and the stage hook)
// ======================================================================================
__device__ __forceinline__ float ffb_border_w(int d) {   // {0.14, 0.14, 0.4472, 0.4472, 0.4472}, 1 beyond
    return d < 2 ? 0.14f : (d < 5 ? 0.4472f : 1.f);
}

// R planes: channel c of pixel (x, y) at R[c * plane + y * rp + x].
__device__ __forceinline__ void ffb_compute_M(const float* __restrict__ R0, const float* __restrict__ R1,
                                              size_t plane, int rp, int w, int h, int x, int y,
                                              float dx, float dy, float m[5]) {
    float fx = (float)x + dx, fy = (float)y + dy;
    const float x1f = floorf(fx), y1f = floorf(fy);
    const int x1 = (int)x1f, y1 = (int)y1f;
    fx -= x1f;
    fy -= y1f;
    const float* q = R0 + (size_t)y * rp + x;
    const float r00 = __ldg(q), r01 = __ldg(q + plane), r02 = __ldg(q + 2 * plane), r03 = __ldg(q + 3 * plane),
                r04 = __ldg(q + 4 * plane);
    float r2, r3, r4, r5, r6;
    if ((unsigned)x1 < (unsigned)(w - 1) && (unsigned)y1 < (unsigned)(h - 1)) {
        const float a00 = (1.f - fx) * (1.f - fy), a01 = fx * (1.f - fy), a10 = (1.f - fx) * fy, a11 = fx * fy;
        const float* p = R1 + (size_t)y1 * rp + x1;
#define FFB_SAMP(c) (a00 * __ldg(p + (c)*plane) + a01 * __ldg(p + (c)*plane + 1) + a10 * __ldg(p + (c)*plane + rp) + a11 * __ldg(p + (c)*plane + rp + 1))
        r2 = FFB_SAMP(0);
        r3 = FFB_SAMP(1);
        r4 = (r02 + FFB_SAMP(2)) * 0.5f;
        r5 = (r03 + FFB_SAMP(3)) * 0.5f;
        r6 = (r04 + FFB_SAMP(4)) * 0.25f;
#undef FFB_SAMP
    } else {
        r2 = r3 = 0.f;
        r4 = r02;
        r5 = r03;
        r6 = r04 * 0.5f;
    }
    r2 = (r00 - r2) * 0.5f;
    r3 = (r01 - r3) * 0.5f;
    r2 += r4 * dy + r6 * dx;
    r3 += r6 * dy + r5 * dx;
    if ((unsigned)(x - 5) >= (unsigned)(w - 10) || (unsigned)(y - 5) >= (unsigned)(h - 10)) {
        const float s = ffb_border_w(x) * ffb_border_w(w - x - 1) * ffb_border_w(y) * ffb_border_w(h - y - 1);
        r2 *= s; r3 *= s; r4 *= s; r5 *= s; r6 *= s;
    }
    m[0] = r4 * r4 + r6 * r6;
    m[1] = (r4 + r5) * r6;
    m[2] = r5 * r5 + r6 * r6;
    m[3] = r4 * r2 + r6 * r3;
    m[4] = r6 * r2 + r5 * r3;
}

struct FfbMatArgs {
    const float* R0; const float* R1; size_t plane; int rp; int w, h;
    const float2* flow; int fp;
    float* M;   // 5 planes, same geometry as R
};
__global__ void __launch_bounds__(256) k_update_matrices(FfbMatArgs a) {
    const int x = blockIdx.x * 32 + (threadIdx.x & 31);
    const int y = blockIdx.y * 8 + (threadIdx.x >> 5);
    if (x >= a.w || y >= a.h) return;
    float2 d = make_float2(0.f, 0.f);
    if (a.flow) d = a.flow[(size_t)y * a.fp + x];
    float m[5];
    ffb_compute_M(a.R0, a.R1, a.plane, a.rp, a.w, a.h, x, y, d.x, d.y, m);
#pragma unroll
    for (int c = 0; c < 5; ++c) a.M[c * a.plane + (size_t)y * a.rp + x] = m[c];
}

// ======================================================================================
// K3  fused flow iteration: matrices -> 15x15 box mean (replicate border) -> 2x2 solve
// ======================================================================================
// One CTA owns a strip of SW output columns (plus a 7-column halo on each side: one thread per
// M column) and marches down a segment of SH rows, U rows per step.  The matrices never touch HBM:
//   * each thread gathers the inputs of the 5-vector M of its column, two rows at a time.  All loads are
//     unconditional (the R1 footprint is clamped into the image and the out-of-bounds fallback is
//     selected afterwards), so the 20 loads of a row pair are issued back to back; the flow of the next
//     step is prefetched one step ahead (it feeds the gather addresses),
//   * a Kahan-compensated running sum over the last 15 rows is kept per column (the column ring of
//     raw M values lives in shared memory so the row leaving the window can be subtracted),
//   * the vertical sums are published to a shared row buffer,
//   * the first U * (SW / HO) threads form the horizontal 15-sums for HO adjacent outputs from aligned
//     16-byte shared loads, solve the 2x2 system and store the flow vectors.  The horizontal phase of
//     step s-1 runs at the top of step s, before that step's loads are issued (fewer live registers).
// Warps whose 32 columns lie entirely beyond the strip's last needed column (the last strip of a level,
// narrow levels) skip the gather and the vertical sums; they only meet the barriers.
struct FfbIterArgs {
    FfbRing R;              // frame expansions: pair j uses elements PS*j (prev) and PS*j + 1 (next)
    int plane; int rp; int w, h;                     // plane = rp * h floats (< 2^31 / 5)
    const float2* fin; size_t fin_stride; int fip;   // flow in (NULL = zero), strides in float2
    FfbRing fout; int fop;                           // flow out ring (element j), pitch in float2
    int SW;                 // output columns per strip (multiple of HO, <= NT - 14)
    int SH;                 // rows per segment (even)
    // A1e fused (exact 2:1 levels only): when up_src != NULL the incoming flow is the coarser level's
    // result, up-sampled and doubled on the fly instead of being read from `fin`.
    const float2* up_src; size_t up_stride; int usp; int wc, hc;
};

// Shared row buffer of the vertical sums, one row of NT positions per (buffer, row of the step, channel).
// HO = 4: position p is stored at p.  HO = 8: a task reads the six 16-byte vectors 2g .. 2g+5 (g = task
// index), i.e. lanes are 32 bytes apart and a quarter-warp would hit every bank twice; the even and the
// odd vectors are therefore stored in two separate halves, so that the k-th load of consecutive tasks
// reads consecutive vectors (conflict-free), and the halves are 16 banks apart so that the 32 scalar
// stores of a publishing warp (16 to each half) do not collide either.
template <int NT, int HO>
struct FfbHrowLayout {
    static constexpr int HALF = NT / 2;
    static constexpr int HOFF = HO == 8 ? (HALF % 32 == 16 ? HALF : (HALF + 31) / 32 * 32 + 16) : 0;
    static constexpr int PITCH = HO == 8 ? HOFF + HALF : NT + 4;            // floats per (row, channel)
    static constexpr int RSTRIDE = HO == 8 ? 5 * PITCH + ((24 - (5 * PITCH) % 32) + 32) % 32 : 5 * PITCH;   // per row of a step
    __device__ __forceinline__ static int idx(int p) {
        return HO == 8 ? ((p >> 2) & 1) * HOFF + ((p >> 3) << 2) + (p & 3) : p;
    }
};

template <int NT, int U, int HO>
__host__ __device__ constexpr size_t ffb_flow_iter_smem() {
    // U = 2: the row buffer is double-buffered (one barrier per step); U = 4: single buffer, two barriers
    return sizeof(float) * ((U == 2 ? 2 : 1) * U * FfbHrowLayout<NT, HO>::RSTRIDE + FFB_WIN * 5 * NT);
}

// Raw inputs of one matrix update, as loaded (all loads unconditional).
struct FfbGather {
    float r0[5];      // R0 at the pixel
    float t[5][4];    // R1 footprint per channel: (y1,x1) (y1,x1+1) (y1+1,x1) (y1+1,x1+1), clamped into the image
    float fx, fy;     // fractional parts
    float dx, dy;
    int inside;
};

// Expansion layout (written by k_polyexp): per frame-level a float4 image A[h][rp] holding
// (d/dy, d/dx, yy, xx) per pixel followed by a float plane B[h][rp] holding xy.  A 2x2 bilinear
// footprint is then 4 x 16-byte + 4 x 4-byte loads off two row addresses instead of 20 scalar loads.
__device__ __forceinline__ void ffb_gather_issue(const float4* __restrict__ A0, const float* __restrict__ B0,
                                                 const float4* __restrict__ A1, const float* __restrict__ B1,
                                                 int rp, int w, int h, int x, int y, float2 d, FfbGather& g) {
    float fx = (float)x + d.x, fy = (float)y + d.y;
    const float x1f = floorf(fx), y1f = floorf(fy);
    const int x1 = (int)x1f, y1 = (int)y1f;
    g.fx = fx - x1f;
    g.fy = fy - y1f;
    g.dx = d.x;
    g.dy = d.y;
    g.inside = ((unsigned)x1 < (unsigned)(w - 1)) && ((unsigned)y1 < (unsigned)(h - 1));
    const int xs = min(max(x1, 0), w - 2), ys = min(max(y1, 0), h - 2);
    const unsigned o0 = (unsigned)(y * rp + x), o1 = (unsigned)(ys * rp + xs);
    const float4 q = __ldg(A0 + o0);
    const float q4 = __ldg(B0 + o0);
    const float4 t00 = __ldg(A1 + o1);
    const float4 t01 = __ldg(A1 + o1 + 1);
    const float4 t10 = __ldg(A1 + o1 + rp);
    const float4 t11 = __ldg(A1 + o1 + rp + 1);
    g.r0[0] = q.x; g.r0[1] = q.y; g.r0[2] = q.z; g.r0[3] = q.w; g.r0[4] = q4;
    g.t[0][0] = t00.x; g.t[0][1] = t01.x; g.t[0][2] = t10.x; g.t[0][3] = t11.x;
    g.t[1][0] = t00.y; g.t[1][1] = t01.y; g.t[1][2] = t10.y; g.t[1][3] = t11.y;
    g.t[2][0] = t00.z; g.t[2][1] = t01.z; g.t[2][2] = t10.z; g.t[2][3] = t11.z;
    g.t[3][0] = t00.w; g.t[3][1] = t01.w; g.t[3][2] = t10.w; g.t[3][3] = t11.w;
    g.t[4][0] = __ldg(B1 + o1);
    g.t[4][1] = __ldg(B1 + o1 + 1);
    g.t[4][2] = __ldg(B1 + o1 + rp);
    g.t[4][3] = __ldg(B1 + o1 + rp + 1);
}

__device__ __forceinline__ void ffb_gather_finish(const FfbGather& g, int w, int h, int x, int y, float m[5]) {
    const float fx = g.fx, fy = g.fy;
    const float a00 = (1.f - fx) * (1.f - fy), a01 = fx * (1.f - fy), a10 = (1.f - fx) * fy, a11 = fx * fy;
    float s[5];
#pragma unroll
    for (int c = 0; c < 5; ++c) s[c] = a00 * g.t[c][0] + a01 * g.t[c][1] + a10 * g.t[c][2] + a11 * g.t[c][3];
    float r2, r3, r4, r5, r6;
    if (g.inside) {
        r2 = s[0];
        r3 = s[1];
        r4 = (g.r0[2] + s[2]) * 0.5f;
        r5 = (g.r0[3] + s[3]) * 0.5f;
        r6 = (g.r0[4] + s[4]) * 0.25f;
    } else {
        r2 = r3 = 0.f;
        r4 = g.r0[2];
        r5 = g.r0[3];
        r6 = g.r0[4] * 0.5f;
    }
    r2 = (g.r0[0] - r2) * 0.5f;
    r3 = (g.r0[1] - r3) * 0.5f;
    r2 += r4 * g.dy + r6 * g.dx;
    r3 += r6 * g.dy + r5 * g.dx;
    if ((unsigned)(x - 5) >= (unsigned)(w - 10) || (unsigned)(y - 5) >= (unsigned)(h - 10)) {
        const float sc = ffb_border_w(x) * ffb_border_w(w - x - 1) * ffb_border_w(y) * ffb_border_w(h - y - 1);
        r2 *= sc; r3 *= sc; r4 *= sc; r5 *= sc; r6 *= sc;
    }
    m[0] = r4 * r4 + r6 * r6;
    m[1] = (r4 + r5) * r6;
    m[2] = r5 * r5 + r6 * r6;
    m[3] = r4 * r2 + r6 * r3;
    m[4] = r6 * r2 + r5 * r3;
}

// cv::resize(INTER_LINEAR) source index / weight for an exact 2:1 up-sampling (dst_n == 2 * src_n)
__device__ __forceinline__ void ffb_up2(int d, int src_n, int& i0, int& i1, float& al) {
    i0 = (d - 1) >> 1;                 // d = 0 -> -1
    al = (d & 1) ? 0.25f : 0.75f;
    if (i0 < 0) { i0 = 0; al = 0.f; }
    if (i0 >= src_n - 1) { i0 = src_n - 1; al = 0.f; }
    i1 = min(i0 + 1, src_n - 1);
}

// box mean -> 2x2 solve of one output (sums of the window of the five matrix channels; sc = 1 / winsize^2)
__device__ __forceinline__ float2 ffb_solve(float s0, float s1, float s2, float s3, float s4,
                                            float sc = 1.f / (float)(FFB_WIN * FFB_WIN)) {
    const float g11 = s0 * sc, g12 = s1 * sc, g22 = s2 * sc, h1 = s3 * sc, h2 = s4 * sc;
    // det = g11*g22 - g12*g12 with an exact-product correction (Kahan's ad-bc)
    const float wq = g12 * g12;
    const float e = __fmaf_rn(-g12, g12, wq);
    const float fd = __fmaf_rn(g11, g22, -wq);
    const float den = (fd + e) + 1e-3f;
    float idet = __fdividef(1.f, den);              // approximate reciprocal ...
    idet = idet * __fmaf_rn(-den, idet, 2.f);       // ... plus one Newton step (<= 1 ulp, no slow path)
    float2 o;
    o.x = (g11 * h2 - g12 * h1) * idet;
    o.y = (g22 * h1 - g12 * h2) * idet;
    return o;
}

// PS (pair stride): pair j reads the expansions in ring elements PS*j and PS*j + 1.  1: consecutive frames of a bracket
// (frame j+1 is `next` of pair j and `prev` of pair j+1); 2: independent pairs, staged as prev_0, next_0, prev_1, ...
// REV (slot order): pair j reads element PS*j + REV as R0 and PS*j + !REV as R1; REV = true is the backward flow of a
// pair (frame j+1 -> frame j of a bracket, next_j -> prev_j of independent pairs).
template <int NT, int U, int MINB, bool UP2X, int HO, int PS, bool REV>
__global__ void __launch_bounds__(NT, MINB) k_flow_iter(FfbIterArgs a) {
    static_assert(HO == 4 || HO == 8, "outputs per horizontal task");
    static_assert(U == 2 || U == 4, "rows per step");
    using HL = FfbHrowLayout<NT, HO>;
    constexpr int NB = U == 2 ? 2 : 1;               // row buffers
    // dynamic shared memory (exceeds the 48 KB static limit): row buffer first (16-byte aligned), then the ring
    FFB_DYN_SMEM(float, smem_f);
    float* hrow = smem_f;                                               // [NB][U] rows of RSTRIDE floats: [5][PITCH]
    typedef float (*RingT)[5][NT];
    RingT ring = reinterpret_cast<RingT>(smem_f + NB * U * HL::RSTRIDE);   // [FFB_WIN][5][NT]
    const int tid = threadIdx.x;
    const int pair = blockIdx.x;      // fastest-varying: see the launcher
    const float4* A0 = reinterpret_cast<const float4*>(ffb_ring_at(a.R, PS * pair + (REV ? 1 : 0)));
    const float4* A1 = reinterpret_cast<const float4*>(ffb_ring_at(a.R, PS * pair + (REV ? 0 : 1)));
    const float* B0 = reinterpret_cast<const float*>(A0 + a.plane);
    const float* B1 = reinterpret_cast<const float*>(A1 + a.plane);
    const float2* fin = a.fin ? a.fin + (size_t)pair * a.fin_stride : nullptr;
    float2* fout = reinterpret_cast<float2*>(ffb_ring_at(a.fout, pair));
    const int w = a.w, h = a.h;
    const int xo0 = (int)blockIdx.y * a.SW;
    const int useful = min(a.SW, w - xo0);                  // outputs of this strip
    const int xc = ffb_clampi(xo0 - FFB_WIN_R + tid, 0, w - 1);
    // a warp is live when at least one of its columns is a matrix column the strip's outputs need
    const bool live = (tid & ~31) < useful + 2 * FFB_WIN_R;
    const int hpos = HL::idx(tid);
    const int y0 = blockIdx.z * a.SH;
    const int y1 = min(y0 + a.SH, h);
    const int nfeed = (y1 - y0) + 2 * FFB_WIN_R;
    const int nsteps = (nfeed + U - 1) / U;
    // horizontal-phase role of this thread (fixed for the whole kernel)
    const int groups = (useful + HO - 1) / HO;
    const bool hz = tid < U * groups;
    const int hu = hz ? tid / groups : 0;
    const int hg = hz ? tid - hu * groups : 0;
    const int hx = xo0 + HO * hg;

    if (live) {
#pragma unroll
        for (int s = 0; s < FFB_WIN; ++s)
#pragma unroll
            for (int c = 0; c < 5; ++c) ring[s][c][tid] = 0.f;
    }
    if (HO == 4 && tid < 4) {      // positions NT .. NT+3 are read (not used) by the last task's 16-byte loads
#pragma unroll
        for (int b = 0; b < NB * U; ++b)
#pragma unroll
            for (int c = 0; c < 5; ++c) hrow[b * HL::RSTRIDE + c * HL::PITCH + NT + tid] = 0.f;
    }
    float vs[5] = {0.f, 0.f, 0.f, 0.f, 0.f}, comp[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
    int slot = 0;

    // horizontal sums + solve + store of the U rows published by step `s` into buffer `buf`
    auto horizontal = [&](int s, int buf) {
        const int i = s * U + hu;
        if (!hz || i < 2 * FFB_WIN_R || i >= nfeed) return;
        const int yo = y0 + i - 2 * FFB_WIN_R;
        const float* hb = hrow + (buf * U + hu) * HL::RSTRIDE;
        if (HO == 8) {
            // 8 adjacent outputs per task: 22 window elements from six 16-byte shared loads per channel
            // (three from the even half, three from the odd half);
            // sum_j = (e7..e14) + (e_j..e6) + (e15..e_{14+j})
            float sum8[5][8];
#pragma unroll
            for (int c = 0; c < 5; ++c) {
                const float4* he = reinterpret_cast<const float4*>(hb + c * HL::PITCH + 4 * hg);
                const float4* ho = reinterpret_cast<const float4*>(hb + c * HL::PITCH + HL::HOFF + 4 * hg);
                const float4 q0 = he[0], q1 = ho[0], q2 = he[1], q3 = ho[1], q4 = he[2], q5 = ho[2];
                const float e[24] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w, q2.x, q2.y, q2.z, q2.w,
                                     q3.x, q3.y, q3.z, q3.w, q4.x, q4.y, q4.z, q4.w, q5.x, q5.y, q5.z, q5.w};
                const float common = ((e[7] + e[8]) + (e[9] + e[10])) + ((e[11] + e[12]) + (e[13] + e[14]));
                float L[8], R[8];
                L[7] = 0.f;
                L[6] = e[6];
#pragma unroll
                for (int j = 5; j >= 0; --j) L[j] = e[j] + L[j + 1];
                R[0] = 0.f;
                R[1] = e[15];
#pragma unroll
                for (int j = 2; j < 8; ++j) R[j] = R[j - 1] + e[14 + j];
                sum8[c][0] = common + L[0];
                sum8[c][7] = common + R[7];
#pragma unroll
                for (int j = 1; j < 7; ++j) sum8[c][j] = common + (L[j] + R[j]);
            }
            float2 o8[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) o8[j] = ffb_solve(sum8[0][j], sum8[1][j], sum8[2][j], sum8[3][j], sum8[4][j]);
            float2* dst8 = fout + (yo * a.fop + hx);
            if (hx + 7 < w) {   // hx % 8 == 0, flow rows and buffers are 32-byte aligned (checked by the launcher)
                ffb_store_f8(reinterpret_cast<float*>(dst8), make_float4(o8[0].x, o8[0].y, o8[1].x, o8[1].y),
                             make_float4(o8[2].x, o8[2].y, o8[3].x, o8[3].y));
                ffb_store_f8(reinterpret_cast<float*>(dst8 + 4), make_float4(o8[4].x, o8[4].y, o8[5].x, o8[5].y),
                             make_float4(o8[6].x, o8[6].y, o8[7].x, o8[7].y));
            } else {
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    if (hx + j < w) dst8[j] = o8[j];
            }
        } else {
        float sum[5][4];
#pragma unroll
        for (int c = 0; c < 5; ++c) {
            const float4* hp = reinterpret_cast<const float4*>(hb + c * HL::PITCH + 4 * hg);
            const float4 q0 = hp[0], q1 = hp[1], q2 = hp[2], q3 = hp[3], q4 = hp[4];
            // window of output 0 = elements 0..14; each next output drops one, adds one
            const float mid = ((q0.w + q1.x) + (q1.y + q1.z)) + ((q1.w + q2.x) + (q2.y + q2.z)) +
                              ((q2.w + q3.x) + (q3.y + q3.z));          // elements 3..14
            sum[c][0] = mid + ((q0.x + q0.y) + q0.z);
            sum[c][1] = mid + ((q0.y + q0.z) + q3.w);
            sum[c][2] = mid + ((q0.z + q3.w) + q4.x);
            sum[c][3] = mid + ((q3.w + q4.x) + q4.y);
        }
        float2 o[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) o[j] = ffb_solve(sum[0][j], sum[1][j], sum[2][j], sum[3][j], sum[4][j]);
        float2* dst = fout + (yo * a.fop + hx);
        if (hx + 3 < w) {   // hx % 4 == 0, flow rows and buffers are 32-byte aligned (checked by the launcher)
            ffb_store_f8(reinterpret_cast<float*>(dst), make_float4(o[0].x, o[0].y, o[1].x, o[1].y),
                         make_float4(o[2].x, o[2].y, o[3].x, o[3].y));
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (hx + j < w) dst[j] = o[j];
        }
        }
    };

    // A1e fused (UP2X): the incoming flow is the coarser level's result, bilinearly up-sampled and
    // doubled on the fly.  Only instantiated for exact 2:1 level geometry, where cv::resize's table is
    // closed-form: output d reads source (d-1)>>1 (+1) with weight 0.75 (d even) / 0.25 (d odd),
    // clamped at both ends -- no table loads in the address chain.
    const float2* ups = UP2X ? a.up_src + (size_t)pair * a.up_stride : nullptr;
    int ux0 = 0, ux1 = 0;
    float ual = 0.f;
    if (UP2X) ffb_up2(xc, a.wc, ux0, ux1, ual);
    // flow vectors of feed rows i0, i0 + 1 of the segment (i0 even) at this thread's column
    auto load_flow2 = [&](int i0, float2& da, float2& db) {
        const int ya = ffb_clampi(y0 - FFB_WIN_R + i0, 0, h - 1), yb = ffb_clampi(y0 - FFB_WIN_R + i0 + 1, 0, h - 1);
        if (UP2X) {
            // The launcher makes SH even, so the two rows are an (odd, even) pair of image rows (or both clamped
            // to the same border row): they interpolate between the SAME two coarse rows, with weights
            // 0.25 / 0.75.  Fetch and x-interpolate those rows once for both (same arithmetic as k_upsample_flow).
            int uy0, uy1, vy0, vy1;
            float be0, be1;
            ffb_up2(ya, a.hc, uy0, uy1, be0);
            ffb_up2(yb, a.hc, vy0, vy1, be1);
            const float2 p00 = __ldg(ups + (uy0 * a.usp + ux0)), p01 = __ldg(ups + (uy0 * a.usp + ux1));
            const float2 p10 = __ldg(ups + (uy1 * a.usp + ux0)), p11 = __ldg(ups + (uy1 * a.usp + ux1));
            const float tx = p00.x * (1.f - ual) + p01.x * ual, ty = p00.y * (1.f - ual) + p01.y * ual;
            const float bx = p10.x * (1.f - ual) + p11.x * ual, by = p10.y * (1.f - ual) + p11.y * ual;
            da.x = (tx * (1.f - be0) + bx * be0) * 2.f;
            da.y = (ty * (1.f - be0) + by * be0) * 2.f;
            if (vy0 == uy0 && vy1 == uy1) {
                db.x = (tx * (1.f - be1) + bx * be1) * 2.f;
                db.y = (ty * (1.f - be1) + by * be1) * 2.f;
            } else {   // not reached with an even SH; kept so that any segmentation stays correct
                const float2 q00 = __ldg(ups + (vy0 * a.usp + ux0)), q01 = __ldg(ups + (vy0 * a.usp + ux1));
                const float2 q10 = __ldg(ups + (vy1 * a.usp + ux0)), q11 = __ldg(ups + (vy1 * a.usp + ux1));
                const float sx = q00.x * (1.f - ual) + q01.x * ual, sy = q00.y * (1.f - ual) + q01.y * ual;
                const float cx = q10.x * (1.f - ual) + q11.x * ual, cy = q10.y * (1.f - ual) + q11.y * ual;
                db.x = (sx * (1.f - be1) + cx * be1) * 2.f;
                db.y = (sy * (1.f - be1) + cy * be1) * 2.f;
            }
        } else if (fin) {
            da = __ldg(fin + (ya * a.fip + xc));
            db = __ldg(fin + (yb * a.fip + xc));
        } else {
            da = db = make_float2(0.f, 0.f);
        }
    };

    float2 d[U], dn[U];
    if (live) {
#pragma unroll
        for (int u = 0; u < U; u += 2) load_flow2(u, d[u], d[u + 1]);
    }
    // issue the gather of feed rows s*U + hh, + 1 (20 independent loads)
    auto issue_pair = [&](int s, int hh, FfbGather (&g)[2]) {
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int yc = ffb_clampi(y0 - FFB_WIN_R + s * U + hh + u, 0, h - 1);
            ffb_gather_issue(A0, B0, A1, B1, a.rp, w, h, xc, yc, d[hh + u], g[u]);
        }
    };
    for (int s = 0; s < nsteps; ++s) {
        const int buf = NB == 2 ? (s & 1) : 0;
        // the horizontal phase of the previous step runs before this step's loads are issued
        // (lower register pressure; the other resident warps cover the load latency)
        if (s > 0) horizontal(s - 1, NB == 2 ? (buf ^ 1) : 0);
        FfbGather g[2];
        if (live) issue_pair(s, 0, g);
#pragma unroll
        for (int hh = 0; hh < U; hh += 2) {
            float vrow[2][5];
            if (live) {
                load_flow2((s + 1) * U + hh, dn[hh], dn[hh + 1]);      // flow prefetch of step s+1 (feeds its gather addresses)
                // ---- matrices + vertical running sums (Kahan-compensated add of  new - leaving)
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    const int i = s * U + hh + u;
                    if (i < nfeed) {
                        const int yc = ffb_clampi(y0 - FFB_WIN_R + i, 0, h - 1);
                        float m[5];
                        ffb_gather_finish(g[u], w, h, xc, yc, m);
#pragma unroll
                        for (int c = 0; c < 5; ++c) {
                            const float old = ring[slot][c][tid];
                            ring[slot][c][tid] = m[c];
                            const float yk = (m[c] - old) - comp[c];
                            const float t = vs[c] + yk;
                            comp[c] = (t - vs[c]) - yk;
                            vs[c] = t;
                        }
                        slot = slot + 1 == FFB_WIN ? 0 : slot + 1;
                    }
#pragma unroll
                    for (int c = 0; c < 5; ++c) vrow[u][c] = vs[c];
                }
            }
            // single row buffer: the horizontal phase of step s-1 must have read it before it is overwritten
            if (NB == 1 && hh == 0) __syncthreads();
            if (live) {
#pragma unroll
                for (int u = 0; u < 2; ++u)
#pragma unroll
                    for (int c = 0; c < 5; ++c) hrow[(buf * U + hh + u) * HL::RSTRIDE + c * HL::PITCH + hpos] = vrow[u][c];
                if (hh + 2 < U) issue_pair(s, hh + 2, g);      // (issuing these before the barrier spills: -17 %)
            }
        }
        __syncthreads();
#pragma unroll
        for (int u = 0; u < U; ++u) d[u] = dn[u];
    }
    horizontal(nsteps - 1, NB == 2 ? ((nsteps - 1) & 1) : 0);
}

// ======================================================================================
// K3'  flow iteration for window sizes other than 15: matrices to HBM, then box sum + solve
// ======================================================================================
// k_flow_matrices: one thread per pixel gathers the production expansion layout (ffb_gather_*) and writes
// M = (G11, G12, G22, h1, h2) as five planes of rp x h floats per pair.
struct FfbMatrixArgs {
    FfbRing R; int plane; int rp; int w, h;          // as FfbIterArgs
    const float2* fin; size_t fin_stride; int fip;   // flow in (NULL = zero), strides in float2
    float* M; size_t m_stride;                       // per pair: 5 planes of `plane` floats
};

template <int PS, bool REV>   // pair stride and slot order, as k_flow_iter's
__global__ void __launch_bounds__(256) k_flow_matrices(FfbMatrixArgs a) {
    const int x = blockIdx.x * 32 + (threadIdx.x & 31);
    const int y = blockIdx.y * 8 + (threadIdx.x >> 5);
    if (x >= a.w || y >= a.h) return;
    const int pair = blockIdx.z;
    const float4* A0 = reinterpret_cast<const float4*>(ffb_ring_at(a.R, PS * pair + (REV ? 1 : 0)));
    const float4* A1 = reinterpret_cast<const float4*>(ffb_ring_at(a.R, PS * pair + (REV ? 0 : 1)));
    const float* B0 = reinterpret_cast<const float*>(A0 + a.plane);
    const float* B1 = reinterpret_cast<const float*>(A1 + a.plane);
    const float2 d = a.fin ? __ldg(a.fin + (size_t)pair * a.fin_stride + (size_t)y * a.fip + x) : make_float2(0.f, 0.f);
    FfbGather g;
    ffb_gather_issue(A0, B0, A1, B1, a.rp, a.w, a.h, x, y, d, g);
    float m[5];
    ffb_gather_finish(g, a.w, a.h, x, y, m);
    float* M = a.M + (size_t)pair * a.m_stride + (size_t)y * a.rp + x;
#pragma unroll
    for (int c = 0; c < 5; ++c) M[(size_t)c * a.plane] = m[c];
}

// k_box_solve: (2r+1) x (2r+1) box sums of M with replicate border, then the 2x2 solve with scale 1 / winsize^2
// (an even winsize sums 2 * (winsize / 2) + 1 taps, as OpenCV does).  One CTA = BOX_NT matrix columns (a strip of
// BOX_NT - 2r outputs) marching down a segment of SH rows; each thread keeps the vertical sums of its column in double
// (add the entering row, subtract the leaving one -- OpenCV keeps double sliding sums too), the outputs sum 2r+1 of
// them from shared memory in double.
constexpr int BOX_NT = 256;
struct FfbBoxArgs {
    const float* M; size_t m_stride; int plane; int rp; int w, h;
    int r; float scale;
    FfbRing fout; int fop;   // flow out ring (element = pair), pitch in float2
    int SW, SH;              // outputs per strip (BOX_NT - 2r), rows per segment
};

__global__ void __launch_bounds__(BOX_NT) k_box_solve(FfbBoxArgs a) {
    __shared__ double vrow[5][BOX_NT];
    const int tid = threadIdx.x;
    const int pair = blockIdx.x;
    const int w = a.w, h = a.h, r = a.r;
    const float* M = a.M + (size_t)pair * a.m_stride;
    float2* fout = reinterpret_cast<float2*>(ffb_ring_at(a.fout, pair));
    const int xo0 = (int)blockIdx.y * a.SW;
    const int useful = min(a.SW, w - xo0);
    const bool live = tid < useful + 2 * r;
    const int xc = ffb_clampi(xo0 - r + tid, 0, w - 1);
    const int y0 = (int)blockIdx.z * a.SH, y1 = min(y0 + a.SH, h);
    double vs[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
    if (live) {
        for (int i = -r; i <= r; ++i) {
            const float* p = M + (size_t)ffb_clampi(y0 + i, 0, h - 1) * a.rp + xc;
#pragma unroll
            for (int c = 0; c < 5; ++c) vs[c] += (double)__ldg(p + (size_t)c * a.plane);
        }
    }
    for (int y = y0; y < y1; ++y) {
#pragma unroll
        for (int c = 0; c < 5; ++c) vrow[c][tid] = vs[c];
        __syncthreads();
        if (tid < useful) {
            float s[5];
#pragma unroll
            for (int c = 0; c < 5; ++c) {
                double t = 0.0;
                for (int j = 0; j <= 2 * r; ++j) t += vrow[c][tid + j];
                s[c] = (float)t;
            }
            fout[(size_t)y * a.fop + xo0 + tid] = ffb_solve(s[0], s[1], s[2], s[3], s[4], a.scale);
        }
        __syncthreads();
        if (live && y + 1 < y1) {
            const float* pin = M + (size_t)ffb_clampi(y + 1 + r, 0, h - 1) * a.rp + xc;
            const float* pout = M + (size_t)ffb_clampi(y - r, 0, h - 1) * a.rp + xc;
#pragma unroll
            for (int c = 0; c < 5; ++c)
                vs[c] += (double)__ldg(pin + (size_t)c * a.plane) - (double)__ldg(pout + (size_t)c * a.plane);
        }
    }
}

// ======================================================================================
// K3b forward-backward consistency of pairs whose forward and backward final flows are resident
// ======================================================================================
// Sundaram, Brox & Keutzer (ECCV 2010).  One thread per pixel (x, y) of pair j: the forward flow f sends it to
// t = (x + fx, y + fy).  A target outside [0, w-1] x [0, h-1] (NaN included) is inconsistent; otherwise the backward
// flow is sampled bilinearly at t (b) and the pixel is consistent when |f + b|^2 <= alpha (|f|^2 + |b|^2) + beta.
// Every operation is one fp32 rounding in this order, with no contraction, so that a float32 restatement gives the same
// bits; the consistent pixels of a pair are counted with integer atomics, so the count is deterministic.
struct FfbCheckArgs {
    FfbRing fw, bw; int fp;     // forward / backward flows (element = pair), pitch in float2
    int w, h;
    FfbRing mask; int mp;       // mask bytes 1 / 0 (element = pair), pitch in bytes; mask.base NULL: no mask
    unsigned* count;            // consistent pixels of pair j added to count[j] (NULL: not counted)
    float alpha, beta;
};

__global__ void __launch_bounds__(256) k_fb_check(FfbCheckArgs a) {
    const int x = blockIdx.x * 32 + (threadIdx.x & 31);
    const int y = blockIdx.y * 8 + (threadIdx.x >> 5);
    const int pair = blockIdx.z;
    bool ok = false;
    if (x < a.w && y < a.h) {
        const float2* F = reinterpret_cast<const float2*>(ffb_ring_at(a.fw, pair));
        const float2* Bk = reinterpret_cast<const float2*>(ffb_ring_at(a.bw, pair));
        const float2 f = __ldg(F + (size_t)y * a.fp + x);
        const float tx = __fadd_rn((float)x, f.x), ty = __fadd_rn((float)y, f.y);
        if (tx >= 0.f && tx <= (float)(a.w - 1) && ty >= 0.f && ty <= (float)(a.h - 1)) {
            const float x0f = floorf(tx), y0f = floorf(ty);
            const int x0 = (int)x0f, y0 = (int)y0f;
            const int x1 = min(x0 + 1, a.w - 1), y1 = min(y0 + 1, a.h - 1);
            const float ax = __fsub_rn(tx, x0f), ay = __fsub_rn(ty, y0f);
            const float rx = __fsub_rn(1.f, ax), ry = __fsub_rn(1.f, ay);
            const float2 b00 = __ldg(Bk + (size_t)y0 * a.fp + x0), b01 = __ldg(Bk + (size_t)y0 * a.fp + x1);
            const float2 b10 = __ldg(Bk + (size_t)y1 * a.fp + x0), b11 = __ldg(Bk + (size_t)y1 * a.fp + x1);
            const float bx = __fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(b00.x, rx), __fmul_rn(b01.x, ax)), ry),
                                       __fmul_rn(__fadd_rn(__fmul_rn(b10.x, rx), __fmul_rn(b11.x, ax)), ay));
            const float by = __fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(b00.y, rx), __fmul_rn(b01.y, ax)), ry),
                                       __fmul_rn(__fadd_rn(__fmul_rn(b10.y, rx), __fmul_rn(b11.y, ax)), ay));
            const float ex = __fadd_rn(f.x, bx), ey = __fadd_rn(f.y, by);
            const float e = __fadd_rn(__fmul_rn(ex, ex), __fmul_rn(ey, ey));
            const float nf = __fadd_rn(__fmul_rn(f.x, f.x), __fmul_rn(f.y, f.y));
            const float nb = __fadd_rn(__fmul_rn(bx, bx), __fmul_rn(by, by));
            ok = e <= __fadd_rn(__fmul_rn(a.alpha, __fadd_rn(nf, nb)), a.beta);
        }
        if (a.mask.base) ffb_ring_at(a.mask, pair)[(size_t)y * a.mp + x] = ok ? 1 : 0;
    }
    if (a.count) {      // a warp is one row of 32 pixels: one atomic per warp
        unsigned n = ok ? 1u : 0u;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) n += __shfl_xor_sync(0xffffffffu, n, o);
        if ((threadIdx.x & 31) == 0 && n) atomicAdd(a.count + pair, n);
    }
}

// ======================================================================================
// K4  swapped-axis "divergence" argmax + magnitude sum   (A3 + A4)
// ======================================================================================
struct FfbDivArgs {
    FfbRing flow; int fp; int w, h;     // pitch in float2
    int rows_per_block;
    unsigned long long* pkey;           // [pairs][gridDim.x]
    double* psum;                       // [pairs][gridDim.x]
};

// One thread = 4 adjacent pixels of a row: the flow vectors of the row above, the row itself and the row
// below arrive as three 32-byte loads (rows are 32-byte aligned, pitch % 4 == 0); the horizontal
// neighbours of the group's end pixels come from the adjacent lanes (one scalar load at the warp ends).
__global__ void __launch_bounds__(256) k_divmag(FfbDivArgs a) {
    __shared__ unsigned long long skey[8];
    __shared__ double ssum[8];
    const int pair = blockIdx.z;
    const float2* F = reinterpret_cast<const float2*>(ffb_ring_at(a.flow, pair));
    const int w = a.w, h = a.h, fp = a.fp;
    const int ylo = blockIdx.x * a.rows_per_block, yhi = min(ylo + a.rows_per_block, h);
    const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;
    const int lane = threadIdx.x & 31;
    // per-thread maximum as (|div| bits, pixel index): a thread visits its pixels in increasing index order, so a
    // strict comparison keeps the first maximum; the 64-bit key is only built once at the end
    unsigned best_a = 0u, best_i = 0u;
    double msum = 0.0;
    for (int y = ylo + ty; y < yhi; y += 4) {
        const float2* row = F + (size_t)y * fp;
        const float2* up = F + (size_t)(y > 0 ? y - 1 : 0) * fp;
        const float2* dn = F + (size_t)(y < h - 1 ? y + 1 : h - 1) * fp;
        const float ysc = (y > 0 && y < h - 1) ? 0.5f : 1.f;
        // the trip count is the same for all lanes of a warp (the shuffles below need the whole warp)
        for (int xw = 4 * (tx - lane); xw < w; xw += 256) {
            const int x = xw + 4 * lane;
            const bool active = x < w;
            float cxv[4], cyv[4], uav[4], ubv[4];
            if (active) {
                float4 lo, hi;
                ffb_load_f8(reinterpret_cast<const float*>(row + x), lo, hi);
                cxv[0] = lo.x; cyv[0] = lo.y; cxv[1] = lo.z; cyv[1] = lo.w; cxv[2] = hi.x; cyv[2] = hi.y; cxv[3] = hi.z; cyv[3] = hi.w;
                ffb_load_f8(reinterpret_cast<const float*>(up + x), lo, hi);
                uav[0] = lo.x; uav[1] = lo.z; uav[2] = hi.x; uav[3] = hi.z;
                ffb_load_f8(reinterpret_cast<const float*>(dn + x), lo, hi);
                ubv[0] = lo.x; ubv[1] = lo.z; ubv[2] = hi.x; ubv[3] = hi.z;
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) cxv[j] = cyv[j] = uav[j] = ubv[j] = 0.f;
            }
            float lft = __shfl_up_sync(0xffffffffu, cyv[3], 1);       // v at x - 1
            float rgt = __shfl_down_sync(0xffffffffu, cyv[0], 1);     // v at x + 4
            if (active) {
                if (lane == 0 && x > 0) lft = __ldg(row + (x - 1)).y;
                if (lane == 31 && x + 4 < w) rgt = __ldg(row + (x + 4)).y;
                float m4 = 0.f;      // magnitudes of the (up to) 4 pixels, added in fp32 before they join the fp64 sum
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int xj = x + j;
                    if (xj < w) {
                        // np.gradient: (f[i+1]-f[i-1])/2 inside, one-sided first differences at the ends
                        const float vl = xj > 0 ? (j > 0 ? cyv[j > 0 ? j - 1 : 0] : lft) : cyv[0];
                        const float vr = xj < w - 1 ? (j < 3 ? cyv[j < 3 ? j + 1 : 3] : rgt) : cyv[j];
                        const float xsc = (xj > 0 && xj < w - 1) ? 0.5f : 1.f;
                        const float gu = __fmul_rn(__fsub_rn(ubv[j], uav[j]), ysc);
                        const float gv = __fmul_rn(__fsub_rn(vr, vl), xsc);
                        const unsigned av = __float_as_uint(fabsf(__fadd_rn(gu, gv)));
                        if (av > best_a) { best_a = av; best_i = (unsigned)(y * w + xj); }
                        m4 = __fadd_rn(m4, sqrtf(__fmaf_rn(cxv[j], cxv[j], __fmul_rn(cyv[j], cyv[j]))));
                    }
                }
                msum += (double)m4;
            }
        }
    }
    // (bits(|div|) << 32) | ~index: the largest key is the largest |div|, ties broken by the smallest index.  A thread
    // that saw only zeros (or nothing) offers pixel 0 of ITS OWN range, which loses against any real pixel 0 tie-break
    // only if its own first index is larger -- so it offers the smallest index it visited instead (or none).
    const bool any = ylo + ty < yhi && 4 * tx < w;
    if (best_a == 0u && any) best_i = (unsigned)((ylo + ty) * w + 4 * tx);
    unsigned long long best = any ? (((unsigned long long)best_a << 32) | (unsigned long long)(0xFFFFFFFFu - best_i)) : 0ull;
    best = ffb_warp_max_u64(best);
    msum = ffb_warp_sum(msum);
    const int warp = threadIdx.x >> 5;
    if (lane == 0) { skey[warp] = best; ssum[warp] = msum; }
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long b = skey[0];
        double s = ssum[0];
        for (int i = 1; i < 8; ++i) { b = skey[i] > b ? skey[i] : b; s += ssum[i]; }
        a.pkey[(size_t)pair * gridDim.x + blockIdx.x] = b;
        a.psum[(size_t)pair * gridDim.x + blockIdx.x] = s;
    }
}

struct FfbP1Args {
    FfbRing flow; int fp; int w, h;
    const unsigned long long* pkey; const double* psum; int nblk;
    int pov; float cut_threshold;
    int out0;                 // index of the batch's first pair inside the bracket arrays
    int* cx; int* cy; float* val; float* mean_mag; unsigned char* cut;
};

__global__ void __launch_bounds__(32) k_phase1_finish(FfbP1Args a) {
    const int pair = blockIdx.x;
    const int lane = threadIdx.x;
    unsigned long long best = 0ull;
    double s = 0.0;
    for (int i = lane; i < a.nblk; i += 32) {
        const unsigned long long k = a.pkey[(size_t)pair * a.nblk + i];
        best = k > best ? k : best;
        s += a.psum[(size_t)pair * a.nblk + i];
    }
    best = ffb_warp_max_u64(best);
    s = ffb_warp_sum(s);
    if (lane == 0) {
        const int w = a.w, h = a.h;
        const int o = a.out0 + pair;
        const float mm = (float)(s / ((double)w * (double)h));
        a.mean_mag[o] = mm;
        a.cut[o] = mm > a.cut_threshold ? 1 : 0;
        if (a.pov) {   // F:880-882
            a.cx[o] = w / 2;
            a.cy[o] = h - 1;
            a.val[o] = 0.f;
        } else {
            const unsigned idx = 0xFFFFFFFFu - (unsigned)(best & 0xFFFFFFFFull);
            const int y = (int)(idx / (unsigned)w), x = (int)(idx - (unsigned)y * (unsigned)w);
            const float2* F = reinterpret_cast<const float2*>(ffb_ring_at(a.flow, pair));
            const float ua = F[(size_t)(y > 0 ? y - 1 : 0) * a.fp + x].x;
            const float ub = F[(size_t)(y < h - 1 ? y + 1 : h - 1) * a.fp + x].x;
            const float vl = F[(size_t)y * a.fp + (x > 0 ? x - 1 : 0)].y;
            const float vr = F[(size_t)y * a.fp + (x < w - 1 ? x + 1 : w - 1)].y;
            const float gu = __fmul_rn(__fsub_rn(ub, ua), (y > 0 && y < h - 1) ? 0.5f : 1.f);
            const float gv = __fmul_rn(__fsub_rn(vr, vl), (x > 0 && x < w - 1) ? 0.5f : 1.f);
            a.cx[o] = x;
            a.cy[o] = y;
            a.val[o] = __fadd_rn(gu, gv);
        }
    }
}

// ======================================================================================
// A5  +-6 centre mean (F:1203-1214)
// ======================================================================================
// cx, cy hold the raw centres of n consecutive pairs of one bracket (the whole bracket, or -- for a shard of
// it -- the shard plus up to 6 pairs on each side); centre j is written to centers[2 * (j - out_shift)].
__global__ void __launch_bounds__(128) k_smooth_centers(const int* cx, const int* cy, int n, int j0, int j1, int out_shift,
                                                        double* centers /* [..][2] */) {
    const int j = j0 + blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= j1) return;
    const int lo = max(0, j - 6), hi = min(n, j + 7);
    long long sx = 0, sy = 0;
    for (int i = lo; i < hi; ++i) { sx += cx[i]; sy += cy[i]; }
    centers[2 * (j - out_shift)] = (double)sx / (double)(hi - lo);
    centers[2 * (j - out_shift) + 1] = (double)sy / (double)(hi - lo);
}

// ======================================================================================
// K5  balanced weighted radial projection mean   (A6)
// ======================================================================================
// result = 1/(HW) * sum_y wy(y) * [ sum_x u*wx(x)*(x-cx) + (y-cy) * sum_x v*wx(x) ]
// with wx = (W-x)/W for x > cx else x/W (same for y); POV mode: wx = wy = 1.
struct FfbRadArgs {
    FfbRing flow; int fp; int w, h;
    int rows_per_block;
    const double* centers;       // [bracket pairs][2]
    const unsigned char* cut;    // [bracket pairs]
    int out0;                    // bracket index of ring element 0 of this launch
    int pov;
    double* partial;             // [pairs][gridDim.y * gridDim.x]
};

__global__ void __launch_bounds__(256) k_radial(FfbRadArgs a) {
    __shared__ double ssum[8];
    const int pair = blockIdx.z;
    const int o = a.out0 + pair;
    const int nblk = gridDim.x * gridDim.y;
    const int bid = blockIdx.y * gridDim.x + blockIdx.x;
    if (a.cut[o]) {   // F:766-767: a cut contributes exactly 0.0 and its flow is never read
        if (threadIdx.x == 0) a.partial[(size_t)pair * nblk + bid] = 0.0;
        return;
    }
    const float2* F = reinterpret_cast<const float2*>(ffb_ring_at(a.flow, pair));
    const double cx = a.centers[2 * o], cy = a.centers[2 * o + 1];
    const int w = a.w, h = a.h;
    const int x = blockIdx.x * 256 + threadIdx.x;
    const int ylo = blockIdx.y * a.rows_per_block, yhi = min(ylo + a.rows_per_block, h);
    double acc = 0.0;
    if (x < w) {
        const double wxd = a.pov ? 1.0 : (((double)x > cx) ? (double)(w - x) / (double)w : (double)x / (double)w);
        const float wx = (float)wxd;
        const float ax = (float)(wxd * ((double)x - cx));
        const double inv_h = 1.0 / (double)h;      // one division per thread, not one per row
#pragma unroll 8
        for (int y = ylo; y < yhi; ++y) {
            const float2 f = __ldg(F + (size_t)y * a.fp + x);
            const double wy = a.pov ? 1.0 : (double)(((double)y > cy) ? h - y : y) * inv_h;
            const float dyf = (float)((double)y - cy);
            const float t = __fmaf_rn(f.x, ax, __fmul_rn(__fmul_rn(f.y, wx), dyf));
            acc += (double)t * wy;
        }
    }
    acc = ffb_warp_sum(acc);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) ssum[warp] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int i = 0; i < 8; ++i) s += ssum[i];
        a.partial[(size_t)pair * nblk + bid] = s;
    }
}

__global__ void __launch_bounds__(32) k_radial_finish(const double* partial, int nblk, int w, int h, int out0,
                                                      double* scalar) {
    const int pair = blockIdx.x;
    double s = 0.0;
    for (int i = threadIdx.x; i < nblk; i += 32) s += partial[(size_t)pair * nblk + i];
    s = ffb_warp_sum(s);
    if (threadIdx.x == 0) scalar[out0 + pair] = s / ((double)w * (double)h);
}

// ======================================================================================
// N2  frame pre-processing: decoded BGR frame -> 256 x 256 gray  (F:173-189, F:1057-1082)
// ======================================================================================
// cv2.resize(INTER_LINEAR) in OpenCV's 8-bit fixed-point arithmetic (11-bit weights, horizontal pass
// in int, vertical  (((b0*(H0>>4))>>16) + ((b1*(H1>>4))>>16) + 2) >> 2 ) on the RGB channels, then
// cv2.cvtColor(RGB2GRAY) = (9798 R + 19235 G + 3735 B + 16384) >> 15.  Integer work: bit-exact.
// VR mode: the resize target is 512 x 512 and only its bottom-left 256 x 256 quadrant is produced.
struct FfbPreArgs {
    const uint8_t* src; size_t src_frame_stride; int src_pitch;   // BGR, 3 bytes per pixel
    uint8_t* dst; size_t dst_frame_stride; int dst_pitch;          // gray OW x OH
    const int* xt;    // [4][TW]: x0, x1, a0, a1 per resized column
    const int* yt;    // [4][TH]: y0, y1, b0, b1 per resized row
    int TW, TH;       // resize target (256 x 256, 512 x 512 in VR mode, or the source size)
    int x_off, y_off; // first resized column / row that is kept (VR: the bottom-left quadrant)
    int OW, OH;       // size of the kept window = size of the gray output
};

__global__ void __launch_bounds__(256) k_preprocess(FfbPreArgs a) {
    const int x = blockIdx.x * 32 + (threadIdx.x & 31);
    const int y = blockIdx.y * 8 + (threadIdx.x >> 5);
    if (x >= a.OW || y >= a.OH) return;
    const int ry = y + a.y_off, rx = x + a.x_off;
    const int x0 = a.xt[rx] * 3, x1 = a.xt[a.TW + rx] * 3, a0 = a.xt[2 * a.TW + rx], a1 = a.xt[3 * a.TW + rx];
    const int y0 = a.yt[ry], y1 = a.yt[a.TH + ry], b0 = a.yt[2 * a.TH + ry], b1 = a.yt[3 * a.TH + ry];
    const uint8_t* src = a.src + (size_t)blockIdx.z * a.src_frame_stride;
    const uint8_t* r0 = src + (size_t)y0 * a.src_pitch;
    const uint8_t* r1 = src + (size_t)y1 * a.src_pitch;
    int rgb[3];
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {          // ch indexes RGB; the source is BGR
        const int o = 2 - ch;
        const int h0 = (int)__ldg(r0 + x0 + o) * a0 + (int)__ldg(r0 + x1 + o) * a1;
        const int h1 = (int)__ldg(r1 + x0 + o) * a0 + (int)__ldg(r1 + x1 + o) * a1;
        rgb[ch] = (((b0 * (h0 >> 4)) >> 16) + ((b1 * (h1 >> 4)) >> 16) + 2) >> 2;
    }
    const int gray = (9798 * rgb[0] + 19235 * rgb[1] + 3735 * rgb[2] + 16384) >> 15;
    a.dst[(size_t)blockIdx.z * a.dst_frame_stride + (size_t)y * a.dst_pitch + x] = (uint8_t)gray;
}

// ======================================================================================
// X9  warp by a dense flow: cv2.remap(src, flow, None, INTER_LINEAR | WARP_RELATIVE_MAP) on uint8 frames
// ======================================================================================
// cv2's 8-bit arithmetic in integers, bit-exact.  Per axis, with f the flow component at output pixel x:
//   R  = cvRound(32 f)                    NaN, +-inf and |32 f| >= 2^31 give INT_MIN (cvRound on x86; __float2int_rn
//                                         would saturate instead, and map NaN to 0)
//   x0 = saturate_short((R >> 5) + x)     the left tap column (cv2 adds the integer grid after rounding: rounding
//   ax = R & 31                           x + f in float32 first would differ where that sum rounds)
// cv2's 15-bit weights are the products (32 - ax | ax) (32 - ay | ay) * 32: exact, summing to 32768 (the entry of
// ax = ay = 0 holds 32767 and a 1, which still returns the tap itself), so the output
// (sum w_k v_k + 16384) >> 15 equals (sum W_k v_k + 512) >> 10 with W_k the 10-bit products, per channel.
// Borders: constant -- a tap outside the frame reads the border value; replicate -- each tap's coordinates are
// clamped.  Frames are narrower and lower than 32767 px (cv2's limit), so x0 + 1 never overflows a short's range.
// One thread = 4 consecutive output pixels of a row (a warp = 128 pixels): their flows are one 256-bit load when the
// flow rows are 32-byte aligned, their outputs one 32-bit store per channel when the output rows are 4-byte aligned.
struct FfbRemapArgs {
    const uint8_t* src; size_t src_stride, src_pitch;   // image i at src + i * src_stride, C bytes per pixel
    FfbRing flow; size_t fp;                           // flow of image i: ring element i, rows fp bytes apart
    uint8_t* dst; size_t dst_stride, dst_pitch;
    int w, h;
    int border_value;
    bool flow_v8, dst_v4;
};

__device__ __forceinline__ int ffb_remap_round(float f) {
    const float s = __fmul_rn(f, 32.f);   // exact: a power of two
    return s >= -2147483648.f && s < 2147483648.f ? (int)rintf(s) : -2147483647 - 1;
}

template <int C, bool REPLICATE>
__device__ __forceinline__ void ffb_remap_px(const FfbRemapArgs& a, const uint8_t* S, int x, int y, float fx, float fy,
                                             uint8_t* out) {
    const int rx = ffb_remap_round(fx), ry = ffb_remap_round(fy);
    const int x0 = ffb_clampi((rx >> 5) + x, -32768, 32767), y0 = ffb_clampi((ry >> 5) + y, -32768, 32767);
    const int wx[2] = {32 - (rx & 31), rx & 31}, wy[2] = {32 - (ry & 31), ry & 31};
    int acc[C];
#pragma unroll
    for (int c = 0; c < C; ++c) acc[c] = 0;
#pragma unroll
    for (int dy = 0; dy < 2; ++dy) {
#pragma unroll
        for (int dx = 0; dx < 2; ++dx) {
            const int w = wx[dx] * wy[dy];
            int tx = x0 + dx, ty = y0 + dy;
            if (REPLICATE) {
                tx = ffb_clampi(tx, 0, a.w - 1);
                ty = ffb_clampi(ty, 0, a.h - 1);
            } else if (tx < 0 || tx >= a.w || ty < 0 || ty >= a.h) {
#pragma unroll
                for (int c = 0; c < C; ++c) acc[c] += w * a.border_value;
                continue;
            }
            const uint8_t* p = S + (size_t)ty * a.src_pitch + (size_t)tx * C;
#pragma unroll
            for (int c = 0; c < C; ++c) acc[c] += w * (int)__ldg(p + c);
        }
    }
#pragma unroll
    for (int c = 0; c < C; ++c) out[c] = (uint8_t)((acc[c] + 512) >> 10);
}

template <int C, bool REPLICATE>
__global__ void __launch_bounds__(256) k_remap_flow(FfbRemapArgs a) {
    const int x = (blockIdx.x * 32 + (threadIdx.x & 31)) * 4;
    const int y = blockIdx.y * 8 + (threadIdx.x >> 5);
    if (x >= a.w || y >= a.h) return;
    const int img = blockIdx.z;
    const int n = min(4, a.w - x);
    const float* F = reinterpret_cast<const float*>(ffb_ring_at(a.flow, img) + (size_t)y * a.fp) + 2 * x;
    float f[8];
    if (a.flow_v8 && n == 4) {
        float4 lo, hi;
        ffb_load_f8(F, lo, hi);
        f[0] = lo.x; f[1] = lo.y; f[2] = lo.z; f[3] = lo.w; f[4] = hi.x; f[5] = hi.y; f[6] = hi.z; f[7] = hi.w;
    } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) f[i] = i < 2 * n ? __ldg(F + i) : 0.f;
    }
    const uint8_t* S = a.src + (size_t)img * a.src_stride;
    uint8_t out[4 * C];
#pragma unroll
    for (int i = 0; i < 4; ++i)
        if (i < n) ffb_remap_px<C, REPLICATE>(a, S, x + i, y, f[2 * i], f[2 * i + 1], out + i * C);
    uint8_t* D = a.dst + (size_t)img * a.dst_stride + (size_t)y * a.dst_pitch + (size_t)x * C;
    if (a.dst_v4 && n == 4) {
#pragma unroll
        for (int c = 0; c < C; ++c)
            reinterpret_cast<unsigned*>(D)[c] = (unsigned)out[4 * c] | (unsigned)out[4 * c + 1] << 8 |
                                                (unsigned)out[4 * c + 2] << 16 | (unsigned)out[4 * c + 3] << 24;
    } else {
#pragma unroll
        for (int i = 0; i < 4 * C; ++i)
            if (i < n * C) D[i] = out[i];
    }
}
