// ffb_common.h -- shared host/device declarations for the sm_100a kernels.
#pragma once

#ifdef FFB_EMU
#include "cuda_emu.h"   // tests/emu: host emulation used only by the CPU test-suite
#define FFB_LAUNCH(kernel, grid, block, smem, stream, ...) \
    emu::launch((grid), (block), (smem), [=]() { kernel(__VA_ARGS__); })
#define FFB_DYN_SMEM(type, name) type* name = reinterpret_cast<type*>(emu::g_dyn_smem)
#else
#include <cuda_runtime.h>
#define FFB_LAUNCH(kernel, grid, block, smem, stream, ...) \
    kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__)
#define FFB_DYN_SMEM(type, name) \
    extern __shared__ __align__(16) unsigned char ffb_dyn_smem_raw[]; \
    type* name = reinterpret_cast<type*>(ffb_dyn_smem_raw)
#endif

#include <stddef.h>
#include <stdint.h>

// ---- 256-bit global store (sm_100+, STG.E.ENL2.256): eight floats at a 32-byte aligned address.
// A thread that owns 32 contiguous bytes fills a whole DRAM/L2 sector with one instruction instead of
// half a sector with each of two 16-byte stores.
#ifdef FFB_EMU
static inline void ffb_store_f8(float* p, float4 lo, float4 hi) {
    reinterpret_cast<float4*>(p)[0] = lo;
    reinterpret_cast<float4*>(p)[1] = hi;
}
#else
__device__ __forceinline__ void ffb_store_f8(float* p, float4 lo, float4 hi) {
    asm volatile("st.global.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "f"(lo.x), "f"(lo.y), "f"(lo.z),
                 "f"(lo.w), "f"(hi.x), "f"(hi.y), "f"(hi.z), "f"(hi.w)
                 : "memory");
}
#endif

// 256-bit read-only global load (LDG.E.ENL2.256.CONSTANT): eight floats from a 32-byte aligned address
#ifdef FFB_EMU
static inline void ffb_load_f8(const float* p, float4& lo, float4& hi) {
    lo = reinterpret_cast<const float4*>(p)[0];
    hi = reinterpret_cast<const float4*>(p)[1];
}
#else
__device__ __forceinline__ void ffb_load_f8(const float* p, float4& lo, float4& hi) {
    asm volatile("ld.global.nc.v8.f32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=f"(lo.x), "=f"(lo.y), "=f"(lo.z), "=f"(lo.w), "=f"(hi.x), "=f"(hi.y), "=f"(hi.z), "=f"(hi.w)
                 : "l"(p));
}
#endif

// FFB_MAX_LEVELS sizes the single-pass pyramid (k_pyramid_pow2, levels 0..3); a context's level table holds up to
// FFB_PLAN_LEVELS levels.  FFB_WIN is the window of the fused k_flow_iter (other window sizes take k_flow_matrices +
// k_box_solve).
#define FFB_MAX_LEVELS 4
#define FFB_PLAN_LEVELS 16
#define FFB_WIN 15
#define FFB_WIN_R 7

// Half of a symmetric 1-D kernel: k[0] is the centre tap, k[i] the taps at +-i.
struct FfbTaps {
    int r;
    float k[10];
};

// Polynomial-expansion constants of a (2N+1)-tap expansion (FarnebackPrepareGaussian, computed on the host in double).
template <int N>
struct FfbPolyConsts {
    float g[N + 1];
    float xg[N + 1];
    float xxg[N + 1];
    float ig11, ig03, ig33, ig55;
};

// A ring of equally sized device buffers: element j lives at base + ((first + j) % mod) * stride.
struct FfbRing {
    char* base;
    size_t stride;   // bytes
    int first;
    int mod;
};
__host__ __device__ __forceinline__ char* ffb_ring_at(const FfbRing& r, int j) {
    return r.base + (size_t)((r.first + j) % r.mod) * r.stride;
}

static __host__ __device__ __forceinline__ int ffb_round_up(int v, int m) { return (v + m - 1) / m * m; }
