// Shared helpers for the inerf_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/inerf_b200.h"

namespace inerf {

void set_error(const char* fmt, ...);

inline int fail(int code, const char* msg) {
    set_error("%s", msg);
    return code;
}

// Launch-error check: returns a positive cudaError_t through the C ABI.
inline int check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("%s: %s", what, cudaGetErrorString(e));
        return (int)e;
    }
    return INERF_OK;
}

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

inline int num_sms() {
    static thread_local int cached_dev = -1, cached = 0;
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev != cached_dev) {
        cudaDeviceGetAttribute(&cached, cudaDevAttrMultiProcessorCount, dev);
        cached_dev = dev;
    }
    return cached > 0 ? cached : 148;
}

// FaceNeRF parameter slots (include/inerf_b200.h, INERF_N_PARAMS)
enum { P_PTS_W = 0, P_VIEWS_W = 16, P_ALPHA_W = 22, P_ALPHA_B = 23, P_RGB_W = 24, P_RGB_B = 25 };
inline int pts_w(int i) { return 2 * i; }
inline int pts_b(int i) { return 2 * i + 1; }
inline int views_w(int i) { return 16 + 2 * i; }
inline int views_b(int i) { return 17 + 2 * i; }

// Offsets (floats) inside the folded-bias buffer written by inerf_mlp_fold_cond.
struct CondLayout {
    int W, H;          // 256, 128
    __host__ __device__ int pts(int i) const { return i * W; }
    __host__ __device__ int views(int i) const { return 8 * W + i * H; }
    __host__ __device__ int alpha_b() const { return 8 * W + 3 * H; }
    __host__ __device__ int rgb_b() const { return 8 * W + 3 * H + 1; }
    __host__ __device__ constexpr int total() const { return 8 * W + 3 * H + 4; }
};

// `cond` of one call: the COND_FLOATS folded fp32 biases (CondLayout{256, 128}), then two bias-tile sets for the tensor-core kernels
// (fold_cond.cuh): the bf16 set, then the fp16x2 set.  A set holds one tile per (layer, half): 4 KB for the 8 pts_linears (128 rows),
// 2 KB for the 3 views_linears (64 rows).
constexpr int COND_FLOATS = CondLayout{256, 128}.total();
constexpr int BIAS_TILE_BYTES = 16 * 4096 + 6 * 2048;
__host__ __device__ constexpr uint32_t bias_tile_offset(int layer, int half) {
    return layer < 8 ? (2 * layer + half) * 4096u : 65536u + (2 * (layer - 8) + half) * 2048u;
}

inline int check_dims(const InerfNetDims* d) {
    if (!d) return fail(INERF_E_ARG, "dims is NULL");
    if (d->width != 256 || d->depth != 8 || d->in_xyz != 63 || d->in_views != 27)
        return fail(INERF_E_UNSUPPORTED, "only D=8, W=256, in_xyz=63, in_views=27 FaceNeRF is built");
    if (d->dim_aud < 0 || d->dim_expr < 0 || d->dim_latent < 0 || d->dim_aud + d->dim_expr + d->dim_latent > 1024)
        return fail(INERF_E_SHAPE, "conditioning dims out of range");
    return INERF_OK;
}

}  // namespace inerf

// ---------------------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ float4 ldg_stream4(const float4* p) {
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
                 : "l"(p));
    return r;
}

__device__ __forceinline__ float ldg_stream(const float* p) {
    float r;
    asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(r) : "l"(p));
    return r;
}
