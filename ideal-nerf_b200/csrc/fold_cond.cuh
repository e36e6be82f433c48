// Conditioning fold (SURVEY.md Appendix B; face_nerf.py:44-56,69): the per-call constant columns [aud | expr/3 | latent] of pts_linears.0 / .5 and
// views_linears.0 become biases, written as fp32 (CondLayout) and as the operand tiles of the two tensor-core kernels.  The block body is
// shared by fold_cond_kernel (mlp_fp32.cu, launched by inerf_mlp_fold_cond: one net per launch) and the set-up kernel of
// inerf_render_rays_fused (render_fused.cu: both nets of a render_rays call plus the rays and coarse depths in ONE launch).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.cuh"

namespace inerf {

struct FoldArgs {
    const float* w[INERF_N_PARAMS];
    const float* aud; const float* expr; const float* latent;
    int da, de, dl;
    float* cond;
};
int mlp_fold_cond_launch(const FoldArgs& f, cudaStream_t st);      // mlp_fp32.cu

// Row `r` of a bias tile for the tensor-core kernel (mlp_bf16.cu): K-major, non-swizzled [rows][16] bf16 stored as 8x8 core
// matrices, columns (hi, lo, 0, ..., 0) with hi + lo = the fp32 bias to 16 mantissa bits.
__device__ __forceinline__ void write_bias_tile_row(uint8_t* tile, int r, float b) {
    const __nv_bfloat16 hi = __float2bfloat16_rn(b);
    const __nv_bfloat16 lo = __float2bfloat16_rn(b - __bfloat162float(hi));
    const uint32_t w0 = (uint32_t)__bfloat16_as_ushort(hi) | ((uint32_t)__bfloat16_as_ushort(lo) << 16);
    uint8_t* p = tile + (r >> 3) * 256 + (r & 7) * 16;
    *reinterpret_cast<uint4*>(p) = make_uint4(w0, 0u, 0u, 0u);
    *reinterpret_cast<uint4*>(p + 128) = make_uint4(0u, 0u, 0u, 0u);
}

// The same row for the fp32-gate tensor-core kernel (mlp_f16x2.cu): fp16, columns (hi, mid, lo, 0, ...) = the bias split in three fp16
// numbers (exact to 2^-33 relative for |b| >= 2^-14); these tiles follow the bf16 ones in `cond`.
__device__ __forceinline__ void write_bias_tile_row_f16x3(uint8_t* tile, int r, float b) {
    const __half hi = __float2half_rn(b);
    const float r1 = b - __half2float(hi);
    const __half mid = __float2half_rn(r1);
    const __half lo = __float2half_rn(r1 - __half2float(mid));
    const uint32_t w0 = (uint32_t)__half_as_ushort(hi) | ((uint32_t)__half_as_ushort(mid) << 16);
    uint8_t* p = tile + (r >> 3) * 256 + (r & 7) * 16;
    *reinterpret_cast<uint4*>(p) = make_uint4(w0, (uint32_t)__half_as_ushort(lo), 0u, 0u);
    *reinterpret_cast<uint4*>(p + 128) = make_uint4(0u, 0u, 0u, 0u);
}

// One block of the fold: bx in [0, 12) = layer (8 pts_linears, 3 views_linears, the two head biases), by in [0, 8) = row group; 256 threads;
// c = 1024 floats of shared memory.
__device__ __forceinline__ void fold_cond_block(const FoldArgs& f, int bx, int by, float* c) {
    uint8_t* tiles = reinterpret_cast<uint8_t*>(f.cond + COND_FLOATS);
    const int C = f.da + f.de + f.dl;
    for (int i = threadIdx.x; i < C; i += blockDim.x) {
        float v;
        if (i < f.da) v = f.aud[i];
        else if (i < f.da + f.de) v = __fdiv_rn(__fmul_rn(f.expr[i - f.da], 1.0f), 3.0f);   // expr * 1 / 3  (face_nerf.py:49)
        else v = f.latent[i - f.da - f.de];
        c[i] = v;
    }
    __syncthreads();
    const CondLayout cl{256, 128};
    const int b = bx, lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    if (b < 8) {                                  // pts_linears.b
        const float* W = f.w[2 * b];
        const float* B = f.w[2 * b + 1];
        const int ldw = (b == 0) ? 63 + C : (b == 5 ? 319 + C : 256);
        const bool folded = (b == 0 || b == 5) && C > 0;
        for (int n = by * 32 + warp; n < by * 32 + 32; n += nwarp) {      // grid.y = 8 row groups: the rows are independent
            float s = 0.f;
            if (folded)
                for (int j = lane; j < C; j += 32) s = fmaf(W[(size_t)n * ldw + 63 + j], c[j], s);
            s = warp_sum(s);
            if (lane == 0) {
                f.cond[cl.pts(b) + n] = B[n] + s;
                write_bias_tile_row(tiles + bias_tile_offset(b, n >> 7), n & 127, B[n] + s);
                write_bias_tile_row_f16x3(tiles + BIAS_TILE_BYTES + bias_tile_offset(b, n >> 7), n & 127, B[n] + s);
            }
        }
    } else if (b < 11) {                          // views_linears.(b-8)
        const int v = b - 8;
        const float* W = f.w[P_VIEWS_W + 2 * v];
        const float* B = f.w[P_VIEWS_W + 2 * v + 1];
        const int ldw = 283 + f.de;
        for (int n = by * 16 + warp; n < by * 16 + 16; n += nwarp) {
            float s = 0.f;
            if (v == 0)
                for (int j = lane; j < f.de; j += 32) s = fmaf(W[(size_t)n * ldw + 283 + j], c[f.da + j], s);
            s = warp_sum(s);
            if (lane == 0) {
                f.cond[cl.views(v) + n] = B[n] + s;
                write_bias_tile_row(tiles + bias_tile_offset(b, n >> 6), n & 63, B[n] + s);
                write_bias_tile_row_f16x3(tiles + BIAS_TILE_BYTES + bias_tile_offset(b, n >> 6), n & 63, B[n] + s);
            }
        }
    } else if (threadIdx.x < 4 && by == 0) {
        f.cond[cl.alpha_b() + threadIdx.x] = threadIdx.x == 0 ? f.w[P_ALPHA_B][0] : f.w[P_RGB_B][threadIdx.x - 1];
    }
}

}  // namespace inerf
