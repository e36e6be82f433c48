// Device-side pieces of raw2outputs shared by composite.cu (inerf_composite_fwd / _bwd) and render_fused.cu (inerf_render_rays_fused).
// Reference: NeRFs/HeadNeRF/train/baseline.py:325-375, NeRFs/TorsoNeRF/test_torso.py:352-402.
#pragma once
#include "common.cuh"

namespace inerf {

// Reduce 8 per-lane values across the warp with 9 shuffles.  Afterwards lane 4*q holds the full
// sum of quantity q (replicated on lanes 4q..4q+3).
__device__ __forceinline__ float reduce8(float (&v)[8], int lane) {
    const bool hi16 = lane & 16, hi8 = lane & 8, hi4 = lane & 4;
    float a[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        float send = hi16 ? v[j] : v[j + 4];
        float keep = hi16 ? v[j + 4] : v[j];
        a[j] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
    }
    float b[2];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        float send = hi8 ? a[j] : a[j + 2];
        float keep = hi8 ? a[j + 2] : a[j];
        b[j] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
    }
    float send = hi4 ? b[0] : b[1];
    float keep = hi4 ? b[1] : b[0];
    float c = keep + __shfl_xor_sync(0xffffffffu, send, 4);
    c += __shfl_xor_sync(0xffffffffu, c, 2);
    c += __shfl_xor_sync(0xffffffffu, c, 1);
    return c;
}

// exp / sigmoid through the SFU (ex2.approx, rcp.approx): <= 2 ulp on ex2 plus the rounding of x*log2(e), i.e. an absolute
// error below 3e-7 on alpha and on the colours -- three orders under the 1e-3 gate, and 60 fewer issue slots per
// 32 samples than the IEEE expf + division (the kernel was issue bound, not HBM bound, with those).
__device__ __forceinline__ float fast_exp(float x) {                                             // FMUL + MUFU.EX2
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x * 1.4426950408889634f));
    return r;
}
__device__ __forceinline__ float sigmoidf_(float x) { return __fdividef(1.0f, 1.0f + fast_exp(-x)); }

struct Sample {
    float alpha, q, dist, s;   // s = sigma + noise (pre-relu)
};

__device__ __forceinline__ Sample make_sample(float sigma, float noise, float z, float znext, float norm, bool last,
                                              bool valid) {
    Sample o;
    o.s = sigma + noise;
    o.dist = (last ? 1e10f : (znext - z)) * norm;
    float e = fast_exp(-(fmaxf(o.s, 0.0f) + 1e-6f) * o.dist);
    o.alpha = valid ? 1.0f - e : 0.0f;
    o.q = valid ? (1.0f - o.alpha) + 1e-10f : 1.0f;
    return o;
}

// inclusive multiplicative scan over the warp
__device__ __forceinline__ float warp_scan_mul(float p, int lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        float t = __shfl_up_sync(0xffffffffu, p, o);
        if (lane >= o) p *= t;
    }
    return p;
}

// inclusive additive suffix scan over the warp (lane l gets sum over lanes >= l)
__device__ __forceinline__ float warp_suffix_add(float p, int lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        float t = __shfl_down_sync(0xffffffffu, p, o);
        if (lane + o < 32) p += t;
    }
    return p;
}

// Forward for even S (every production shape: 64, 192): lane l owns the two ADJACENT samples 2l, 2l+1 of each
// 64-sample chunk, so raw arrives as one 256-bit load per lane (LDG.256, 1 KB contiguous per warp), z / weights as
// 64-bit accesses, and the transmittance scan runs once per 64 samples on the per-lane product q_a*q_b -- half the
// shuffles and selects per sample of the one-sample-per-lane form above (which stays for odd S).
struct Raw2 { float4 a, b; };

__device__ __forceinline__ Raw2 ldg_stream8(const float4* p) {
    Raw2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(r.a.x), "=f"(r.a.y), "=f"(r.a.z), "=f"(r.a.w), "=f"(r.b.x), "=f"(r.b.y), "=f"(r.b.z), "=f"(r.b.w)
                 : "l"(p));
    return r;
}

__device__ __forceinline__ float2 ldg_stream2(const float* p) {
    float2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0,%1}, [%2];" : "=f"(r.x), "=f"(r.y) : "l"(p));
    return r;
}

// One ray of raw2outputs for even S, executed by one warp (the body of composite_fwd2_kernel; also the first half of the fused
// compositor + importance sampler and the NaN-flagging final compositor of inerf_render_rays_fused, render_fused.cu).  weights may be
// NULL (the fine pass of an inference render only needs its last entry); last_weight: NULL or (n).  z_c0 / w_c0 return the lane's two
// depths / weights of chunk 0 (S = 64: the whole ray).  Returns a bit mask of the non-finite outputs this lane wrote
// (1 rgb, 2 disp, 4 acc, 8 depth, 16 last_weight).
// SIG = 1 or 4: the sigma-only form (the coarse pass of a render that discards its colour).  Only the densities are read, sample i's at
// ((const float*)raw)[i * SIG + SIG - 1] -- a density-only buffer (1) or the sigma lane of a full raw (4) -- and rgb, rgb_fg, bc_rgb
// are not touched; weights, depth, disp, acc and last_weight are the bits of the full form (reduce8 sums each quantity on its own).
template <int C, int SIG = 0>
__device__ __forceinline__ uint32_t composite2_ray(
    const float4* __restrict__ raw, const float* __restrict__ z, const float* __restrict__ rays_d, int d_stride,
    const float* __restrict__ bc_rgb, const float* __restrict__ noise, int ray, int s, int white_bkgd,
    float* __restrict__ rgb, float* __restrict__ disp, float* __restrict__ acc, float* __restrict__ depth,
    float* __restrict__ weights, float* __restrict__ rgb_fg, float* __restrict__ last_weight, int lane, float2& z_c0, float2& w_c0) {
    const size_t base = (size_t)ray * s;

    Raw2 rv[C];
    float2 zv[C], nv[C];
#pragma unroll
    for (int c = 0; c < C; ++c) {
        const int i = c * 64 + 2 * lane;                       // s is even: i < s  <=>  i + 1 < s
        const bool ok = i < s;
        if (ok) {
            if constexpr (SIG == 0) {
                rv[c] = ldg_stream8(raw + base + i);
            } else {
                const float* sg = reinterpret_cast<const float*>(raw) + (base + i) * SIG + (SIG - 1);
                const float2 s2 = SIG == 1 ? ldg_stream2(sg) : make_float2(ldg_stream(sg), ldg_stream(sg + SIG));
                rv[c].a = make_float4(0.f, 0.f, 0.f, s2.x);
                rv[c].b = make_float4(0.f, 0.f, 0.f, s2.y);
            }
            zv[c] = ldg_stream2(z + base + i);
            nv[c] = noise ? ldg_stream2(noise + base + i) : make_float2(0.f, 0.f);
        } else {
            rv[c].a = rv[c].b = make_float4(0.f, 0.f, 0.f, 0.f);
            zv[c] = nv[c] = make_float2(0.f, 0.f);
        }
    }
    const float* dptr = rays_d + (size_t)ray * d_stride;
    const float dx = dptr[0], dy = dptr[1], dz = dptr[2];
    const float norm = sqrtf(dx * dx + dy * dy + dz * dz);
    const float bcr = SIG ? 0.f : bc_rgb[ray * 3], bcg = SIG ? 0.f : bc_rgb[ray * 3 + 1], bcb = SIG ? 0.f : bc_rgb[ray * 3 + 2];

    float carry = 1.0f;
    uint32_t bad = 0;
    float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int c = 0; c < C; ++c) {
        const int i = c * 64 + 2 * lane;
        const bool valid = i < s, last_b = i + 1 == s - 1;     // the ray's last sample is always a `b`
        float znext = __shfl_down_sync(0xffffffffu, zv[c].x, 1);
        if (c + 1 < C) {
            const float z0 = __shfl_sync(0xffffffffu, zv[c + 1 < C ? c + 1 : c].x, 0);
            if (lane == 31) znext = z0;
        }
        const Sample sa = make_sample(rv[c].a.w, nv[c].x, zv[c].x, zv[c].y, norm, false, valid);
        const Sample sb = make_sample(rv[c].b.w, nv[c].y, zv[c].y, znext, norm, last_b, valid);
        const float incl = warp_scan_mul(sa.q * sb.q, lane);
        float excl = __shfl_up_sync(0xffffffffu, incl, 1);
        if (lane == 0) excl = 1.0f;
        const float Ta = carry * excl;
        const float Tb = Ta * sa.q;
        carry *= __shfl_sync(0xffffffffu, incl, 31);
        const float wa = sa.alpha * Ta, wb = sb.alpha * Tb;
        if (valid && weights) *reinterpret_cast<float2*>(weights + base + i) = make_float2(wa, wb);
        if (last_b && last_weight) { last_weight[ray] = wb; if (!isfinite(wb)) bad |= 16u; }
        if (c == 0) { z_c0 = zv[0]; w_c0 = make_float2(wa, wb); }
        if constexpr (SIG == 0) {
            const float ar = sigmoidf_(rv[c].a.x), ag = sigmoidf_(rv[c].a.y), ab = sigmoidf_(rv[c].a.z);
            const float br = sigmoidf_(rv[c].b.x), bg = sigmoidf_(rv[c].b.y), bb = sigmoidf_(rv[c].b.z);
            const float fr = wa * ar + (last_b ? 0.f : wb * br);   // foreground sums exclude the background sample
            const float fg = wa * ag + (last_b ? 0.f : wb * bg);
            const float fb = wa * ab + (last_b ? 0.f : wb * bb);
            v[5] += fr; v[6] += fg; v[7] += fb;
            v[0] += last_b ? fr + wb * bcr : fr;
            v[1] += last_b ? fg + wb * bcg : fg;
            v[2] += last_b ? fb + wb * bcb : fb;
        }
        v[3] += wa * zv[c].x + wb * zv[c].y;
        v[4] += wa + wb;
    }
    const float tot = reduce8(v, lane);                            // lane 4q holds quantity q
    const float acc_t = __shfl_sync(0xffffffffu, tot, 16);
    const float depth_t = __shfl_sync(0xffffffffu, tot, 12);
    const int q = lane >> 2;
    if ((lane & 3) == 0) {
        if (q < 3) {
            if constexpr (SIG == 0) {
                const float v_ = white_bkgd ? tot + (1.0f - acc_t) : tot;
                rgb[ray * 3 + q] = v_;
                if (!isfinite(v_)) bad |= 1u;
            }
        } else if (q == 3) {
            const float dp = __fdiv_rn(1.0f, fmaxf(1e-10f, __fdiv_rn(depth_t, acc_t)));
            depth[ray] = depth_t;
            disp[ray] = dp;
            if (!isfinite(dp)) bad |= 2u;
            if (!isfinite(depth_t)) bad |= 8u;
        } else if (q == 4) {
            acc[ray] = acc_t;
            if (!isfinite(acc_t)) bad |= 4u;
        } else if (!SIG && rgb_fg) rgb_fg[ray * 3 + (q - 5)] = tot;
    }
    return bad;
}

}  // namespace inerf
