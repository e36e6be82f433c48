// Ray generation / packing, positional encoding, stratified coarse depths, head/torso blend.
//
// All arithmetic that feeds the bit-exact sample_pdf gate uses explicit round-to-nearest
// intrinsics (__fmul_rn/__fadd_rn are never contracted into FMA), so the depths equal the
// reference's tensor-op-at-a-time fp32 values (SURVEY.md Appendix A1-A2).
#include "common.cuh"
#include "philox.cuh"
#include "rays_parts.cuh"

using namespace inerf;

// ---------------------------------------------------------------------------------------------
// get_rays + packing.  helper.py:228-243, audio_exp_nerf.py:409-427
// ---------------------------------------------------------------------------------------------
// rays of the pixels [first, first + count) of the row-major H x W grid; rays[0] is pixel `first`
__global__ void get_rays_kernel(int W, int first, int count, float focal, float cx, float cy, const float* __restrict__ c2w,
                                int rs, float near_, float far_, float* __restrict__ rays) {
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= count) return;
    int row = (first + idx) / W, col = (first + idx) - row * W;
    float d[3];
    pixel_dir((float)row, (float)col, focal, cx, cy, c2w, rs, d);
    store_ray(rays + (size_t)idx * 11, c2w[3], c2w[rs + 3], c2w[2 * rs + 3], d[0], d[1], d[2], near_, far_);
}

__global__ void pack_rays_kernel(const float* __restrict__ o, const float* __restrict__ d, int n, float near_,
                                 float far_, float* __restrict__ rays) {
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n) return;
    store_ray(rays + (size_t)idx * 11, o[idx * 3], o[idx * 3 + 1], o[idx * 3 + 2], d[idx * 3], d[idx * 3 + 1],
              d[idx * 3 + 2], near_, far_);
}

// Rays of SELECTED pixels only (training batches): the reference builds the full H x W ray grid for every sample and then indexes
// N_rand of them (audio_exp_nerf.py:123-139,189-191); same arithmetic as get_rays_kernel, one thread per selected pixel.
__global__ void get_rays_at_kernel(const long long* __restrict__ coords, int n, float focal, float cx, float cy,
                                   const float* __restrict__ c2w, int rs, float near_, float far_, float* __restrict__ rays) {
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n) return;
    const float row = (float)coords[2 * idx], col = (float)coords[2 * idx + 1];
    float d[3];
    pixel_dir(row, col, focal, cx, cy, c2w, rs, d);
    store_ray(rays + (size_t)idx * 11, c2w[3], c2w[rs + 3], c2w[2 * rs + 3], d[0], d[1], d[2], near_, far_);
}

extern "C" int inerf_get_rays_at(const int64_t* coords, int n, float focal, float cx, float cy, const float* c2w, int c2w_row_stride,
                                 float near_, float far_, float* rays, void* stream) {
    if (n < 0 || c2w_row_stride < 4) return fail(INERF_E_SHAPE, "inerf_get_rays_at: bad n / c2w_row_stride");
    if (n == 0) return INERF_OK;
    if (!coords || !c2w || !rays) return fail(INERF_E_ARG, "inerf_get_rays_at: NULL pointer");
    get_rays_at_kernel<<<(n + 255) / 256, 256, 0, as_stream(stream)>>>(reinterpret_cast<const long long*>(coords), n, focal, cx, cy, c2w,
                                                                      c2w_row_stride, near_, far_, rays);
    return check_launch("inerf_get_rays_at");
}

extern "C" int inerf_get_rays(int H, int W, float focal, float cx, float cy, const float* c2w, int c2w_row_stride,
                              float near_, float far_, float* rays, void* stream) {
    if (!c2w || !rays) return fail(INERF_E_ARG, "inerf_get_rays: NULL pointer");
    if (H <= 0 || W <= 0 || (int64_t)H * W > (1 << 30) || c2w_row_stride < 4)
        return fail(INERF_E_SHAPE, "inerf_get_rays: bad H/W/c2w_row_stride");
    int n = H * W;
    get_rays_kernel<<<(n + 255) / 256, 256, 0, as_stream(stream)>>>(W, 0, n, focal, cx, cy, c2w, c2w_row_stride, near_, far_, rays);
    return check_launch("inerf_get_rays");
}

extern "C" int inerf_get_rays_range(int H, int W, float focal, float cx, float cy, const float* c2w, int c2w_row_stride,
                                    float near_, float far_, int first, int count, float* rays, void* stream) {
    if (H <= 0 || W <= 0 || (int64_t)H * W > (1 << 30) || c2w_row_stride < 4) return fail(INERF_E_SHAPE, "inerf_get_rays_range: bad H/W/c2w_row_stride");
    if (first < 0 || count < 0 || (int64_t)first + count > (int64_t)H * W) return fail(INERF_E_SHAPE, "inerf_get_rays_range: [first, first+count) outside the frame");
    if (count == 0) return INERF_OK;
    if (!c2w || !rays) return fail(INERF_E_ARG, "inerf_get_rays_range: NULL pointer");
    get_rays_kernel<<<(count + 255) / 256, 256, 0, as_stream(stream)>>>(W, first, count, focal, cx, cy, c2w, c2w_row_stride, near_, far_, rays);
    return check_launch("inerf_get_rays_range");
}

extern "C" int inerf_pack_rays(const float* rays_o, const float* rays_d, int n, float near_, float far_, float* rays,
                               void* stream) {
    if (n < 0) return fail(INERF_E_SHAPE, "inerf_pack_rays: n < 0");
    if (n == 0) return INERF_OK;
    if (!rays_o || !rays_d || !rays) return fail(INERF_E_ARG, "inerf_pack_rays: NULL pointer");
    pack_rays_kernel<<<(n + 255) / 256, 256, 0, as_stream(stream)>>>(rays_o, rays_d, n, near_, far_, rays);
    return check_launch("inerf_pack_rays");
}

// ---------------------------------------------------------------------------------------------
// positional encoding.  helper.py:174-224
// ---------------------------------------------------------------------------------------------
__global__ void posenc_kernel(const float* __restrict__ x, int64_t n, int dims, int n_freqs, float* __restrict__ out) {
    int width = dims * (1 + 2 * n_freqs);
    int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n * width) return;
    int64_t row = idx / width;
    int j = (int)(idx - row * width);
    float v;
    if (j < dims) {
        v = x[row * dims + j];
    } else {
        int q = (j - dims) / dims;           // 2*freq + (0: sin, 1: cos)
        int c = (j - dims) - q * dims;
        float a = __fmul_rn(x[row * dims + c], exp2f((float)(q >> 1)));   // 2^k scaling is exact
        v = (q & 1) ? cosf(a) : sinf(a);
    }
    out[idx] = v;
}

extern "C" int inerf_posenc(const float* x, int64_t n, int dims, int n_freqs, float* out, void* stream) {
    if (n < 0 || dims <= 0 || dims > 64 || n_freqs < 0 || n_freqs > 32)
        return fail(INERF_E_SHAPE, "inerf_posenc: bad n/dims/n_freqs");
    if (n == 0) return INERF_OK;
    if (!x || !out) return fail(INERF_E_ARG, "inerf_posenc: NULL pointer");
    int64_t total = n * dims * (1 + 2 * n_freqs);
    if ((total + 255) / 256 > 0x7fffffffLL) return fail(INERF_E_SHAPE, "inerf_posenc: too many elements");
    posenc_kernel<<<(unsigned)((total + 255) / 256), 256, 0, as_stream(stream)>>>(x, n, dims, n_freqs, out);
    return check_launch("inerf_posenc");
}

// ---------------------------------------------------------------------------------------------
// stratified coarse depths.  audio_exp_nerf.py:306-328
// ---------------------------------------------------------------------------------------------
template <bool RNG>
__global__ void sample_coarse_kernel(const float* __restrict__ rays, int n, int ray_stride, int s,
                                     const float* __restrict__ t_vals, const float* __restrict__ t_rand,
                                     const unsigned long long* __restrict__ rng_state, int lindisp, float* __restrict__ z) {
    int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (int64_t)n * s) return;
    int ray = (int)(idx / s);
    int i = (int)(idx - (int64_t)ray * s);
    float near_ = rays[(size_t)ray * ray_stride + 6], far_ = rays[(size_t)ray * ray_stride + 7];
    float zi = coarse_z(near_, far_, t_vals[i], lindisp);
    if (RNG || t_rand) {
        // mids = .5*(z[1:]+z[:-1]); upper = [mids, z[-1]]; lower = [z[0], mids]; z = lower + (upper-lower)*r
        float lo = zi, hi = zi;
        if (i > 0) lo = __fmul_rn(0.5f, __fadd_rn(zi, coarse_z(near_, far_, t_vals[i - 1], lindisp)));
        if (i < s - 1) hi = __fmul_rn(0.5f, __fadd_rn(coarse_z(near_, far_, t_vals[i + 1], lindisp), zi));
        float r;
        if constexpr (RNG) {                                // draw idx of the stream: word idx & 3 of Philox block idx >> 2
            const Philox4 q = philox_at(rng_state, (uint64_t)idx >> 2, INERF_RNG_STREAM_COARSE);
            const uint32_t w = (idx & 2) ? ((idx & 1) ? q.w : q.z) : ((idx & 1) ? q.y : q.x);
            r = u01(w);
        } else {
            r = t_rand[idx];
        }
        if (i == s - 1) r = 1.0f;                           // t_rand[..., -1] = 1.0  (:326)
        zi = __fadd_rn(lo, __fmul_rn(__fsub_rn(hi, lo), r));
    }
    z[idx] = zi;
}

extern "C" int inerf_sample_coarse(const float* rays, int n, int ray_stride, int s, const float* t_vals,
                                   const float* t_rand, int lindisp, float* z, void* stream) {
    if (n < 0 || s <= 0 || s > 4096 || ray_stride < 8) return fail(INERF_E_SHAPE, "inerf_sample_coarse: bad n/s/stride");
    if (n == 0) return INERF_OK;
    if (!rays || !t_vals || !z) return fail(INERF_E_ARG, "inerf_sample_coarse: NULL pointer");
    int64_t total = (int64_t)n * s;
    sample_coarse_kernel<false><<<(unsigned)((total + 255) / 256), 256, 0, as_stream(stream)>>>(rays, n, ray_stride, s, t_vals, t_rand,
                                                                                               nullptr, lindisp, z);
    return check_launch("inerf_sample_coarse");
}

// In-kernel jitter, four consecutive samples of a ray per thread (s % 4 == 0): ONE Philox block feeds the four draws -- the one-sample
// form above evaluates a whole block per sample and is issue bound (ncu: 97 us per 202 500 x 64 samples, 74 % issue slots) -- and the row
// leaves as a 128-bit store.  Same draw numbering (word i & 3 of block i >> 2), so both forms return the same bits.
__global__ void sample_coarse_rng4_kernel(const float* __restrict__ rays, int n, int ray_stride, int s, const float* __restrict__ t_vals,
                                          const unsigned long long* __restrict__ rng_state, int lindisp, float* __restrict__ z) {
    const int64_t q4 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;      // Philox block = group of four samples
    const int per_ray = s >> 2;
    if (q4 >= (int64_t)n * per_ray) return;
    const int ray = (int)(q4 / per_ray);
    const int i0 = (int)(q4 - (int64_t)ray * per_ray) << 2;
    const float near_ = rays[(size_t)ray * ray_stride + 6], far_ = rays[(size_t)ray * ray_stride + 7];
    float zc[6];                                                             // depths i0 - 1 .. i0 + 4
#pragma unroll
    for (int j = 0; j < 6; ++j) {
        const int i = min(max(i0 - 1 + j, 0), s - 1);
        zc[j] = coarse_z(near_, far_, t_vals[i], lindisp);
    }
    const Philox4 q = philox_at(rng_state, (uint64_t)q4, INERF_RNG_STREAM_COARSE);
    const uint32_t w[4] = {q.x, q.y, q.z, q.w};
    float out[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int i = i0 + j;
        const float zi = zc[j + 1];
        const float lo = i > 0 ? __fmul_rn(0.5f, __fadd_rn(zi, zc[j])) : zi;
        const float hi = i < s - 1 ? __fmul_rn(0.5f, __fadd_rn(zc[j + 2], zi)) : zi;
        const float r = (i == s - 1) ? 1.0f : u01(w[j]);
        out[j] = __fadd_rn(lo, __fmul_rn(__fsub_rn(hi, lo), r));
    }
    reinterpret_cast<float4*>(z)[q4] = make_float4(out[0], out[1], out[2], out[3]);
}

extern "C" int inerf_sample_coarse_rng(const float* rays, int n, int ray_stride, int s, const float* t_vals, const uint64_t* rng_state,
                                       int lindisp, float* z, void* stream) {
    if (n < 0 || s <= 0 || s > 4096 || ray_stride < 8) return fail(INERF_E_SHAPE, "inerf_sample_coarse_rng: bad n/s/stride");
    if (n == 0) return INERF_OK;
    if (!rays || !t_vals || !z || !rng_state) return fail(INERF_E_ARG, "inerf_sample_coarse_rng: NULL pointer");
    int64_t total = (int64_t)n * s;
    if ((s & 3) == 0 && ((uintptr_t)z & 15) == 0) {
        sample_coarse_rng4_kernel<<<(unsigned)((total / 4 + 255) / 256), 256, 0, as_stream(stream)>>>(
            rays, n, ray_stride, s, t_vals, reinterpret_cast<const unsigned long long*>(rng_state), lindisp, z);
        return check_launch("inerf_sample_coarse_rng");
    }
    sample_coarse_kernel<true><<<(unsigned)((total + 255) / 256), 256, 0, as_stream(stream)>>>(
        rays, n, ray_stride, s, t_vals, nullptr, reinterpret_cast<const unsigned long long*>(rng_state), lindisp, z);
    return check_launch("inerf_sample_coarse_rng");
}

// ---------------------------------------------------------------------------------------------
// RNG state upkeep and the NaN / Inf scan of render_rays' outputs (audio_exp_nerf.py:367-369)
// ---------------------------------------------------------------------------------------------
__global__ void rng_advance_kernel(unsigned long long* state, unsigned long long inc) { state[1] += inc; }

extern "C" int inerf_rng_advance(uint64_t* rng_state, uint64_t increment, void* stream) {
    if (!rng_state) return fail(INERF_E_ARG, "inerf_rng_advance: NULL pointer");
    rng_advance_kernel<<<1, 1, 0, as_stream(stream)>>>(reinterpret_cast<unsigned long long*>(rng_state), (unsigned long long)increment);
    return check_launch("inerf_rng_advance");
}

struct ScanArgs { const float* x[INERF_MAX_SCAN]; long long n[INERF_MAX_SCAN]; int k; };

__global__ void flag_nonfinite_kernel(ScanArgs a, int* __restrict__ flags) {
    const float* x = a.x[blockIdx.y];
    const long long n = a.n[blockIdx.y];
    bool bad = false;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        bad |= !isfinite(x[i]);
    if (__syncthreads_or(bad) && threadIdx.x == 0) atomicOr(flags, 1 << blockIdx.y);
}

extern "C" int inerf_flag_nonfinite(const float* const* xs_host, const int64_t* ns_host, int k, int32_t* flags, void* stream) {
    if (k < 0 || k > INERF_MAX_SCAN) return fail(INERF_E_SHAPE, "inerf_flag_nonfinite: 0 <= k <= INERF_MAX_SCAN tensors");
    if (k == 0) return INERF_OK;
    if (!xs_host || !ns_host || !flags) return fail(INERF_E_ARG, "inerf_flag_nonfinite: NULL pointer");
    ScanArgs a{};
    long long nmax = 0;
    for (int i = 0; i < k; ++i) {
        if (ns_host[i] < 0 || (ns_host[i] > 0 && !xs_host[i])) return fail(INERF_E_ARG, "inerf_flag_nonfinite: NULL tensor / negative size");
        a.x[i] = xs_host[i]; a.n[i] = ns_host[i];
        nmax = ns_host[i] > nmax ? ns_host[i] : nmax;
    }
    a.k = k;
    if (nmax == 0) return INERF_OK;
    long long blocks = (nmax + 1023) / 1024;
    if (blocks > 592) blocks = 592;
    flag_nonfinite_kernel<<<dim3((unsigned)blocks, k), 256, 0, as_stream(stream)>>>(a, flags);
    return check_launch("inerf_flag_nonfinite");
}

// ---------------------------------------------------------------------------------------------
// head/torso blend.  train_torso.py:269-270
// ---------------------------------------------------------------------------------------------
// one value of rgb_head * last_weight_torso[..., None] + rgb_fg_torso; shared by blend_kernel and head_torso_to8b_kernel so that both
// entry points round the same way
__device__ __forceinline__ float blend_value(float head, float lw, float fg) { return __fadd_rn(__fmul_rn(head, lw), fg); }

// (255 * clip(x, 0, 1)).astype(uint8): float -> int truncates like astype
__device__ __forceinline__ uint8_t to8b_value(float x) { return (uint8_t)(int)__fmul_rn(255.f, fminf(fmaxf(x, 0.f), 1.f)); }

__global__ void blend_kernel(const float* __restrict__ rgb_head, const float* __restrict__ lw,
                             const float* __restrict__ fg, int n, float* __restrict__ rgb) {
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n * 3) return;
    rgb[idx] = blend_value(rgb_head[idx], lw[idx / 3], fg[idx]);
}

extern "C" int inerf_head_torso_blend(const float* rgb_head, const float* last_weight_torso, const float* rgb_fg_torso,
                                      int n, float* rgb, void* stream) {
    if (n < 0) return fail(INERF_E_SHAPE, "inerf_head_torso_blend: n < 0");
    if (n == 0) return INERF_OK;
    if (!rgb_head || !last_weight_torso || !rgb_fg_torso || !rgb)
        return fail(INERF_E_ARG, "inerf_head_torso_blend: NULL pointer");
    blend_kernel<<<(n * 3 + 255) / 256, 256, 0, as_stream(stream)>>>(rgb_head, last_weight_torso, rgb_fg_torso, n, rgb);
    return check_launch("inerf_head_torso_blend");
}

// ---------------------------------------------------------------------------------------------
// torso-stage loss seed: the two composites of train_torso.py:269-270, their mean squared errors and the gradients that reach the torso
// pair, in one pass.  The composite is blend_value (the bits of blend_kernel), the per-value gradient the expression of mse_pair_kernel;
// one thread per ray, so last_weight's gradient is summed over the ray's three values in registers.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) head_torso_mse_pair_kernel(
    const float* __restrict__ head, const float* __restrict__ head0, const float* __restrict__ lw, const float* __restrict__ lw0,
    const float* __restrict__ fg, const float* __restrict__ fg0, const float* __restrict__ tgt, long long n, float inv_m,
    float* __restrict__ g_lw, float* __restrict__ g_lw0, float* __restrict__ g_fg, float* __restrict__ g_fg0, float* __restrict__ loss) {
    float s0 = 0.f, s1 = 0.f;
    for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (long long)gridDim.x * blockDim.x) {
        const float w = lw[r], w0 = lw0[r];
        float gw = 0.f, gw0 = 0.f;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const long long i = 3 * r + c;
            const float t = tgt[i], h = head[i], h0 = head0[i];
            const float d0 = blend_value(h, w, fg[i]) - t, d1 = blend_value(h0, w0, fg0[i]) - t;
            s0 = fmaf(d0, d0, s0);
            s1 = fmaf(d1, d1, s1);
            const float g0 = 2.0f * d0 * inv_m, g1 = 2.0f * d1 * inv_m;
            g_fg[i] = g0;
            g_fg0[i] = g1;
            gw = __fadd_rn(gw, __fmul_rn(g0, h));
            gw0 = __fadd_rn(gw0, __fmul_rn(g1, h0));
        }
        g_lw[r] = gw;
        g_lw0[r] = gw0;
    }
    s0 = warp_sum(s0);
    s1 = warp_sum(s1);
    __shared__ float sh[2][8];
    const int lane = threadIdx.x & 31, wi = threadIdx.x >> 5;
    if (lane == 0) { sh[0][wi] = s0; sh[1][wi] = s1; }
    __syncthreads();
    if (threadIdx.x < 2) {
        float t = 0.f;
        for (int j = 0; j < 8; ++j) t += sh[threadIdx.x][j];
        atomicAdd(loss + threadIdx.x, t * inv_m);
    }
}

extern "C" int inerf_head_torso_mse_pair(const float* rgb_head, const float* rgb_head0, const float* last_weight, const float* last_weight0,
                                         const float* rgb_fg, const float* rgb_fg0, const float* target, int64_t n, float* g_last_weight,
                                         float* g_last_weight0, float* g_rgb_fg, float* g_rgb_fg0, float* loss2, void* stream) {
    if (n <= 0) return fail(INERF_E_SHAPE, "inerf_head_torso_mse_pair: need at least one ray");
    if (!rgb_head || !rgb_head0 || !last_weight || !last_weight0 || !rgb_fg || !rgb_fg0 || !target || !g_last_weight || !g_last_weight0 ||
        !g_rgb_fg || !g_rgb_fg0 || !loss2)
        return fail(INERF_E_ARG, "inerf_head_torso_mse_pair: NULL pointer");
    cudaError_t e = cudaMemsetAsync(loss2, 0, 2 * sizeof(float), as_stream(stream));
    if (e != cudaSuccess) { set_error("inerf_head_torso_mse_pair: %s", cudaGetErrorString(e)); return (int)e; }
    const int grid = (int)((n + 255) / 256 < 4 * (long long)num_sms() ? (n + 255) / 256 : 4 * (long long)num_sms());
    head_torso_mse_pair_kernel<<<grid, 256, 0, as_stream(stream)>>>(rgb_head, rgb_head0, last_weight, last_weight0, rgb_fg, rgb_fg0, target, n,
                                                                   1.0f / (float)(3 * n), g_last_weight, g_last_weight0, g_rgb_fg, g_rgb_fg0,
                                                                   loss2);
    return check_launch("inerf_head_torso_mse_pair");
}

// ---------------------------------------------------------------------------------------------
// to8b: (255 * clip(x, 0, 1)).astype(uint8)   helper.py:154 (used on every rendered frame, eval_aud_exp_nerf.py:490)
// ---------------------------------------------------------------------------------------------
__global__ void to8b_kernel(const float* __restrict__ x, long long n, uint8_t* __restrict__ out) {
    const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i >= n) return;
    if (i + 3 < n && ((uintptr_t)(x + i) & 15) == 0 && ((uintptr_t)(out + i) & 3) == 0) {
        const float4 v = *reinterpret_cast<const float4*>(x + i);
        *reinterpret_cast<uchar4*>(out + i) = make_uchar4(to8b_value(v.x), to8b_value(v.y), to8b_value(v.z), to8b_value(v.w));
    } else {
        for (long long j = i; j < n && j < i + 4; ++j) out[j] = to8b_value(x[j]);
    }
}

extern "C" int inerf_to8b(const float* x, int64_t n, uint8_t* out, void* stream) {
    if (n < 0) return fail(INERF_E_SHAPE, "inerf_to8b: n < 0");
    if (n == 0) return INERF_OK;
    if (!x || !out) return fail(INERF_E_ARG, "inerf_to8b: NULL pointer");
    const long long threads = (n + 3) / 4;
    to8b_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, as_stream(stream)>>>(x, n, out);
    return check_launch("inerf_to8b");
}

// ---------------------------------------------------------------------------------------------
// blend + to8b in one pass: the composited head + torso frame of test_torso.py:523-524 leaves a band as bytes.  Four values per thread
// like to8b_kernel; value i belongs to ray i / 3.  out_rgb (optional) receives the fp32 blend.
// ---------------------------------------------------------------------------------------------
__global__ void head_torso_to8b_kernel(const float* __restrict__ rgb_head, const float* __restrict__ lw, const float* __restrict__ fg,
                                       long long n_values, uint8_t* __restrict__ out, float* __restrict__ rgb) {
    const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i >= n_values) return;
    if (i + 3 < n_values && (((uintptr_t)(rgb_head + i) | (uintptr_t)(fg + i) | (rgb ? (uintptr_t)(rgb + i) : 0)) & 15) == 0 &&
        ((uintptr_t)(out + i) & 3) == 0) {
        // values i .. i + 3 span rays `ray` (value i) and `ray + 1` (value i + 3, always: i + 3 - 3 * ray >= 3)
        const long long ray = i / 3;
        const int m = (int)(i - ray * 3);
        const float4 h = *reinterpret_cast<const float4*>(rgb_head + i), f = *reinterpret_cast<const float4*>(fg + i);
        const float w0 = lw[ray], w1 = lw[ray + 1];
        const float4 c = make_float4(blend_value(h.x, w0, f.x), blend_value(h.y, m + 1 < 3 ? w0 : w1, f.y),
                                     blend_value(h.z, m + 2 < 3 ? w0 : w1, f.z), blend_value(h.w, w1, f.w));
        if (rgb) *reinterpret_cast<float4*>(rgb + i) = c;
        *reinterpret_cast<uchar4*>(out + i) = make_uchar4(to8b_value(c.x), to8b_value(c.y), to8b_value(c.z), to8b_value(c.w));
    } else {
        for (long long j = i; j < n_values && j < i + 4; ++j) {
            const float c = blend_value(rgb_head[j], lw[j / 3], fg[j]);
            if (rgb) rgb[j] = c;
            out[j] = to8b_value(c);
        }
    }
}

extern "C" int inerf_head_torso_to8b(const float* rgb_head, const float* last_weight_torso, const float* rgb_fg_torso, int64_t n,
                                     uint8_t* out_u8, float* out_rgb, void* stream) {
    if (n < 0) return fail(INERF_E_SHAPE, "inerf_head_torso_to8b: n < 0");
    if (n > 0x7fffffffLL * 256 * 4 / 3) return fail(INERF_E_SHAPE, "inerf_head_torso_to8b: too many rays for one launch");
    if (n == 0) return INERF_OK;
    if (!rgb_head || !last_weight_torso || !rgb_fg_torso || !out_u8) return fail(INERF_E_ARG, "inerf_head_torso_to8b: NULL pointer");
    const long long threads = (3 * n + 3) / 4;
    head_torso_to8b_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, as_stream(stream)>>>(rgb_head, last_weight_torso, rgb_fg_torso,
                                                                                           3 * n, out_u8, out_rgb);
    return check_launch("inerf_head_torso_to8b");
}
