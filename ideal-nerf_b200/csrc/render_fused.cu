// inerf_render_rays_fused: the whole inference render_rays (coarse + fine) enqueued by one C call, with the small stages fused.
//
// Reference: Network.render_rays, NeRFs/HeadNeRF/train/audio_exp_nerf.py:297-371 (torso: NeRFs/TorsoNeRF/train_torso.py:290-363);
// get_rays helper.py:228-243; raw2outputs baseline.py:325-375; sample_pdf helper.py:269-313; the NaN scan :367-369.
//
// What is fused (the two FaceNeRF launches are the kernels of inerf_mlp_fwd, 97 % of a frame; this file is about everything else):
//   * set-up kernel  = conditioning fold of both nets (2 x 96 blocks) + the rays of this call's pixels + the jittered coarse depths
//                      (was: get_rays_range, sample_coarse_rng, 2 x fold_cond = 4 launches);
//   * composite_sample_64_128_kernel = raw2outputs of the coarse pass + sample_pdf / merge / std with in-kernel draws: one warp per
//                      ray, the lane keeps its two weights in registers between the two halves, so the (n, 64) weights never reach
//                      HBM (was: composite_fwd + importance_sample_rng; 512 B/ray less traffic);
//   * composite_final_kernel = raw2outputs of the fine pass writing the maps and last_weight only (the (n, 192) weights tensor is
//                      optional: 768 B/ray less), OR-ing the NaN / Inf flags and bumping the RNG offset (was: composite_fwd +
//                      rng_advance [+ flag_nonfinite]).
// Without rgb0 (args->rgb0 == NULL: a frame or video render, which keeps only the fine colour) the coarse pass needs sigma alone: in bf16
// mode the coarse net runs its density-only build (L0-L7 and the alpha head, one float per point), in the other modes the full net, and
// the coarse compositor reads sigma only (composite2_ray's SIG form): the same weights, disp0, acc0, z_std and merged depths, bit for bit.
// A rank that renders a 25 k-ray band of a frame (8 GPUs) spends as long in these small launches as in their work, so the count matters
// there.  Every fused kernel runs the same device functions as its stand-alone twin: bit-identical outputs (tests/test_gpu_parity.py).
#include "common.cuh"
#include "composite_parts.cuh"
#include "fold_cond.cuh"
#include "mlp_common.cuh"
#include "philox.cuh"
#include "rays_parts.cuh"
#include "sample_parts.cuh"

using namespace inerf;

namespace {

constexpr int FOLD_BLOCKS = 12 * 8;      // blocks of one net's fold (fold_cond_block: 12 layers x 8 row groups)

struct SetupArgs {
    FoldArgs fold[2];
    int n_fold;                          // nets to fold (2)
    int gen, W, first;                   // gen != 0: generate the rays of pixels [first, first + n)
    float focal, cx, cy, near_, far_;
    const float* c2w; int rs;
    float* rays_out;
    const float* rays_in; int ray_stride;
    int n, s, do_z;                      // do_z != 0: jittered depths, four samples per thread
    const float* t_vals;
    const unsigned long long* rng_state;
    float* z;
};

__global__ void __launch_bounds__(256) render_setup_kernel(const __grid_constant__ SetupArgs a) {
    __shared__ float c[1024];
    const int nf = a.n_fold * FOLD_BLOCKS;
    if ((int)blockIdx.x < nf) {
        const int net = blockIdx.x / FOLD_BLOCKS, r = blockIdx.x - net * FOLD_BLOCKS;
        fold_cond_block(a.fold[net], r % 12, r / 12, c);
        return;
    }
    const int per_ray = a.do_z ? (a.s >> 2) : 1;                     // threads per ray
    const long long q4 = (long long)(blockIdx.x - nf) * 256 + threadIdx.x;
    if (q4 >= (long long)a.n * per_ray) return;
    const int ray = (int)(q4 / per_ray);
    const int i0 = (int)(q4 - (long long)ray * per_ray) << 2;
    float near_ = a.near_, far_ = a.far_;
    if (a.gen) {
        if (i0 == 0) {
            const int pix = a.first + ray, row = pix / a.W, col = pix - row * a.W;
            float d[3];
            pixel_dir((float)row, (float)col, a.focal, a.cx, a.cy, a.c2w, a.rs, d);
            store_ray(a.rays_out + (size_t)ray * 11, a.c2w[3], a.c2w[a.rs + 3], a.c2w[2 * a.rs + 3], d[0], d[1], d[2], near_, far_);
        }
    } else {
        near_ = a.rays_in[(size_t)ray * a.ray_stride + 6];
        far_ = a.rays_in[(size_t)ray * a.ray_stride + 7];
    }
    if (!a.do_z) return;
    // the arithmetic of sample_coarse_rng4_kernel (rays.cu): same draw numbering, same bits
    const int s = a.s;
    float zc[6];
#pragma unroll
    for (int j = 0; j < 6; ++j) {
        const int i = min(max(i0 - 1 + j, 0), s - 1);
        zc[j] = coarse_z(near_, far_, a.t_vals[i], 0);
    }
    const Philox4 q = philox_at(a.rng_state, (uint64_t)q4, INERF_RNG_STREAM_COARSE);
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
    reinterpret_cast<float4*>(a.z)[q4] = make_float4(out[0], out[1], out[2], out[3]);
}

struct CompArgs {
    const float4* raw; const float* z; const float* rays; int ray_stride; const float* bc_rgb;
    int n, s, white_bkgd;
    float *rgb, *disp, *acc, *depth, *weights, *rgb_fg, *last_weight;
    const unsigned long long* rng_state;      // sampler: draws; final: NULL
    unsigned long long* rng_bump;             // final: the state whose offset this launch advances (NULL: none)
    float *z_merged, *z_std;
    int* flags;
};

// coarse pass: raw2outputs (S = 64) + sample_pdf / merge / std (128 in-kernel draws); one warp per ray.  SIG: composite2_ray's
// sigma-only form (1: density-only raw, 4: the sigma lane of a full raw) or 0, the full form with rgb0
template <int SIG>
__global__ void __launch_bounds__(256) composite_sample_64_128_kernel(const CompArgs a) {
    __shared__ __align__(16) float smem[8 * IMP64_WARP_FLOATS];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int ray = blockIdx.x * 8 + wib;
    if (ray >= a.n) return;
    float2 z2, w2;
    const uint32_t bad = composite2_ray<1, SIG>(a.raw, a.z, a.rays + 3, a.ray_stride, a.bc_rgb, nullptr, ray, 64, a.white_bkgd, a.rgb, a.disp,
                                                a.acc, a.depth, a.weights, a.rgb_fg, a.last_weight, lane, z2, w2);
    const float sd = importance_rng_64_128_ray(z2, w2, ray, lane, smem + wib * IMP64_WARP_FLOATS, a.rng_state, INERF_RNG_STREAM_PDF, nullptr,
                                               a.z_merged, a.z_std);
    if (a.flags) {
        uint32_t f = ((bad & 1u) ? INERF_NF_RGB0 : 0u) | ((bad & 2u) ? INERF_NF_DISP0 : 0u) | ((bad & 4u) ? INERF_NF_ACC0 : 0u);
        if (lane == 0 && !isfinite(sd)) f |= INERF_NF_Z_STD;
        if (f) atomicOr(a.flags, (int)f);
    }
}

// coarse pass of the general path without rgb0: raw2outputs of the densities alone (composite2_ray's SIG form) writing disp0, acc0,
// depth0 and the weights that inerf_importance_sample reads -- the bits inerf_composite_fwd writes there
template <int C, int SIG>
__global__ void __launch_bounds__(256) composite_sigma_kernel(const CompArgs a) {
    const int lane = threadIdx.x & 31;
    const int ray = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (ray >= a.n) return;
    float2 z2, w2;
    composite2_ray<C, SIG>(a.raw, a.z, a.rays + 3, a.ray_stride, nullptr, nullptr, ray, a.s, a.white_bkgd, nullptr, a.disp, a.acc, a.depth,
                           a.weights, nullptr, nullptr, lane, z2, w2);
}

template <int SIG>
void launch_composite_sigma(const CompArgs& a, cudaStream_t st) {
    const int c2 = (a.s + 63) / 64;      // n_samples <= 254
    if (c2 <= 1) composite_sigma_kernel<1, SIG><<<(a.n + 7) / 8, 256, 0, st>>>(a);
    else if (c2 == 2) composite_sigma_kernel<2, SIG><<<(a.n + 7) / 8, 256, 0, st>>>(a);
    else if (c2 == 3) composite_sigma_kernel<3, SIG><<<(a.n + 7) / 8, 256, 0, st>>>(a);
    else composite_sigma_kernel<4, SIG><<<(a.n + 7) / 8, 256, 0, st>>>(a);
}

// fine pass: raw2outputs writing maps + last_weight (weights optional), the NaN / Inf flags, the RNG bump
template <int C>
__global__ void __launch_bounds__(256) composite_final_kernel(const CompArgs a) {
    if (a.rng_bump && blockIdx.x == 0 && threadIdx.x == 0) a.rng_bump[1] += 1ull;      // every reader of the state ran in an earlier launch
    const int lane = threadIdx.x & 31;
    const int ray = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (ray >= a.n) return;
    float2 z2, w2;
    const uint32_t bad = composite2_ray<C>(a.raw, a.z, a.rays + 3, a.ray_stride, a.bc_rgb, nullptr, ray, a.s, a.white_bkgd, a.rgb, a.disp,
                                           a.acc, a.depth, a.weights, a.rgb_fg, a.last_weight, lane, z2, w2);
    if (a.flags && bad) {
        const uint32_t f = ((bad & 1u) ? INERF_NF_RGB_MAP : 0u) | ((bad & 2u) ? INERF_NF_DISP_MAP : 0u) | ((bad & 4u) ? INERF_NF_ACC_MAP : 0u) |
                           ((bad & 16u) ? INERF_NF_LAST_WEIGHT : 0u);
        if (f) atomicOr(a.flags, (int)f);
    }
}

// z_std scan for the paths whose sampler is a stand-alone kernel
__global__ void flag_zstd_kernel(const float* __restrict__ x, int n, int* flags) {
    bool bad = false;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) bad |= !isfinite(x[i]);
    if (__syncthreads_or(bad) && threadIdx.x == 0) atomicOr(flags, (int)INERF_NF_Z_STD);
}

inline size_t up256(size_t b) { return (b + 255) & ~(size_t)255; }

struct Workspace {
    size_t rays, cond_c, cond_f, z_c, raw_c, w_c, z_s, z_m, raw_f, depth0, total;
};

int plan(const InerfRenderArgs* a, Workspace& w) {
    if (!a) return fail(INERF_E_ARG, "inerf_render_rays_fused: args is NULL");
    if (a->n < 0 || a->n_samples < 4 || (a->n_samples & 1) || a->n_importance <= 0 || ((a->n_samples + a->n_importance) & 1) ||
        a->n_samples + a->n_importance > 256)
        return fail(INERF_E_SHAPE, "inerf_render_rays_fused: needs an even n_samples >= 4, n_importance > 0 and an even n_samples + n_importance <= 256");
    size_t cf = 0;
    int rc = inerf_mlp_cond_floats(&a->coarse.dims, &cf);
    if (rc) return rc;
    rc = check_dims(&a->fine.dims);
    if (rc) return rc;
    const size_t n = (size_t)a->n, s1 = (size_t)a->n_samples, st = s1 + (size_t)a->n_importance;
    const bool fused_cs = a->perturb && a->n_samples == 64 && a->n_importance == 128;
    const bool dens = !a->rgb0 && a->mode == INERF_MLP_BF16;      // the coarse net's density-only build: one float per point
    size_t o = 0;
    auto take = [&o](size_t bytes) { const size_t at = o; o += up256(bytes); return at; };
    w.rays = take(a->gen_rays ? n * 11 * 4 : 0);
    w.cond_c = take(cf * 4);
    w.cond_f = take(cf * 4);
    w.z_c = take(n * s1 * 4);
    w.raw_c = take(n * s1 * (dens ? 4 : 16));
    w.w_c = take(fused_cs ? 0 : n * s1 * 4);
    w.z_s = take(a->perturb ? 0 : n * (size_t)a->n_importance * 4);
    w.z_m = take(a->z_vals ? 0 : n * st * 4);
    w.raw_f = take(n * st * 16);
    w.depth0 = take(n * 4);
    w.total = o;
    return INERF_OK;
}

int fill_fold(FoldArgs& f, const InerfRenderNet& net, float* cond, const char* which) {
    const InerfNetDims& d = net.dims;
    if (!net.params_host) return fail(INERF_E_ARG, "inerf_render_rays_fused: params_host is NULL");
    if ((d.dim_aud > 0 && !net.aud) || (d.dim_expr > 0 && !net.expr) || (d.dim_latent > 0 && !net.latent)) {
        set_error("inerf_render_rays_fused: %s net: conditioning vector missing for a non-zero dim", which);
        return INERF_E_ARG;
    }
    for (int i = 0; i < INERF_N_PARAMS; ++i) {
        if (!net.params_host[i]) return fail(INERF_E_ARG, "inerf_render_rays_fused: NULL parameter pointer");
        f.w[i] = net.params_host[i];
    }
    f.aud = net.aud; f.expr = net.expr; f.latent = net.latent;
    f.da = d.dim_aud; f.de = d.dim_expr; f.dl = d.dim_latent;
    f.cond = cond;
    return INERF_OK;
}

}  // namespace

extern "C" int inerf_render_workspace_bytes(const InerfRenderArgs* args, size_t* bytes) {
    if (!bytes) return fail(INERF_E_ARG, "inerf_render_workspace_bytes: NULL");
    Workspace w{};
    const int rc = plan(args, w);
    if (rc) return rc;
    *bytes = w.total;
    return INERF_OK;
}

namespace {
// ev: NULL, or six events recorded on the stream before stage 1 and after each of the five stages (inerf_debug_render_stage_ms)
int render_rays_fused(const InerfRenderArgs* a, void* stream, cudaEvent_t* ev) {
    Workspace w{};
    int rc = plan(a, w);
    if (rc) return rc;
    if (a->mode == INERF_MLP_F16X2_EMB)
        return fail(INERF_E_UNSUPPORTED, "inerf_render_rays_fused: INERF_MLP_F16X2_EMB is an embedded-row mode; the fused render takes INERF_MLP_F16X2");
    if (a->n == 0) return INERF_OK;
    if (!a->workspace || a->workspace_bytes < w.total) return fail(INERF_E_ARG, "inerf_render_rays_fused: workspace missing or smaller than inerf_render_workspace_bytes");
    if ((uintptr_t)a->workspace & 255) return fail(INERF_E_ALIGN, "inerf_render_rays_fused: workspace must be 256-byte aligned");
    if (!a->bc_rgb || !a->t_vals || !a->rgb_map || !a->disp_map || !a->acc_map || !a->depth_map || !a->last_weight || !a->disp0 || !a->acc0 ||
        !a->z_std)
        return fail(INERF_E_ARG, "inerf_render_rays_fused: NULL pointer");
    if (a->perturb ? !a->rng_state : !a->u_vals) return fail(INERF_E_ARG, "inerf_render_rays_fused: rng_state (perturb) / u_vals (deterministic) missing");
    const bool with_fg = a->rgb_map_fg != nullptr;
    if (with_fg != (a->rgb_map_fg0 != nullptr) || with_fg != (a->last_weight0 != nullptr))
        return fail(INERF_E_ARG, "inerf_render_rays_fused: rgb_map_fg, rgb_map_fg0 and last_weight0 are given together or not at all");
    if (with_fg && !a->rgb0) return fail(INERF_E_ARG, "inerf_render_rays_fused: the torso extras need rgb0 (rgb_map_fg0 is a coarse colour)");
    if (a->gen_rays) {
        if (a->H <= 0 || a->W <= 0 || (int64_t)a->H * a->W > (1 << 30) || a->c2w_row_stride < 4 || a->first < 0 ||
            (int64_t)a->first + a->n > (int64_t)a->H * a->W)
            return fail(INERF_E_SHAPE, "inerf_render_rays_fused: [first, first + n) outside the H x W frame / bad c2w_row_stride");
        if (!a->c2w) return fail(INERF_E_ARG, "inerf_render_rays_fused: c2w is NULL");
    } else if (!a->rays || a->ray_stride < 11) {
        return fail(INERF_E_ARG, "inerf_render_rays_fused: rays missing or ray_stride < 11");
    }
    if (a->z_vals && ((uintptr_t)a->z_vals & 15)) return fail(INERF_E_ALIGN, "inerf_render_rays_fused: z_vals must be 16-byte aligned");

    cudaStream_t st = as_stream(stream);
    auto mark = [&](int i) { if (ev) cudaEventRecord(ev[i], st); };
    mark(0);
    uint8_t* ws = reinterpret_cast<uint8_t*>(a->workspace);
    auto F = [ws](size_t off) { return reinterpret_cast<float*>(ws + off); };
    const int n = a->n, s1 = a->n_samples, ni = a->n_importance, stot = s1 + ni;
    const float* rays = a->gen_rays ? F(w.rays) : a->rays;
    const int stride = a->gen_rays ? 11 : a->ray_stride;
    float* z_c = F(w.z_c);
    float* z_m = a->z_vals ? a->z_vals : F(w.z_m);
    unsigned long long* rng = reinterpret_cast<unsigned long long*>(a->rng_state);

    // ---- 1. set-up: folds + rays + jittered depths -------------------------------------------------------------------------------
    SetupArgs sa{};
    rc = fill_fold(sa.fold[0], a->coarse, F(w.cond_c), "coarse");
    if (rc) return rc;
    rc = fill_fold(sa.fold[1], a->fine, F(w.cond_f), "fine");
    if (rc) return rc;
    sa.n_fold = 2;
    const bool fast_z = a->perturb && !a->lindisp && (s1 & 3) == 0;
    sa.gen = a->gen_rays; sa.W = a->W; sa.first = a->first;
    sa.focal = a->focal; sa.cx = a->cx; sa.cy = a->cy; sa.near_ = a->near_; sa.far_ = a->far_;
    sa.c2w = a->c2w; sa.rs = a->c2w_row_stride;
    sa.rays_out = a->gen_rays ? F(w.rays) : nullptr;
    sa.rays_in = a->rays; sa.ray_stride = a->ray_stride;
    sa.n = n; sa.s = s1; sa.do_z = fast_z;
    sa.t_vals = a->t_vals; sa.rng_state = rng; sa.z = z_c;
    {
        const long long work = fast_z ? (long long)n * (s1 >> 2) : (a->gen_rays ? (long long)n : 0);
        const unsigned blocks = (unsigned)(2 * FOLD_BLOCKS + (work + 255) / 256);
        render_setup_kernel<<<blocks, 256, 0, st>>>(sa);
        rc = check_launch("inerf_render_rays_fused[set-up]");
        if (rc) return rc;
    }
    if (!fast_z) {
        rc = a->perturb ? inerf_sample_coarse_rng(rays, n, stride, s1, a->t_vals, a->rng_state, a->lindisp, z_c, stream)
                        : inerf_sample_coarse(rays, n, stride, s1, a->t_vals, nullptr, a->lindisp, z_c, stream);
        if (rc) return rc;
    }

    mark(1);
    // ---- 2. coarse FaceNeRF ------------------------------------------------------------------------------------------------------
    // without rgb0 the compositor reads sigma alone: the density-only buffer (bf16) or the sigma lane of the full raw
    const int sig = a->rgb0 ? 0 : (a->mode == INERF_MLP_BF16 ? 1 : 4);
    rc = sig == 1 ? mlp_fwd_density(&a->coarse.dims, a->coarse.params_host, a->coarse.packed, F(w.cond_c), rays, stride, z_c, n, s1, F(w.raw_c), st)
                  : inerf_mlp_fwd(a->mode, &a->coarse.dims, a->coarse.params_host, a->coarse.packed, F(w.cond_c), rays, stride, z_c, n, s1, F(w.raw_c),
                                  stream);
    if (rc) return rc;

    mark(2);
    // ---- 3. coarse raw2outputs + importance sampling -------------------------------------------------------------------------------
    CompArgs ca{};
    ca.raw = reinterpret_cast<const float4*>(F(w.raw_c)); ca.z = z_c; ca.rays = rays; ca.ray_stride = stride; ca.bc_rgb = a->bc_rgb;
    ca.n = n; ca.s = s1; ca.white_bkgd = a->white_bkgd;
    ca.rgb = a->rgb0; ca.disp = a->disp0; ca.acc = a->acc0; ca.depth = F(w.depth0);
    ca.weights = nullptr; ca.rgb_fg = a->rgb_map_fg0; ca.last_weight = a->last_weight0;
    ca.rng_state = rng; ca.z_merged = z_m; ca.z_std = a->z_std; ca.flags = a->nonfinite;
    if (a->perturb && s1 == 64 && ni == 128) {
        if (sig == 0) composite_sample_64_128_kernel<0><<<(n + 7) / 8, 256, 0, st>>>(ca);
        else if (sig == 1) composite_sample_64_128_kernel<1><<<(n + 7) / 8, 256, 0, st>>>(ca);
        else composite_sample_64_128_kernel<4><<<(n + 7) / 8, 256, 0, st>>>(ca);
        rc = check_launch("inerf_render_rays_fused[coarse compositor + sampler]");
        if (rc) return rc;
    } else {
        float* w_c = F(w.w_c);
        if (sig == 0) {
            rc = inerf_composite_fwd(F(w.raw_c), z_c, rays + 3, stride, a->bc_rgb, nullptr, n, s1, a->white_bkgd, a->rgb0, a->disp0, a->acc0,
                                     F(w.depth0), w_c, a->rgb_map_fg0, stream);
        } else {
            ca.weights = w_c;
            if (sig == 1) launch_composite_sigma<1>(ca, st); else launch_composite_sigma<4>(ca, st);
            rc = check_launch("inerf_render_rays_fused[coarse compositor, sigma only]");
        }
        if (rc) return rc;
        if (a->last_weight0) {
            cudaError_t e = cudaMemcpy2DAsync(a->last_weight0, 4, w_c + (s1 - 1), (size_t)s1 * 4, 4, (size_t)n, cudaMemcpyDeviceToDevice, st);
            if (e != cudaSuccess) { set_error("inerf_render_rays_fused: last_weight0 copy: %s", cudaGetErrorString(e)); return (int)e; }
        }
        rc = a->perturb ? inerf_importance_sample_rng(z_c, w_c, n, s1, ni, a->rng_state, INERF_RNG_STREAM_PDF, nullptr, z_m, a->z_std, stream)
                        : inerf_importance_sample(z_c, w_c, n, s1, ni, a->u_vals, 0, INERF_PDF_EXACT_TORCH_CPU, F(w.z_s), nullptr, z_m, a->z_std,
                                                  stream);
        if (rc) return rc;
        if (a->nonfinite) {      // z_std here; the coarse maps of this path are scanned after the final compositor
            flag_zstd_kernel<<<(n + 1023) / 1024 < 148 ? (n + 1023) / 1024 : 148, 256, 0, st>>>(a->z_std, n, a->nonfinite);
            rc = check_launch("inerf_render_rays_fused[z_std scan]");
            if (rc) return rc;
        }
    }

    mark(3);
    // ---- 4. fine FaceNeRF --------------------------------------------------------------------------------------------------------
    rc = inerf_mlp_fwd(a->mode, &a->fine.dims, a->fine.params_host, a->fine.packed, F(w.cond_f), rays, stride, z_m, n, stot, F(w.raw_f), stream);
    if (rc) return rc;

    mark(4);
    // ---- 5. final raw2outputs (+ flags, + RNG bump) ----------------------------------------------------------------------------------
    CompArgs fa{};
    fa.raw = reinterpret_cast<const float4*>(F(w.raw_f)); fa.z = z_m; fa.rays = rays; fa.ray_stride = stride; fa.bc_rgb = a->bc_rgb;
    fa.n = n; fa.s = stot; fa.white_bkgd = a->white_bkgd;
    fa.rgb = a->rgb_map; fa.disp = a->disp_map; fa.acc = a->acc_map; fa.depth = a->depth_map;
    fa.weights = a->weights; fa.rgb_fg = a->rgb_map_fg; fa.last_weight = a->last_weight;
    fa.rng_bump = a->perturb ? rng : nullptr;
    fa.flags = a->nonfinite;
    if (fa.weights && ((uintptr_t)fa.weights & 7)) return fail(INERF_E_ALIGN, "inerf_render_rays_fused: weights must be 8-byte aligned");
    {
        const dim3 grid((n + 7) / 8), block(256);
        const int c2 = (stot + 63) / 64;
        if (c2 <= 1) composite_final_kernel<1><<<grid, block, 0, st>>>(fa);
        else if (c2 == 2) composite_final_kernel<2><<<grid, block, 0, st>>>(fa);
        else if (c2 == 3) composite_final_kernel<3><<<grid, block, 0, st>>>(fa);
        else composite_final_kernel<4><<<grid, block, 0, st>>>(fa);
        rc = check_launch("inerf_render_rays_fused[final compositor]");
        if (rc) return rc;
    }
    if (a->nonfinite && !(a->perturb && s1 == 64 && ni == 128)) {      // the coarse maps of the stand-alone path
        // inerf_flag_nonfinite sets bit i for tensor i: three empty entries put the maps on INERF_NF_RGB0 / _DISP0 / _ACC0
        const float* xs6[6] = {nullptr, nullptr, nullptr, a->rgb0, a->disp0, a->acc0};
        const int64_t ns6[6] = {0, 0, 0, a->rgb0 ? (int64_t)n * 3 : 0, n, n};
        rc = inerf_flag_nonfinite(xs6, ns6, 6, a->nonfinite, stream);
        if (rc) return rc;
    }
    mark(5);
    return INERF_OK;
}
}  // namespace

extern "C" int inerf_render_rays_fused(const InerfRenderArgs* a, void* stream) { return render_rays_fused(a, stream, nullptr); }

extern "C" int inerf_debug_render_stage_ms(const InerfRenderArgs* a, void* stream, float* ms_host5) {
    if (!ms_host5) return fail(INERF_E_ARG, "inerf_debug_render_stage_ms: NULL");
    cudaEvent_t ev[6];
    for (int i = 0; i < 6; ++i)
        if (cudaEventCreate(&ev[i]) != cudaSuccess) return fail(INERF_E_ARG, "inerf_debug_render_stage_ms: cudaEventCreate failed");
    int rc = render_rays_fused(a, stream, ev);
    if (rc == INERF_OK && a && a->n > 0) {
        cudaError_t e = cudaEventSynchronize(ev[5]);
        if (e != cudaSuccess) { set_error("inerf_debug_render_stage_ms: %s", cudaGetErrorString(e)); rc = (int)e; }
        for (int i = 0; i < 5 && rc == INERF_OK; ++i) cudaEventElapsedTime(&ms_host5[i], ev[i], ev[i + 1]);
    }
    for (int i = 0; i < 6; ++i) cudaEventDestroy(ev[i]);
    return rc;
}
