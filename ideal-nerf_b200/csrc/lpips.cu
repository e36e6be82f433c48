// LPIPS v0.1 with the AlexNet trunk (Zhang et al. 2018) of rendered uint8 frames against ground-truth uint8 frames, on the device and
// graph-capturable.  The contract is written down in include/inerf_b200.h above inerf_lpips; oracle/lpips_ref.py restates it in float64.
//
// Per call, for the B rows at once (image 2b = pred[b], image 2b + 1 = gt_frames[frame_index[b]]):
//   conv1 -> head1, pool -> conv2 -> head2, pool -> conv3 -> head3 -> conv4 -> head4 -> conv5 -> head5, then one reduction kernel.
// conv_kernel is one FP32 implicit GEMM (M = output channels, N = output pixels of both images of a row, K = C_in k^2), templated on the
// layer geometry: a 64 x 64 tile per 256-thread CTA, 4 x 4 outputs per thread, operand tiles of 16 k-steps double-buffered in shared
// memory, bias and ReLU fused.  The conv1 instance gathers its operand from the uint8 frames directly (BGR bytes to RGB, the im2tensor /
// ScalingLayer affine, zero padding in the scaled space), so no float copy of a frame exists.  Feature maps are fp32 (image, C, h, w) in
// the workspace.  head_kernel scores one layer: per position both images' channel norms, the squared difference of the normalised vectors
// dotted with lin_k, and one partial sum per CTA in a fixed order; lpips_sum_kernel adds the partials of each layer in index order and
// divides by h_k w_k.  No atomics: results are bit-identical from run to run and between eager calls and graph replay.
#include <algorithm>

#include "common.cuh"

using namespace inerf;

namespace {

constexpr int kBM = 64, kBN = 64, kBK = 16;          // conv tile: output channels x output pixels x reduction steps
constexpr int kConvThreads = 256;
constexpr int kHeadThreads = 256;
constexpr int kHeadWarps = kHeadThreads / 32;
constexpr int kHeadPos = 32;                          // positions per head CTA
constexpr int kPoolThreads = 256;
constexpr int kSumThreads = 128;
constexpr int kMinSide = 31;                          // conv1 must give >= 7 outputs so that both 3 / 2 max pools leave >= 1

__host__ __device__ constexpr int conv_out(int n, int k, int s, int p) { return (n + 2 * p - k) / s + 1; }
__host__ __device__ constexpr int pool_out(int n) { return (n - 3) / 2 + 1; }

// Side of each layer's map for an input side n: f1, f2, f3 (= f4 = f5).
struct Sides {
    int s[3];
    explicit Sides(int n) {
        s[0] = conv_out(n, 11, 4, 2);
        s[1] = pool_out(s[0]);
        s[2] = pool_out(s[1]);
    }
};

// The workspace, in floats from its start: the seven maps, then the per-CTA partial sums of the five heads.  Every region starts on a
// 256-byte boundary.
struct Layout {
    size_t f1, q1, f2, q2, f3, f4, f5, part[5], total;     // offsets and total in floats
    int h[3], w[3], tiles[5];                             // map sides of f1, f2, f3 (= f4 = f5); head CTAs per row of each layer
    Layout(int B, int H, int W) {
        const Sides sh(H), sw(W);
        for (int i = 0; i < 3; ++i) h[i] = sh.s[i], w[i] = sw.s[i];
        size_t at = 0;
        auto take = [&](size_t n) { const size_t o = at; at += (n + 63) / 64 * 64; return o; };
        const size_t imgs = 2 * (size_t)B;
        f1 = take(imgs * 64 * h[0] * w[0]);
        q1 = take(imgs * 64 * h[1] * w[1]);
        f2 = take(imgs * 192 * h[1] * w[1]);
        q2 = take(imgs * 192 * h[2] * w[2]);
        f3 = take(imgs * 384 * h[2] * w[2]);
        f4 = take(imgs * 256 * h[2] * w[2]);
        f5 = take(imgs * 256 * h[2] * w[2]);
        for (int k = 0; k < 5; ++k) {
            const int i = k < 2 ? k : 2;
            tiles[k] = (h[i] * w[i] + kHeadPos - 1) / kHeadPos;
            part[k] = take((size_t)B * tiles[k]);
        }
        total = at;
    }
};

// One row's source bytes for conv1: pred[b], or gt_frames[frame_index[b]] -- pred[b] itself when the index is out of range (that row's
// score is set to 0 at the end; reading its own bytes keeps every load in bounds).
struct U8Src {
    const uint8_t* pred;
    const uint8_t* gt;
    const int64_t* frame_index;
    int n_frames;
};

template <int CIN, int COUT, int KS, int S, int P, bool U8>
__global__ void __launch_bounds__(kConvThreads) conv_kernel(const float* __restrict__ in, U8Src src, const float* __restrict__ wt,
                                                            const float* __restrict__ bias, float* __restrict__ out, int Hi, int Wi, int Ho,
                                                            int Wo) {
    constexpr int KK = KS * KS, K = CIN * KK, NK = (K + kBK - 1) / kBK;
    static_assert(COUT % kBM == 0, "output channels must fill the M tiles");
    __shared__ __align__(16) float As[2][kBK][kBM];
    __shared__ __align__(16) float Bs[2][kBK][kBN];

    const int t = threadIdx.x;
    const int b = blockIdx.z, m0 = blockIdx.y * kBM, n0 = blockIdx.x * kBN;
    const int hw = Ho * Wo, N = 2 * hw;

    // operand B (the im2col column): this thread loads column nl of the tile at k-steps kb, kb + 4, kb + 8, kb + 12
    const int nl = t & (kBN - 1), kb = t >> 6;
    const int n = n0 + nl;
    const bool n_ok = n < N;
    const int side = n_ok && n >= hw, p = n - side * hw;
    const int oy = p / Wo, ox = p - oy * Wo;
    const int iy0 = oy * S - P, ix0 = ox * S - P;
    const float* fin = nullptr;
    const uint8_t* uin = nullptr;
    if constexpr (U8) {
        const size_t frame = (size_t)Hi * Wi * 3;
        if (side == 0) {
            uin = src.pred + (size_t)b * frame;
        } else {
            const long long f = src.frame_index[b];
            uin = (f >= 0 && f < src.n_frames) ? src.gt + (size_t)f * frame : src.pred + (size_t)b * frame;
        }
    } else {
        fin = in + (size_t)(2 * b + side) * CIN * Hi * Wi;
    }
    // operand A (the weights, row-major (COUT, K)): this thread loads k-steps ka .. ka + 3 of output channel m0 + ma
    const int ma = t >> 2, ka = (t & 3) * 4;
    const float* wrow = wt + (size_t)(m0 + ma) * K;

    float ra[4], rb[4];
    auto load = [&](int k0) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int k = k0 + ka + j;
            ra[j] = (K % kBK == 0 || k < K) ? __ldg(wrow + k) : 0.f;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int k = k0 + kb + 4 * j;
            float v = 0.f;
            if (n_ok && (K % kBK == 0 || k < K)) {
                const int ci = k / KK, r = k - ci * KK, ky = r / KS, kx = r - ky * KS;
                const int iy = iy0 + ky, ix = ix0 + kx;
                if (iy >= 0 && iy < Hi && ix >= 0 && ix < Wi) {
                    if constexpr (U8) {
                        // AlexNet channel ci (R, G, B) is byte 2 - ci of a BGR pixel; lpips' im2tensor, then its ScalingLayer
                        const float x = (float)__ldg(uin + ((size_t)iy * Wi + ix) * 3 + (2 - ci)) / 127.5f - 1.f;
                        const float shift = ci == 0 ? -0.030f : ci == 1 ? -0.088f : -0.188f;
                        const float scale = ci == 0 ? 0.458f : ci == 1 ? 0.448f : 0.450f;
                        v = (x - shift) / scale;
                    } else {
                        v = __ldg(fin + ((size_t)ci * Hi + iy) * Wi + ix);
                    }
                }
            }
            rb[j] = v;
        }
    };
    auto store = [&](int buf) {
#pragma unroll
        for (int j = 0; j < 4; ++j) As[buf][ka + j][ma] = ra[j];
#pragma unroll
        for (int j = 0; j < 4; ++j) Bs[buf][kb + 4 * j][nl] = rb[j];
    };

    const int tm = t >> 4, tn = t & 15;                   // this thread's outputs: channels m0 + 4 tm + i, pixels n0 + 4 tn + j
    float acc[4][4] = {};
    load(0);
    store(0);
    __syncthreads();
    for (int kt = 0; kt < NK; ++kt) {
        const int buf = kt & 1;
        if (kt + 1 < NK) load((kt + 1) * kBK);
#pragma unroll
        for (int kk = 0; kk < kBK; ++kk) {
            const float4 a = *reinterpret_cast<const float4*>(&As[buf][kk][tm * 4]);
            const float4 v = *reinterpret_cast<const float4*>(&Bs[buf][kk][tn * 4]);
            const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        if (kt + 1 < NK) store(buf ^ 1);                  // buf ^ 1 was last read in iteration kt - 1, before the barrier below it
        __syncthreads();
    }

#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int m = m0 + tm * 4 + i;
        const float bm = __ldg(bias + m);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int nn = n0 + tn * 4 + j;
            if (nn >= N) continue;
            const int s = nn >= hw, pp = nn - s * hw;
            out[((size_t)(2 * b + s) * COUT + m) * hw + pp] = fmaxf(acc[i][j] + bm, 0.f);
        }
    }
}

// 3 x 3 max pool, stride 2, no padding, of `planes` (h, w) planes.
__global__ void __launch_bounds__(kPoolThreads) pool_kernel(const float* __restrict__ in, float* __restrict__ out, size_t planes, int h, int w,
                                                            int ho, int wo) {
    const size_t total = planes * ho * wo;
    for (size_t i = (size_t)blockIdx.x * kPoolThreads + threadIdx.x; i < total; i += (size_t)gridDim.x * kPoolThreads) {
        const size_t pl = i / ((size_t)ho * wo);
        const int r = (int)(i - pl * ho * wo), y = r / wo, x = r - y * wo;
        const float* src = in + pl * h * w + (size_t)(2 * y) * w + 2 * x;
        float v = src[0];
#pragma unroll
        for (int dy = 0; dy < 3; ++dy)
#pragma unroll
            for (int dx = 0; dx < 3; ++dx) v = fmaxf(v, src[dy * w + dx]);
        out[i] = v;
    }
}

// One LPIPS layer on kHeadPos consecutive positions of row blockIdx.y: lane = position (coalesced reads of each channel plane), warp w =
// the channels w, w + kHeadWarps, ...  Both images' squared norms are added over the warps, then each thread adds lin[c] d_c^2 over its
// channels with d = a / (|a| + 1e-10) - g / (|g| + 1e-10); the CTA's total over its positions goes to partial[row * tiles + blockIdx.x].
// Every sum runs in a fixed order.
template <int C>
__global__ void __launch_bounds__(kHeadThreads) head_kernel(const float* __restrict__ f, const float* __restrict__ lin, int hw, int tiles,
                                                            float* __restrict__ partial) {
    __shared__ float s_a[kHeadWarps][kHeadPos], s_g[kHeadWarps][kHeadPos];
    __shared__ float s_den[2][kHeadPos];
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5, b = blockIdx.y, p = blockIdx.x * kHeadPos + lane;
    const bool ok = p < hw;
    const float* a = f + (size_t)(2 * b) * C * hw + p;
    const float* g = a + (size_t)C * hw;
    float na = 0.f, ng = 0.f;
    if (ok)
        for (int c = warp; c < C; c += kHeadWarps) {
            const float x = a[(size_t)c * hw], y = g[(size_t)c * hw];
            na = fmaf(x, x, na);
            ng = fmaf(y, y, ng);
        }
    s_a[warp][lane] = na;
    s_g[warp][lane] = ng;
    __syncthreads();
    if (warp == 0) {
        float sa = 0.f, sg = 0.f;
#pragma unroll
        for (int w = 0; w < kHeadWarps; ++w) {
            sa += s_a[w][lane];
            sg += s_g[w][lane];
        }
        s_den[0][lane] = sqrtf(sa) + 1e-10f;
        s_den[1][lane] = sqrtf(sg) + 1e-10f;
    }
    __syncthreads();
    const float da = s_den[0][lane], dg = s_den[1][lane];
    float v = 0.f;
    if (ok)
        for (int c = warp; c < C; c += kHeadWarps) {
            const float d = a[(size_t)c * hw] / da - g[(size_t)c * hw] / dg;
            v = fmaf(__ldg(lin + c), d * d, v);
        }
    s_a[warp][lane] = v;                                  // s_a's norms were read by warp 0 before the barrier above
    __syncthreads();
    if (warp == 0) {
        float sum = 0.f;
#pragma unroll
        for (int w = 0; w < kHeadWarps; ++w) sum += s_a[w][lane];
        sum = warp_sum(sum);
        if (lane == 0) partial[(size_t)b * tiles + blockIdx.x] = sum;
    }
}

struct SumArgs {
    const float* part[5];
    int tiles[5];
    int hw[5];
};

// out[b] = sum over the five layers, in order, of (the layer's partials of row b, summed in order) / (h_k w_k); 0 for an out-of-range
// frame index.
__global__ void __launch_bounds__(kSumThreads) lpips_sum_kernel(SumArgs a, const int64_t* __restrict__ frame_index, int n_frames, int B,
                                                                float* __restrict__ out) {
    const int b = blockIdx.x * kSumThreads + threadIdx.x;
    if (b >= B) return;
    const long long f = frame_index[b];
    float total = 0.f;
    if (f >= 0 && f < n_frames) {
#pragma unroll
        for (int k = 0; k < 5; ++k) {
            const float* q = a.part[k] + (size_t)b * a.tiles[k];
            float s = 0.f;
            for (int i = 0; i < a.tiles[k]; ++i) s += q[i];
            total += s / (float)a.hw[k];
        }
    }
    out[b] = total;
}

template <int CIN, int COUT, int KS, int S, int P, bool U8>
void launch_conv(const float* in, U8Src src, const float* w, const float* bias, float* out, int B, int Hi, int Wi, int Ho, int Wo,
                 cudaStream_t s) {
    const dim3 grid((unsigned)((2 * Ho * Wo + kBN - 1) / kBN), COUT / kBM, (unsigned)B);
    conv_kernel<CIN, COUT, KS, S, P, U8><<<grid, kConvThreads, 0, s>>>(in, src, w, bias, out, Hi, Wi, Ho, Wo);
}

template <int C>
void launch_head(const float* f, const float* lin, int B, int hw, int tiles, float* partial, cudaStream_t s) {
    head_kernel<C><<<dim3((unsigned)tiles, (unsigned)B), kHeadThreads, 0, s>>>(f, lin, hw, tiles, partial);
}

void launch_pool(const float* in, float* out, size_t planes, int h, int w, int ho, int wo, cudaStream_t s) {
    const size_t total = planes * ho * wo;
    const unsigned blocks = (unsigned)std::min<size_t>((total + kPoolThreads - 1) / kPoolThreads, (size_t)num_sms() * 16);
    pool_kernel<<<blocks, kPoolThreads, 0, s>>>(in, out, planes, h, w, ho, wo);
}

int check_shape(const char* what, int32_t B, int32_t H, int32_t W) {
    if (B < 0) {
        set_error("%s: negative B", what);
        return INERF_E_ARG;
    }
    if (H < kMinSide || W < kMinSide || (int64_t)H * W > INERF_IMAGE_METRICS_MAX_PIXELS || B > INERF_LPIPS_MAX_ROWS) {
        set_error("%s: %d rows of %d x %d frames (need H, W >= %d, H * W <= %d, B <= %d)", what, B, H, W, kMinSide,
                  INERF_IMAGE_METRICS_MAX_PIXELS, INERF_LPIPS_MAX_ROWS);
        return INERF_E_SHAPE;
    }
    return INERF_OK;
}

}  // namespace

extern "C" int inerf_lpips_workspace_bytes(int32_t B, int32_t H, int32_t W, size_t* bytes) {
    if (!bytes) return fail(INERF_E_ARG, "inerf_lpips_workspace_bytes: NULL pointer");
    if (int rc = check_shape("inerf_lpips_workspace_bytes", B, H, W)) return rc;
    *bytes = Layout(B, H, W).total * sizeof(float);
    return INERF_OK;
}

extern "C" int inerf_lpips(const float* const* params_host, const uint8_t* pred, const uint8_t* gt_frames, const int64_t* frame_index,
                           int32_t B, int32_t H, int32_t W, int32_t n_frames, void* workspace, size_t workspace_bytes, float* out,
                           void* stream) {
    if (!params_host || !pred || !gt_frames || !frame_index || !workspace || !out) return fail(INERF_E_ARG, "inerf_lpips: NULL pointer");
    for (int i = 0; i < INERF_LPIPS_N_PARAMS; ++i)
        if (!params_host[i]) return fail(INERF_E_ARG, "inerf_lpips: NULL parameter pointer");
    if (n_frames < 0) return fail(INERF_E_ARG, "inerf_lpips: negative n_frames");
    if (int rc = check_shape("inerf_lpips", B, H, W)) return rc;
    const Layout L(B, H, W);
    if (workspace_bytes < L.total * sizeof(float)) {
        set_error("inerf_lpips: workspace of %zu bytes, need %zu", workspace_bytes, L.total * sizeof(float));
        return INERF_E_SHAPE;
    }
    if (B == 0) return INERF_OK;

    cudaStream_t s = as_stream(stream);
    float* ws = static_cast<float*>(workspace);
    const float* const* pp = params_host;
    const U8Src src{pred, gt_frames, frame_index, n_frames};
    const U8Src none{nullptr, nullptr, nullptr, 0};
    const size_t imgs = 2 * (size_t)B;
    const int hw[3] = {L.h[0] * L.w[0], L.h[1] * L.w[1], L.h[2] * L.w[2]};
    float* f1 = ws + L.f1;
    float* q1 = ws + L.q1;
    float* f2 = ws + L.f2;
    float* q2 = ws + L.q2;
    float* f3 = ws + L.f3;
    float* f4 = ws + L.f4;
    float* f5 = ws + L.f5;

    launch_conv<3, 64, 11, 4, 2, true>(nullptr, src, pp[0], pp[1], f1, B, H, W, L.h[0], L.w[0], s);
    launch_head<64>(f1, pp[10], B, hw[0], L.tiles[0], ws + L.part[0], s);
    launch_pool(f1, q1, imgs * 64, L.h[0], L.w[0], L.h[1], L.w[1], s);
    launch_conv<64, 192, 5, 1, 2, false>(q1, none, pp[2], pp[3], f2, B, L.h[1], L.w[1], L.h[1], L.w[1], s);
    launch_head<192>(f2, pp[11], B, hw[1], L.tiles[1], ws + L.part[1], s);
    launch_pool(f2, q2, imgs * 192, L.h[1], L.w[1], L.h[2], L.w[2], s);
    launch_conv<192, 384, 3, 1, 1, false>(q2, none, pp[4], pp[5], f3, B, L.h[2], L.w[2], L.h[2], L.w[2], s);
    launch_head<384>(f3, pp[12], B, hw[2], L.tiles[2], ws + L.part[2], s);
    launch_conv<384, 256, 3, 1, 1, false>(f3, none, pp[6], pp[7], f4, B, L.h[2], L.w[2], L.h[2], L.w[2], s);
    launch_head<256>(f4, pp[13], B, hw[2], L.tiles[3], ws + L.part[3], s);
    launch_conv<256, 256, 3, 1, 1, false>(f4, none, pp[8], pp[9], f5, B, L.h[2], L.w[2], L.h[2], L.w[2], s);
    launch_head<256>(f5, pp[14], B, hw[2], L.tiles[4], ws + L.part[4], s);

    SumArgs a;
    for (int k = 0; k < 5; ++k) {
        a.part[k] = ws + L.part[k];
        a.tiles[k] = L.tiles[k];
        a.hw[k] = hw[k < 2 ? k : 2];
    }
    lpips_sum_kernel<<<(unsigned)((B + kSumThreads - 1) / kSumThreads), kSumThreads, 0, s>>>(a, frame_index, n_frames, B, out);
    return check_launch("inerf_lpips");
}
