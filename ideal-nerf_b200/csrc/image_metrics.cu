// Image quality of rendered uint8 frames against ground-truth uint8 frames: exact SSE over three regions and the SSIM of Wang et al. 2004
// (11-tap Gaussian, sigma 1.5), on the device and graph-capturable.  The contract is written down in include/inerf_b200.h above
// inerf_image_metrics; oracle/image_metrics_ref.py restates it in numpy float64.  inerf_masked_sse (end of the file; oracle/masked_sse_ref.py)
// gives the exact SSE over a per-frame pixel mask instead of boxes: the torso region of data.torso_bits.
//
// One CTA scores one 32 x 32 tile of one frame.  It stages the tile plus its 5-pixel halo of both images in shared memory as bytes, sums
// the tile's squared errors in integers, then per channel runs the separable filter -- a horizontal pass over the 42 halo rows, then a
// vertical pass -- for the five moments (mu_x, mu_y, E[x^2], E[y^2], E[xy]) in fp32, and adds the SSIM of every tile position whose
// window lies inside the frame.  The tile's totals reach the frame's with one int64 / fp64 atomic each.
//
// fp32 moments: the variances are differences E[x^2] - mu^2 of numbers up to 255^2, whose rounding error (~4e-3) is not small against
// C2 = 58.5 where the window is flat.  Each image therefore enters the filter shifted by its own byte at the tile's first pixel (the
// variances and the covariance do not change under a shift; the means get it back): in a flat or smooth neighbourhood the shifted
// values are small and so is the cancellation.
#include "common.cuh"

using namespace inerf;

namespace {

constexpr int kTile = 32;                   // positions per side of a CTA's tile
constexpr int kHalo = 5;                    // radius of the 11-tap window
constexpr int kTaps = 2 * kHalo + 1;
constexpr int kSpan = kTile + 2 * kHalo;    // 42 input rows / columns a tile reads
constexpr int kPitch = kSpan + 2;
constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr float kC1 = 6.5025f;              // (0.01 * 255)^2
constexpr float kC2 = 58.5225f;             // (0.03 * 255)^2

struct Taps {
    float w[kTaps];
};

__device__ __forceinline__ long long warp_sum_ll(long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Pixels of the inclusive box {r0, r1, c0, c1} inside the H x W frame.
__device__ __forceinline__ long long box_pixels(const int32_t* b, int H, int W) {
    const int r0 = max(b[0], 0), r1 = min(b[1], H - 1), c0 = max(b[2], 0), c1 = min(b[3], W - 1);
    return (long long)max(r1 - r0 + 1, 0) * max(c1 - c0 + 1, 0);
}

__global__ void __launch_bounds__(kThreads) image_metrics_kernel(const uint8_t* __restrict__ pred, const uint8_t* __restrict__ gt,
                                                                 const int64_t* __restrict__ frame_index, const int32_t* __restrict__ bounds,
                                                                 int H, int W, int n_frames, int tiles_x, int tiles, const Taps g,
                                                                 long long* sse, long long* npix, double* ssim_sum) {
    __shared__ uint8_t s_img[2][3][kSpan][kPitch];       // pred, gt; per channel; halo rows / columns outside the frame are 0
    __shared__ float s_h[5][kSpan][kTile];              // horizontal-pass moments of one channel
    __shared__ long long s_red_i[3][kWarps];
    __shared__ float s_red_f[kWarps];

    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int b = blockIdx.x / tiles, tile = blockIdx.x - b * tiles;
    const int y0 = (tile / tiles_x) * kTile, x0 = (tile % tiles_x) * kTile;
    const long long f = frame_index[b];
    const bool live = f >= 0 && f < n_frames;
    const int32_t* bx = (bounds && live) ? bounds + f * 8 : nullptr;
    if (tile == 0 && t == 0) {
        npix[b * 3] = live ? (long long)H * W : 0;
        if (bounds) {
            npix[b * 3 + 1] = bx ? box_pixels(bx, H, W) : 0;
            npix[b * 3 + 2] = bx ? box_pixels(bx + 4, H, W) : 0;
        }
    }
    if (!live) return;                                  // sse and ssim_sum were zeroed before the launch

    const size_t hw = (size_t)H * W;
    const uint8_t* pa = pred + (size_t)b * hw * 3;
    const uint8_t* pb = gt + (size_t)f * hw * 3;
    for (int i = t; i < kSpan * kSpan * 3; i += kThreads) {
        const int r = i / (kSpan * 3), rem = i - r * (kSpan * 3), col = rem / 3, c = rem - col * 3;
        const int gy = y0 - kHalo + r, gx = x0 - kHalo + col;
        uint8_t va = 0, vb = 0;
        if (gy >= 0 && gy < H && gx >= 0 && gx < W) {
            const size_t o = ((size_t)gy * W + gx) * 3 + c;
            va = pa[o];
            vb = pb[o];
        }
        s_img[0][c][r][col] = va;
        s_img[1][c][r][col] = vb;
    }
    __syncthreads();

    // squared errors of the tile's pixels: full frame, face rect R, mouth box M (an int32 holds a tile's 1024 x 3 x 255^2)
    int e_full = 0, e_rect = 0, e_mouth = 0;
    for (int p = t; p < kTile * kTile; p += kThreads) {
        const int ly = p / kTile, lx = p - ly * kTile, gy = y0 + ly, gx = x0 + lx;
        if (gy >= H || gx >= W) continue;
        int e = 0;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const int d = (int)s_img[0][c][ly + kHalo][lx + kHalo] - (int)s_img[1][c][ly + kHalo][lx + kHalo];
            e += d * d;
        }
        e_full += e;
        if (bx) {
            if (gy >= bx[0] && gy <= bx[1] && gx >= bx[2] && gx <= bx[3]) e_rect += e;
            if (gy >= bx[4] && gy <= bx[5] && gx >= bx[6] && gx <= bx[7]) e_mouth += e;
        }
    }

    float s_acc = 0.f;
    for (int c = 0; c < 3; ++c) {
        const float sha = (float)s_img[0][c][kHalo][kHalo], shb = (float)s_img[1][c][kHalo][kHalo];
        for (int i = t; i < kSpan * kTile; i += kThreads) {
            const int r = i / kTile, x = i - r * kTile;
            float m0 = 0.f, m1 = 0.f, m2 = 0.f, m3 = 0.f, m4 = 0.f;
#pragma unroll
            for (int k = 0; k < kTaps; ++k) {
                const float a = (float)s_img[0][c][r][x + k] - sha, v = (float)s_img[1][c][r][x + k] - shb;
                m0 = fmaf(g.w[k], a, m0);
                m1 = fmaf(g.w[k], v, m1);
                m2 = fmaf(g.w[k], a * a, m2);              // a * a, v * v, a * v are exact: |a|, |v| <= 255
                m3 = fmaf(g.w[k], v * v, m3);
                m4 = fmaf(g.w[k], a * v, m4);
            }
            s_h[0][r][x] = m0;
            s_h[1][r][x] = m1;
            s_h[2][r][x] = m2;
            s_h[3][r][x] = m3;
            s_h[4][r][x] = m4;
        }
        __syncthreads();
        const int lx = lane, gx = x0 + lx;
        for (int ly = warp; ly < kTile; ly += kWarps) {
            const int gy = y0 + ly;
            if (gy < kHalo || gy >= H - kHalo || gx < kHalo || gx >= W - kHalo) continue;
            float m0 = 0.f, m1 = 0.f, m2 = 0.f, m3 = 0.f, m4 = 0.f;
#pragma unroll
            for (int k = 0; k < kTaps; ++k) {
                m0 = fmaf(g.w[k], s_h[0][ly + k][lx], m0);
                m1 = fmaf(g.w[k], s_h[1][ly + k][lx], m1);
                m2 = fmaf(g.w[k], s_h[2][ly + k][lx], m2);
                m3 = fmaf(g.w[k], s_h[3][ly + k][lx], m3);
                m4 = fmaf(g.w[k], s_h[4][ly + k][lx], m4);
            }
            const float va = m2 - m0 * m0, vb = m3 - m1 * m1, cov = m4 - m0 * m1;
            const float ua = m0 + sha, ub = m1 + shb;
            s_acc += ((2.f * ua * ub + kC1) * (2.f * cov + kC2)) / ((ua * ua + ub * ub + kC1) * (va + vb + kC2));
        }
        __syncthreads();                                // s_h is rewritten by the next channel
    }

    const long long w_full = warp_sum_ll(e_full), w_rect = warp_sum_ll(e_rect), w_mouth = warp_sum_ll(e_mouth);
    const float w_ssim = warp_sum(s_acc);
    if (lane == 0) {
        s_red_i[0][warp] = w_full;
        s_red_i[1][warp] = w_rect;
        s_red_i[2][warp] = w_mouth;
        s_red_f[warp] = w_ssim;
    }
    __syncthreads();
    if (t == 0) {
        long long e[3] = {0, 0, 0};
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) {
            e[0] += s_red_i[0][w];
            e[1] += s_red_i[1][w];
            e[2] += s_red_i[2][w];
            s += s_red_f[w];
        }
        for (int j = 0; j < (bounds ? 3 : 1); ++j)
            if (e[j]) atomicAdd(reinterpret_cast<unsigned long long*>(sse + b * 3 + j), (unsigned long long)e[j]);
        if (s != 0.f) atomicAdd(ssim_sum + b, (double)s);
    }
}

// ---- SSE over a per-frame pixel mask (inerf_masked_sse) ---------------------------------------------------------------------------------
// One 256-thread CTA scores kMaskPixels consecutive pixels of one row of the batch; the 32 lanes of a warp read 32 consecutive pixels, whose
// mask bits are one word (read once per warp, broadcast), so only pixels in the mask load their bytes.
constexpr int kMaskThreads = 256;
constexpr int kMaskPixels = 4 * kMaskThreads;

__global__ void __launch_bounds__(kMaskThreads) masked_sse_kernel(const uint8_t* __restrict__ pred, const uint8_t* __restrict__ gt,
                                                                  const int64_t* __restrict__ frame_index, const uint32_t* __restrict__ bits,
                                                                  int hw, int words, int n_frames, int chunks, long long* sse,
                                                                  long long* npix) {
    __shared__ long long s_e[kMaskThreads / 32];
    __shared__ int s_n[kMaskThreads / 32];
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int b = blockIdx.x / chunks, p0 = (blockIdx.x - b * chunks) * kMaskPixels;
    const long long f = frame_index[b];
    if (f < 0 || f >= n_frames) return;                 // sse and npix were zeroed before the launch
    const uint8_t* pa = pred + (size_t)b * hw * 3;
    const uint8_t* pb = gt + (size_t)f * hw * 3;
    const uint32_t* m = bits + (size_t)f * words;
    const int p1 = min(p0 + kMaskPixels, hw);
    int e = 0, n = 0;                                   // at most 4 pixels x 3 x 255^2 per thread
    for (int p = p0 + t; p < p1; p += kMaskThreads) {
        if (!((__ldg(m + (p >> 5)) >> (p & 31)) & 1u)) continue;
        const size_t o = (size_t)p * 3;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const int d = (int)pa[o + c] - (int)pb[o + c];
            e += d * d;
        }
        ++n;
    }
    const long long w_e = warp_sum_ll(e);
    int w_n = n;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) w_n += __shfl_xor_sync(0xffffffffu, w_n, o);
    if (lane == 0) {
        s_e[warp] = w_e;
        s_n[warp] = w_n;
    }
    __syncthreads();
    if (t == 0) {
        long long te = 0, tn = 0;
#pragma unroll
        for (int w = 0; w < kMaskThreads / 32; ++w) {
            te += s_e[w];
            tn += s_n[w];
        }
        if (te) atomicAdd(reinterpret_cast<unsigned long long*>(sse + b), (unsigned long long)te);
        if (tn) atomicAdd(reinterpret_cast<unsigned long long*>(npix + b), (unsigned long long)tn);
    }
}

}  // namespace

extern "C" int inerf_image_metrics(const uint8_t* pred, const uint8_t* gt_frames, const int64_t* frame_index, const int32_t* bounds,
                                   int32_t B, int32_t H, int32_t W, int32_t n_frames, int64_t* sse, int64_t* npix, double* ssim_sum,
                                   void* stream) {
    if (!pred || !gt_frames || !frame_index || !sse || !npix || !ssim_sum) return fail(INERF_E_ARG, "inerf_image_metrics: NULL pointer");
    if (B < 0 || n_frames < 0) return fail(INERF_E_ARG, "inerf_image_metrics: negative B or n_frames");
    if (H < kTaps || W < kTaps || (int64_t)H * W > INERF_IMAGE_METRICS_MAX_PIXELS) {
        set_error("inerf_image_metrics: %d x %d frames (need H, W >= %d and H * W <= %d)", H, W, kTaps, INERF_IMAGE_METRICS_MAX_PIXELS);
        return INERF_E_SHAPE;
    }
    const int tiles_x = (W + kTile - 1) / kTile, tiles = tiles_x * ((H + kTile - 1) / kTile);
    if ((int64_t)B * tiles > 0x7fffffff) return fail(INERF_E_SHAPE, "inerf_image_metrics: B * tiles exceeds the grid");
    if (B == 0) return INERF_OK;
    Taps g;
    double w[kTaps], sum = 0.;                           // scipy.ndimage's kernel: exp(-x^2 / (2 sigma^2)), normalised in fp64
    for (int k = 0; k < kTaps; ++k) sum += (w[k] = exp(-0.5 * (k - kHalo) * (k - kHalo) / (1.5 * 1.5)));
    for (int k = 0; k < kTaps; ++k) g.w[k] = (float)(w[k] / sum);
    cudaStream_t s = as_stream(stream);
    cudaError_t e = bounds ? cudaMemsetAsync(sse, 0, (size_t)B * 3 * sizeof(int64_t), s)
                           : cudaMemset2DAsync(sse, 3 * sizeof(int64_t), 0, sizeof(int64_t), (size_t)B, s);    // column 0 only
    if (e == cudaSuccess) e = cudaMemsetAsync(ssim_sum, 0, (size_t)B * sizeof(double), s);
    if (e != cudaSuccess) {
        set_error("inerf_image_metrics: %s", cudaGetErrorString(e));
        return (int)e;
    }
    image_metrics_kernel<<<(unsigned)(B * tiles), kThreads, 0, s>>>(pred, gt_frames, frame_index, bounds, H, W, n_frames, tiles_x, tiles, g,
                                                                    reinterpret_cast<long long*>(sse), reinterpret_cast<long long*>(npix),
                                                                    ssim_sum);
    return check_launch("inerf_image_metrics");
}

extern "C" int inerf_masked_sse(const uint8_t* pred, const uint8_t* gt_frames, const int64_t* frame_index, const uint32_t* bits, int32_t B,
                                int32_t H, int32_t W, int32_t n_frames, int64_t* sse, int64_t* npix, void* stream) {
    if (!pred || !gt_frames || !frame_index || !bits || !sse || !npix) return fail(INERF_E_ARG, "inerf_masked_sse: NULL pointer");
    if (B < 0 || n_frames < 0) return fail(INERF_E_ARG, "inerf_masked_sse: negative B or n_frames");
    if (H < kTaps || W < kTaps || (int64_t)H * W > INERF_IMAGE_METRICS_MAX_PIXELS) {
        set_error("inerf_masked_sse: %d x %d frames (need H, W >= %d and H * W <= %d)", H, W, kTaps, INERF_IMAGE_METRICS_MAX_PIXELS);
        return INERF_E_SHAPE;
    }
    const int hw = H * W, chunks = (hw + kMaskPixels - 1) / kMaskPixels;
    if ((int64_t)B * chunks > 0x7fffffff) return fail(INERF_E_SHAPE, "inerf_masked_sse: B * chunks exceeds the grid");
    if (B == 0) return INERF_OK;
    cudaStream_t s = as_stream(stream);
    cudaError_t e = cudaMemsetAsync(sse, 0, (size_t)B * sizeof(int64_t), s);
    if (e == cudaSuccess) e = cudaMemsetAsync(npix, 0, (size_t)B * sizeof(int64_t), s);
    if (e != cudaSuccess) {
        set_error("inerf_masked_sse: %s", cudaGetErrorString(e));
        return (int)e;
    }
    masked_sse_kernel<<<(unsigned)(B * chunks), kMaskThreads, 0, s>>>(pred, gt_frames, frame_index, bits, hw, (hw + 31) / 32, n_frames, chunks,
                                                                      reinterpret_cast<long long*>(sse), reinterpret_cast<long long*>(npix));
    return check_launch("inerf_masked_sse");
}
