// FaceNeRF MLP, fp32 mode: exact-arithmetic path (FFMA, fp32 everywhere) + conditioning fold.  The C-ABI dispatch of every MLP mode
// is in mlp_api.cu.
//
// Reference: models/face_nerf.py:40-80 (forward), NeRFs/HeadNeRF/train/audio_exp_nerf.py:332,376-394
// (points, embedding, netchunk loop), NeRFs/HeadNeRF/helper.py:174-204 (positional encoding).
//
// The fp32 mode is the "max-abs <= 1e-3 vs the reference" mode of BASELINE.json and the on-device
// yardstick for the bf16 tensor-core kernel (mlp_bf16.cu).  One CTA owns a tile of 64 points and
// keeps every activation in shared memory from the positional encoding to the (r,g,b,sigma) output;
// only the weights stream in (from L2, nn.Linear layout, no repack so training can update them in
// place).  Each layer is a 64 x N x K register-tiled SGEMM: 256 threads, 8 points x 8 (or 4)
// features per thread, K consumed in 16-wide slices double-buffered through shared memory.
//
// Conditioning (aud | expr/3 | latent) is constant over the call, so its weight columns are folded
// into the biases once per call by inerf_mlp_fold_cond (SURVEY.md Appendix B) and the per-point
// network is 63->256, 4x(256->256), 319->256, 2x(256->256), {256->1, 283->128, 2x(128->128), 128->3}.
#include <cuda_bf16.h>

#include <cuda_fp16.h>

#include "mlp_common.cuh"
#include "fold_cond.cuh"

using namespace inerf;

namespace {

constexpr int TM = 64;            // points per tile
constexpr int KC = 16;            // K slice
constexpr int NTHREADS = 256;

// activation element (k, m) of a [K][64] k-major buffer; 16-byte chunks are XOR-swizzled by k/4 so
// that the epilogue's column-of-rows float4 stores are bank-conflict free.
__device__ __forceinline__ int act_idx(int k, int m) { return k * TM + ((((m >> 2) ^ (k >> 2)) & 15) << 2) + (m & 3); }

struct Seg {
    const float* src;   // smem activations [K][64]
    int k;              // rows used
    int wcol;           // first weight column
};

template <int N>
__device__ __forceinline__ void load_w_regs(float (&r)[N / 16], const float* __restrict__ W, int ldw, const Seg& sg,
                                            int k0, int tid) {
    constexpr int PER = N / 16;
    const int n = tid % N, kk0 = (tid / N) * PER;
    const float* row = W + (size_t)n * ldw + sg.wcol + k0 + kk0;
#pragma unroll
    for (int i = 0; i < PER; ++i) r[i] = (k0 + kk0 + i < sg.k) ? __ldg(row + i) : 0.0f;
}

template <int N>
__device__ __forceinline__ void store_w_smem(const float (&r)[N / 16], float* ws, int tid) {
    constexpr int PER = N / 16;
    const int n = tid % N, kk0 = (tid / N) * PER;
#pragma unroll
    for (int i = 0; i < PER; ++i) ws[(kk0 + i) * N + n] = r[i];
}

// out[n][m] = act( sum_k W[n][wcol+k] * in[k][m] + bias[n] )   for one 64-point tile.
// N = 256: thread owns features {4tn..4tn+3} U {128+4tn..}, N = 128: {4tn..4tn+3}; points 8tm..8tm+7.
template <int N>
__device__ void gemm_layer(const float* __restrict__ W, int ldw, const Seg* segs, int nseg,
                           const float* __restrict__ bias, float* __restrict__ out, float* __restrict__ wsm,
                           float* __restrict__ save = nullptr) {
    constexpr int NT = N / 32;
    const int tid = threadIdx.x, tn = tid & 31, tm = tid >> 5;
    float acc[NT][8];
#pragma unroll
    for (int j = 0; j < NT; ++j)
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[j][i] = 0.f;

    int nchunks = 0;
    for (int sidx = 0; sidx < nseg; ++sidx) nchunks += (segs[sidx].k + KC - 1) / KC;

    float wr[N / 16];
    int seg_i = 0, k0 = 0;
    load_w_regs<N>(wr, W, ldw, segs[0], 0, tid);
    store_w_smem<N>(wr, wsm, tid);
    __syncthreads();
    for (int c = 0; c < nchunks; ++c) {
        // position of the next chunk
        int nseg_i = seg_i, nk0 = k0 + KC;
        if (nk0 >= segs[seg_i].k) { nseg_i = seg_i + 1; nk0 = 0; }
        const bool more = c + 1 < nchunks;
        if (more) load_w_regs<N>(wr, W, ldw, segs[nseg_i], nk0, tid);

        const float* ws = wsm + (c & 1) * (KC * N);
        const float* in = segs[seg_i].src;
        const int kmax = min(KC, segs[seg_i].k - k0);
#pragma unroll 4
        for (int kk = 0; kk < KC; ++kk) {
            if (kk < kmax) {
                const int k = k0 + kk;
                const int sw = (k >> 2) & 15;
                const float4 a0 = *reinterpret_cast<const float4*>(in + k * TM + (((2 * tm) ^ sw) << 2));
                const float4 a1 = *reinterpret_cast<const float4*>(in + k * TM + (((2 * tm + 1) ^ sw) << 2));
                const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
                float b[NT];
                const float4 b0 = *reinterpret_cast<const float4*>(ws + kk * N + 4 * tn);
                b[0] = b0.x; b[1] = b0.y; b[2] = b0.z; b[3] = b0.w;
                if constexpr (NT == 8) {
                    const float4 b1 = *reinterpret_cast<const float4*>(ws + kk * N + 128 + 4 * tn);
                    b[4] = b1.x; b[5] = b1.y; b[6] = b1.z; b[7] = b1.w;
                }
#pragma unroll
                for (int j = 0; j < NT; ++j)
#pragma unroll
                    for (int i = 0; i < 8; ++i) acc[j][i] = fmaf(b[j], a[i], acc[j][i]);
            }
        }
        if (more) store_w_smem<N>(wr, wsm + ((c + 1) & 1) * (KC * N), tid);
        seg_i = nseg_i; k0 = nk0;
        __syncthreads();
    }
    // epilogue: bias + ReLU, write the next layer's k-major activations
#pragma unroll
    for (int j = 0; j < NT; ++j) {
        const int n = 4 * tn + (j & 3) + 128 * (j >> 2);
        const float b = __ldg(bias + n);
#pragma unroll
        for (int i = 0; i < 8; ++i) { const float v = acc[j][i] + b; acc[j][i] = v < 0.f ? 0.f : v; }      // F.relu: a NaN stays a NaN (fmaxf would swallow it)
        const int sw = (n >> 2) & 15;
        *reinterpret_cast<float4*>(out + n * TM + (((2 * tm) ^ sw) << 2)) = make_float4(acc[j][0], acc[j][1], acc[j][2], acc[j][3]);
        *reinterpret_cast<float4*>(out + n * TM + (((2 * tm + 1) ^ sw) << 2)) = make_float4(acc[j][4], acc[j][5], acc[j][6], acc[j][7]);
    }
    if (save) {      // training: keep the post-ReLU activations, point-major rows of SAVE_W floats (coalesced 512 B per warp store)
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            float* row = save + (size_t)(8 * tm + i) * SAVE_W + 4 * tn;
#pragma unroll
            for (int jg = 0; jg < NT / 4; ++jg)
                *reinterpret_cast<float4*>(row + 128 * jg) = make_float4(acc[4 * jg][i], acc[4 * jg + 1][i], acc[4 * jg + 2][i], acc[4 * jg + 3][i]);
        }
    }
    __syncthreads();
}

// dot products of NOUT tiny output rows with a [K][64] activation buffer; result in red[o][m]
template <int NOUT>
__device__ void small_head(const float* __restrict__ W, int K, const float* __restrict__ in, float* __restrict__ red) {
    const int tid = threadIdx.x, m = tid & 63, part = tid >> 6;
    const int kq = K / 4;
    float acc[NOUT];
#pragma unroll
    for (int o = 0; o < NOUT; ++o) acc[o] = 0.f;
    for (int k = part * kq; k < (part + 1) * kq; ++k) {
        const float a = in[act_idx(k, m)];
#pragma unroll
        for (int o = 0; o < NOUT; ++o) acc[o] = fmaf(__ldg(W + o * K + k), a, acc[o]);
    }
#pragma unroll
    for (int o = 0; o < NOUT; ++o) red[(o * 4 + part) * TM + m] = acc[o];
    __syncthreads();
}

template <bool EMBEDDED>
__global__ void __launch_bounds__(NTHREADS, 1) mlp_fp32_kernel(MlpArgs a) {
    extern __shared__ __align__(16) float sm[];
    float* H0 = sm;                      // [256][64]
    float* H1 = H0 + 256 * TM;           // [256][64]
    float* PE = H1 + 256 * TM;           // [64][64]   gamma_10(p), 63 rows used
    float* DIR = PE + 64 * TM;           // [32][64]   gamma_4(viewdir), 27 rows used
    float* WS = DIR + 32 * TM;           // 2 x [16][256]
    float* RED = WS + 2 * KC * 256;      // [16][64] head partials
    float* OUTB = RED + 16 * TM;         // [64][4]

    const int tid = threadIdx.x;
    const CondLayout cl{256, 128};
    const long long ntiles = (a.P + TM - 1) / TM;
    const int C = a.cond_dim;

    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        // ---- inputs: positional encodings of the tile's points --------------------------------
        {
            const int m = tid & 63, part = tid >> 6;
            long long p = tile * TM + m;
            const bool ok = p < a.P;
            if (!ok) p = a.P - 1;
            if constexpr (EMBEDDED) {
                const float* xr = a.x + p * 90;
                for (int k = part; k < 64; k += 4) PE[act_idx(k, m)] = (k < 63) ? xr[k] : 0.f;
                for (int k = part; k < 32; k += 4) DIR[act_idx(k, m)] = (k < 27) ? xr[63 + k] : 0.f;
            } else {
                const long long ray = p / a.s;
                const float* r = a.rays + ray * a.ray_stride;
                const float zz = a.z[p];
                float pos[3], vd[3];
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    pos[c] = __fadd_rn(r[c], __fmul_rn(r[3 + c], zz));     // o + d*z   (:332)
                    vd[c] = r[a.ray_stride - 3 + c];                       // rays[:, -3:]
                }
                if (part == 0) {
#pragma unroll
                    for (int c = 0; c < 3; ++c) { PE[act_idx(c, m)] = pos[c]; DIR[act_idx(c, m)] = vd[c]; }
                    PE[act_idx(63, m)] = 0.f;
                }
                if (part == 1)
                    for (int k = 27; k < 32; ++k) DIR[act_idx(k, m)] = 0.f;
                for (int f = part; f < 10; f += 4) {
                    const float sc = (float)(1 << f);
#pragma unroll
                    for (int c = 0; c < 3; ++c) {
                        float sn, cs;
                        sincosf(pos[c] * sc, &sn, &cs);
                        PE[act_idx(3 + 6 * f + c, m)] = sn;
                        PE[act_idx(6 + 6 * f + c, m)] = cs;
                    }
                }
                {
                    const int f = part;                                    // 4 view frequencies, 4 parts
                    const float sc = (float)(1 << f);
#pragma unroll
                    for (int c = 0; c < 3; ++c) {
                        float sn, cs;
                        sincosf(vd[c] * sc, &sn, &cs);
                        DIR[act_idx(3 + 6 * f + c, m)] = sn;
                        DIR[act_idx(6 + 6 * f + c, m)] = cs;
                    }
                }
            }
        }
        __syncthreads();
        float* sv = a.save ? a.save + (size_t)tile * TM * SAVE_W : nullptr;     // this tile's rows of the activation store
        if (sv) {                                      // inputs of the dW GEMMs: gamma(p) (64 cols, last = 0) and gamma(v) (32 cols)
            const int m = tid >> 2, kq = tid & 3;
            float* row = sv + (size_t)m * SAVE_W + SAVE_PE;
            for (int k = kq * 24; k < kq * 24 + 24; ++k) row[k] = (k < 64) ? PE[act_idx(k, m)] : DIR[act_idx(k - 64, m)];
        }

        // ---- trunk -----------------------------------------------------------------------------
        Seg sg[2];
        sg[0] = {PE, 63, 0};
        gemm_layer<256>(a.w[0], 63 + C, sg, 1, a.cond + cl.pts(0), H0, WS, sv);
        float* cur = H0;
        float* nxt = H1;
        for (int l = 1; l < 8; ++l) {
            if (l == 5) {
                sg[0] = {PE, 63, 0};
                sg[1] = {cur, 256, 63 + C};
                gemm_layer<256>(a.w[2 * l], 319 + C, sg, 2, a.cond + cl.pts(l), nxt, WS, sv ? sv + l * 256 : nullptr);
            } else {
                sg[0] = {cur, 256, 0};
                gemm_layer<256>(a.w[2 * l], 256, sg, 1, a.cond + cl.pts(l), nxt, WS, sv ? sv + l * 256 : nullptr);
            }
            float* t = cur; cur = nxt; nxt = t;
        }
        // cur = relu(pts_linears.7(...));  sigma = alpha_linear(cur)
        small_head<1>(a.w[P_ALPHA_W], 256, cur, RED);
        if (tid < TM) {
            float s = (RED[0 * TM + tid] + RED[1 * TM + tid]) + (RED[2 * TM + tid] + RED[3 * TM + tid]);
            OUTB[tid * 4 + 3] = s + a.cond[cl.alpha_b()];
        }
        // ---- view branch -----------------------------------------------------------------------
        sg[0] = {cur, 256, 0};
        sg[1] = {DIR, 27, 256};
        gemm_layer<128>(a.w[P_VIEWS_W], 283 + a.dim_expr, sg, 2, a.cond + cl.views(0), nxt, WS, sv ? sv + 2048 : nullptr);
        sg[0] = {nxt, 128, 0};
        gemm_layer<128>(a.w[P_VIEWS_W + 2], 128, sg, 1, a.cond + cl.views(1), cur, WS, sv ? sv + 2048 + 128 : nullptr);
        sg[0] = {cur, 128, 0};
        gemm_layer<128>(a.w[P_VIEWS_W + 4], 128, sg, 1, a.cond + cl.views(2), nxt, WS, sv ? sv + 2048 + 256 : nullptr);
        small_head<3>(a.w[P_RGB_W], 128, nxt, RED);
        if (tid < 3 * TM) {
            const int o = tid / TM, m = tid - o * TM;
            float s = (RED[(o * 4 + 0) * TM + m] + RED[(o * 4 + 1) * TM + m]) +
                      (RED[(o * 4 + 2) * TM + m] + RED[(o * 4 + 3) * TM + m]);
            OUTB[m * 4 + o] = s + a.cond[cl.rgb_b() + o];
        }
        __syncthreads();
        if (tid < TM) {
            const long long p = tile * TM + tid;
            if (p < a.P) reinterpret_cast<float4*>(a.out)[p] = *reinterpret_cast<const float4*>(OUTB + tid * 4);
        }
        __syncthreads();
    }
}

constexpr size_t FP32_SMEM = (size_t)(2 * 256 * TM + 64 * TM + 32 * TM + 2 * KC * 256 + 16 * TM + TM * 4) * sizeof(float);

// ---------------------------------------------------------------------------------------------
// conditioning fold
// ---------------------------------------------------------------------------------------------
__global__ void fold_cond_kernel(FoldArgs f) {
    __shared__ float c[1024];
    fold_cond_block(f, blockIdx.x, blockIdx.y, c);
}

}  // namespace

namespace inerf {

int mlp_fp32_launch(const MlpArgs& a, bool embedded, cudaStream_t st) {
    static thread_local int configured_dev = -1;
    int dev = 0;
    cudaGetDevice(&dev);
    if (configured_dev != dev) {
        cudaError_t e1 = cudaFuncSetAttribute(mlp_fp32_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FP32_SMEM);
        cudaError_t e2 = cudaFuncSetAttribute(mlp_fp32_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FP32_SMEM);
        if (e1 != cudaSuccess || e2 != cudaSuccess) {
            set_error("mlp_fp32: cudaFuncSetAttribute(%zu B smem): %s", FP32_SMEM, cudaGetErrorString(e1 != cudaSuccess ? e1 : e2));
            return (int)(e1 != cudaSuccess ? e1 : e2);
        }
        configured_dev = dev;
    }
    long long ntiles = (a.P + TM - 1) / TM;
    int grid = (int)(ntiles < (long long)num_sms() ? ntiles : (long long)num_sms());
    if (embedded) mlp_fp32_kernel<true><<<grid, NTHREADS, FP32_SMEM, st>>>(a);
    else mlp_fp32_kernel<false><<<grid, NTHREADS, FP32_SMEM, st>>>(a);
    return check_launch("inerf_mlp_fwd[fp32]");
}

int mlp_fold_cond_launch(const FoldArgs& f, cudaStream_t st) {
    fold_cond_kernel<<<dim3(12, 8), 256, 0, st>>>(f);
    return check_launch("inerf_mlp_fold_cond");
}

}  // namespace inerf

