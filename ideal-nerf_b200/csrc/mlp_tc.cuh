// What the tensor-core FaceNeRF kernels share (mlp_bf16.cu, mlp_f16x2.cu; the backward chain of mlp_bf16_bwd.cu uses the ring): the
// weight-stage ring, the forward layer geometry, the stage schedule that lays out the packed weight blob, and its pack kernel.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "mlp_common.cuh"
#include "sm100_ptx.cuh"

namespace inerf {

// The weight-stage ring in shared memory: NSTAGE stages of 16 KB (one 128-row x 64-column K-block).  The CTA-pair build splits every
// stage across the two CTAs of a cluster (each holds HALF of its rows), so the same ring is twice as deep.
template <bool PAIR, int NSTAGE> struct Ring { static constexpr int N = PAIR ? 2 * NSTAGE : NSTAGE, BYTES = PAIR ? 8192 : 16384; };

// ---- forward layer geometry (compile-time; build_tc_schedule lays out the packed blob in the same order) --------------------------
__host__ __device__ constexpr int lay_N(int l) { return l < 8 ? 256 : 128; }
__host__ __device__ constexpr int lay_act_kb(int l) { return l == 0 ? 0 : (l <= 8 ? 4 : 2); }     // activation K-blocks (64 wide)
__host__ __device__ constexpr bool lay_pe(int l) { return l == 0 || l == 5; }                     // + the gamma(p) K-block
__host__ __device__ constexpr bool lay_x(int l, bool emb) { return lay_pe(l) || (emb && l == 8); }   // + a PE-buffer K-block (gamma(p) or gamma(v))
__host__ __device__ constexpr int lay_prev_N(int l) { return l == 0 ? 128 : lay_N(l - 1); }       // L0 follows V2 of the previous iteration

// One weight stage as the producer streams it: the image at `offset` in the packed blob, n8 * 8 rows; `first`: the first stage of its
// (layer, half), whose bias tile is streamed with it.
struct TcStage {
    uint32_t offset;
    uint8_t n8, first, layer, half;
};
static_assert(sizeof(TcStage) == 8, "stage record");

// How pack_kernel fills one stage image: weight rows [n0, n0 + rows), columns wcol .. wcol + 63 (kmax valid, the rest zero);
// lo (fp16x2 blobs): the low fp16 half of the split instead of the high one.
struct TcPack {
    int w_index, ldw, n0, rows, wcol, kmax, lo;
    uint32_t offset;
};

constexpr int MAX_TC_STAGES = 160;     // 78 K-blocks at most (the embedded-row schedule), x 2 parts for fp16x2

struct TcSchedule {
    int n_stages;
    uint32_t total_bytes;
    TcStage st[MAX_TC_STAGES];
    TcPack pack[MAX_TC_STAGES];
};

// The stage order of both forward kernels: layer by layer, half by half, the activation K-blocks in order and the PE-buffer block last;
// with parts = 2 (fp16x2) each K-block is two stages, hi then lo.  emb: the embedded-row schedule -- V0 gains a last K-block per half,
// the view columns 256..282 of views_linears.0 (kmax = 27) against the gamma(v) image in the PE buffer; every other stage, and the order
// of all stages, is the fused-entry schedule's.
inline TcSchedule build_tc_schedule(const InerfNetDims* d, bool emb, int parts) {
    struct LayerDesc { int w_index, ldw, wcol_act; };
    const int C = d->dim_aud + d->dim_expr + d->dim_latent, E = d->dim_expr;
    LayerDesc L[11];
    L[0] = {0, 63 + C, 0};
    for (int l = 1; l < 8; ++l) L[l] = {2 * l, 256, 0};
    L[5] = {10, 319 + C, 63 + C};
    L[8] = {P_VIEWS_W, 283 + E, 0};
    L[9] = {P_VIEWS_W + 2, 128, 0};
    L[10] = {P_VIEWS_W + 4, 128, 0};
    TcSchedule S{};
    uint32_t off = 0;
    int n = 0;
    for (int l = 0; l < 11; ++l) {
        const int NH = lay_N(l) / 2, n_kb = lay_act_kb(l) + (lay_x(l, emb) ? 1 : 0);
        for (int h = 0; h < 2; ++h)
            for (int i = 0; i < n_kb; ++i)
                for (int part = 0; part < parts; ++part, ++n) {
                    const bool x = i == lay_act_kb(l);
                    S.st[n] = TcStage{off, (uint8_t)(NH / 8), (uint8_t)(i == 0 && part == 0), (uint8_t)l, (uint8_t)h};
                    S.pack[n] = TcPack{L[l].w_index, L[l].ldw, h * NH, NH, x ? (l == 8 ? 256 : 0) : L[l].wcol_act + i * 64,
                                       x ? (l == 8 ? 27 : 63) : 64, part, off};
                    off += (uint32_t)NH * 128u;
                }
    }
    S.n_stages = n;
    S.total_bytes = off;
    return S;
}

// ---- packing ------------------------------------------------------------------------------------------------------------------
// The table travels as a kernel parameter (by value): nothing is copied from pageable host memory, so the launch can be captured in a
// CUDA graph (train.TrainStep re-packs the weights after every optimiser step).  80 rows next to the 26 weight pointers fit the 4 KB
// parameter space; longer tables take several launches.
constexpr int PACK_PER_LAUNCH = 80;
struct TcPackArgs {
    const float* w[INERF_N_PARAMS];
    TcPack st[PACK_PER_LAUNCH];
    uint8_t* blob;
};
static_assert(sizeof(TcPackArgs) <= 4000, "kernel parameter space");

// F16: fp16 (hi, or the remainder v - hi for lo rows) instead of bf16; 128B-swizzled K-major images
template <bool F16>
__global__ void pack_kernel(const __grid_constant__ TcPackArgs pa) {
    const TcPack st = pa.st[blockIdx.x];
    const float* W = pa.w[st.w_index];
    for (int i = threadIdx.x; i < st.rows * 64; i += blockDim.x) {
        const int r = i >> 6, c = i & 63;
        const float v = (c < st.kmax) ? W[(size_t)(st.n0 + r) * st.ldw + st.wcol + c] : 0.f;
        uint8_t* dst = pa.blob + st.offset + sm100::sw128_offset(r, c);
        if constexpr (F16) {
            const __half hi = __float2half_rn(v);
            *reinterpret_cast<__half*>(dst) = st.lo ? __float2half_rn(v - __half2float(hi)) : hi;
        } else {
            *reinterpret_cast<__nv_bfloat16*>(dst) = __float2bfloat16_rn(v);
        }
    }
}

template <bool F16>
int pack_tc_schedule(const TcSchedule& S, const float* const* params_host, void* packed, cudaStream_t st, const char* what) {
    if ((uintptr_t)packed & 15) return fail(INERF_E_ALIGN, "inerf_mlp_pack: packed must be 16-byte aligned");
    for (int first = 0; first < S.n_stages; first += PACK_PER_LAUNCH) {
        TcPackArgs pa{};
        for (int i = 0; i < INERF_N_PARAMS; ++i) pa.w[i] = params_host[i];
        const int cnt = S.n_stages - first < PACK_PER_LAUNCH ? S.n_stages - first : PACK_PER_LAUNCH;
        for (int i = 0; i < cnt; ++i) pa.st[i] = S.pack[first + i];
        pa.blob = reinterpret_cast<uint8_t*>(packed);
        pack_kernel<F16><<<cnt, 256, 0, st>>>(pa);
        if (int rc = check_launch(what)) return rc;
    }
    return INERF_OK;
}

}  // namespace inerf
