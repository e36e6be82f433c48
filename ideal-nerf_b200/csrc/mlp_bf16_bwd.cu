// FaceNeRF backward, bf16 tensor-core mode, the chain:  delta_{l-1} = (delta_l . W_l[:, activation columns]) * [H_{l-1} > 0]
//
// Reference: torch.autograd of models/face_nerf.py:40-80 inside loss.backward() (NeRFs/HeadNeRF/train/audio_exp_nerf.py:549),
// restated on the folded network (SURVEY.md Appendix B).  No dX for layer 0 and for the gamma(p) / gamma(v) / conditioning columns
// (points are data, z_samples are detached in the reference).
//
// Same machine as the forward kernel (mlp_bf16.cu): one persistent CTA per SM, 256 points per iteration as two 128-row slots, the
// deltas live in shared memory in place of the activations (bf16, K-major, 128-byte swizzle), TRANSPOSED weights stream in through the
// bulk-copy ring in MMA issue order, fp32 accumulators in TMEM, two output halves per layer so an epilogue overlaps the other half.
// Ten GEMM layers, back to front:
//   j0: d_v2 (128) -> v1 (128)     j1: d_v1 -> v0 (128)     j2: d_v0 (128) -> h7 (256), + d_sigma (x) alpha_linear.weight as a rank-1 MMA
//   j3..j9: d_h7 -> h6 -> ... -> h0 (256 -> 256; j5 uses the h4 columns of the skip layer pts_linears.5)
// The epilogue multiplies by the ReLU mask the forward stored (one bit per activation), rounds to bf16, writes the delta back to shared
// memory for the next GEMM and to HBM as a 16 KB image per 64 features for the dW kernel (mlp_bf16_dw.cu).  Four "init" warps turn
// d_raw into d_v2 = (d_rgb . rgb_linear.weight) * mask, the d_sigma operand tile and the d_raw image of the next iteration.
#include <cuda_bf16.h>
#include <stdlib.h>

#include "mlp_tc.cuh"

using namespace inerf;
using namespace sm100;

namespace {

constexpr int NSTAGE = 4;
constexpr int STAGE_BYTES = 16384;
// CTA-pair build (PAIR = true, see mlp_bf16.cu): each CTA of a cluster of two holds HALF of the rows of every weight stage; the same 64 KB
// ring is eight stages deep
template <bool PAIR> using RingOf = Ring<PAIR, NSTAGE>;
constexpr int NTH = 512;
constexpr int N_EPI = 256, N_INIT = 128;
constexpr int NLAY = 10;

__host__ __device__ constexpr int bl_N(int j) { return j < 2 ? 128 : 256; }              // output width (activation the delta belongs to)
__host__ __device__ constexpr int bl_kb(int j) { return j < 3 ? 2 : 4; }                 // input delta width / 64
__host__ __device__ constexpr int bl_prev_N(int j) { return j == 0 ? 128 : bl_N(j - 1); }
__host__ __device__ constexpr int bl_out_layer(int j) { return 9 - j; }                  // forward layer whose pre-activation gradient layer j produces
__host__ __device__ constexpr int bl_w_layer(int j) { return 10 - j; }                   // forward layer whose weight it multiplies by

constexpr int OFF_ACT = 0;                                   // [2][4][16384]
constexpr int OFF_W = 131072;                                // [NSTAGE][16384]
constexpr int OFF_DS = OFF_W + NSTAGE * STAGE_BYTES;         // [2][4096]  d_sigma tiles (A of the rank-1 MMA), no-swizzle [128][16]
constexpr int OFF_AWT = OFF_DS + 2 * 4096;                   // [2][4096]  alpha_linear.weight tiles (B of the rank-1 MMA), one per output half
constexpr int OFF_RW = OFF_AWT + 2 * 4096;                   // rgb_linear.weight 3 x 128 floats
constexpr int OFF_BAR = OFF_RW + 1536;
constexpr int SMEM_BWD = OFF_BAR + 256;
static_assert(SMEM_BWD <= 232448, "shared memory budget");

struct Bars {
    uint64_t wfull[8], wempty[8];
    uint64_t pfull[8];       // pair build, leader only: the PEER's half of the stage has landed (relayed by the peer's warp 1)
    uint64_t cbar[3];        // C0, C1, C2 (pair build: multicast to both CTAs)
    uint64_t ebar[2];        // E0, E1 (8 epilogue warps; pair build: the leader's, 8 + 8 warps)
    uint64_t init_ready;     // 4 init warps, once per iteration (pair build: the leader's, 4 + 4 warps)
    uint64_t init_free;      // commit after the last MMA of the iteration
    uint32_t tmem_base;
};
static_assert(sizeof(Bars) <= 256, "barrier block");

struct BwdChainArgs {
    const void* packed_t;          // transposed weight stages + the two alpha tiles (inerf_mlp_pack, INERF_MLP_BF16_BWD)
    const float* rgb_w;            // rgb_linear.weight (3,128)
    const uint32_t* mask;          // [n_tiles][TRAIN_MASK_WORDS][128]
    const float* d_raw;            // [P][4]
    uint8_t* delta_img;            // [n_tiles][TRAIN_IMGS][16384]
    long long P;
    uint32_t n_stage_bytes_total;  // offset of the alpha tiles inside packed_t
};

struct BStep { uint8_t n8, first, layer, half; uint32_t offset; };
constexpr int MAX_BSTEPS = 96;
__constant__ BStep c_bsteps[MAX_BSTEPS];

__device__ __forceinline__ void bwait(uint64_t* bar, uint32_t parity) {
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity))
        if (clock64() - t0 > 8000000000LL) __trap();          // ~4 s: a lost arrival must not hang the GPU
}

// issuer-side wait on an event whose arrivals may come from the peer CTA; the single-CTA build waits with the bounded bwait
template <bool PAIR>
__device__ __forceinline__ void wait_ev_bounded(uint64_t* bar, uint32_t parity) {
    if constexpr (PAIR) mbar_wait_cluster(bar, parity);
    else bwait(bar, parity);
}

struct IssueCtx {
    Bars* bars;
    uint32_t a_lo, w_lo, hi, tmem_base, ds_lo, awt_lo;
    uint32_t stage, wpar, layer_ctr, iter_ctr;
};

template <int J, bool PAIR>
__device__ __forceinline__ void issue_layer(IssueCtx& c) {
    constexpr int NSTAGE = RingOf<PAIR>::N, STAGE_BYTES = RingOf<PAIR>::BYTES;
    constexpr int N = bl_N(J), NH = N / 2, NKB = bl_kb(J);
    constexpr int KB_PER_HALF_PREV = bl_prev_N(J) / 128;
    constexpr int N_OUT_H0 = NH / 64;
    constexpr int N_FIRST = NKB < N_OUT_H0 ? NKB : N_OUT_H0;
    constexpr uint32_t IDESC = umma_idesc_bf16(PAIR ? 256 : 128, NH);
    Bars* bars = c.bars;
    const uint32_t par_prev = (c.layer_ctr - 1) & 1;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
#pragma unroll
        for (int i = 0; i < NKB; ++i) {
            if (h == 0 && c.layer_ctr > 0) {
                if (J == 0 || bl_N(J) > bl_prev_N(J)) {        // new iteration, or a layer WIDER than the previous one: its first half
                    // overwrites accumulator columns that both halves of the previous epilogue read
                    if (i == 0) { wait_ev_bounded<PAIR>(&bars->ebar[0], par_prev); wait_ev_bounded<PAIR>(&bars->ebar[1], par_prev); }
                } else {
                    if (i == 0) wait_ev_bounded<PAIR>(&bars->ebar[0], par_prev);
                    if (i == KB_PER_HALF_PREV) wait_ev_bounded<PAIR>(&bars->ebar[1], par_prev);
                }
            }
            if (J == 0 && h == 0 && i == 0) wait_ev_bounded<PAIR>(&bars->init_ready, c.iter_ctr & 1);
            bwait(&bars->wfull[c.stage], c.wpar);
            if constexpr (PAIR) mbar_wait_cluster(&bars->pfull[c.stage], c.wpar);
            tc_fence_after();
            if (elect_one()) {
                if (J == 2 && i == 0) {
                    // d h7 += d_sigma (x) alpha_linear.weight: A row = (s_hi, s_hi, s_lo, s_lo, 0...), B row = (w_hi, w_lo, w_hi, w_lo, 0...)
#pragma unroll
                    for (int slot = 0; slot < 2; ++slot)
                        umma_any<PAIR>(c.tmem_base + slot * 256 + h * NH, c.ds_lo + slot * (4096 >> 4), c.awt_lo + h * (4096 >> 4), HI_NOSWZ, IDESC, 0u);
                }
                const uint32_t b_lo = c.w_lo + c.stage * (STAGE_BYTES >> 4);
#pragma unroll
                for (int slot = 0; slot < 2; ++slot) {
                    const uint32_t a_lo = c.a_lo + slot * (65536 >> 4) + i * (16384 >> 4);
                    const uint32_t d = c.tmem_base + slot * 256 + h * NH;
#pragma unroll
                    for (int k = 0; k < 4; ++k) umma_any<PAIR>(d, a_lo + 2 * k, b_lo + 2 * k, c.hi, IDESC, (J != 2 && i == 0 && k == 0) ? 0u : 1u);
                }
                commit_any<PAIR>(&bars->wempty[c.stage]);
                const bool last = (i == NKB - 1);
                if (h == 0 && last) commit_any<PAIR>(&bars->cbar[0]);
                if (h == 1 && i == N_FIRST - 1) commit_any<PAIR>(&bars->cbar[1]);
                if (h == 1 && last) commit_any<PAIR>(&bars->cbar[2]);
                if (h == 1 && last && J == NLAY - 1) commit_any<PAIR>(&bars->init_free);
            }
            __syncwarp();
            if (++c.stage == NSTAGE) { c.stage = 0; c.wpar ^= 1; }
        }
    }
    ++c.layer_ctr;
}

// PAIR = true: clusters of two CTAs, one tcgen05.mma.cta_group::2 over the 2 x 128 rows of the pair, the (transposed) weight stages split
// across the pair; a pair iteration is two 256-point chunks, CTA r takes chunk 2 it + r (the forward kernel's pair build, mlp_bf16.cu).
template <bool PAIR>
__global__ void __launch_bounds__(NTH, 1) mlp_bf16_bwd_chain_kernel(BwdChainArgs a, int n_steps) {
    constexpr int NSTAGE = RingOf<PAIR>::N, STAGE_BYTES = RingOf<PAIR>::BYTES;
    extern __shared__ __align__(1024) uint8_t sm[];
    if ((smem_u32(sm) & 1023u) != 0) __trap();
    Bars* bars = reinterpret_cast<Bars*>(sm + OFF_BAR);
    float* s_rw = reinterpret_cast<float*>(sm + OFF_RW);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t rank = PAIR ? cluster_ctarank() : 0u;
    const long long n_iter = PAIR ? (a.P + 511) / 512 : (a.P + 255) / 256;
    const long long it_first = PAIR ? (long long)(blockIdx.x >> 1) : (long long)blockIdx.x;
    const long long it_step = PAIR ? (long long)(gridDim.x >> 1) : (long long)gridDim.x;
#define CHUNK_OF(it_) (PAIR ? 2 * (it_) + (long long)rank : (it_))

    for (int i = tid; i < 384; i += NTH) s_rw[i] = a.rgb_w[i];
    {   // the alpha tiles are constants of the call: straight copy of their packed image (pair build: this CTA's half of the rows of each
        // tile, placed at the tile's base, as the B operand of a cta_group::2 MMA is split)
        const uint8_t* src = reinterpret_cast<const uint8_t*>(a.packed_t) + a.n_stage_bytes_total;
        constexpr int HALF = PAIR ? 2048 : 4096;
        for (int i = tid; i < 2 * HALF / 16; i += NTH) {
            const int tile = i / (HALF / 16), o = i - tile * (HALF / 16);
            reinterpret_cast<uint4*>(sm + OFF_AWT + tile * 4096)[o] = reinterpret_cast<const uint4*>(src + tile * 4096 + rank * HALF)[o];
        }
    }
    fence_proxy_async_smem();
    if (tid == 0) {
        for (int s = 0; s < NSTAGE; ++s) { mbar_init(&bars->wfull[s], 1); mbar_init(&bars->wempty[s], 1); mbar_init(&bars->pfull[s], 1); }
        for (int j = 0; j < 3; ++j) mbar_init(&bars->cbar[j], 1);
        for (int j = 0; j < 2; ++j) mbar_init(&bars->ebar[j], PAIR ? 2 * (N_EPI / 32) : N_EPI / 32);
        mbar_init(&bars->init_ready, PAIR ? 2 * (N_INIT / 32) : N_INIT / 32);
        mbar_init(&bars->init_free, 1);
        fence_mbar_init();
    }
    if (warp == 2) {
        if constexpr (PAIR) { tmem_alloc_pair(&bars->tmem_base, 512); }
        else { tmem_alloc(&bars->tmem_base, 512); tmem_relinquish(); }
    }
    tc_fence_before();
    __syncthreads();
    if constexpr (PAIR) cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = bars->tmem_base;

    if (warp == 0) {
        // ================= weight producer ===========================================================================
        if (lane == 0) {
            const uint8_t* blob = reinterpret_cast<const uint8_t*>(a.packed_t);
            uint32_t g = 0;
            constexpr uint32_t SPLIT = PAIR ? 2u : 1u;      // pair build: this CTA's half of the rows of every stage
            for (long long it = it_first; it < n_iter; it += it_step)
                for (int s = 0; s < n_steps; ++s, ++g) {
                    const uint32_t stage = g % NSTAGE, round = g / NSTAGE;
                    bwait(&bars->wempty[stage], (round & 1) ^ 1);
                    const uint32_t bytes = (uint32_t)c_bsteps[s].n8 * 8u * 128u / SPLIT;
                    mbar_arrive_expect_tx(&bars->wfull[stage], bytes);
                    bulk_g2s(sm + OFF_W + stage * STAGE_BYTES, blob + c_bsteps[s].offset + rank * bytes, bytes, &bars->wfull[stage]);
                }
        }
    } else if (warp == 1 && PAIR && rank != 0) {
        // ================= relay (peer CTA of a pair): tell the leader when MY half of a weight stage has landed ======================
        if (lane == 0) {
            uint32_t g = 0;
            for (long long it = it_first; it < n_iter; it += it_step)
                for (int s = 0; s < n_steps; ++s, ++g) {
                    bwait(&bars->wfull[g % NSTAGE], (g / NSTAGE) & 1);
                    mbar_arrive_remote(&bars->pfull[g % NSTAGE], 0);
                }
        }
    } else if (warp == 1) {
        // ================= MMA issuer ===================================================================================
        IssueCtx c;
        c.bars = bars;
        c.hi = (uint32_t)(umma_desc_sw128(0) >> 32);
        c.a_lo = (uint32_t)umma_desc_sw128(smem_u32(sm + OFF_ACT));
        c.w_lo = (uint32_t)umma_desc_sw128(smem_u32(sm + OFF_W));
        c.ds_lo = desc_lo_noswz(smem_u32(sm + OFF_DS));
        c.awt_lo = desc_lo_noswz(smem_u32(sm + OFF_AWT));
        c.tmem_base = tmem_base;
        c.stage = 0; c.wpar = 0; c.layer_ctr = 0; c.iter_ctr = 0;
        for (long long it = it_first; it < n_iter; it += it_step, ++c.iter_ctr) {
            // layers 3..8 have the same geometry (256 x 256 after a 256-wide layer): one copy of the issue code, run six times,
            // keeps the kernel's SASS inside the instruction cache (see the forward kernel)
            issue_layer<0, PAIR>(c); issue_layer<1, PAIR>(c); issue_layer<2, PAIR>(c);
#pragma unroll 1
            for (int r = 0; r < 6; ++r) issue_layer<3, PAIR>(c);
            issue_layer<9, PAIR>(c);
        }
    } else if (warp >= 4 && warp < 12) {
        // ================= epilogue: one row per thread ==================================================================
        const int slot = (warp - 4) >> 2;
        const int row = ((warp & 3) << 5) + lane;
        const uint32_t t_lane = tmem_base + ((uint32_t)((warp & 3) << 5) << 16) + slot * 256;
        uint8_t* act = sm + OFF_ACT + slot * 65536;
        const uint32_t row_off = (row >> 3) * 1024 + (row & 7) * 128;
        const uint32_t rsw = row & 7;
        uint32_t layer_ctr = 0;
        for (long long it = it_first; it < n_iter; it += it_step) {
            // pair build: the peer's last chunk may lie wholly past the end -- it reads tile 0's masks and writes nothing
            const bool chunk_ok = !PAIR || CHUNK_OF(it) * 256 < a.P;
            const size_t T = chunk_ok ? (size_t)CHUNK_OF(it) * 2 + slot : 0;
            for (int j = 0; j < NLAY; ++j, ++layer_ctr) {
                const int N = j < 2 ? 128 : 256, NH = N >> 1, lo = 9 - j;      // lo: forward layer this delta belongs to
                const uint32_t par = layer_ctr & 1;
                // ReLU masks of this row for the whole layer (8 or 4 words), loaded before the accumulators are ready
                uint32_t mw[8];
                const uint32_t* mp = a.mask + (T * TRAIN_MASK_WORDS + train_mask_of(lo)) * 128 + row;
#pragma unroll
                for (int w = 0; w < 8; ++w) mw[w] = (w < (N >> 5)) ? __ldg(mp + w * 128) : 0u;
                uint8_t* gimg_base = a.delta_img + (T * TRAIN_IMGS + train_img_of(lo)) * 16384;
#pragma unroll 1
                for (int h = 0; h < 2; ++h) {
                    bwait(&bars->cbar[h == 0 ? 0 : 2], par);
                    __syncwarp();
                    tc_fence_after();
                    uint32_t packed[64];
                    const int nchunk = NH >> 5;
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        if (c < nchunk) {
                            uint32_t r[32];
                            tmem_ld32(t_lane + h * NH + c * 32, r);
                            tmem_wait_ld();
                            const uint32_t m = (h == 0) ? mw[c] : (NH == 128 ? mw[4 + c] : mw[2 + c]);      // word f0 / 32
#pragma unroll
                            for (int q = 0; q < 16; ++q) {
                                const float v0 = (m & (0x80000000u >> (2 * q))) ? __uint_as_float(r[2 * q]) : 0.f;
                                const float v1 = (m & (0x80000000u >> (2 * q + 1))) ? __uint_as_float(r[2 * q + 1]) : 0.f;
                                packed[c * 16 + q] = pack_bf16x2(v0, v1);
                            }
                        }
                    }
                    tc_fence_before();
                    if (j == NLAY - 1 && !chunk_ok) {
                        // nothing to store
                    } else if (j == NLAY - 1) {
                        // d_h0 feeds no further GEMM: straight to HBM (the init warps of the next iteration may already be refilling the
                        // shared-memory K-blocks, so they are not used as a staging buffer here)
#pragma unroll
                        for (int c = 0; c < 4; ++c) {
                            const int f0 = h * NH + c * 32, ch0 = (f0 & 63) >> 3;
                            uint8_t* gk = gimg_base + (f0 >> 6) * 16384 + row_off;
#pragma unroll
                            for (int q = 0; q < 4; ++q)
                                *reinterpret_cast<uint4*>(gk + (((ch0 + q) ^ rsw) << 4)) =
                                    make_uint4(packed[c * 16 + q * 4], packed[c * 16 + q * 4 + 1], packed[c * 16 + q * 4 + 2], packed[c * 16 + q * 4 + 3]);
                        }
                    } else {
                        if (h == 0) bwait(&bars->cbar[1], par);
                        // the delta image for dW: each warp bulk-copies its own 32 rows of the K-blocks it writes (4 KB per K-block image), so no
                        // barrier couples the warps.  Before overwriting them lane 0 waits until the copy that last read these rows has left
                        // shared memory: two copies back (same half of the previous layer), or the latest where the layer widens (j == 2).
                        if (lane == 0) { if (h == 0 && j == 2) bulk_wait_read_all(); else bulk_wait_read_but_one(); }
                        __syncwarp();
#pragma unroll
                        for (int c = 0; c < 4; ++c) {
                            if (c < nchunk) {
                                const int f0 = h * NH + c * 32;
                                uint8_t* kb = act + (f0 >> 6) * 16384 + row_off;
                                const int ch0 = (f0 & 63) >> 3;
#pragma unroll
                                for (int q = 0; q < 4; ++q)
                                    *reinterpret_cast<uint4*>(kb + (((ch0 + q) ^ rsw) << 4)) =
                                        make_uint4(packed[c * 16 + q * 4], packed[c * 16 + q * 4 + 1], packed[c * 16 + q * 4 + 2], packed[c * 16 + q * 4 + 3]);
                            }
                        }
                        fence_proxy_async_smem();
                        __syncwarp();
                        if (lane == 0) {
                            const int kb0 = (h * NH) >> 6, nkb = NH >> 6;
                            const uint32_t wrow = (uint32_t)(warp & 3) * 4096u;
                            if (chunk_ok)
                                for (int k = 0; k < nkb; ++k) bulk_s2g(gimg_base + (kb0 + k) * 16384 + wrow, act + (kb0 + k) * 16384 + wrow, 4096u);
                            bulk_commit();
                            // last copy of the iteration: the init warps refill K-blocks 0,1 once the final layer's MMAs are done, so the copy
                            // of those K-blocks (the previous half's) must have left shared memory before this half releases that layer
                            if (j == NLAY - 2 && h == 1) bulk_wait_read_but_one();
                        }
                    }
                    __syncwarp();
                    if (lane == 0) { if constexpr (PAIR) mbar_arrive_remote(&bars->ebar[h], 0); else mbar_arrive(&bars->ebar[h]); }
                }
            }
        }
        if (lane == 0) bulk_wait_all();
    } else if (warp >= 12) {
        // ================= init: d_raw -> d_v2, d_sigma tile, d_raw image ==================================================
        // Phase 1 (any time): d_v2 and the d_raw image of row t of both slots go to HBM (the dW kernel needs them there anyway).
        // Phase 2 (after the last MMA of the previous iteration has read the shared-memory deltas): the thread reads its own two
        // 256-byte rows back (L2 hits) into the A-operand K-blocks 0,1 -- holding them in registers across the wait would need 128.
        const int t = tid - 12 * 32;             // row of both slots
        const uint32_t trow = (t >> 3) * 1024 + (t & 7) * 128, tsw = t & 7;
        uint32_t iter_ctr = 0;
        for (long long it = it_first; it < n_iter; it += it_step, ++iter_ctr) {
            const long long chunk = CHUNK_OF(it);
            const bool chunk_ok = !PAIR || chunk * 256 < a.P;      // a chunk wholly past the end: zero deltas, tile 0's masks, no stores
            float dsig[2];
#pragma unroll 1
            for (int sl = 0; sl < 2; ++sl) {
                const long long p = chunk * 256 + sl * 128 + t;
                const size_t T = chunk_ok ? (size_t)chunk * 2 + sl : 0;
                const float4 dr = (p < a.P) ? reinterpret_cast<const float4*>(a.d_raw)[p] : make_float4(0.f, 0.f, 0.f, 0.f);
                dsig[sl] = dr.w;
                const uint32_t* mp = a.mask + (T * TRAIN_MASK_WORDS + train_mask_of(10)) * 128 + t;
                uint8_t* g2 = a.delta_img + (T * TRAIN_IMGS + train_img_of(10)) * 16384 + trow;
#pragma unroll
                for (int w = 0; w < 4; ++w) {                  // 32 features per mask word = 4 x 16-byte chunks
                    const uint32_t m = __ldg(mp + w * 128);
                    uint32_t pk[16];
#pragma unroll
                    for (int q = 0; q < 16; ++q) {
                        const int n = w * 32 + 2 * q;
                        float v0 = fmaf(dr.x, s_rw[n], fmaf(dr.y, s_rw[128 + n], dr.z * s_rw[256 + n]));
                        float v1 = fmaf(dr.x, s_rw[n + 1], fmaf(dr.y, s_rw[128 + n + 1], dr.z * s_rw[256 + n + 1]));
                        if (!(m & (0x80000000u >> (2 * q)))) v0 = 0.f;
                        if (!(m & (0x80000000u >> (2 * q + 1)))) v1 = 0.f;
                        pk[q] = pack_bf16x2(v0, v1);
                    }
                    uint8_t* gk = g2 + (w >> 1) * 16384;
                    const int ch0 = (w & 1) * 4;
#pragma unroll
                    for (int q = 0; q < 4; ++q)
                        if (chunk_ok) *reinterpret_cast<uint4*>(gk + (((ch0 + q) ^ tsw) << 4)) = make_uint4(pk[4 * q], pk[4 * q + 1], pk[4 * q + 2], pk[4 * q + 3]);
                }
                uint8_t* go = a.delta_img + (T * TRAIN_IMGS + TRAIN_IMG_DOUT) * 16384 + trow;      // columns 0..3 = d_rgb, d_sigma; zero elsewhere
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    uint4 v = make_uint4(0u, 0u, 0u, 0u);
                    if (q == 0) { v.x = pack_bf16x2(dr.x, dr.y); v.y = pack_bf16x2(dr.z, dr.w); }
                    if (chunk_ok) *reinterpret_cast<uint4*>(go + ((q ^ tsw) << 4)) = v;
                }
            }
            if (iter_ctr > 0) bwait(&bars->init_free, (iter_ctr - 1) & 1);
#pragma unroll 1
            for (int sl = 0; sl < 2; ++sl) {
                const size_t T = chunk_ok ? (size_t)chunk * 2 + sl : 0;
                const uint8_t* g2 = a.delta_img + (T * TRAIN_IMGS + train_img_of(10)) * 16384 + trow;
                uint8_t* dst = sm + OFF_ACT + sl * 65536 + trow;
                uint4 v[16];
#pragma unroll
                for (int q = 0; q < 16; ++q)
                    v[q] = chunk_ok ? *reinterpret_cast<const uint4*>(g2 + (q >> 3) * 16384 + ((q & 7) << 4)) : make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
                for (int q = 0; q < 16; ++q) *reinterpret_cast<uint4*>(dst + (q >> 3) * 16384 + ((q & 7) << 4)) = v[q];
                // d_sigma tile row: (hi, hi, lo, lo, 0, 0, 0, 0 | 0 x 8)
                const __nv_bfloat16 hi = __float2bfloat16_rn(dsig[sl]);
                const __nv_bfloat16 lo = __float2bfloat16_rn(dsig[sl] - __bfloat162float(hi));
                const uint32_t hh = (uint32_t)__bfloat16_as_ushort(hi) * 0x10001u, ll = (uint32_t)__bfloat16_as_ushort(lo) * 0x10001u;
                uint8_t* ds = sm + OFF_DS + sl * 4096 + (t >> 3) * 256 + (t & 7) * 16;
                *reinterpret_cast<uint4*>(ds) = make_uint4(hh, ll, 0u, 0u);
                *reinterpret_cast<uint4*>(ds + 128) = make_uint4(0u, 0u, 0u, 0u);
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) { if constexpr (PAIR) mbar_arrive_remote(&bars->init_ready, 0); else mbar_arrive(&bars->init_ready); }
        }
    }

    tc_fence_before();
    __syncthreads();
    if constexpr (PAIR) {
        cluster_sync_all();      // nobody leaves while the peer may still arrive on / multicast to this CTA
        if (warp == 2) tmem_dealloc_pair(tmem_base, 512);
    } else {
        if (warp == 2) tmem_dealloc(tmem_base, 512);
    }
#undef CHUNK_OF
}

// ---------------------------------------------------------------------------------------------
// schedule + transposed weight packing (host)
// ---------------------------------------------------------------------------------------------
struct BPack { int w_index, ldw, k0, n0, rows; uint32_t offset; };      // image[r][c] = W[(k0 + c) * ldw + n0 + r], rows x 64

struct BSchedule {
    int n_steps;
    BStep steps[MAX_BSTEPS];
    BPack pack[MAX_BSTEPS];
    uint32_t stage_bytes;      // the two alpha tiles follow
};

BSchedule build_bschedule(const InerfNetDims* d) {
    const int C = d->dim_aud + d->dim_expr + d->dim_latent, E = d->dim_expr;
    BSchedule S{};
    uint32_t off = 0;
    int n = 0;
    for (int j = 0; j < NLAY; ++j) {
        const int l = bl_w_layer(j), N = bl_N(j), NH = N / 2, NKB = bl_kb(j);
        const int w_index = l < 8 ? 2 * l : P_VIEWS_W + 2 * (l - 8);
        const int ldw = l == 5 ? 319 + C : (l == 8 ? 283 + E : (l < 8 ? 256 : 128));
        const int ncol0 = l == 5 ? 63 + C : 0;
        for (int h = 0; h < 2; ++h)
            for (int kb = 0; kb < NKB; ++kb) {
                S.steps[n] = BStep{(uint8_t)(NH / 8), (uint8_t)(kb == 0), (uint8_t)j, (uint8_t)h, off};
                S.pack[n] = BPack{w_index, ldw, kb * 64, ncol0 + h * NH, NH, off};
                off += (uint32_t)NH * 128u;
                ++n;
            }
    }
    S.n_steps = n;
    S.stage_bytes = off;
    return S;
}

struct BPackArgs {
    const float* w[INERF_N_PARAMS];
    BPack st[MAX_BSTEPS];
    uint8_t* blob;
    uint32_t alpha_off;
    int n_steps;
};

static_assert(sizeof(BPackArgs) <= 4000, "kernel parameter space");
__global__ void bwd_pack_kernel(const __grid_constant__ BPackArgs pa) {      // argument table by value: graph-capturable, no host copy
    if ((int)blockIdx.x < pa.n_steps) {
        const BPack st = pa.st[blockIdx.x];
        const float* W = pa.w[st.w_index];
        for (int i = threadIdx.x; i < st.rows * 64; i += blockDim.x) {
            const int c = i / st.rows, r = i - c * st.rows;          // consecutive threads walk a weight row: coalesced reads
            const float v = W[(size_t)(st.k0 + c) * st.ldw + st.n0 + r];
            *reinterpret_cast<__nv_bfloat16*>(pa.blob + st.offset + sw128_offset(r, c)) = __float2bfloat16_rn(v);
        }
    } else {
        // alpha tiles: [half][128 rows][16 cols] no-swizzle, row n = (w_hi, w_lo, w_hi, w_lo, 0 ...)
        const float* aw = pa.w[P_ALPHA_W];
        for (int n = threadIdx.x; n < 256; n += blockDim.x) {
            const int h = n >> 7, r = n & 127;
            const __nv_bfloat16 hi = __float2bfloat16_rn(aw[n]);
            const __nv_bfloat16 lo = __float2bfloat16_rn(aw[n] - __bfloat162float(hi));
            const uint32_t w = (uint32_t)__bfloat16_as_ushort(hi) | ((uint32_t)__bfloat16_as_ushort(lo) << 16);
            uint8_t* p = pa.blob + pa.alpha_off + h * 4096 + (r >> 3) * 256 + (r & 7) * 16;
            *reinterpret_cast<uint4*>(p) = make_uint4(w, w, 0u, 0u);
            *reinterpret_cast<uint4*>(p + 128) = make_uint4(0u, 0u, 0u, 0u);
        }
    }
}

}  // namespace

namespace inerf {

int mlp_bf16_bwd_packed_bytes(const InerfNetDims* d, size_t* bytes) {
    BSchedule S = build_bschedule(d);
    *bytes = (size_t)S.stage_bytes + 2 * 4096;
    return INERF_OK;
}

int mlp_bf16_bwd_pack(const InerfNetDims* d, const float* const* params_host, void* packed, cudaStream_t st) {
    if ((uintptr_t)packed & 15) return fail(INERF_E_ALIGN, "inerf_mlp_pack: packed must be 16-byte aligned");
    BSchedule S = build_bschedule(d);
    BPackArgs pa{};
    for (int i = 0; i < INERF_N_PARAMS; ++i) pa.w[i] = params_host[i];
    for (int i = 0; i < S.n_steps; ++i) pa.st[i] = S.pack[i];
    pa.blob = reinterpret_cast<uint8_t*>(packed);
    pa.alpha_off = S.stage_bytes;
    pa.n_steps = S.n_steps;
    bwd_pack_kernel<<<S.n_steps + 1, 256, 0, st>>>(pa);
    return check_launch("inerf_mlp_pack[bf16 bwd]");
}

int mlp_bf16_bwd_chain_launch(const InerfNetDims* dims, const float* const* params_host, const void* packed_t, const uint32_t* mask,
                              const float* d_raw, uint8_t* delta_img, long long P, cudaStream_t st) {
    static thread_local int configured_dev = -1;
    // step sizes / offsets do not depend on the conditioning dims; a function-local static is initialised once, thread-safely
    static const BSchedule S = [] { InerfNetDims d{64, 76, 32, 256, 8, 63, 27}; return build_bschedule(&d); }();
    int rc = setup_once(configured_dev, {(const void*)mlp_bf16_bwd_chain_kernel<false>, (const void*)mlp_bf16_bwd_chain_kernel<true>}, SMEM_BWD,
                        "mlp_bf16_bwd", [] { return cudaMemcpyToSymbol(c_bsteps, S.steps, sizeof(BStep) * MAX_BSTEPS); });
    if (rc) return rc;
    BwdChainArgs a{};
    a.packed_t = packed_t; a.rgb_w = params_host[P_RGB_W]; a.mask = mask; a.d_raw = d_raw; a.delta_img = delta_img; a.P = P;
    a.n_stage_bytes_total = S.stage_bytes;
    const long long n_iter = (P + 255) / 256;
    return mlp_pair_enabled() ? launch_tc(mlp_bf16_bwd_chain_kernel<true>, true, n_iter, NTH, SMEM_BWD, st, "inerf_mlp_bwd[bf16 chain pair]", a, S.n_steps)
                              : launch_tc(mlp_bf16_bwd_chain_kernel<false>, false, n_iter, NTH, SMEM_BWD, st, "inerf_mlp_bwd[bf16 chain]", a, S.n_steps);
}

}  // namespace inerf
