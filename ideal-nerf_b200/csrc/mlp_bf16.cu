// FaceNeRF MLP, bf16 mode: the fused tensor-core kernel (tcgen05.mma, accumulators in TMEM, weights
// streamed by the TMA engine, activations resident in shared memory from the positional encoding
// to the (r,g,b,sigma) output).
//
// Reference: models/face_nerf.py:40-80, NeRFs/HeadNeRF/train/audio_exp_nerf.py:332,376-394,
// NeRFs/HeadNeRF/helper.py:174-204.  Folded per-point network (SURVEY.md Appendix B):
//   L0 63->256, L1-4 256->256, L5 (63+256)->256, L6-7 256->256, alpha 256->1,
//   V0 (256 [+27 view cols])->128, V1-2 128->128, rgb 128->3.
//
// Shipped form: clusters of TWO CTAs (template parameter PAIR, tcgen05 cta_group::2): one M = 256 MMA over both CTAs' rows, the weight
// stages split across the pair -- see the comment above the kernel.  The decomposition below is per CTA and is the same in both forms.
//
// Work decomposition (one persistent CTA per SM, 512 threads):
//   * a CTA iteration owns 256 consecutive points = two 128-row "slots" that advance in lock step,
//     so every streamed weight byte feeds 256 rows (halves the L2->SM weight traffic of a 128-row tile);
//   * every layer is issued as two output halves h0,h1 (N/2 columns each, M=128, K=16 per
//     tcgen05.mma).  The epilogue of half h0 (TMEM -> +bias -> ReLU -> bf16 -> swizzled smem) runs
//     while the tensor pipe computes h1, and the epilogue of h1 overlaps the first K-blocks of the
//     next layer, so the pipe never waits for an epilogue.  Activations are updated IN PLACE:
//     h1 reads the K-blocks that epi(h0) will overwrite first and commits (C1) before they are
//     written; commit C0 = "h0 accumulators complete", C2 = "layer complete";
//   * roles: warp 0 = weight producer (cp.async.bulk, 16 KB stages, mbarrier ring), warp 1 = MMA
//     issuer (one thread), warp 2 = TMEM allocator, warps 4-11 = epilogue (one row per thread, 4 warps
//     per slot), warps 12-15 = positional-encoding producers for the NEXT iteration (2 rows/thread);
//   * gamma(viewdir) is constant per ray, so its 27 columns of views_linears.0 become a per-ray fp32
//     bias vector (computed by the PE warps) added in the V0 epilogue instead of a K=32 MMA block;
//   * alpha_linear (256->1) and rgb_linear (128->3) are fp32 dot products inside the L7 / V2 epilogues.
// Weights are pre-packed (inerf_mlp_pack) as the exact shared-memory image of every stage: bf16,
// K-major, 128-byte swizzle, in MMA issue order, so a stage is ONE contiguous bulk copy.
//
// Embedded-row variant (template parameter EMB, FaceNeRF.forward's x (P, 63+27)): the rows carry their own gamma(v), so there is no
// per-ray view bias.  The 27 view columns of views_linears.0 run as one more K-block at the end of each V0 half, its A operand a
// gamma(v) image that the producer warps write into the PE buffer once L5 (the last reader of gamma(p)) has completed; the commit after
// the last V0 view MMA hands the buffer back for the next iteration's gamma(p).  Packed blob: INERF_MLP_BF16_EMB (two more stages).
#include <cuda_bf16.h>

#include "mlp_tc.cuh"

using namespace inerf;
using namespace sm100;

namespace {

constexpr int NSTAGE = 3;
constexpr int STAGE_BYTES = 16384;
// CTA-pair build (PAIR = true): every weight stage is split across the two CTAs of a cluster (each holds HALF of its rows), so the same
// 48 KB ring is six stages deep
template <bool PAIR> using RingOf = Ring<PAIR, NSTAGE>;
constexpr int MAX_STEPS = 80;
constexpr int RMAX = 4;            // rays a 128-row slot can touch (s >= 43)
constexpr int NTHREADS_BF16 = 512;
constexpr int N_EPI = 256, N_PE = 128;

__constant__ TcStage c_steps[MAX_STEPS];
__constant__ TcStage c_steps_emb[MAX_STEPS];      // the embedded-row schedule (one more K-block per V0 half)
template <bool EMB> __device__ __forceinline__ const TcStage& step_at(int s) { return EMB ? c_steps_emb[s] : c_steps[s]; }

// smem map (bytes from the 1024-aligned base)
constexpr int OFF_ACT = 0;                               // [2][4][16384]
constexpr int OFF_PE = 131072;                           // [2][16384]
constexpr int OFF_W = 163840;                            // [NSTAGE][16384]
constexpr int OFF_ONES = OFF_W + NSTAGE * STAGE_BYTES;   // A operand of the bias MMAs: 128 x 16 bf16 ones, no-swizzle core-matrix layout
constexpr int OFF_BT = OFF_ONES + 4096;                  // [2][4096] bias tiles (B operand of the bias MMAs), streamed per layer half
constexpr int OFF_SB = OFF_BT + 2 * 4096;                // alpha_linear.bias, rgb_linear.bias (4 floats)
constexpr int OFF_AW = OFF_SB + 16;                      // alpha_linear.weight 256 floats
constexpr int OFF_RW = OFF_AW + 1024;                    // rgb_linear.weight 3x128 floats
constexpr int OFF_DIRB = OFF_RW + 1536;                  // [2][RMAX][128] floats
constexpr int OFF_BAR = OFF_DIRB + 2 * RMAX * 128 * 4;   // mbarriers
constexpr int SMEM_BYTES = OFF_BAR + 320;
constexpr int SMEM_ALLOC = SMEM_BYTES;
static_assert(SMEM_ALLOC <= 232448, "shared memory budget");

struct Bars {
    uint64_t wfull[RingOf<true>::N], wempty[RingOf<true>::N];
    uint64_t pfull[RingOf<true>::N];   // pair build, leader only: the PEER's half of the stage has landed (relayed by the peer's warp 1)
    uint64_t cbar[3];        // C0, C1, C2   (tcgen05.commit, once per layer; pair build: multicast to both CTAs)
    uint64_t ebar[2];        // E0, E1       (8 epilogue warps, once per layer; pair build: the leader's, 8 + 8 warps)
    uint64_t pe_ready;       // 128 PE threads, once per iteration (pair build: the leader's, 4 + 4 warps)
    uint64_t pe_free;        // commit after the last MMA that reads the PE block
    uint64_t dirb_ready;     // 128 PE threads
    uint64_t dirb_free;      // 8 epilogue warps
    uint64_t bfull[2], bempty[2];   // bias-tile ring
    uint64_t pbfull[2];      // pair build, leader only: the peer's half of the bias tile has landed
    uint32_t tmem_base;
};
static_assert(sizeof(Bars) <= 320, "barrier block");

struct LayerInfo { int N, bias_off; };

__device__ __forceinline__ LayerInfo layer_info(int l) {
    LayerInfo r;
    if (l < 8) { r.N = 256; r.bias_off = l * 256; }
    else { r.N = 128; r.bias_off = 8 * 256 + (l - 8) * 128; }
    return r;
}

// One 32-column chunk of an epilogue: +bias (+per-ray view bias), ReLU, bf16 pack; KIND 1 also accumulates
// alpha_linear, KIND 3 rgb_linear, in fp32 from the un-rounded activations.
template <int KIND, bool SAVE>
__device__ __forceinline__ void epi_convert(const uint32_t (&r)[32], uint32_t* __restrict__ packed16,
                                            const float* __restrict__ dsrc, const float* __restrict__ aw, const float* __restrict__ rw,
                                            float& alpha, float& rgb0, float& rgb1, float& rgb2, uint32_t& neg_bits) {
#pragma unroll
    for (int j = 0; j < 32; j += 4) {
        float v[4] = {__uint_as_float(r[j]), __uint_as_float(r[j + 1]), __uint_as_float(r[j + 2]), __uint_as_float(r[j + 3])};
        if constexpr (KIND == 2) {
            const float4 d = *reinterpret_cast<const float4*>(dsrc + j);
            v[0] += d.x; v[1] += d.y; v[2] += d.z; v[3] += d.w;
        }
        if constexpr (SAVE) {      // sign bits, first value in the top bit: one funnel shift per value
#pragma unroll
            for (int t = 0; t < 4; ++t) neg_bits = __funnelshift_l(__float_as_uint(v[t]), neg_bits, 1);
        }
        if constexpr (KIND == 1) {
            const float4 w = *reinterpret_cast<const float4*>(aw + j);
            alpha = fmaf(relu_nan(v[0]), w.x, alpha); alpha = fmaf(relu_nan(v[1]), w.y, alpha);
            alpha = fmaf(relu_nan(v[2]), w.z, alpha); alpha = fmaf(relu_nan(v[3]), w.w, alpha);
        }
        if constexpr (KIND == 3) {
            const float q[4] = {relu_nan(v[0]), relu_nan(v[1]), relu_nan(v[2]), relu_nan(v[3])};
            const float4 w0 = *reinterpret_cast<const float4*>(rw + j);
            const float4 w1 = *reinterpret_cast<const float4*>(rw + 128 + j);
            const float4 w2 = *reinterpret_cast<const float4*>(rw + 256 + j);
            rgb0 = fmaf(q[0], w0.x, rgb0); rgb0 = fmaf(q[1], w0.y, rgb0); rgb0 = fmaf(q[2], w0.z, rgb0); rgb0 = fmaf(q[3], w0.w, rgb0);
            rgb1 = fmaf(q[0], w1.x, rgb1); rgb1 = fmaf(q[1], w1.y, rgb1); rgb1 = fmaf(q[2], w1.z, rgb1); rgb1 = fmaf(q[3], w1.w, rgb1);
            rgb2 = fmaf(q[0], w2.x, rgb2); rgb2 = fmaf(q[1], w2.y, rgb2); rgb2 = fmaf(q[2], w2.z, rgb2); rgb2 = fmaf(q[3], w2.w, rgb2);
        }
        packed16[(j >> 1)] = pack_bf16x2_relu(v[0], v[1]);
        packed16[(j >> 1) + 1] = pack_bf16x2_relu(v[2], v[3]);
    }
}

struct IssueCtx {
    Bars* bars;
    uint32_t a_lo, pe_lo, w_lo, hi;      // descriptor halves of the activation / PE / weight-ring bases
    uint32_t tmem_base;
    uint32_t stage, wpar;                // weight ring position and the parity of its current round
    uint32_t ones_lo, bt_lo, bslot, bpar;   // bias MMA operands (no-swizzle descriptors) and the bias ring position
    uint32_t layer_ctr, iter_ctr;
};

// All MMAs of layer L for both 128-row slots, straight-line: every descriptor offset, wait and commit below is a compile-time
// constant of (L, half, K-block), so a step costs ~10 uniform-datapath instructions per tcgen05.mma instead of a table decode.
// (The table-driven form was issue-latency bound: ~150 dependent SASS instructions per 8-MMA step on ONE thread, ~1000 cycles
// against the 512 the tensor pipe needs -- profiles/r01_mlp_ablation.txt.)
// EMB: the embedded-row schedule.  pe_ready and pe_free then complete twice per iteration (gamma(p) for L0 / L5, gamma(v) for V0), so
// the issuer's waits have fixed parities: 0 before L0, 1 before V0's view K-block.
template <int L, bool PAIR, bool EMB = false>
__device__ __forceinline__ void issue_layer(IssueCtx& c) {
    constexpr int NSTAGE = RingOf<PAIR>::N, STAGE_BYTES = RingOf<PAIR>::BYTES;
    constexpr int N = lay_N(L), NH = N / 2, NKB = lay_act_kb(L), CNT = NKB + (lay_x(L, EMB) ? 1 : 0);
    constexpr int KB_PER_HALF_PREV = lay_prev_N(L) / 128;     // activation K-blocks written by ONE half of the previous epilogue
    constexpr int N_OUT_H0 = NH / 64;                          // K-blocks epi(h0) of THIS layer overwrites
    constexpr int N_FIRST = NKB < N_OUT_H0 ? NKB : N_OUT_H0;   // leading K-blocks of h1 that epi(h0) will overwrite
    constexpr uint32_t IDESC = umma_idesc_bf16(PAIR ? 256 : 128, NH);
    Bars* bars = c.bars;
    const uint32_t par_prev = (c.layer_ctr - 1) & 1;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
#pragma unroll
        for (int i = 0; i < CNT; ++i) {
            const bool is_pe = (i == NKB);                     // the PE block comes last in both halves
            if (h == 0 && c.layer_ctr > 0) {                   // each epilogue event is waited ONCE per layer, at its first use
                if (L == 0) {                                  // new iteration: both accumulator halves of V2 drained
                    if (i == 0) { wait_ev<PAIR>(&bars->ebar[0], par_prev); wait_ev<PAIR>(&bars->ebar[1], par_prev); }
                } else if (!is_pe) {
                    if (i == 0) wait_ev<PAIR>(&bars->ebar[0], par_prev);
                    if (i == KB_PER_HALF_PREV) wait_ev<PAIR>(&bars->ebar[1], par_prev);
                }
            }
            if (L == 0 && h == 0 && i == 0) wait_ev<PAIR>(&bars->pe_ready, EMB ? 0u : c.iter_ctr & 1);
            if (EMB && L == 8 && h == 0 && is_pe) wait_ev<PAIR>(&bars->pe_ready, 1u);
            mbar_wait(&bars->wfull[c.stage], c.wpar);
            if constexpr (PAIR) mbar_wait_cluster(&bars->pfull[c.stage], c.wpar);
            if (i == 0) {
                mbar_wait(&bars->bfull[c.bslot], c.bpar);
                if constexpr (PAIR) mbar_wait_cluster(&bars->pbfull[c.bslot], c.bpar);
            }
            tc_fence_after();
            if (elect_one()) {
                if (i == 0) {
                    // bias: D = ones[128x16] . tile[NHx16]^T with tile columns (hi, lo, 0, ...) = the folded bias split in two bf16;
                    // this MMA overwrites the accumulator, every weight MMA below accumulates
#pragma unroll
                    for (int slot = 0; slot < 2; ++slot)
                        umma_any<PAIR>(c.tmem_base + slot * 256 + h * NH, c.ones_lo, c.bt_lo + c.bslot * (4096 >> 4), HI_NOSWZ, IDESC, 0u);
                    commit_any<PAIR>(&bars->bempty[c.bslot]);
                }
                const uint32_t b_lo = c.w_lo + c.stage * (STAGE_BYTES >> 4);
#pragma unroll
                for (int slot = 0; slot < 2; ++slot) {
                    const uint32_t a_lo = is_pe ? c.pe_lo + slot * (16384 >> 4) : c.a_lo + slot * (65536 >> 4) + i * (16384 >> 4);
                    const uint32_t d = c.tmem_base + slot * 256 + h * NH;
#pragma unroll
                    for (int k = 0; k < 4; ++k) umma_any<PAIR>(d, a_lo + 2 * k, b_lo + 2 * k, c.hi, IDESC, 1u);
                }
                commit_any<PAIR>(&bars->wempty[c.stage]);
                const bool last = (i == CNT - 1);
                if (h == 0 && last) commit_any<PAIR>(&bars->cbar[0]);
                if (h == 1 && (N_FIRST > 0 ? i == N_FIRST - 1 : last)) commit_any<PAIR>(&bars->cbar[1]);
                if (h == 1 && last) commit_any<PAIR>(&bars->cbar[2]);
                if (h == 1 && last && (L == 5 || (EMB && L == 8))) commit_any<PAIR>(&bars->pe_free);
            }
            __syncwarp();
            if (i == 0) { c.bslot ^= 1; if (c.bslot == 0) c.bpar ^= 1; }
            if (++c.stage == NSTAGE) { c.stage = 0; c.wpar ^= 1; }
        }
    }
    ++c.layer_ctr;
}


__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

// Epilogue of one layer WITHOUT head / view-bias work (L0-L6 and V1: eight of eleven), inference build, both halves as straight-line
// code: tcgen05.ld, 16 conversions and (second half) 4 stores per 32-column chunk, store addresses = eight per-thread bases computed once
// per kernel + immediates, no layer-kind or chunk-count branch between the chunks.  The general loop below spends a third of its stall
// samples on instruction fetch and branch resolution around exactly this body (ncu source counters); instantiating that loop twice was
// slower (register spills), a separate small function is not.  act_row: shared-memory address of this thread's row in K-block 0 of its
// slot; soff[j] = byte offset of 16-byte chunk j of a 128-byte row after the swizzle.
template <int NH, bool PAIR>
__device__ __forceinline__ void epi_plain_layer(Bars* bars, uint32_t par, uint32_t t_lane, uint32_t act_row, const uint32_t (&soff)[8],
                                                int lane) {
    constexpr int NC = NH / 32;      // chunks per half: 4 (N = 256) or 2 (N = 128)
    // ---- first half: convert everything, wait until the second half's MMAs have read the K-blocks it overwrites (C1), store ----------
    mbar_wait(&bars->cbar[0], par);
    __syncwarp();
    tc_fence_after();
    uint32_t packed[NC * 16];
#pragma unroll
    for (int c = 0; c < NC; ++c) {
        uint32_t r[32];
        tmem_ld32(t_lane + c * 32, r);
        tmem_wait_ld();
#pragma unroll
        for (int j = 0; j < 16; ++j) packed[c * 16 + j] = pack_bf16x2_relu(__uint_as_float(r[2 * j]), __uint_as_float(r[2 * j + 1]));
    }
    tc_fence_before();
    mbar_wait(&bars->cbar[1], par);
    __syncwarp();
#pragma unroll
    for (int c = 0; c < NC; ++c)
#pragma unroll
        for (int q = 0; q < 4; ++q)
            sts128(act_row + ((c * 32) >> 6) * 16384 + soff[(((c * 32) & 63) >> 3) + q], packed[c * 16 + q * 4], packed[c * 16 + q * 4 + 1],
                   packed[c * 16 + q * 4 + 2], packed[c * 16 + q * 4 + 3]);
    fence_proxy_async_smem();
    __syncwarp();
    if (lane == 0) { if constexpr (PAIR) mbar_arrive_remote(&bars->ebar[0], 0); else mbar_arrive(&bars->ebar[0]); }
    // ---- second half: nothing reads its K-blocks any more, every chunk is stored as soon as it is converted ----------------------------
    mbar_wait(&bars->cbar[2], par);
    __syncwarp();
    tc_fence_after();
#pragma unroll
    for (int c = 0; c < NC; ++c) {
        uint32_t r[32], pk[16];
        tmem_ld32(t_lane + NH + c * 32, r);
        tmem_wait_ld();
#pragma unroll
        for (int j = 0; j < 16; ++j) pk[j] = pack_bf16x2_relu(__uint_as_float(r[2 * j]), __uint_as_float(r[2 * j + 1]));
#pragma unroll
        for (int q = 0; q < 4; ++q)
            sts128(act_row + ((NH + c * 32) >> 6) * 16384 + soff[(((NH + c * 32) & 63) >> 3) + q], pk[q * 4], pk[q * 4 + 1], pk[q * 4 + 2], pk[q * 4 + 3]);
    }
    tc_fence_before();
    fence_proxy_async_smem();
    __syncwarp();
    if (lane == 0) { if constexpr (PAIR) mbar_arrive_remote(&bars->ebar[1], 0); else mbar_arrive(&bars->ebar[1]); }
}

// Epilogue of L7 in the density-only build (DENS): the alpha head alone, in epi_convert<1>'s FMA order.  Nothing reads h7 (V0 does not
// run), so it is neither converted nor stored and no C1 wait is needed; each half still arrives on its event once its TMEM loads are
// done, because the next iteration's L0 overwrites those accumulators.
template <bool PAIR>
__device__ __forceinline__ void epi_alpha_layer(Bars* bars, uint32_t par, uint32_t t_lane, const float* __restrict__ aw, int lane, float& alpha) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        mbar_wait(&bars->cbar[h == 0 ? 0 : 2], par);
        __syncwarp();
        tc_fence_after();
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            uint32_t r[32];
            tmem_ld32(t_lane + h * 128 + c * 32, r);
            tmem_wait_ld();
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
                const float4 w = *reinterpret_cast<const float4*>(aw + h * 128 + c * 32 + j);
                alpha = fmaf(relu_nan(__uint_as_float(r[j])), w.x, alpha); alpha = fmaf(relu_nan(__uint_as_float(r[j + 1])), w.y, alpha);
                alpha = fmaf(relu_nan(__uint_as_float(r[j + 2])), w.z, alpha); alpha = fmaf(relu_nan(__uint_as_float(r[j + 3])), w.w, alpha);
            }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) { if constexpr (PAIR) mbar_arrive_remote(&bars->ebar[h], 0); else mbar_arrive(&bars->ebar[h]); }
    }
}

// ---------------------------------------------------------------------------------------------
// the kernel
// ---------------------------------------------------------------------------------------------
// PAIR = true (inference build): the kernel runs as clusters of two CTAs.  Every MMA is ONE tcgen05.mma.cta_group::2 over the 2 x 128
// rows of the pair (issued by the leader's warp 1), and the B operand -- the weight stage -- is split across the pair: each CTA streams
// and keeps only HALF of the rows of every stage.  Why: the N = 128 MMAs of the single-CTA form read 8 KB of operands per 64 cycles,
// all 128 B/clk of an SM's shared memory, so the epilogue's activation stores (128 KB per layer) and the weight ring's refills compete
// with the tensor pipe for the same port -- a layer measured 5.2 kcycles against 4.35 of MMA time (profiles/r03_phase_timers.txt), and
// total shared-memory traffic / 128 B/clk reproduces the iteration time.  A pair reads 6 KB per MMA per CTA and writes half the weight
// bytes.  Schedule, layouts, packed blob and epilogue are the single-CTA kernel's: a pair iteration is two 256-point chunks, CTA r takes
// chunk 2 it + r.  Cross-CTA protocol: commits are multicast to both CTAs' barriers; the peer's epilogue / positional-encoding warps
// arrive remotely on the LEADER's event barriers; the peer's (otherwise idle) warp 1 relays "my half of the stage has landed".
//
// DENS = true (density-only build, inference only): the coarse pass of a render that discards the coarse colour needs sigma alone, which
// depends on L0-L7 and the alpha head.  The issuer runs L0-L7 and starts the next iteration (L0 waits E0 / E1 of L7), producer and relay
// stream the stages of L0-L7 -- the first n_steps of the same schedule and blob -- the PE warps skip the per-ray view bias, and the output
// is one float per point, alpha + alpha_linear.bias: the .w of the full build, bit for bit.
template <bool SAVE = false, bool PAIR = false, bool EMB = false, bool DENS = false>
__global__ void __launch_bounds__(NTHREADS_BF16, 1) mlp_bf16_kernel(MlpArgs a, int n_steps, int n_rays) {
    constexpr int NSTAGE = RingOf<PAIR>::N, STAGE_BYTES = RingOf<PAIR>::BYTES;
    static_assert(!(DENS && (SAVE || EMB)), "the density-only build is an inference build of the fused entry");
    // Dynamic shared memory is the only shared allocation of this kernel, so it starts at offset 0 of the CTA's
    // window: 1024-byte aligned as the 128B-swizzle atoms need.  (No pointer re-alignment arithmetic here: it would
    // make the compiler lose the shared address space and emit generic LD/ST for every epilogue access.)
    extern __shared__ __align__(1024) uint8_t sm[];
    if ((smem_u32(sm) & 1023u) != 0) __trap();
    Bars* bars = reinterpret_cast<Bars*>(sm + OFF_BAR);
    float* s_sb = reinterpret_cast<float*>(sm + OFF_SB);
    float* s_aw = reinterpret_cast<float*>(sm + OFF_AW);
    float* s_rw = reinterpret_cast<float*>(sm + OFF_RW);
    float* s_dirb = reinterpret_cast<float*>(sm + OFF_DIRB);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    // iteration space: single CTA: chunk = it, one chunk of 256 points per CTA iteration; pair: chunk = 2 it + rank
    const uint32_t rank = PAIR ? cluster_ctarank() : 0u;
    const long long n_iter = PAIR ? (a.P + 511) / 512 : (a.P + 255) / 256;
    const long long it_first = PAIR ? (long long)(blockIdx.x >> 1) : (long long)blockIdx.x;
    const long long it_step = PAIR ? (long long)(gridDim.x >> 1) : (long long)gridDim.x;
#define CHUNK_OF(it_) (PAIR ? 2 * (it_) + (long long)rank : (it_))

    // ---- one-time setup -------------------------------------------------------------------
    if (tid < 4) s_sb[tid] = a.cond[8 * 256 + 3 * 128 + tid];
    for (int i = tid; i < 256; i += NTHREADS_BF16)           // the ones tile (bf16 1.0 = 0x3F80), read by the async proxy
        reinterpret_cast<uint4*>(sm + OFF_ONES)[i] = make_uint4(0x3F803F80u, 0x3F803F80u, 0x3F803F80u, 0x3F803F80u);
    fence_proxy_async_smem();
    for (int i = tid; i < 256; i += NTHREADS_BF16) s_aw[i] = a.w[P_ALPHA_W][i];
    for (int i = tid; i < 384; i += NTHREADS_BF16) s_rw[i] = a.w[P_RGB_W][i];
    if (tid == 0) {
        for (int s = 0; s < NSTAGE; ++s) { mbar_init(&bars->wfull[s], 1); mbar_init(&bars->wempty[s], 1); mbar_init(&bars->pfull[s], 1); }
        for (int j = 0; j < 3; ++j) mbar_init(&bars->cbar[j], 1);
        for (int j = 0; j < 2; ++j) mbar_init(&bars->ebar[j], PAIR ? 2 * (N_EPI / 32) : N_EPI / 32);
        mbar_init(&bars->pe_ready, PAIR ? 2 * (N_PE / 32) : N_PE);
        mbar_init(&bars->pe_free, 1);
        mbar_init(&bars->dirb_ready, N_PE);
        mbar_init(&bars->dirb_free, N_EPI / 32);
        for (int j = 0; j < 2; ++j) { mbar_init(&bars->bfull[j], 1); mbar_init(&bars->bempty[j], 1); mbar_init(&bars->pbfull[j], 1); }
        fence_mbar_init();
    }
    if (warp == 2) {
        if constexpr (PAIR) {
            tmem_alloc_pair(&bars->tmem_base, 512);
        } else {
            tmem_alloc(&bars->tmem_base, 512);
            tmem_relinquish();
        }
    }
    tc_fence_before();
    __syncthreads();
    if constexpr (PAIR) cluster_sync_all();      // both CTAs' barriers and tensor memory exist before any remote arrive / multicast commit
    tc_fence_after();
    const uint32_t tmem_base = bars->tmem_base;

    if (warp == 0) {
        // ================= weight producer ==================================================
        if (lane == 0) {
            const uint8_t* blob = reinterpret_cast<const uint8_t*>(a.packed);
            const uint8_t* tiles = reinterpret_cast<const uint8_t*>(a.cond + COND_FLOATS);
            uint32_t g = 0, bh = 0;
            // pair build: this CTA's HALF of the rows of every stage / bias tile (rows [rank * NH / 2, (rank + 1) * NH / 2) are the first /
            // second half of the image's bytes: 8-row groups are contiguous)
            constexpr uint32_t SPLIT = PAIR ? 2u : 1u;
            for (long long it = it_first; it < n_iter; it += it_step) {
                for (int s = 0; s < n_steps; ++s, ++g) {
                    const uint32_t stage = g % NSTAGE, round = g / NSTAGE;
                    if (step_at<EMB>(s).first) {       // first step of a (layer, half): its bias tile
                        const uint32_t slot = bh & 1, l = step_at<EMB>(s).layer, h = step_at<EMB>(s).half;
                        const uint32_t bytes = (uint32_t)step_at<EMB>(s).n8 * 8u * 32u / SPLIT;
                        const uint32_t off = bias_tile_offset(l, h) + rank * bytes;
                        mbar_wait(&bars->bempty[slot], ((bh >> 1) & 1) ^ 1);
                        mbar_arrive_expect_tx(&bars->bfull[slot], bytes);
                        bulk_g2s(sm + OFF_BT + slot * 4096, tiles + off, bytes, &bars->bfull[slot]);
                        ++bh;
                    }
                    mbar_wait(&bars->wempty[stage], (round & 1) ^ 1);
                    const uint32_t bytes = (uint32_t)step_at<EMB>(s).n8 * 8u * 128u / SPLIT;
                    mbar_arrive_expect_tx(&bars->wfull[stage], bytes);
                    bulk_g2s(sm + OFF_W + stage * STAGE_BYTES, blob + step_at<EMB>(s).offset + rank * bytes, bytes, &bars->wfull[stage]);
                }
            }
        }
    } else if (warp == 1 && PAIR && rank != 0) {
        // ================= relay (peer CTA of a pair): tell the leader when MY half of a bias tile / weight stage has landed =========
        if (lane == 0) {
            uint32_t g = 0, bh = 0;
            for (long long it = it_first; it < n_iter; it += it_step)
                for (int s = 0; s < n_steps; ++s, ++g) {
                    if (step_at<EMB>(s).first) {
                        mbar_wait(&bars->bfull[bh & 1], (bh >> 1) & 1);
                        mbar_arrive_remote(&bars->pbfull[bh & 1], 0);
                        ++bh;
                    }
                    mbar_wait(&bars->wfull[g % NSTAGE], (g / NSTAGE) & 1);
                    mbar_arrive_remote(&bars->pfull[g % NSTAGE], 0);
                }
        }
    } else if (warp == 1) {
        // ================= MMA issuer (whole warp converged; one elected lane issues) ==========
        IssueCtx c;
        c.bars = bars;
        c.hi = (uint32_t)(umma_desc_sw128(0) >> 32);
        c.a_lo = (uint32_t)umma_desc_sw128(smem_u32(sm + OFF_ACT));
        c.pe_lo = (uint32_t)umma_desc_sw128(smem_u32(sm + OFF_PE));
        c.w_lo = (uint32_t)umma_desc_sw128(smem_u32(sm + OFF_W));
        c.tmem_base = tmem_base;
        c.ones_lo = desc_lo_noswz(smem_u32(sm + OFF_ONES));
        c.bt_lo = desc_lo_noswz(smem_u32(sm + OFF_BT));
        c.bslot = 0; c.bpar = 0;
        c.stage = 0; c.wpar = 0; c.layer_ctr = 0; c.iter_ctr = 0;
        for (long long it = it_first; it < n_iter; it += it_step, ++c.iter_ctr) {
            // Layers of equal geometry share ONE copy of the straight-line issue code (L1-L4, L6, L7 are 256 x 256 after a 256-wide
            // layer; V1, V2 are 128 x 128 after a 128-wide one): 11 inlined copies were 78 KB of SASS streamed once per iteration, which
            // together with the epilogue and PE code overflowed the instruction cache the epilogue warps live in (ncu: stall_no_inst).
            issue_layer<0, PAIR, EMB>(c);
#pragma unroll 1
            for (int seg = 0; seg < 2; ++seg) {
#pragma unroll 1
                for (int r = 0; r < (seg ? 2 : 4); ++r) issue_layer<1, PAIR, EMB>(c);
                if (seg == 0) issue_layer<5, PAIR, EMB>(c);
            }
            if constexpr (!DENS) {
                issue_layer<8, PAIR, EMB>(c);
#pragma unroll 1
                for (int r = 0; r < 2; ++r) issue_layer<9, PAIR, EMB>(c);
            }
        }
    } else if (warp >= 4 && warp < 12) {
        // ================= epilogue: one row per thread ======================================
        const int slot = (warp - 4) >> 2;
        const int row = ((warp & 3) << 5) + lane;
        const uint32_t t_lane = tmem_base + ((uint32_t)((warp & 3) << 5) << 16) + slot * 256;
        uint8_t* act = sm + OFF_ACT + slot * 65536;
        const uint32_t row_off = (row >> 3) * 1024 + (row & 7) * 128;
        const uint32_t rsw = row & 7;
        const uint32_t act_row_u32 = smem_u32(act) + row_off;
        uint32_t soff[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) soff[j] = ((uint32_t)j ^ rsw) << 4;
        uint32_t layer_ctr = 0, iter_ctr = 0;
        for (long long it = it_first; it < n_iter; it += it_step, ++iter_ctr) {
            const long long chunk = CHUNK_OF(it);
            const bool chunk_ok = !PAIR || chunk * 256 < a.P;      // pair build: the peer's last chunk may lie wholly past the end (nothing is saved for it)
            const long long p0 = chunk * 256 + slot * 128;
            long long p = p0 + row;
            const bool in_range = p < a.P;
            if (!in_range) p = a.P - 1;
            const int ray_local = EMB ? 0 : (int)(p / a.s - min(p0, a.P - 1) / a.s);      // embedded rows: no per-ray view bias
            float alpha = 0.f, rgb0 = 0.f, rgb1 = 0.f, rgb2 = 0.f;
            for (int l = 0; l < (DENS ? 8 : 11); ++l, ++layer_ctr) {
                const LayerInfo li = layer_info(l);
                const int NH = li.N >> 1;
                const uint32_t par = layer_ctr & 1;
                if constexpr (!SAVE) {      // inference: the layers without head / view-bias work take the straight-line epilogue
                    if (l <= 6) { epi_plain_layer<128, PAIR>(bars, par, t_lane, act_row_u32, soff, lane); continue; }
                    if constexpr (DENS) { epi_alpha_layer<PAIR>(bars, par, t_lane, s_aw, lane, alpha); continue; }
                    if (l == 9 || (EMB && l == 8)) { epi_plain_layer<64, PAIR>(bars, par, t_lane, act_row_u32, soff, lane); continue; }
                }
                if (!EMB && l == 8) mbar_wait(&bars->dirb_ready, iter_ctr & 1);
#pragma unroll 1
                for (int h = 0; h < 2; ++h) {
                    mbar_wait(&bars->cbar[h == 0 ? 0 : 2], par);
                    __syncwarp();
                    tc_fence_after();
                    uint32_t packed[64];
                    const int nchunk = NH >> 5;      // 4 (N=256) or 2 (N=128)
                    // training: this row's mask words of the half (one pointer per half instead of a 64-bit index product per chunk)
                    uint32_t* mask_half = SAVE ? a.save_mask + (((size_t)chunk * 2 + slot) * TRAIN_MASK_WORDS + train_mask_of(l) + ((h * NH) >> 5)) * 128 + row
                                               : nullptr;
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        if (c < nchunk) {
                            uint32_t r[32];
                            tmem_ld32(t_lane + h * NH + c * 32, r);
                            tmem_wait_ld();
                            const int f0 = h * NH + c * 32;                 // first output feature of the chunk
                            uint32_t neg = 0;
                            switch (l) {                                    // layer kind is warp-uniform: one specialised body per chunk
                                case 7: epi_convert<1, SAVE>(r, &packed[c * 16], nullptr, s_aw + f0, nullptr, alpha, rgb0, rgb1, rgb2, neg); break;
                                case 8:
                                    if constexpr (EMB) epi_convert<0, SAVE>(r, &packed[c * 16], nullptr, nullptr, nullptr, alpha, rgb0, rgb1, rgb2, neg);
                                    else epi_convert<2, SAVE>(r, &packed[c * 16], s_dirb + (slot * RMAX + ray_local) * 128 + f0, nullptr, nullptr, alpha, rgb0, rgb1, rgb2, neg);
                                    break;
                                case 10: epi_convert<3, SAVE>(r, &packed[c * 16], nullptr, nullptr, s_rw + f0, alpha, rgb0, rgb1, rgb2, neg); break;
                                default: epi_convert<0, SAVE>(r, &packed[c * 16], nullptr, nullptr, nullptr, alpha, rgb0, rgb1, rgb2, neg); break;
                            }
                            if (SAVE && chunk_ok)      // training: the ReLU mask word of the chunk (the activations follow as a bulk copy of the smem image)
                                mask_half[c * 128] = ~neg;
                            if (!SAVE && h == 1 && l != 10) {
                                // second half: nothing reads these K-blocks any more (its own MMAs are complete), so each chunk goes to shared
                                // memory as soon as it is converted and drains behind the next chunk's load instead of in front of the fence
                                uint8_t* kb = act + (f0 >> 6) * 16384 + row_off;
                                const int ch0 = (f0 & 63) >> 3;
#pragma unroll
                                for (int q = 0; q < 4; ++q)
                                    *reinterpret_cast<uint4*>(kb + soff[ch0 + q]) =
                                        make_uint4(packed[c * 16 + q * 4], packed[c * 16 + q * 4 + 1], packed[c * 16 + q * 4 + 2], packed[c * 16 + q * 4 + 3]);
                            }
                        }
                    }
                    tc_fence_before();
                    if (l != 10 || SAVE) {
                        if (h == 0) mbar_wait(&bars->cbar[1], par);
                        if constexpr (SAVE) {
                            // training: each warp bulk-copies its own 32 rows of the K-blocks it writes (4 KB per K-block image) to HBM, so no
                            // barrier couples the warps.  Before overwriting them, lane 0 waits until the copy that last read these rows has
                            // left shared memory: that is two copies back (this half's K-blocks were written by the same half of the previous
                            // layer) unless the layer widens (l == 0 after the 128-wide rgb layer), where it is the latest one.
                            if (lane == 0) { if (h == 0 && l == 0) bulk_wait_read_all(); else bulk_wait_read_but_one(); }
                        }
                        __syncwarp();      // h1 has finished reading the K-blocks written below
#pragma unroll
                        for (int c = 0; c < 4; ++c) {
                            if (c < nchunk && (SAVE || h == 0)) {
                                const int f0 = h * NH + c * 32;
                                uint8_t* kb = act + (f0 >> 6) * 16384 + row_off;
                                const int ch0 = (f0 & 63) >> 3;                // first 16-byte chunk inside the 128-byte row
#pragma unroll
                                for (int q = 0; q < 4; ++q) {
                                    uint4 v = make_uint4(packed[c * 16 + q * 4], packed[c * 16 + q * 4 + 1],
                                                         packed[c * 16 + q * 4 + 2], packed[c * 16 + q * 4 + 3]);
                                    *reinterpret_cast<uint4*>(kb + soff[ch0 + q]) = v;
                                }
                            }
                        }
                        fence_proxy_async_smem();
                        if constexpr (SAVE) {
                            __syncwarp();
                            if (lane == 0 && chunk_ok) {
                                const int kb0 = (h * NH) >> 6, nkb = NH >> 6;      // 2 K-blocks per half (N = 256) or 1 (N = 128)
                                const uint32_t wrow = (uint32_t)(warp & 3) * 4096u;      // 32 rows = 4 row groups of 1 KB
                                uint8_t* g = a.save_img + (((size_t)chunk * 2 + slot) * TRAIN_IMGS + train_img_of(l) + kb0) * 16384 + wrow;
                                for (int k = 0; k < nkb; ++k) bulk_s2g(g + k * 16384, act + (kb0 + k) * 16384 + wrow, 4096u);
                                bulk_commit();
                            }
                        }
                    }
                    // one arrival per warp: 256 per-thread arrivals on one mbarrier serialise in the shared-memory pipe and sit on
                    // the layer-to-layer critical path (E1 gates the next layer's third K-block)
                    __syncwarp();
                    if (lane == 0) { if constexpr (PAIR) mbar_arrive_remote(&bars->ebar[h], 0); else mbar_arrive(&bars->ebar[h]); }
                }
                if (!EMB && l == 8) {
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&bars->dirb_free);
                }
            }
            if (DENS && in_range) {
                a.out[p] = alpha + s_sb[0];
            } else if (in_range) {
                float4 o;
                o.x = rgb0 + s_sb[1];
                o.y = rgb1 + s_sb[2];
                o.z = rgb2 + s_sb[3];
                o.w = alpha + s_sb[0];
                reinterpret_cast<float4*>(a.out)[p] = o;
            }
        }
        if constexpr (SAVE) {
            if (lane == 0) bulk_wait_all();
        }
    } else if (EMB && warp >= 12) {
        // ================= embedded rows: gamma(p), then gamma(v), of row t of both slots, copied from x into the PE buffer ======
        // A row of x is 90 floats (360 B; 8-byte aligned when x is 16-byte aligned): gamma(p) = columns 0..62 (image column 63 zero),
        // gamma(v) = columns 63..89 (image columns 27..63 zero).  Each block is in registers before the wait for the buffer, so only the
        // shared-memory stores lie between its release and the pe_ready arrival.  pe_free parities: 0 = L5 has read gamma(p) of this
        // iteration, 1 = V0 has read gamma(v) of the previous one.
        const int t = tid - 12 * 32;
        const uint32_t row_img = (t >> 3) * 1024 + (t & 7) * 128;
        auto store_img = [&](uint8_t* img, const uint32_t* w, int n_chunks) {      // one 128-byte row of a swizzled image, zero-padded
#pragma unroll
            for (int q = 0; q < 8; ++q)
                *reinterpret_cast<uint4*>(img + row_img + ((q ^ (t & 7)) << 4)) =
                    q < n_chunks ? make_uint4(w[4 * q], w[4 * q + 1], w[4 * q + 2], w[4 * q + 3]) : make_uint4(0u, 0u, 0u, 0u);
        };
        auto arrive_ready = [&] {
            fence_proxy_async_smem();
            if constexpr (PAIR) {
                __syncwarp();
                if (lane == 0) mbar_arrive_remote(&bars->pe_ready, 0);
            } else {
                mbar_arrive(&bars->pe_ready);
            }
        };
        for (long long it = it_first; it < n_iter; it += it_step) {
            const long long chunk = CHUNK_OF(it);
            const bool chunk_ok = !PAIR || chunk * 256 < a.P;
            const float* xr[2];
#pragma unroll
            for (int sl = 0; sl < 2; ++sl) {
                long long p = chunk * 256 + sl * 128 + t;
                if (p > a.P - 1) p = a.P - 1;
                xr[sl] = a.x + p * 90;
            }
            uint32_t pk[2][32];
#pragma unroll
            for (int sl = 0; sl < 2; ++sl) {
#pragma unroll
                for (int j = 0; j < 31; ++j) {
                    const float2 v = __ldg(reinterpret_cast<const float2*>(xr[sl]) + j);
                    pk[sl][j] = pack_bf16x2(v.x, v.y);
                }
                pk[sl][31] = pack_bf16x2(__ldg(xr[sl] + 62), 0.f);
            }
            if (it != it_first) mbar_wait(&bars->pe_free, 1u);
#pragma unroll
            for (int sl = 0; sl < 2; ++sl) store_img(sm + OFF_PE + sl * 16384, pk[sl], 8);
            arrive_ready();
            if (SAVE && chunk_ok) {          // training: gamma(p) is the X operand of dW for pts_linears.0 / .5
#pragma unroll
                for (int sl = 0; sl < 2; ++sl)
                    store_img(a.save_img + (((size_t)chunk * 2 + sl) * TRAIN_IMGS + TRAIN_IMG_PE) * 16384, pk[sl], 8);
            }
            uint32_t pv[2][16];
#pragma unroll
            for (int sl = 0; sl < 2; ++sl) {
                float g[28];
                g[0] = __ldg(xr[sl] + 63);
#pragma unroll
                for (int j = 0; j < 13; ++j) {
                    const float2 v = __ldg(reinterpret_cast<const float2*>(xr[sl] + 64) + j);
                    g[1 + 2 * j] = v.x; g[2 + 2 * j] = v.y;
                }
                g[27] = 0.f;
#pragma unroll
                for (int j = 0; j < 14; ++j) pv[sl][j] = pack_bf16x2(g[2 * j], g[2 * j + 1]);
                pv[sl][14] = pv[sl][15] = 0u;
            }
            mbar_wait(&bars->pe_free, 0u);
#pragma unroll
            for (int sl = 0; sl < 2; ++sl) store_img(sm + OFF_PE + sl * 16384, pv[sl], 4);
            arrive_ready();
            if (SAVE && chunk_ok) {          // training: gamma(v) per point, the X operand of dW for the view columns of views_linears.0
#pragma unroll
                for (int sl = 0; sl < 2; ++sl)
                    store_img(a.save_img + (((size_t)chunk * 2 + sl) * TRAIN_IMGS + TRAIN_IMG_DIR) * 16384, pv[sl], 4);
            }
        }
    } else if (warp >= 12) {
        // ================= positional encoding + per-ray view bias producers ==================
        const int t = tid - 12 * 32;                 // 0..127: row of both slots, and output feature of the view bias
        float wdir[27];                              // views_linears.0.weight[t, 256:283], resident in registers
        if constexpr (!DENS) {
            const float* wrow = a.w[P_VIEWS_W] + (size_t)t * (283 + a.dim_expr) + 256;
#pragma unroll
            for (int j = 0; j < 27; ++j) wdir[j] = wrow[j];
        }
        uint32_t iter_ctr = 0;
        for (long long it = it_first; it < n_iter; it += it_step, ++iter_ctr) {
            const long long chunk = CHUNK_OF(it);
            // ---- gamma_10(o + d z) for row t of both slots ---------------------------------------
            uint32_t pk[2][32];
#pragma unroll
            for (int sl = 0; sl < 2; ++sl) {
                long long p = chunk * 256 + sl * 128 + t;
                if (p > a.P - 1) p = a.P - 1;
                const long long ray = p / a.s;
                const float* r = a.rays + ray * a.ray_stride;
                const float zz = a.z[p];
                float v[64];
#pragma unroll
                for (int c = 0; c < 3; ++c) v[c] = __fadd_rn(r[c], __fmul_rn(r[3 + c], zz));
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    // one accurate sincosf per coordinate, then angle doubling: sin 2a = 2 sin a cos a, cos 2a = 1 - 2 sin^2 a.
                    // An angle error doubles per octave, but an amplitude error (sin^2 + cos^2 != 1) is multiplied by 4 sin^2 a, so
                    // the absolute error grows by up to ~3.1x per octave (two steps at most 9.5x): bounded by 3.1^f * 2^-22, ~1e-4 at
                    // octave 7 and ~6e-3 at octave 9 (tests/test_bf16_operands.py measured 1.0e-4 and 9.7e-4 there).  Near a zero of sin / cos that is
                    // many bf16 ulps of the value; against the bf16 rounding (2^-9 relative) of operands of magnitude ~1 it is small,
                    // and it costs 27 short FMA chains instead of 27 range reductions.  (mlp_f16x2.cu and mlp_fp32.cu call sincosf
                    // per octave.)
                    float sn, cs;
                    sincosf(v[c], &sn, &cs);
                    v[3 + c] = sn;
                    v[6 + c] = cs;
#pragma unroll
                    for (int f = 1; f < 10; ++f) {
                        const float s2 = 2.0f * sn * cs, c2 = fmaf(-2.0f * sn, sn, 1.0f);
                        sn = s2; cs = c2;
                        v[3 + 6 * f + c] = sn;
                        v[6 + 6 * f + c] = cs;
                    }
                }
                v[63] = 0.f;
#pragma unroll
                for (int j = 0; j < 32; ++j) pk[sl][j] = pack_bf16x2(v[2 * j], v[2 * j + 1]);
            }
            if (iter_ctr > 0) mbar_wait(&bars->pe_free, (iter_ctr - 1) & 1);
#pragma unroll
            for (int sl = 0; sl < 2; ++sl) {
                uint8_t* dst = sm + OFF_PE + sl * 16384 + (t >> 3) * 1024 + (t & 7) * 128;
#pragma unroll
                for (int q = 0; q < 8; ++q)
                    *reinterpret_cast<uint4*>(dst + ((q ^ (t & 7)) << 4)) =
                        make_uint4(pk[sl][4 * q], pk[sl][4 * q + 1], pk[sl][4 * q + 2], pk[sl][4 * q + 3]);
            }
            fence_proxy_async_smem();
            if constexpr (PAIR) {
                __syncwarp();
                if (lane == 0) mbar_arrive_remote(&bars->pe_ready, 0);
            } else {
                mbar_arrive(&bars->pe_ready);
            }
            const bool chunk_ok = !PAIR || chunk * 256 < a.P;
            if (SAVE && chunk_ok) {          // training: gamma(p) is the X operand of dW for pts_linears.0 / .5
#pragma unroll
                for (int sl = 0; sl < 2; ++sl) {
                    uint8_t* dst = a.save_img + (((size_t)chunk * 2 + sl) * TRAIN_IMGS + TRAIN_IMG_PE) * 16384 + (t >> 3) * 1024 + (t & 7) * 128;
#pragma unroll
                    for (int q = 0; q < 8; ++q)
                        *reinterpret_cast<uint4*>(dst + ((q ^ (t & 7)) << 4)) =
                            make_uint4(pk[sl][4 * q], pk[sl][4 * q + 1], pk[sl][4 * q + 2], pk[sl][4 * q + 3]);
                }
            }
            // ---- per-ray view bias: lane q < 2*RMAX encodes ray q, the warp shares it by shuffle (no V0 in the density-only build) ----
            if constexpr (!DENS) {
                float enc[27];
                const int q = lane;
                if (q < 2 * RMAX) {
                    const int sl = q / RMAX, rl = q - sl * RMAX;
                    long long pfirst = chunk * 256 + sl * 128;
                    if (pfirst > a.P - 1) pfirst = a.P - 1;
                    long long ray = pfirst / a.s + rl;
                    if (ray > n_rays - 1) ray = n_rays - 1;
                    const float* r = a.rays + ray * a.ray_stride + (a.ray_stride - 3);
                    enc[0] = r[0]; enc[1] = r[1]; enc[2] = r[2];
#pragma unroll
                    for (int f = 0; f < 4; ++f)
#pragma unroll
                        for (int c = 0; c < 3; ++c) {
                            float sn, cs;
                            sincosf(enc[c] * (float)(1 << f), &sn, &cs);
                            enc[3 + 6 * f + c] = sn;
                            enc[6 + 6 * f + c] = cs;
                        }
                } else {
#pragma unroll
                    for (int j = 0; j < 27; ++j) enc[j] = 0.f;
                }
                if (SAVE && chunk_ok) {      // training: gamma(v) per POINT, the X operand of dW for the view columns of views_linears.0
#pragma unroll
                    for (int sl = 0; sl < 2; ++sl) {
                        long long p = chunk * 256 + sl * 128 + t, pfirst = chunk * 256 + sl * 128;
                        if (p > a.P - 1) p = a.P - 1;
                        if (pfirst > a.P - 1) pfirst = a.P - 1;
                        const int src = sl * RMAX + (int)(p / a.s - pfirst / a.s);
                        float g[28];
#pragma unroll
                        for (int j = 0; j < 27; ++j) g[j] = __shfl_sync(0xffffffffu, enc[j], src);
                        g[27] = 0.f;
                        uint8_t* dst = a.save_img + (((size_t)chunk * 2 + sl) * TRAIN_IMGS + TRAIN_IMG_DIR) * 16384 + (t >> 3) * 1024 + (t & 7) * 128;
#pragma unroll
                        for (int qq = 0; qq < 8; ++qq) {
                            uint4 v = make_uint4(0u, 0u, 0u, 0u);
                            if (qq < 4) {
                                v.x = pack_bf16x2(g[8 * qq], g[8 * qq + 1]);
                                v.y = pack_bf16x2(g[8 * qq + 2], g[8 * qq + 3]);
                                if (qq < 3) { v.z = pack_bf16x2(g[8 * qq + 4], g[8 * qq + 5]); v.w = pack_bf16x2(g[8 * qq + 6], g[8 * qq + 7]); }
                            }
                            *reinterpret_cast<uint4*>(dst + ((qq ^ (t & 7)) << 4)) = v;
                        }
                    }
                }
                if (iter_ctr > 0) mbar_wait(&bars->dirb_free, (iter_ctr - 1) & 1);
                for (int q2 = 0; q2 < 2 * RMAX; ++q2) {
                    float acc = 0.f;
#pragma unroll
                    for (int j = 0; j < 27; ++j) acc = fmaf(wdir[j], __shfl_sync(0xffffffffu, enc[j], q2), acc);
                    s_dirb[q2 * 128 + t] = acc;
                }
                mbar_arrive(&bars->dirb_ready);
            }
        }
    }

    // ---- teardown ---------------------------------------------------------------------------
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

}  // namespace

namespace inerf {

int mlp_bf16_packed_bytes(const InerfNetDims* d, size_t* bytes, bool embedded) {
    *bytes = (size_t)build_tc_schedule(d, embedded, 1).total_bytes;
    return INERF_OK;
}

int mlp_bf16_pack(const InerfNetDims* d, const float* const* params_host, void* packed, cudaStream_t st, bool embedded) {
    return pack_tc_schedule<false>(build_tc_schedule(d, embedded, 1), params_host, packed, st, "inerf_mlp_pack");
}

template <bool SAVE, bool PAIR, bool EMB, bool DENS = false>
static int launch(const MlpArgs& a, int n_steps, int n_rays, cudaStream_t st, const char* what) {
    return launch_tc(mlp_bf16_kernel<SAVE, PAIR, EMB, DENS>, PAIR, (a.P + 255) / 256, NTHREADS_BF16, SMEM_ALLOC, st, what, a, n_steps, n_rays);
}

// FaceNeRF.forward on embedded rows x (P, 90): a.packed is an INERF_MLP_BF16_EMB blob, a.save_img != NULL selects the saving build
static int launch_embedded(const MlpArgs& a, cudaStream_t st) {
    if (((uintptr_t)a.packed | (uintptr_t)a.x) & 15) return fail(INERF_E_ALIGN, "inerf_mlp_fwd_embedded: packed weights and x must be 16-byte aligned");
    if (a.save_img && !a.save_mask) return fail(INERF_E_ARG, "mlp_bf16: save_mask is NULL");
    static thread_local int configured_dev = -1;
    static const TcSchedule S = [] { InerfNetDims d{64, 76, 32, 256, 8, 63, 27}; return build_tc_schedule(&d, true, 1); }();
    int rc = setup_once(configured_dev,
                        {(const void*)mlp_bf16_kernel<false, false, true>, (const void*)mlp_bf16_kernel<true, false, true>,
                         (const void*)mlp_bf16_kernel<false, true, true>, (const void*)mlp_bf16_kernel<true, true, true>},
                        SMEM_ALLOC, "mlp_bf16", [] { return cudaMemcpyToSymbol(c_steps_emb, S.st, sizeof(TcStage) * MAX_STEPS); });
    if (rc) return rc;
    if (mlp_pair_enabled())
        return a.save_img ? launch<true, true, true>(a, S.n_stages, 0, st, "inerf_mlp_fwd_train[bf16 pair]")
                          : launch<false, true, true>(a, S.n_stages, 0, st, "inerf_mlp_fwd[bf16 pair]");
    return a.save_img ? launch<true, false, true>(a, S.n_stages, 0, st, "inerf_mlp_fwd_train_bf16_embedded")
                      : launch<false, false, true>(a, S.n_stages, 0, st, "inerf_mlp_fwd_embedded[bf16]");
}

int mlp_bf16_launch(const MlpArgs& a, bool embedded, cudaStream_t st, bool density) {
    if (embedded) return launch_embedded(a, st);
    if (a.s < 43) return fail(INERF_E_UNSUPPORTED, "bf16 mode needs at least 43 samples per ray (a 128-row slot may touch at most 4 rays)");
    if ((uintptr_t)a.packed & 15) return fail(INERF_E_ALIGN, "inerf_mlp_fwd: packed weights must be 16-byte aligned");
    static thread_local int configured_dev = -1;
    // the step table does not depend on the conditioning dims; a function-local static is initialised once, thread-safely
    static const TcSchedule S = [] { InerfNetDims d{64, 76, 32, 256, 8, 63, 27}; return build_tc_schedule(&d, false, 1); }();
    static const int n_steps_dens = tc_stages_before(S, 8);      // the stages of L0-L7
    int rc = setup_once(configured_dev,
                        {(const void*)mlp_bf16_kernel<false>, (const void*)mlp_bf16_kernel<true>, (const void*)mlp_bf16_kernel<false, true>,
                         (const void*)mlp_bf16_kernel<true, true>, (const void*)mlp_bf16_kernel<false, false, false, true>,
                         (const void*)mlp_bf16_kernel<false, true, false, true>},
                        SMEM_ALLOC, "mlp_bf16", [] { return cudaMemcpyToSymbol(c_steps, S.st, sizeof(TcStage) * MAX_STEPS); });
    if (rc) return rc;
    const int n_rays = (int)(a.P / a.s);
    if (density) {
        if (a.save_img) return fail(INERF_E_ARG, "mlp_bf16: the density-only build has no saving form");
        return mlp_pair_enabled() ? launch<false, true, false, true>(a, n_steps_dens, n_rays, st, "inerf_mlp_fwd[bf16 pair, density only]")
                                  : launch<false, false, false, true>(a, n_steps_dens, n_rays, st, "inerf_mlp_fwd[bf16, density only]");
    }
    if (a.save_img) {
        if (!a.save_mask) return fail(INERF_E_ARG, "mlp_bf16: save_mask is NULL");
        return mlp_pair_enabled() ? launch<true, true, false>(a, S.n_stages, n_rays, st, "inerf_mlp_fwd_train[bf16 pair]")
                                  : launch<true, false, false>(a, S.n_stages, n_rays, st, "inerf_mlp_fwd_train[bf16]");
    }
    return mlp_pair_enabled() ? launch<false, true, false>(a, S.n_stages, n_rays, st, "inerf_mlp_fwd[bf16 pair]")
                              : launch<false, false, false>(a, S.n_stages, n_rays, st, "inerf_mlp_fwd[bf16]");
}

}  // namespace inerf
