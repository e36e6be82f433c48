// FaceNeRF MLP, fp32-GATE tensor-core mode ("fp16x2"): the fused tcgen05 kernel of mlp_bf16.cu with every operand carried as a
// pair of fp16 numbers, x = x_hi + x_lo (22 significant bits), and every product formed by three tensor-core passes
//     A.W  ~=  A_hi.W_hi + A_lo.W_hi + A_hi.W_lo            (the dropped A_lo.W_lo term is 2^-22 relative)
// accumulated in fp32 in tensor memory -- in TWO accumulators: the tensor core adds into its accumulator with truncation (round toward
// zero), one biased rounding of the running sum per MMA, so the small correction passes (lo.hi, hi.lo: 2^-11 of the result) go to their
// own accumulator, where the same truncation is 2^-11 smaller, and the main accumulator only sees the hi.hi passes (a third of the
// roundings); the epilogue adds the two in fp32 with round-to-nearest (Ootomo & Yokota's error-corrected tensor-core GEMM uses the same
// separation).  With one shared accumulator raw was 1e-5 of scale off the fp32 kernel, against 1.5e-6 for exact accumulation of the
// same split operands (CPU emulation).  This is the mode for north_star's "max-abs <= 1e-3 in fp32" gate at tensor-core speed:
// a single-pass bf16 / fp16 / tf32 kernel cannot meet it on the normalised-density preset, whose sigma ~ N(0, 8^2) amplifies operand
// rounding ~100x (bf16 3.4e-2, fp16 = tf32 1.2e-2 max-abs on rgb_map, CPU emulation of the kernel's rounding points on the reference's
// golden render), while the hi/lo split sits at the algorithm's own fp32 rounding floor (3-7e-4; profiles/r02_precision_modes.txt).
//
// Reference arithmetic: models/face_nerf.py:40-80 (fp32 nn.Linear), NeRFs/HeadNeRF/train/audio_exp_nerf.py:332,376-394 (points,
// positional encoding), NeRFs/HeadNeRF/helper.py:174-204.
//
// Structure (differences from mlp_bf16.cu, whose barrier protocol is kept one to one):
//   * a CTA iteration owns ONE 128-row slot; the shared-memory area that holds the second slot there holds the LOW halves here
//     (activations 2 x 64 KB, gamma(p) 2 x 16 KB), so the memory map and the 3 x 16 KB weight ring are unchanged; TMEM columns
//     [0, 256) hold the main accumulator of the layer (both halves), [256, 512) the correction accumulator;
//   * every weight K-block is streamed as two stages, W_hi then W_lo (the packed blob is twice as large: 2.2 MB / net, from L2);
//     per K-block the issuer emits 12 MMAs (M = 128, N = 128 or 64, K = 16): 4 x A_hi.W_hi, 4 x A_lo.W_hi on the first stage,
//     4 x A_hi.W_lo on the second -- three times the tensor work per point of the bf16 kernel;
//   * the eight epilogue warps share the slot: warps 4-7 and 8-11 read the same 32-lane quarters of tensor memory but different
//     column chunks of each layer half; ReLU + split: hi = the value with its low 13 mantissa bits cleared (exact in fp16), lo = the
//     exact fp32 remainder rounded to fp16, both packed with cvt.rn.relu.f16x2; the alpha / rgb heads are fp32 FMAs on the un-split
//     values, their per-group partial sums meet through shared memory once per iteration;
//   * biases enter through one K = 16 MMA per layer half against a tile of fp16 ones with columns (hi, mid, lo) = the folded fp32
//     bias split in three fp16 (exact to 2^-33);
//   * gamma(p): one sincosf per coordinate and octave (30 per point; the bf16 kernel's angle doubling is accurate to ~3.1^f * 2^-22
//     at octave f, not enough here), split into hi / lo like the activations; gamma(viewdir) as a per-ray fp32 bias vector, as in the bf16 kernel.
// Every mbarrier wait is bounded (~2 s) and traps instead of hanging the GPU.
//
// Embedded-row variant (template parameter EMB, FaceNeRF.forward's x (P, 63+27); inference only): mlp_bf16.cu's embedded-row build in
// hi / lo form.  The producer warps split gamma(p) = x[:, 0:63] and gamma(v) = x[:, 63:90] of their row with split_rn2 instead of
// computing them, so any row count works.  There is no per-ray view bias: the 27 view columns of views_linears.0 run as one more K-block
// (W_hi, W_lo stages, 12 MMAs) at the end of each V0 half, its A operand the gamma(v) hi / lo image that the producers write into the PE
// buffer once L5 (the last reader of gamma(p)) has completed; the commit after the last V0 view MMA hands the buffer back for the next
// iteration's gamma(p).  pe_ready / pe_free therefore complete twice per iteration.  Packed blob: INERF_MLP_F16X2_EMB (four more stages).
#include <cuda_fp16.h>

#include "mlp_tc.cuh"

using namespace inerf;
using namespace sm100;

namespace {

constexpr int NSTAGE = 3;
constexpr int STAGE_BYTES = 16384;
// CTA-pair build (PAIR = true, see mlp_bf16.cu): each CTA of a cluster of two holds HALF of the rows of every weight stage; the same 48 KB
// ring is six stages deep
template <bool PAIR> using RingOf = Ring<PAIR, NSTAGE>;
constexpr int MAX_FSTAGES = 160;     // 76 K-block steps x (hi, lo); the embedded-row schedule has 78
constexpr int RMAX = 4;              // rays a 128-row slot can touch (s >= 43)
constexpr int NTHREADS = 512;
constexpr int N_EPI = 256, N_PE = 128;

__constant__ TcStage c_fstages[MAX_FSTAGES];
__constant__ TcStage c_fstages_emb[MAX_FSTAGES];     // the embedded-row schedule (one more K-block per V0 half)
template <bool EMB> __device__ __forceinline__ const TcStage& fstage_at(int s) { return EMB ? c_fstages_emb[s] : c_fstages[s]; }

// smem map (bytes from the 1024-aligned base) -- mlp_bf16.cu's, with [hi|lo] where it has [slot 0|slot 1]
constexpr int OFF_ACT = 0;                               // [2: hi, lo][4 K-blocks][16384]
constexpr int OFF_PE = 131072;                           // [2: hi, lo][16384]
constexpr int OFF_W = 163840;                            // [NSTAGE][16384]
constexpr int OFF_ONES = OFF_W + NSTAGE * STAGE_BYTES;   // 128 x 16 fp16 ones, no-swizzle core-matrix layout
constexpr int OFF_BT = OFF_ONES + 4096;                  // [2][4096] bias tiles
constexpr int OFF_SB = OFF_BT + 2 * 4096;                // alpha_linear.bias, rgb_linear.bias (4 floats)
constexpr int OFF_AW = OFF_SB + 16;                      // alpha_linear.weight 256 floats
constexpr int OFF_RW = OFF_AW + 1024;                    // rgb_linear.weight 3x128 floats
constexpr int OFF_DIRB = OFF_RW + 1536;                  // [RMAX][128] floats
constexpr int OFF_PART = OFF_DIRB + RMAX * 128 * 4;      // [128 rows] float4: head partial sums of epilogue group 1
constexpr int OFF_BAR = OFF_PART + 128 * 16;             // mbarriers
constexpr int SMEM_BYTES = OFF_BAR + 320;
static_assert(SMEM_BYTES <= 232448, "shared memory budget");

struct Bars {
    uint64_t wfull[6], wempty[6];
    uint64_t pfull[6];       // pair build, leader only: the PEER's half of the stage has landed (relayed by the peer's warp 1)
    uint64_t cbar[3];        // C0, C1, C2   (tcgen05.commit, once per layer; pair build: multicast to both CTAs)
    uint64_t ebar[2];        // E0, E1       (8 epilogue warps, once per layer; pair build: the leader's, 8 + 8 warps)
    uint64_t pe_ready, pe_free, dirb_ready, dirb_free;
    uint64_t bfull[2], bempty[2];
    uint64_t pbfull[2];      // pair build, leader only: the peer's half of the bias tile has landed
    uint32_t tmem_base;
};
static_assert(sizeof(Bars) <= 320, "barrier block");

// The MMA issuer's waits sit on the critical path of the tensor pipe (the bf16 kernel lost 3 % when its issuer got the bounded form):
// the issuer polls with the plain try_wait loop; every wait it depends on is made by a warp that IS bounded, so a protocol error still
// ends in a trap of that warp (and the launch failing), not in a hang.
__device__ __forceinline__ void wait_i(uint64_t* bar, uint32_t parity) { mbar_wait(bar, parity); }

__device__ __forceinline__ void wait_b(uint64_t* bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    const long long t0 = clock64();
    uint32_t spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        if ((++spins & 1023u) == 0 && clock64() - t0 > 4000000000LL) __trap();      // a lost arrival must not hang the GPU
    }
}

// kind::f16 instruction descriptor with fp16 A / B (format 0), fp32 D
__host__ __device__ constexpr uint32_t idesc_f16(int M, int N) { return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24); }

constexpr uint32_t CORR_COL = 256;      // first TMEM column of the correction accumulator
// Compensation of the tensor core's accumulation rounding.  tcgen05.mma adds into its fp32 accumulator with round-toward-zero: each of
// the n MMAs that accumulate into the main accumulator of a layer (1 bias MMA + 4 per K-block: 5 for pts_linears.0, 17 for the 256-wide
// layers and views_linears.0, 21 for the skip layer, 9 for views_linears.1-2) shrinks the running sum by half an ulp on average -- a
// multiplicative bias of ~n x 1.8e-8 per layer that adds up coherently over the 11 layers (measured: raw sigma +7.7e-7 of scale off in
// the mean, 3.5e-6 max, against 1.5e-6 max for the fp32 FFMA kernel; profiles/r02_f16x2_comp.txt).  The epilogue adds the two
// accumulators as fma(main, 1 + comp, correction) -- the same instruction count as the plain add -- with comp = n x 2.9e-8 (the expected
// shrink: n/3 ulps of the final sum, a random walk of partial sums) rounded to fp32 ulps of 1.0 (2^-23): 1 for L0, 4 for the 256-wide
// layers, 2 for V0 / V1-2 (V0's theoretical 4 is indistinguishable in the sweep; the landscape is flat to 5 % around this point).  It
// brings raw to 2.0e-6 max / 5e-7 rms of scale, against 1.5e-6 / 3.3e-7 for the FFMA kernel and 3.5e-6 / 1.0e-6 uncompensated.
__host__ __device__ constexpr float tc_comp_ulps(int l) { return l == 0 ? 1.0f : (l < 8 ? 4.0f : 2.0f); }

// (hi, lo) fp16x2 words of two fp32 values, ReLU applied: hi = the value truncated to 11 significant bits, lo = the exact remainder
__device__ __forceinline__ void split_relu2(float v0, float v1, uint32_t& hi2, uint32_t& lo2) {
    const float h0 = __uint_as_float(__float_as_uint(v0) & 0xFFFFE000u), h1 = __uint_as_float(__float_as_uint(v1) & 0xFFFFE000u);
    const float l0 = v0 - h0, l1 = v1 - h1;                     // exact; same sign as the value, so ReLU clears both halves together
    asm("cvt.rn.relu.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(hi2) : "f"(h1), "f"(h0));
    asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(lo2) : "f"(l1), "f"(l0));
}

// round-to-nearest split without ReLU (positional encoding: values in [-1, 1] and the raw coordinates)
__device__ __forceinline__ void split_rn2(float v0, float v1, uint32_t& hi2, uint32_t& lo2) {
    const __half h0 = __float2half_rn(v0), h1 = __float2half_rn(v1);
    const __half l0 = __float2half_rn(v0 - __half2float(h0)), l1 = __float2half_rn(v1 - __half2float(h1));
    hi2 = (uint32_t)__half_as_ushort(h0) | ((uint32_t)__half_as_ushort(h1) << 16);
    lo2 = (uint32_t)__half_as_ushort(l0) | ((uint32_t)__half_as_ushort(l1) << 16);
}

struct IssueCtx {
    Bars* bars;
    uint32_t a_lo, pe_lo, w_lo, hi;
    uint32_t tmem_base;
    uint32_t stage, wpar;
    uint32_t ones_lo, bt_lo, bslot, bpar;
    uint32_t layer_ctr, iter_ctr;
};

// All MMAs of layer L, straight-line: every descriptor offset, wait and commit is a compile-time constant of (L, half, K-block).
// EMB: the embedded-row schedule.  pe_ready and pe_free then complete twice per iteration (gamma(p) for L0 / L5, gamma(v) for V0), so
// the issuer's waits have fixed parities: 0 before L0, 1 before V0's view K-block.
template <int L, bool PAIR, bool EMB = false>
__device__ __forceinline__ void issue_layer(IssueCtx& c) {
    constexpr int NSTAGE = RingOf<PAIR>::N, STAGE_BYTES = RingOf<PAIR>::BYTES;
    constexpr int N = lay_N(L), NH = N / 2, NKB = lay_act_kb(L), CNT = NKB + (lay_x(L, EMB) ? 1 : 0);
    constexpr int KB_PER_HALF_PREV = lay_prev_N(L) / 128;
    constexpr int N_OUT_H0 = NH / 64;
    constexpr int N_FIRST = NKB < N_OUT_H0 ? NKB : N_OUT_H0;
    constexpr uint32_t IDESC = idesc_f16(PAIR ? 256 : 128, NH);
    Bars* bars = c.bars;
    const uint32_t par_prev = (c.layer_ctr - 1) & 1;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
#pragma unroll
        for (int i = 0; i < CNT; ++i) {
            const bool is_pe = (i == NKB);
            if (h == 0 && c.layer_ctr > 0) {
                if (L == 0) {
                    if (i == 0) { wait_ev<PAIR>(&bars->ebar[0], par_prev); wait_ev<PAIR>(&bars->ebar[1], par_prev); }
                } else if (!is_pe) {
                    if (i == 0) wait_ev<PAIR>(&bars->ebar[0], par_prev);
                    if (i == KB_PER_HALF_PREV) wait_ev<PAIR>(&bars->ebar[1], par_prev);
                }
            }
            if (L == 0 && h == 0 && i == 0) wait_ev<PAIR>(&bars->pe_ready, EMB ? 0u : c.iter_ctr & 1);
            if (EMB && L == 8 && h == 0 && is_pe) wait_ev<PAIR>(&bars->pe_ready, 1u);
            const uint32_t d = c.tmem_base + h * NH, dc = d + CORR_COL;      // main / correction accumulator
            const uint32_t a_hi = is_pe ? c.pe_lo : c.a_lo + i * (16384 >> 4);
            const uint32_t a_lo = is_pe ? c.pe_lo + (16384 >> 4) : c.a_lo + (65536 >> 4) + i * (16384 >> 4);
            // ---- stage 1: W_hi -- A_hi.W_hi -> main, A_lo.W_hi -> correction ------------------------------------------------
            wait_i(&bars->wfull[c.stage], c.wpar);
            if constexpr (PAIR) mbar_wait_cluster(&bars->pfull[c.stage], c.wpar);
            if (i == 0) {
                wait_i(&bars->bfull[c.bslot], c.bpar);
                if constexpr (PAIR) mbar_wait_cluster(&bars->pbfull[c.bslot], c.bpar);
            }
            tc_fence_after();
            if (elect_one()) {
                if (i == 0) {      // bias: D = ones[128x16] . tile[NHx16]^T, tile columns (hi, mid, lo, 0, ...); overwrites the accumulator
                    umma_any<PAIR>(d, c.ones_lo, c.bt_lo + c.bslot * (4096 >> 4), HI_NOSWZ, IDESC, 0u);
                    commit_any<PAIR>(&bars->bempty[c.bslot]);
                }
                const uint32_t b = c.w_lo + c.stage * (STAGE_BYTES >> 4);
#pragma unroll
                for (int k = 0; k < 4; ++k) umma_any<PAIR>(d, a_hi + 2 * k, b + 2 * k, c.hi, IDESC, 1u);
#pragma unroll
                for (int k = 0; k < 4; ++k) umma_any<PAIR>(dc, a_lo + 2 * k, b + 2 * k, c.hi, IDESC, (i == 0 && k == 0) ? 0u : 1u);
                commit_any<PAIR>(&bars->wempty[c.stage]);
            }
            __syncwarp();
            if (i == 0) { c.bslot ^= 1; if (c.bslot == 0) c.bpar ^= 1; }
            if (++c.stage == NSTAGE) { c.stage = 0; c.wpar ^= 1; }
            // ---- stage 2: W_lo -- A_hi.W_lo -> correction -------------------------------------------------------------------
            wait_i(&bars->wfull[c.stage], c.wpar);
            if constexpr (PAIR) mbar_wait_cluster(&bars->pfull[c.stage], c.wpar);
            tc_fence_after();
            if (elect_one()) {
                const uint32_t b = c.w_lo + c.stage * (STAGE_BYTES >> 4);
#pragma unroll
                for (int k = 0; k < 4; ++k) umma_any<PAIR>(dc, a_hi + 2 * k, b + 2 * k, c.hi, IDESC, 1u);
                commit_any<PAIR>(&bars->wempty[c.stage]);
                const bool last = (i == CNT - 1);
                if (h == 0 && last) commit_any<PAIR>(&bars->cbar[0]);
                if (h == 1 && (N_FIRST > 0 ? i == N_FIRST - 1 : last)) commit_any<PAIR>(&bars->cbar[1]);
                if (h == 1 && last) commit_any<PAIR>(&bars->cbar[2]);
                if (h == 1 && last && (L == 5 || (EMB && L == 8))) commit_any<PAIR>(&bars->pe_free);
            }
            __syncwarp();
            if (++c.stage == NSTAGE) { c.stage = 0; c.wpar ^= 1; }
        }
    }
    ++c.layer_ctr;
}

// Sixteen columns of an epilogue: main + correction accumulator (fp32, round to nearest), then
// KIND 0: plain; 1: + alpha_linear partial (L7); 2: + per-ray view bias (V0); 3: + rgb_linear partial (V2); ReLU and hi / lo split
template <int KIND>
__device__ __forceinline__ void epi16(const uint32_t (&r)[16], const uint32_t (&rc)[16], uint32_t* __restrict__ ph, uint32_t* __restrict__ pl,
                                      const float* __restrict__ dsrc, const float* __restrict__ aw, const float* __restrict__ rw,
                                      float& alpha, float& rgb0, float& rgb1, float& rgb2, const float ms) {
#pragma unroll
    for (int j = 0; j < 16; j += 4) {
        float v[4] = {fmaf(__uint_as_float(r[j]), ms, __uint_as_float(rc[j])), fmaf(__uint_as_float(r[j + 1]), ms, __uint_as_float(rc[j + 1])),
                      fmaf(__uint_as_float(r[j + 2]), ms, __uint_as_float(rc[j + 2])), fmaf(__uint_as_float(r[j + 3]), ms, __uint_as_float(rc[j + 3]))};
        if constexpr (KIND == 2) {
            const float4 d = *reinterpret_cast<const float4*>(dsrc + j);
            v[0] += d.x; v[1] += d.y; v[2] += d.z; v[3] += d.w;
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
        split_relu2(v[0], v[1], ph[j >> 1], pl[j >> 1]);
        split_relu2(v[2], v[3], ph[(j >> 1) + 1], pl[(j >> 1) + 1]);
    }
}

// PAIR = true: clusters of two CTAs, one tcgen05.mma.cta_group::2 over the 2 x 128 rows of the pair, the weight stages split across the
// pair (the bf16 kernel's pair build, mlp_bf16.cu; a pair iteration is two 128-point slots, CTA r takes slot 2 it + r).
// EMB = true: rows of a.x (P, 90) with the INERF_MLP_F16X2_EMB schedule (see the header).
template <bool PAIR, bool EMB = false>
__global__ void __launch_bounds__(NTHREADS, 1) mlp_f16x2_kernel(MlpArgs a, int n_stages, int n_rays) {
    constexpr int NSTAGE = RingOf<PAIR>::N, STAGE_BYTES = RingOf<PAIR>::BYTES;
    extern __shared__ __align__(1024) uint8_t sm[];
    if ((smem_u32(sm) & 1023u) != 0) __trap();
    Bars* bars = reinterpret_cast<Bars*>(sm + OFF_BAR);
    float* s_sb = reinterpret_cast<float*>(sm + OFF_SB);
    float* s_aw = reinterpret_cast<float*>(sm + OFF_AW);
    float* s_rw = reinterpret_cast<float*>(sm + OFF_RW);
    float* s_dirb = reinterpret_cast<float*>(sm + OFF_DIRB);
    float4* s_part = reinterpret_cast<float4*>(sm + OFF_PART);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t rank = PAIR ? cluster_ctarank() : 0u;
    const long long n_iter = PAIR ? (a.P + 255) / 256 : (a.P + 127) / 128;
    const long long it_first = PAIR ? (long long)(blockIdx.x >> 1) : (long long)blockIdx.x;
    const long long it_step = PAIR ? (long long)(gridDim.x >> 1) : (long long)gridDim.x;
#define SLOT_OF(it_) (PAIR ? 2 * (it_) + (long long)rank : (it_))

    // ---- one-time setup -------------------------------------------------------------------
    if (tid < 4) s_sb[tid] = a.cond[8 * 256 + 3 * 128 + tid];
    for (int i = tid; i < 256; i += NTHREADS)                 // fp16 1.0 = 0x3C00
        reinterpret_cast<uint4*>(sm + OFF_ONES)[i] = make_uint4(0x3C003C00u, 0x3C003C00u, 0x3C003C00u, 0x3C003C00u);
    fence_proxy_async_smem();
    for (int i = tid; i < 256; i += NTHREADS) s_aw[i] = a.w[P_ALPHA_W][i];
    for (int i = tid; i < 384; i += NTHREADS) s_rw[i] = a.w[P_RGB_W][i];
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
    if constexpr (PAIR) cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = bars->tmem_base;

    if (warp == 0) {
        // ================= weight producer ==================================================
        if (lane == 0) {
            const uint8_t* blob = reinterpret_cast<const uint8_t*>(a.packed);
            const uint8_t* tiles = reinterpret_cast<const uint8_t*>(a.cond + COND_FLOATS) + BIAS_TILE_BYTES;      // after the bf16 tile set
            uint32_t g = 0, bh = 0;
            constexpr uint32_t SPLIT = PAIR ? 2u : 1u;      // pair build: this CTA's half of the rows of every stage / bias tile
            for (long long it = it_first; it < n_iter; it += it_step) {
                for (int s = 0; s < n_stages; ++s, ++g) {
                    const uint32_t stage = g % NSTAGE, round = g / NSTAGE;
                    const TcStage fs = fstage_at<EMB>(s);
                    if (fs.first) {
                        const uint32_t slot = bh & 1, l = fs.layer, h = fs.half;
                        const uint32_t bytes = (uint32_t)fs.n8 * 8u * 32u / SPLIT;
                        const uint32_t off = bias_tile_offset(l, h) + rank * bytes;
                        wait_b(&bars->bempty[slot], ((bh >> 1) & 1) ^ 1);
                        mbar_arrive_expect_tx(&bars->bfull[slot], bytes);
                        bulk_g2s(sm + OFF_BT + slot * 4096, tiles + off, bytes, &bars->bfull[slot]);
                        ++bh;
                    }
                    wait_b(&bars->wempty[stage], (round & 1) ^ 1);
                    const uint32_t bytes = (uint32_t)fs.n8 * 8u * 128u / SPLIT;
                    mbar_arrive_expect_tx(&bars->wfull[stage], bytes);
                    bulk_g2s(sm + OFF_W + stage * STAGE_BYTES, blob + fs.offset + rank * bytes, bytes, &bars->wfull[stage]);
                }
            }
        }
    } else if (warp == 1 && PAIR && rank != 0) {
        // ================= relay (peer CTA of a pair): tell the leader when MY half of a bias tile / weight stage has landed =========
        if (lane == 0) {
            uint32_t g = 0, bh = 0;
            for (long long it = it_first; it < n_iter; it += it_step)
                for (int s = 0; s < n_stages; ++s, ++g) {
                    if (fstage_at<EMB>(s).first) {
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
            issue_layer<0, PAIR, EMB>(c);
#pragma unroll 1
            for (int seg = 0; seg < 2; ++seg) {
#pragma unroll 1
                for (int r = 0; r < (seg ? 2 : 4); ++r) issue_layer<1, PAIR, EMB>(c);
                if (seg == 0) issue_layer<5, PAIR, EMB>(c);
            }
            issue_layer<8, PAIR, EMB>(c);
#pragma unroll 1
            for (int r = 0; r < 2; ++r) issue_layer<9, PAIR, EMB>(c);
        }
    } else if (warp >= 4 && warp < 12) {
        // ================= epilogue: one row per thread, the two warp groups split the column chunks ======================
        const int grp = (warp - 4) >> 2;
        const int row = ((warp & 3) << 5) + lane;
        const uint32_t t_lane = tmem_base + ((uint32_t)((warp & 3) << 5) << 16);
        uint8_t* act = sm + OFF_ACT;
        const uint32_t row_off = (row >> 3) * 1024 + (row & 7) * 128;
        const uint32_t rsw = row & 7;
        uint32_t layer_ctr = 0, iter_ctr = 0;
        for (long long it = it_first; it < n_iter; it += it_step, ++iter_ctr) {
            const long long p0 = SLOT_OF(it) * 128;
            long long p = p0 + row;
            const bool in_range = p < a.P;
            if (!in_range) p = a.P - 1;
            const int ray_local = EMB ? 0 : (int)(p / a.s - min(p0, a.P - 1) / a.s);      // embedded rows: no per-ray view bias
            float alpha = 0.f, rgb0 = 0.f, rgb1 = 0.f, rgb2 = 0.f;
            for (int l = 0; l < 11; ++l, ++layer_ctr) {
                const int NH = (l < 8 ? 256 : 128) >> 1;
                const int npg = NH >> 6;                       // chunks per group and half: 2 (N = 256) or 1 (N = 128)
                const uint32_t par = layer_ctr & 1;
                // 1 + tc_comp_ulps(l) ulps of 1.0, exactly.  Written as float arithmetic the same value let the compiler specialise the
                // epilogue per scale: 3 % slower (profiles/r13_scaffolding_removal_ab.txt)
                const float ms = __uint_as_float(0x3F800000u + (uint32_t)tc_comp_ulps(l));
                if (!EMB && l == 8) wait_b(&bars->dirb_ready, iter_ctr & 1);
#pragma unroll 1
                for (int h = 0; h < 2; ++h) {
                    wait_b(&bars->cbar[h == 0 ? 0 : 2], par);
                    __syncwarp();
                    tc_fence_after();
                    uint32_t ph[32], pl[32];
#pragma unroll
                    for (int cc = 0; cc < 2; ++cc) {
                        if (cc < npg) {
                            const int f0 = h * NH + (grp * npg + cc) * 32;       // first output feature of the chunk
#pragma unroll
                            for (int q16 = 0; q16 < 2; ++q16) {
                                const int f = f0 + q16 * 16;
                                uint32_t r[16], rc[16];
                                tmem_ld16(t_lane + f, r);
                                tmem_ld16(t_lane + CORR_COL + f, rc);
                                tmem_wait_ld();
                                uint32_t* oh = &ph[cc * 16 + q16 * 8];
                                uint32_t* ol = &pl[cc * 16 + q16 * 8];
                                switch (l) {
                                    case 7: epi16<1>(r, rc, oh, ol, nullptr, s_aw + f, nullptr, alpha, rgb0, rgb1, rgb2, ms); break;
                                    case 8:
                                        if constexpr (EMB) epi16<0>(r, rc, oh, ol, nullptr, nullptr, nullptr, alpha, rgb0, rgb1, rgb2, ms);
                                        else epi16<2>(r, rc, oh, ol, s_dirb + ray_local * 128 + f, nullptr, nullptr, alpha, rgb0, rgb1, rgb2, ms);
                                        break;
                                    case 10: epi16<3>(r, rc, oh, ol, nullptr, nullptr, s_rw + f, alpha, rgb0, rgb1, rgb2, ms); break;
                                    default: epi16<0>(r, rc, oh, ol, nullptr, nullptr, nullptr, alpha, rgb0, rgb1, rgb2, ms); break;
                                }
                            }
                        }
                    }
                    tc_fence_before();
                    if (l != 10) {
                        if (h == 0) wait_b(&bars->cbar[1], par);      // h1 has finished reading the K-blocks written below
                        __syncwarp();
#pragma unroll
                        for (int cc = 0; cc < 2; ++cc) {
                            if (cc < npg) {
                                const int f0 = h * NH + (grp * npg + cc) * 32;
                                uint8_t* kb = act + (f0 >> 6) * 16384 + row_off;
                                const int ch0 = (f0 & 63) >> 3;
#pragma unroll
                                for (int q = 0; q < 4; ++q) {
                                    const uint32_t o = ((ch0 + q) ^ rsw) << 4;
                                    *reinterpret_cast<uint4*>(kb + o) =
                                        make_uint4(ph[cc * 16 + q * 4], ph[cc * 16 + q * 4 + 1], ph[cc * 16 + q * 4 + 2], ph[cc * 16 + q * 4 + 3]);
                                    *reinterpret_cast<uint4*>(kb + 65536 + o) =
                                        make_uint4(pl[cc * 16 + q * 4], pl[cc * 16 + q * 4 + 1], pl[cc * 16 + q * 4 + 2], pl[cc * 16 + q * 4 + 3]);
                                }
                            }
                        }
                        fence_proxy_async_smem();
                    }
                    __syncwarp();
                    if (lane == 0) { if constexpr (PAIR) mbar_arrive_remote(&bars->ebar[h], 0); else mbar_arrive(&bars->ebar[h]); }
                }
                if (!EMB && l == 8) {
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&bars->dirb_free);
                }
            }
            // The two groups hold partial sums of the heads: group 1 hands its part over through shared memory.  One buffer is enough:
            // group 1 writes it again only after the next iteration's layers, whose E barriers need group 0's arrivals, i.e. after
            // group 0 has read it.
            float4* part = s_part;
            if (grp == 1) part[row] = make_float4(rgb0, rgb1, rgb2, alpha);
            named_bar_sync(1, N_EPI);
            if (grp == 0 && in_range) {
                const float4 q = part[row];
                float4 o;
                o.x = (rgb0 + q.x) + s_sb[1];
                o.y = (rgb1 + q.y) + s_sb[2];
                o.z = (rgb2 + q.z) + s_sb[3];
                o.w = (alpha + q.w) + s_sb[0];
                reinterpret_cast<float4*>(a.out)[p] = o;
            }
        }
    } else if (EMB && warp >= 12) {
        // ================= embedded rows: gamma(p), then gamma(v), of row t of the slot, split from x into the PE buffer ==========
        // A row of x is 90 floats (360 B; 8-byte aligned when x is 16-byte aligned): gamma(p) = columns 0..62 (image column 63 zero),
        // gamma(v) = columns 63..89 (image columns 27..63 zero); each value is split into its fp16 hi / lo pair.  Each block is in
        // registers before the wait for the buffer, so only the shared-memory stores lie between its release and the pe_ready arrival.
        // pe_free parities: 0 = L5 has read gamma(p) of this iteration, 1 = V0 has read gamma(v) of the previous one.
        const int t = tid - 12 * 32;
        uint8_t* dst = sm + OFF_PE + (t >> 3) * 1024 + (t & 7) * 128;
        auto store_and_arrive = [&](const uint32_t* wh, const uint32_t* wl, int n_chunks) {      // one row of both images, zero-padded
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const uint32_t o = (q ^ (t & 7)) << 4;
                const bool v = q < n_chunks;
                *reinterpret_cast<uint4*>(dst + o) = v ? make_uint4(wh[4 * q], wh[4 * q + 1], wh[4 * q + 2], wh[4 * q + 3]) : make_uint4(0u, 0u, 0u, 0u);
                *reinterpret_cast<uint4*>(dst + 16384 + o) =
                    v ? make_uint4(wl[4 * q], wl[4 * q + 1], wl[4 * q + 2], wl[4 * q + 3]) : make_uint4(0u, 0u, 0u, 0u);
            }
            fence_proxy_async_smem();
            if constexpr (PAIR) {
                __syncwarp();
                if (lane == 0) mbar_arrive_remote(&bars->pe_ready, 0);
            } else {
                mbar_arrive(&bars->pe_ready);
            }
        };
        for (long long it = it_first; it < n_iter; it += it_step) {
            long long p = SLOT_OF(it) * 128 + t;
            if (p > a.P - 1) p = a.P - 1;
            const float* xr = a.x + p * 90;
            uint32_t pkh[32], pkl[32];
#pragma unroll
            for (int j = 0; j < 31; ++j) {
                const float2 v = __ldg(reinterpret_cast<const float2*>(xr) + j);
                split_rn2(v.x, v.y, pkh[j], pkl[j]);
            }
            split_rn2(__ldg(xr + 62), 0.f, pkh[31], pkl[31]);
            if (it != it_first) wait_b(&bars->pe_free, 1u);
            store_and_arrive(pkh, pkl, 8);
            uint32_t pvh[16], pvl[16];
            {
                float g[28];
                g[0] = __ldg(xr + 63);
#pragma unroll
                for (int j = 0; j < 13; ++j) {
                    const float2 v = __ldg(reinterpret_cast<const float2*>(xr + 64) + j);
                    g[1 + 2 * j] = v.x; g[2 + 2 * j] = v.y;
                }
                g[27] = 0.f;
#pragma unroll
                for (int j = 0; j < 14; ++j) split_rn2(g[2 * j], g[2 * j + 1], pvh[j], pvl[j]);
                pvh[14] = pvh[15] = pvl[14] = pvl[15] = 0u;
            }
            wait_b(&bars->pe_free, 0u);
            store_and_arrive(pvh, pvl, 4);
        }
    } else if (warp >= 12) {
        // ================= positional encoding + per-ray view bias producers ==================
        const int t = tid - 12 * 32;                 // 0..127: row of the slot, and output feature of the view bias
        float wdir[27];
        {
            const float* wrow = a.w[P_VIEWS_W] + (size_t)t * (283 + a.dim_expr) + 256;
#pragma unroll
            for (int j = 0; j < 27; ++j) wdir[j] = wrow[j];
        }
        uint32_t iter_ctr = 0;
        for (long long it = it_first; it < n_iter; it += it_step, ++iter_ctr) {
            // ---- gamma_10(o + d z) of row t, every octave with its own sincosf (2^k scaling is exact) -----------------------
            uint32_t pkh[32], pkl[32];
            {
                long long p = SLOT_OF(it) * 128 + t;
                if (p > a.P - 1) p = a.P - 1;
                const long long ray = p / a.s;
                const float* r = a.rays + ray * a.ray_stride;
                const float zz = a.z[p];
                float v[64];
#pragma unroll
                for (int c = 0; c < 3; ++c) v[c] = __fadd_rn(r[c], __fmul_rn(r[3 + c], zz));
#pragma unroll
                for (int f = 0; f < 10; ++f)
#pragma unroll
                    for (int c = 0; c < 3; ++c) {
                        float sn, cs;
                        sincosf(v[c] * (float)(1 << f), &sn, &cs);
                        v[3 + 6 * f + c] = sn;
                        v[6 + 6 * f + c] = cs;
                    }
                v[63] = 0.f;
#pragma unroll
                for (int j = 0; j < 32; ++j) split_rn2(v[2 * j], v[2 * j + 1], pkh[j], pkl[j]);
            }
            if (iter_ctr > 0) wait_b(&bars->pe_free, (iter_ctr - 1) & 1);
            {
                uint8_t* dst = sm + OFF_PE + (t >> 3) * 1024 + (t & 7) * 128;
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const uint32_t o = (q ^ (t & 7)) << 4;
                    *reinterpret_cast<uint4*>(dst + o) = make_uint4(pkh[4 * q], pkh[4 * q + 1], pkh[4 * q + 2], pkh[4 * q + 3]);
                    *reinterpret_cast<uint4*>(dst + 16384 + o) = make_uint4(pkl[4 * q], pkl[4 * q + 1], pkl[4 * q + 2], pkl[4 * q + 3]);
                }
            }
            fence_proxy_async_smem();
            if constexpr (PAIR) {
                __syncwarp();
                if (lane == 0) mbar_arrive_remote(&bars->pe_ready, 0);
            } else {
                mbar_arrive(&bars->pe_ready);
            }
            // ---- per-ray view bias: lane q < RMAX encodes ray q of the slot, the warp shares it by shuffle ----
            {
                float enc[27];
                if (lane < RMAX) {
                    long long pfirst = SLOT_OF(it) * 128;
                    if (pfirst > a.P - 1) pfirst = a.P - 1;
                    long long ray = pfirst / a.s + lane;
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
                if (iter_ctr > 0) wait_b(&bars->dirb_free, (iter_ctr - 1) & 1);
                for (int q2 = 0; q2 < RMAX; ++q2) {
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
#undef SLOT_OF
}

}  // namespace

namespace inerf {

int mlp_f16x2_packed_bytes(const InerfNetDims* d, size_t* bytes, bool embedded) {
    *bytes = (size_t)build_tc_schedule(d, embedded, 2).total_bytes;
    return INERF_OK;
}

int mlp_f16x2_pack(const InerfNetDims* d, const float* const* params_host, void* packed, cudaStream_t st, bool embedded) {
    return pack_tc_schedule<true>(build_tc_schedule(d, embedded, 2), params_host, packed, st, "inerf_mlp_pack[fp16x2]");
}

int mlp_f16x2_launch(const MlpArgs& a, bool embedded, cudaStream_t st) {
    if (embedded) {
        if (((uintptr_t)a.packed | (uintptr_t)a.x) & 15) return fail(INERF_E_ALIGN, "inerf_mlp_fwd_embedded: packed weights and x must be 16-byte aligned");
    } else {
        if (a.s < 43) return fail(INERF_E_UNSUPPORTED, "fp16x2 mode needs at least 43 samples per ray (a 128-row slot may touch at most 4 rays)");
        if ((uintptr_t)a.packed & 15) return fail(INERF_E_ALIGN, "inerf_mlp_fwd: packed weights must be 16-byte aligned");
    }
    static thread_local int configured_dev = -1;
    // offsets do not depend on the conditioning dims
    static const TcSchedule S = [] { InerfNetDims d{64, 76, 32, 256, 8, 63, 27}; return build_tc_schedule(&d, false, 2); }();
    static const TcSchedule SE = [] { InerfNetDims d{64, 76, 32, 256, 8, 63, 27}; return build_tc_schedule(&d, true, 2); }();
    int rc = setup_once(configured_dev,
                        {(const void*)mlp_f16x2_kernel<false>, (const void*)mlp_f16x2_kernel<true>, (const void*)mlp_f16x2_kernel<false, true>,
                         (const void*)mlp_f16x2_kernel<true, true>},
                        SMEM_BYTES, "mlp_f16x2", [] {
                            cudaError_t e = cudaMemcpyToSymbol(c_fstages, S.st, sizeof(TcStage) * MAX_FSTAGES);
                            return e == cudaSuccess ? cudaMemcpyToSymbol(c_fstages_emb, SE.st, sizeof(TcStage) * MAX_FSTAGES) : e;
                        });
    if (rc) return rc;
    const int n_stages = embedded ? SE.n_stages : S.n_stages;
    const int n_rays = embedded ? 0 : (int)(a.P / a.s);
    const bool pair = mlp_pair_enabled();
    const auto kernel = pair ? (embedded ? mlp_f16x2_kernel<true, true> : mlp_f16x2_kernel<true>)
                             : (embedded ? mlp_f16x2_kernel<false, true> : mlp_f16x2_kernel<false>);
    const char* what = embedded ? (pair ? "inerf_mlp_fwd_embedded[fp16x2 pair]" : "inerf_mlp_fwd_embedded[fp16x2]")
                                : (pair ? "inerf_mlp_fwd[fp16x2 pair]" : "inerf_mlp_fwd[fp16x2]");
    return launch_tc(kernel, pair, (a.P + 127) / 128, NTHREADS, SMEM_BYTES, st, what, a, n_stages, n_rays);
}

}  // namespace inerf
