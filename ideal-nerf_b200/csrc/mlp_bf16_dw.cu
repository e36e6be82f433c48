// FaceNeRF backward, bf16 tensor-core mode, weight gradients:  dW_l[n][k] = sum_p delta_l[p][n] * X_l[p][k],  db_l[n] = sum_p delta_l[p][n].
//
// Reference: torch.autograd of models/face_nerf.py:40-80 inside loss.backward() (NeRFs/HeadNeRF/train/audio_exp_nerf.py:549).
//
// Both operands are stored POINT-major, as the 16 KB images [128 points][64 features] (bf16, 128-byte swizzle) the forward and chain
// kernels keep in shared memory (mlp_common.cuh, TRAIN_IMGS per 128-point tile).  Read as MN-major UMMA operands they are exactly
// delta^T and X: M = the delta features, N = the X features, K = the points, so dW is one long-K tcgen05 GEMM per (layer, 128 delta
// features) with NO transposition pass: D[128 x N] (fp32, TMEM) accumulates over a range of tiles, then goes to the nn.Linear-layout
// gradient with fp32 reductions (red.global.add).  db comes from one extra N = 16 MMA per K step against a tile of ones.
//
// Work items = (task, range of tiles), handed out through an atomic counter; one CTA = producer warp (cp.async.bulk of the A / B
// images, 2 x 96 KB stages), issuer warp, 4 epilogue warps.  HBM bound: 48-96 KB per 128 points per task against 8 MMAs.
#include <cuda_bf16.h>

#include "mlp_common.cuh"
#include "sm100_ptx.cuh"

using namespace inerf;
using namespace sm100;

namespace {

constexpr int DW_THREADS = 192;
constexpr int STAGE_A = 32768, STAGE_B = 65536, STAGE = STAGE_A + STAGE_B, NST = 2;
constexpr int OFF_ONES = NST * STAGE;              // 16 x 16 bf16 ones, K-major no-swizzle (512 B)
constexpr int OFF_BARS = OFF_ONES + 512;
constexpr int DW_SMEM = OFF_BARS + 128;
constexpr int MAX_TASKS = 32;

struct DwTask {
    int a_img;          // first delta image of the A block (2 consecutive images = 128 delta features)
    int b_img, b_imgs;  // first X image and how many (N = 64 * b_imgs)
    int w_index, ldw, wcol, kvalid;     // gradient tensor, its leading dimension, first column, valid columns of N
    int row_lo, row_hi, out_row0;       // D rows [row_lo, row_hi) go to gradient rows out_row0 + (row - row_lo)
    int bias_index;                     // gradient tensor of the bias (or -1)
};

struct DwArgs {
    const uint8_t* delta_img;
    const uint8_t* acts_img;
    float* g[INERF_N_PARAMS];
    DwTask task[MAX_TASKS];
    int n_tasks, n_chunks, tiles_per_chunk;
    long long n_tiles;
    int* counter;
};

__device__ __forceinline__ uint32_t desc_lo_mn(uint32_t smem_addr) { return ((smem_addr & 0x3FFFF) >> 4) | ((16384u >> 4) << 16); }
constexpr uint32_t HI_MN_SW128 = (1024u >> 4) | (1u << 14) | ((uint32_t)SWIZZLE_128B << 29);

__device__ __forceinline__ void umma_lohi(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
        "mov.b64 da, {%1, %2};\n\tmov.b64 db, {%3, %4};\n\t"
        "setp.ne.b32 p, %6, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}" ::"r"(tmem_d),
        "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(acc)
        : "memory");
}

__device__ __forceinline__ void bounded_wait(uint64_t* bar, uint32_t parity) {
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity))
        if (clock64() - t0 > 8000000000LL) __trap();          // ~4 s: a lost arrival must not hang the GPU
}

struct DwBars {
    uint64_t full[NST], empty[NST];
    uint64_t done;          // all MMAs of the item complete
    uint64_t drained;       // epilogue has read the accumulators (4 warps)
    uint32_t tmem_base;
    int item;               // broadcast of the work counter
};

static_assert(sizeof(DwArgs) <= 4000, "kernel parameter space");
// The task table is a kernel parameter (by value): no copy from pageable host memory, so the launch is graph-capturable.
__global__ void __launch_bounds__(DW_THREADS, 1) mlp_bf16_dw_kernel(const __grid_constant__ DwArgs a) {
    extern __shared__ __align__(1024) uint8_t sm[];
    if ((smem_u32(sm) & 1023u) != 0) __trap();
    DwBars* bars = reinterpret_cast<DwBars*>(sm + OFF_BARS);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    for (int i = tid; i < 32; i += DW_THREADS)
        reinterpret_cast<uint4*>(sm + OFF_ONES)[i] = make_uint4(0x3F803F80u, 0x3F803F80u, 0x3F803F80u, 0x3F803F80u);
    fence_proxy_async_smem();
    if (tid == 0) {
        for (int s = 0; s < NST; ++s) { mbar_init(&bars->full[s], 1); mbar_init(&bars->empty[s], 1); }
        mbar_init(&bars->done, 1);
        mbar_init(&bars->drained, 4);
        fence_mbar_init();
    }
    if (warp == 2) { tmem_alloc(&bars->tmem_base, 512); tmem_relinquish(); }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = bars->tmem_base;
    const int n_items = a.n_tasks * a.n_chunks;

    uint32_t g = 0, n_done = 0;           // stage counter (producer and issuer advance it identically), items finished by this CTA
    while (true) {
        // ---- next work item (all warps agree through shared memory) -----------------------------------------------------
        __syncthreads();
        if (tid == 0) bars->item = atomicAdd(a.counter, 1);
        __syncthreads();
        const int item = bars->item;
        if (item >= n_items) break;
        const int chunk = item / a.n_tasks;
        const DwTask& t = a.task[item - chunk * a.n_tasks];
        const long long t0 = (long long)chunk * a.tiles_per_chunk;
        const long long t1 = min(a.n_tiles, t0 + a.tiles_per_chunk);
        const int N = 64 * t.b_imgs;

        if (warp == 0) {
            // ================= producer ===========================================================================
            if (lane == 0) {
                for (long long tile = t0; tile < t1; ++tile, ++g) {
                    const uint32_t s = g % NST, round = g / NST;
                    bounded_wait(&bars->empty[s], (round & 1) ^ 1);
                    const uint32_t bytes_b = (uint32_t)t.b_imgs * 16384u;
                    mbar_arrive_expect_tx(&bars->full[s], STAGE_A + bytes_b);
                    bulk_g2s(sm + s * STAGE, a.delta_img + ((size_t)tile * TRAIN_IMGS + t.a_img) * 16384, STAGE_A, &bars->full[s]);
                    bulk_g2s(sm + s * STAGE + STAGE_A, a.acts_img + ((size_t)tile * TRAIN_IMGS + t.b_img) * 16384, bytes_b, &bars->full[s]);
                }
            } else {
                g += (uint32_t)(t1 - t0);
            }
            g = __shfl_sync(0xffffffffu, g, 0);
        } else if (warp == 1) {
            // ================= MMA issuer ===========================================================================
            // D (cols 0..N-1) and the column sums (cols 256..271) are overwritten by the first K step: wait until the epilogue
            // of the previous item has drained them
            if (n_done > 0) bounded_wait(&bars->drained, (n_done - 1) & 1);
            tc_fence_after();
            const uint32_t idesc = umma_idesc_bf16(128, N) | (1u << 15) | (1u << 16);       // A, B MN-major
            const uint32_t idesc_b = umma_idesc_bf16(128, 16) | (1u << 15);                  // A MN-major, ones K-major
            const uint32_t ones_lo = ((smem_u32(sm + OFF_ONES) & 0x3FFFF) >> 4) | ((128u >> 4) << 16);
            for (long long tile = t0; tile < t1; ++tile, ++g) {
                const uint32_t s = g % NST, round = g / NST;
                bounded_wait(&bars->full[s], round & 1);
                tc_fence_after();
                if (elect_one()) {
                    const uint32_t a_lo = desc_lo_mn(smem_u32(sm + s * STAGE)), b_lo = desc_lo_mn(smem_u32(sm + s * STAGE + STAGE_A));
#pragma unroll
                    for (int k = 0; k < 8; ++k) {          // 16 points per step: 2 x 8 rows of 128 B = 2048 B
                        const uint32_t acc = (tile == t0 && k == 0) ? 0u : 1u;
                        umma_lohi(tmem_base, a_lo + k * 128, HI_MN_SW128, b_lo + k * 128, HI_MN_SW128, idesc, acc);
                        umma_lohi(tmem_base + 256, a_lo + k * 128, HI_MN_SW128, ones_lo, HI_NOSWZ, idesc_b, acc);
                    }
                    umma_commit(&bars->empty[s]);
                    if (tile == t1 - 1) umma_commit(&bars->done);
                }
                __syncwarp();
            }
        } else {
            // ================= epilogue: TMEM -> fp32 reductions into the nn.Linear-layout gradients ==================
            const int q = warp & 3;                                        // TMEM lane quarter this warp may read
            const int row = q * 32 + lane;
            bounded_wait(&bars->done, n_done & 1);
            tc_fence_after();
            // The accumulator arrives one ROW per lane; reducing it into the gradient from there would make every red.add touch 32
            // different rows (32 sectors per instruction, ~20 us per work item).  So each warp first parks its 32 rows in the (now idle)
            // stage buffers -- [32][N + 4] fp32, the 16-byte pad keeps the 128-bit stores of 8 consecutive rows on distinct banks --
            // and then walks them row by row with the lanes across 32 consecutive columns: fully coalesced reductions.
            float* park = reinterpret_cast<float*>(sm) + (size_t)q * 32 * (256 + 4);
            const int ldp = N + 4;
            const uint32_t t_lane = tmem_base + ((uint32_t)(q * 32) << 16);
            for (int c0 = 0; c0 < N; c0 += 32) {
                uint32_t r[32];
                tmem_ld32(t_lane + c0, r);
                tmem_wait_ld();
#pragma unroll
                for (int j = 0; j < 32; j += 4)
                    *reinterpret_cast<uint4*>(park + lane * ldp + c0 + j) = make_uint4(r[j], r[j + 1], r[j + 2], r[j + 3]);
            }
            __syncwarp();
            for (int rr = 0; rr < 32; ++rr) {
                const int orow = q * 32 + rr;
                if (orow < t.row_lo || orow >= t.row_hi) continue;      // warp-uniform
                float* G = a.g[t.w_index] + (size_t)(t.out_row0 + orow - t.row_lo) * t.ldw + t.wcol;
                const float* src = park + rr * ldp;
                for (int c0 = 0; c0 < N; c0 += 32)
                    if (c0 + lane < t.kvalid) atomicAdd(G + c0 + lane, src[c0 + lane]);
            }
            const bool row_ok = row >= t.row_lo && row < t.row_hi;
            if (t.bias_index >= 0) {
                uint32_t r[32];
                tmem_ld32(t_lane + 256, r);          // 16 valid columns, all equal to the column sum; read 32 (allocated) and use [0]
                tmem_wait_ld();
                if (row_ok) atomicAdd(a.g[t.bias_index] + t.out_row0 + row - t.row_lo, __uint_as_float(r[0]));
            }
            tc_fence_before();
            fence_proxy_async_smem();      // the parked rows were generic-proxy accesses to buffers the next bulk loads (async proxy) overwrite
            __syncwarp();
            if (lane == 0) mbar_arrive(&bars->drained);
        }
        ++n_done;
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) tmem_dealloc(tmem_base, 512);
}

}  // namespace

namespace inerf {

size_t mlp_bf16_dw_scratch_bytes() { return 16; }      // the work-item counter

// delta_img / acts_img: [n_tiles][TRAIN_IMGS][16384].  grads_host: zero-initialised (or accumulating) gradient tensors, nn.Linear layout.
// scratch: device, mlp_bf16_dw_scratch_bytes().
int mlp_bf16_dw_launch(const InerfNetDims* dims, float* const* grads_host, const uint8_t* delta_img, const uint8_t* acts_img,
                       long long n_tiles, void* scratch, cudaStream_t st) {
    static thread_local int configured_dev = -1;
    int rc = setup_once(configured_dev, {(const void*)mlp_bf16_dw_kernel}, DW_SMEM, "mlp_bf16_dw");
    if (rc) return rc;
    const int C = dims->dim_aud + dims->dim_expr + dims->dim_latent, E = dims->dim_expr;
    DwArgs d{};
    d.delta_img = delta_img; d.acts_img = acts_img; d.n_tiles = n_tiles;
    for (int i = 0; i < INERF_N_PARAMS; ++i) d.g[i] = grads_host[i];
    int nt = 0;
    auto add = [&](int a_img, int b_img, int b_imgs, int w_index, int ldw, int wcol, int kvalid, int row_lo, int row_hi, int out_row0, int bias_index) {
        d.task[nt++] = DwTask{a_img, b_img, b_imgs, w_index, ldw, wcol, kvalid, row_lo, row_hi, out_row0, bias_index};
    };
    // heavy tasks first (N = 256), partners (the two halves of a layer read the same X images) adjacent
    for (int l = 1; l < 8; ++l)
        for (int h = 0; h < 2; ++h) {
            if (l == 5) add(train_img_of(5) + 2 * h, train_img_of(4), 4, 10, 319 + C, 63 + C, 256, 0, 128, 128 * h, -1);
            else add(train_img_of(l) + 2 * h, train_img_of(l - 1), 4, 2 * l, 256, 0, 256, 0, 128, 128 * h, 2 * l + 1);
        }
    add(train_img_of(8), train_img_of(7), 4, P_VIEWS_W, 283 + E, 0, 256, 0, 128, 0, P_VIEWS_W + 1);                 // views_linears.0 <- h7
    add(TRAIN_IMG_DOUT, train_img_of(7), 4, P_ALPHA_W, 256, 0, 256, 3, 4, 0, P_ALPHA_B);                           // alpha_linear (sigma = column 3 of d_raw)
    add(train_img_of(9), train_img_of(8), 2, P_VIEWS_W + 2, 128, 0, 128, 0, 128, 0, P_VIEWS_W + 3);                 // views_linears.1
    add(train_img_of(10), train_img_of(9), 2, P_VIEWS_W + 4, 128, 0, 128, 0, 128, 0, P_VIEWS_W + 5);                // views_linears.2
    add(TRAIN_IMG_DOUT, train_img_of(10), 2, P_RGB_W, 128, 0, 128, 0, 3, 0, P_RGB_B);                               // rgb_linear
    for (int h = 0; h < 2; ++h) {
        add(train_img_of(0) + 2 * h, TRAIN_IMG_PE, 1, 0, 63 + C, 0, 63, 0, 128, 128 * h, 1);                        // pts_linears.0 <- gamma(p)
        add(train_img_of(5) + 2 * h, TRAIN_IMG_PE, 1, 10, 319 + C, 0, 63, 0, 128, 128 * h, 11);                     // pts_linears.5 <- gamma(p)
    }
    add(train_img_of(8), TRAIN_IMG_DIR, 1, P_VIEWS_W, 283 + E, 256, 27, 0, 128, 0, -1);                            // views_linears.0 <- gamma(v)
    d.n_tasks = nt;
    // ~4 items per SM on the heavy tasks; every task uses the same tile ranges so partner tasks stream the same images together
    int chunks = (int)((4LL * num_sms() + nt - 1) / nt);
    if ((long long)chunks > n_tiles) chunks = (int)n_tiles;
    if (chunks < 1) chunks = 1;
    d.tiles_per_chunk = (int)((n_tiles + chunks - 1) / chunks);
    d.n_chunks = (int)((n_tiles + d.tiles_per_chunk - 1) / d.tiles_per_chunk);
    d.counter = reinterpret_cast<int*>(scratch);
    cudaError_t e = cudaMemsetAsync(d.counter, 0, 16, st);
    if (e != cudaSuccess) { set_error("mlp_bf16_dw: %s", cudaGetErrorString(e)); return (int)e; }
    const int items = d.n_tasks * d.n_chunks;
    const int grid = items < num_sms() ? items : num_sms();
    mlp_bf16_dw_kernel<<<grid, DW_THREADS, DW_SMEM, st>>>(d);
    return check_launch("inerf_mlp_bwd[bf16 dW]");
}

}  // namespace inerf
