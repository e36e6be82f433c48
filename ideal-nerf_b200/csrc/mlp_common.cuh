// Shared declarations of the FaceNeRF MLP kernels.
#pragma once
#include <stdlib.h>

#include <initializer_list>
#include <utility>

#include "common.cuh"

namespace inerf {

// Training-time stores (point-major rows).  acts: h0..h7 (8x256) | v0..v2 (3x128) | gamma(p) (64) | gamma(v) (32)
constexpr int SAVE_W = 2528, SAVE_PE = 2432, SAVE_DIR = 2496;
// deltas: gradient w.r.t. every pre-activation, same column map as the first 2432 columns of acts
constexpr int DELTA_W = 2432;

// Kernel-side view of one FaceNeRF call.
struct MlpArgs {
    const float* w[INERF_N_PARAMS];   // nn.Linear layout (out,in), device pointers
    const float* cond;                // folded biases (CondLayout)
    const void* packed;               // mode-specific packed weights (bf16 path)
    // fused-PE input: points p = o + d*z
    const float* rays; int ray_stride;
    const float* z; int s;
    // embedded input (FaceNeRF.forward signature): x (P, 90)
    const float* x;
    long long P;                      // number of points
    float* out;                       // (P,4)
    int cond_dim;                     // dim_aud + dim_expr + dim_latent
    int dim_expr;
    float* save;                      // optional (fp32 path, training): activation store [ceil(P/64)*64][SAVE_W]
    float* trace;                     // optional (bf16 path): post-activation values of the first 256 points, [11][256][256]
    // optional (bf16 path, training): per 128-point tile T = point/128, the activations as the forward kernel holds them in shared
    // memory -- TRAIN_IMGS 16 KB images [128 points][64 features] bf16, K-major, 128-byte swizzle -- and the ReLU masks
    uint8_t* save_img;                // [n_tiles][TRAIN_IMGS][16384]
    uint32_t* save_mask;              // [n_tiles][TRAIN_MASK_WORDS][128]: bit (31-j) of word w = pre-activation 32w+j of the row is >= 0
    float tc_comp;                    // fp16x2 kernel, calibration runs only: uniform main-accumulator scale - 1 (< 0: use tc_ulps)
    float tc_ulps[4];                 // fp16x2 kernel: main-accumulator compensation in ulps of 1.0 for {L0, L1-7, V0, V1-2}
};

// image index inside a tile: h0..h7 at 4l+kb, v0..v2 at 32+2v+kb, gamma(p) (63 cols) at 38, gamma(v) (27 cols) at 39; the backward
// kernels store the deltas with the same map and d_raw (r,g,b,sigma in columns 0..3) at 38
constexpr int TRAIN_IMGS = 40, TRAIN_IMG_PE = 38, TRAIN_IMG_DIR = 39, TRAIN_IMG_DOUT = 38, TRAIN_MASK_WORDS = 76;
__host__ __device__ constexpr int train_img_of(int l) { return l < 8 ? 4 * l : 32 + 2 * (l - 8); }
__host__ __device__ constexpr int train_mask_of(int l) { return l < 8 ? 8 * l : 64 + 4 * (l - 8); }

// ---- launch plumbing of the tensor-core kernels ----------------------------------------------------------------------------------
// The CTA-pair builds (clusters of two, tcgen05 cta_group::2) run by default; INERF_MLP_PAIR=0, read once per process, keeps the
// single-CTA builds: the bit-exact reference of the pair builds, and what the trace / ablation builds run.
inline bool mlp_pair_enabled() {
    static const bool env = [] { const char* e = getenv("INERF_MLP_PAIR"); return !e || atoi(e) != 0; }();
    return env && num_sms() >= 2;
}

// Once per device and host thread for each launch site (`configured_dev`: the site's thread_local, -1 at first): the dynamic
// shared-memory limit of every kernel in `kernels`, then `more` (when given; e.g. a stage table to constant memory).  Errors read
// "<what>: setup: ...".
inline int setup_once(int& configured_dev, std::initializer_list<const void*> kernels, int smem_bytes, const char* what,
                      cudaError_t (*more)() = nullptr) {
    int dev = 0;
    cudaGetDevice(&dev);
    if (configured_dev == dev) return INERF_OK;
    cudaError_t e = cudaSuccess;
    for (const void* k : kernels)
        if (e == cudaSuccess) e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
    if (e == cudaSuccess && more) e = more();
    if (e != cudaSuccess) { set_error("%s: setup: %s", what, cudaGetErrorString(e)); return (int)e; }
    configured_dev = dev;
    return INERF_OK;
}

// Launches `kernel` for `n_iter` single-CTA iterations: as one CTA per iteration up to one per SM, or with `pair` as clusters of two
// CTAs, one per two iterations, up to one per two SMs.  `what` names the launch in error messages.
template <typename... KArgs, typename... Args>
int launch_tc(void (*kernel)(KArgs...), bool pair, long long n_iter, int nthreads, int smem_bytes, cudaStream_t st, const char* what,
              Args&&... args) {
    const long long n = pair ? (n_iter + 1) / 2 : n_iter, cap = pair ? num_sms() / 2 : num_sms();
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)((pair ? 2 : 1) * (n < cap ? n : cap)));
    cfg.blockDim = dim3(nthreads);
    cfg.dynamicSmemBytes = smem_bytes;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = pair ? 1 : 0;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
    if (e != cudaSuccess) { set_error("%s: %s", what, cudaGetErrorString(e)); return (int)e; }
    return check_launch(what);
}

int mlp_fp32_launch(const MlpArgs& a, bool embedded, cudaStream_t st);
// embedded: rows of a.x (P, 90) with an INERF_MLP_BF16_EMB blob; otherwise points of rays/z.  a.save_img != NULL: the activation-saving build
int mlp_bf16_launch(const MlpArgs& a, bool embedded, cudaStream_t st);
int mlp_fp32_bwd_launch(const InerfNetDims* dims, const float* const* params_host, float* const* grads_host,
                        const float* aud, const float* expr, const float* latent, const float* acts, float* deltas,
                        const float* d_raw, long long P, float* d_cond, void* dw_args_dev, cudaStream_t st);
size_t mlp_fp32_bwd_args_bytes();
// fp32-gate tensor-core mode (mlp_f16x2.cu).  embedded: the INERF_MLP_F16X2_EMB blob / rows of a.x (P, 90) instead of the fused entry's
// INERF_MLP_F16X2 blob / points of rays, z
int mlp_f16x2_packed_bytes(const InerfNetDims* d, size_t* bytes, bool embedded = false);
int mlp_f16x2_pack(const InerfNetDims* d, const float* const* params_host, void* packed, cudaStream_t st, bool embedded = false);
int mlp_f16x2_launch(const MlpArgs& a, bool embedded, cudaStream_t st);
int mlp_bf16_hang_info(int32_t* out8);
// bf16 training path (mlp_bf16_bwd.cu, mlp_bf16_dw.cu, mlp_fp32_bwd.cu)
int mlp_bf16_bwd_packed_bytes(const InerfNetDims* d, size_t* bytes);
int mlp_bf16_bwd_pack(const InerfNetDims* d, const float* const* params_host, void* packed, cudaStream_t st);
int mlp_bf16_bwd_chain_launch(const InerfNetDims* dims, const float* const* params_host, const void* packed_t, const uint32_t* mask,
                              const float* d_raw, uint8_t* delta_img, long long P, cudaStream_t st);
size_t mlp_bf16_dw_scratch_bytes();
int mlp_bf16_dw_launch(const InerfNetDims* dims, float* const* grads_host, const uint8_t* delta_img, const uint8_t* acts_img,
                       long long n_tiles, void* scratch, cudaStream_t st);
int mlp_bwd_cond_launch(const InerfNetDims* dims, const float* const* params_host, float* const* grads_host, const float* aud,
                        const float* expr, const float* latent, float* d_cond, cudaStream_t st);
// embedded: the INERF_MLP_BF16_EMB blob of FaceNeRF.forward's embedded-row kernel instead of the fused entry's INERF_MLP_BF16 blob
int mlp_bf16_packed_bytes(const InerfNetDims* d, size_t* bytes, bool embedded = false);
int mlp_bf16_pack(const InerfNetDims* d, const float* const* params_host, void* packed, cudaStream_t st, bool embedded = false);

}  // namespace inerf
