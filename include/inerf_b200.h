/*
 * inerf_b200.h -- C ABI of the B200-native IDEAL-NeRF render_rays hot path.
 *
 * The reference (GaryGky/IDEAL-NeRF) has no FFI: its boundary is the Python call surface of
 * NeRFs/HeadNeRF/train/audio_exp_nerf.py (Network.render_rays and friends), NeRFs/HeadNeRF/helper.py,
 * NeRFs/HeadNeRF/train/baseline.py and models/face_nerf.py.  Every entry point below replaces one
 * stage of that surface and cites the reference lines it stands in for.  The Python package
 * `ideal-nerf_b200/` keeps the reference's names and signatures and calls these through ctypes
 * (INTEGRATION.md shows the binding).
 *
 * Conventions
 *   - plain C, POD arguments only; every pointer is a DEVICE pointer to contiguous row-major fp32
 *     unless the name ends in `_host` or the comment says otherwise;
 *   - `stream` is a cudaStream_t passed as void*; entry points only enqueue work, they never
 *     synchronise, allocate or free device memory;
 *   - return 0 on success, a negative INERF_E_* on bad arguments, a positive cudaError_t when the
 *     CUDA runtime reports a launch error; inerf_last_error() gives the message (thread local);
 *   - re-entrant per (device, stream); no global mutable state besides the last-error string.
 *
 * Limits (every one is reported as INERF_E_UNSUPPORTED / INERF_E_SHAPE with a message, never silently worked around):
 *   - FaceNeRF geometry: D = 8, W = 256, skips = [4], in_xyz = 63, in_views = 27, use_viewdirs (the configuration of every reference
 *     script); conditioning dims are free (head 64 + 76 + 32, torso 106 + 0 + 0, ...);
 *   - on the fused (rays, z) entry inerf_mlp_fwd the tensor-core modes (INERF_MLP_BF16, INERF_MLP_F16X2) need s >= 43 samples per
 *     ray (a 128-row slot may touch at most four rays); inerf_mlp_fwd_embedded runs INERF_MLP_FP32, INERF_MLP_BF16 and
 *     INERF_MLP_F16X2_EMB on any number of rows (each tensor-core mode with its embedded-row blob);
 *   - training entry points exist for INERF_MLP_FP32 and INERF_MLP_BF16, on both entries (INERF_MLP_F16X2 is an inference mode);
 *   - sample_pdf: 2 <= n_bins <= 1024, n_imp <= 1024, the per-ray working set within 48 KB of shared memory; s <= 4096 elsewhere.
 */
#ifndef INERF_B200_H
#define INERF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define INERF_VERSION 100 /* 0.1.0 */

enum {
    INERF_OK = 0,
    INERF_E_ARG = -1,         /* null pointer / negative size */
    INERF_E_SHAPE = -2,       /* size outside what the kernels support */
    INERF_E_ALIGN = -3,       /* pointer not aligned as required */
    INERF_E_UNSUPPORTED = -4, /* mode / dims not built */
    INERF_E_DEVICE = -5       /* current device is not sm_100 */
};

/* MLP arithmetic modes (north_star: fp32 gate <= 1e-3 max-abs, bf16-MLP gate <= 0.05 dB PSNR) */
enum {
    INERF_MLP_FP32 = 0, /* fp32 FFMA, weights read in nn.Linear layout                         */
    INERF_MLP_BF16 = 1, /* bf16 operands, fp32 accumulate in TMEM, tcgen05.mma (packed weights) */
    INERF_MLP_BF16_BWD = 2, /* inerf_mlp_packed_bytes / inerf_mlp_pack only: the TRANSPOSED stage images of the bf16 backward chain */
    INERF_MLP_F16X2 = 3, /* fp32-gate tensor-core mode: every operand an fp16 (hi, lo) pair, three tcgen05 passes per product
                           (hi.hi + lo.hi + hi.lo), fp32 accumulate in TMEM -- meets the <= 1e-3 max-abs gate (inference entry only) */
    INERF_MLP_BF16_EMB = 4, /* inerf_mlp_packed_bytes / inerf_mlp_pack only: the stage images of the bf16 kernel on EMBEDDED rows
                              (inerf_mlp_fwd_embedded, inerf_mlp_fwd_train_bf16_embedded): the INERF_MLP_BF16 schedule plus one
                              K-block per half of views_linears.0 for its 27 view columns */
    INERF_MLP_F16X2_EMB = 5 /* the fp16x2 mode on EMBEDDED rows (inference only): the mode of inerf_mlp_fwd_embedded and of its blob
                               (inerf_mlp_packed_bytes / inerf_mlp_pack), the INERF_MLP_F16X2 schedule plus one (hi, lo) K-block per half
                               of views_linears.0 for its 27 view columns; inerf_mlp_fwd and InerfRenderArgs reject it */
};

/* sample_pdf summation policies (SURVEY.md 7-1) */
enum {
    INERF_PDF_EXACT_TORCH_CPU = 0, /* bit-reproduces torch.sum / torch.cumsum on CPU (the oracle) */
    INERF_PDF_FAST = 1             /* warp-shuffle fp32 sum                                       */
};

/* FaceNeRF geometry, models/face_nerf.py:9-36.  Only D=8, W=256, skips=[4], in_xyz=63,
 * in_views=27, use_viewdirs=True (the configuration every reference script builds) is supported. */
typedef struct InerfNetDims {
    int32_t dim_aud;    /* 64 head; 106 torso (train_torso.py:213-221) */
    int32_t dim_expr;   /* 76 head (79 in train_torso.py:203); 0 torso */
    int32_t dim_latent; /* 32 head; 0 torso                             */
    int32_t width;      /* 256 */
    int32_t depth;      /* 8   */
    int32_t in_xyz;     /* 63  */
    int32_t in_views;   /* 27  */
} InerfNetDims;

/* Parameter pointers of one FaceNeRF in state_dict order (models/face_nerf.py:27-36):
 *   [0..15]  pts_linears.{0..7}.{weight,bias}
 *   [16..21] views_linears.{0..2}.{weight,bias}
 *   [22,23]  alpha_linear.{weight,bias}
 *   [24,25]  rgb_linear.{weight,bias}
 * feature_linear is never applied by the reference forward (face_nerf.py:34) and is not passed.
 * The array itself lives in HOST memory; its entries are DEVICE pointers (nn.Linear layout, (out,in)). */
#define INERF_N_PARAMS 26

int inerf_version(void);
const char* inerf_last_error(void);
/* 0 when the current CUDA device is compute capability 10.x, INERF_E_DEVICE otherwise. */
int inerf_device_check(void);
/* sizeof of the structs of this header as the library was compiled: 0 InerfNetDims, 1 InerfRenderNet, 2 InerfRenderArgs,
 * 4 InerfPixelSampleArgs (0 for any other value, 3 included: bindings written against the three-struct header check that 3 reports 0) -- lets a foreign-language binding check its struct layout at load time. */
size_t inerf_sizeof(int which);

/* ---- rays ----------------------------------------------------------------------------------- */

/* get_rays + ray packing for a full HxW frame.
 * Replaces helper.py:228-243 (get_rays) followed by audio_exp_nerf.py:409-427 (viewdirs, near/far
 * columns).  c2w: device, 3 rows of 4 floats with `c2w_row_stride` floats between rows.
 * rays: (H*W, 11) = [o(3), d(3), near, far, d/|d|(3)]. */
int inerf_get_rays(int H, int W, float focal, float cx, float cy, const float* c2w, int c2w_row_stride,
                   float near_, float far_, float* rays, void* stream);

/* The same rays for n SELECTED pixels only: coords (n,2) int64 = (row, col).  Replaces the full-grid get_rays + index of the
 * training sampler (audio_exp_nerf.py:123-139 + :189-191).  rays: (n, 11). */
int inerf_get_rays_at(const int64_t* coords, int n, float focal, float cx, float cy, const float* c2w, int c2w_row_stride,
                      float near_, float far_, float* rays, void* stream);

/* The same rays for the pixels [first, first + count) of the row-major H x W grid only (one rank's band of a frame whose rays are
 * sharded over several GPUs: SURVEY.md 8e).  rays: (count, 11); rays[0] is pixel `first`.  Same bits as inerf_get_rays. */
int inerf_get_rays_range(int H, int W, float focal, float cx, float cy, const float* c2w, int c2w_row_stride,
                         float near_, float far_, int first, int count, float* rays, void* stream);

/* Ray packing from caller-supplied origins/directions (training batches).
 * Replaces audio_exp_nerf.py:409-427.  rays_o, rays_d: (n,3); rays: (n,11). */
int inerf_pack_rays(const float* rays_o, const float* rays_d, int n, float near_, float far_, float* rays,
                    void* stream);

/* Positional encoding gamma(x) = [x, sin(2^0 x), cos(2^0 x), ..., sin(2^(L-1) x), cos(2^(L-1) x)].
 * Replaces helper.py:174-224 (Embedder.embed via get_embedder).  x: (n, dims), out: (n, dims*(1+2L)). */
int inerf_posenc(const float* x, int64_t n, int dims, int n_freqs, float* out, void* stream);

/* to8b(x) = (255 * clip(x, 0, 1)).astype(uint8).  Replaces helper.py:154 on the rendered frame (eval_aud_exp_nerf.py:490,
 * test_torso.py:524): the image leaves the GPU as n bytes instead of 4n.  x: n floats; out: n bytes. */
int inerf_to8b(const float* x, int64_t n, uint8_t* out, void* stream);

/* Stratified coarse depths.  Replaces audio_exp_nerf.py:306-328 (baseline.py:385-410).
 * rays: (n, ray_stride) with near/far in columns 6,7.  t_vals: (s) = torch.linspace(0,1,s) (a host
 * generated table -- SURVEY.md 7-1).  t_rand: NULL (perturb == 0) or (n, s) uniform draws; the last
 * column is forced to 1.0 as the reference does at :326.  z: (n, s). */
int inerf_sample_coarse(const float* rays, int n, int ray_stride, int s, const float* t_vals,
                        const float* t_rand, int lindisp, float* z, void* stream);

/* ---- in-kernel random draws (perturb > 0) ---------------------------------------------------
 * The stochastic branches of render_rays draw with torch.rand from the global generator (audio_exp_nerf.py:321-328: the
 * stratified jitter; helper.py:282-283: the inverse-CDF draws).  The *_rng entry points make those draws inside the kernel with
 * Philox4x32-10, so no (N, S) tensor of draws is written to and read back from HBM and the whole step can live in a CUDA graph.
 * rng_state: DEVICE pointer to two uint64 {seed, offset}; counter = (draw index, offset + (stream_id << 56)), key = seed.
 * inerf_rng_advance adds `increment` to the offset (one tiny launch, graph-capturable) so the next step draws fresh numbers. */
#define INERF_RNG_STREAM_COARSE 1u /* stratified jitter of inerf_sample_coarse_rng */
#define INERF_RNG_STREAM_PDF 2u    /* default stream of inerf_importance_sample_rng */
#define INERF_RNG_STREAM_PIXELS 3u /* per-pixel keys of inerf_sample_train_pixels */
int inerf_rng_advance(uint64_t* rng_state, uint64_t increment, void* stream);

/* inerf_sample_coarse with t_rand = U[0,1) drawn in the kernel (word (i & 3) of Philox block (i >> 2), i = ray * s + sample; the
 * last sample of every ray uses 1.0 as the reference does at :326). */
int inerf_sample_coarse_rng(const float* rays, int n, int ray_stride, int s, const float* t_vals, const uint64_t* rng_state,
                            int lindisp, float* z, void* stream);

/* NaN / Inf scan of up to INERF_MAX_SCAN tensors in ONE launch: bit i of *flags is OR-ed in when xs[i] (ns[i] floats) holds a
 * non-finite value.  Replaces the nine `.any()` host synchronisations of audio_exp_nerf.py:367-369 with a device flag the caller
 * reads once (or never).  xs_host / ns_host: HOST arrays of k device pointers / element counts; flags: DEVICE int32, not cleared. */
#define INERF_MAX_SCAN 16
int inerf_flag_nonfinite(const float* const* xs_host, const int64_t* ns_host, int k, int32_t* flags, void* stream);

/* ---- compositing ---------------------------------------------------------------------------- */

/* raw2outputs forward.  Replaces baseline.py:325-375 and, with rgb_fg != NULL, the torso variant
 * test_torso.py:352-402.
 * raw (n,s,4) [r,g,b,sigma] pre-activation; z (n,s); rays_d: pointer to the first direction with
 * `rays_d_stride` floats between rays (3 for an (n,3) tensor, 11 for rays+3); bc_rgb (n,3);
 * noise: NULL or (n,s) already scaled by raw_noise_std.
 * Outputs: rgb (n,3), disp (n), acc (n), depth (n), weights (n,s), rgb_fg (n,3) or NULL. */
int inerf_composite_fwd(const float* raw, const float* z, const float* rays_d, int rays_d_stride,
                        const float* bc_rgb, const float* noise, int n, int s, int white_bkgd, float* rgb,
                        float* disp, float* acc, float* depth, float* weights, float* rgb_fg, void* stream);

/* raw2outputs backward (the reference's is autograd of baseline.py:339-375).
 * Any of the incoming gradients may be NULL (treated as zero).  Writes d_raw (n,s,4). */
int inerf_composite_bwd(const float* raw, const float* z, const float* rays_d, int rays_d_stride,
                        const float* bc_rgb, const float* noise, int n, int s, int white_bkgd,
                        const float* g_rgb, const float* g_disp, const float* g_acc, const float* g_depth,
                        const float* g_weights, const float* g_rgb_fg, float* d_raw, void* stream);

/* Training loss seed: loss2[0] = F.mse_loss(rgb, target), loss2[1] = F.mse_loss(rgb0, target) and their gradients
 * g = 2 (x - target) / n_elems in one pass.  Replaces audio_exp_nerf.py:540-546 (and the first backward nodes of :550).
 * rgb, rgb0, target, g_rgb, g_rgb0: n_elems floats (n_elems = 3 * N_rand); loss2: 2 floats (zeroed here). */
int inerf_mse_pair(const float* rgb, const float* rgb0, const float* target, int64_t n_elems, float* g_rgb, float* g_rgb0,
                   float* loss2, void* stream);

/* Head/torso blend rgb = rgb_head * last_weight_torso[:,None] + rgb_fg_torso.
 * Replaces train_torso.py:269-270 / test_torso.py:523. */
int inerf_head_torso_blend(const float* rgb_head, const float* last_weight_torso, const float* rgb_fg_torso,
                           int n, float* rgb, void* stream);

/* Torso-stage loss seed, the counterpart of inerf_mse_pair for the composites of train_torso.py:269-270, for n rays:
 * com = rgb_head * last_weight[:,None] + rgb_fg (the bits of inerf_head_torso_blend), loss2[0] = mean((com - target)^2) over 3n values,
 * loss2[1] the same for the coarse set (rgb_head0, last_weight0, rgb_fg0);  g_com = 2 (com - target) / (3n);  g_rgb_fg = g_com;
 * g_last_weight[i] = sum_c g_com[i,c] * rgb_head[i,c]  (and the "0" set).  The head is frozen in this stage: no gradient w.r.t. rgb_head.
 * All (n,3) / (n) fp32 contiguous, any alignment; loss2: 2 floats (zeroed here).  n <= 0 is a shape error. */
int inerf_head_torso_mse_pair(const float* rgb_head, const float* rgb_head0, const float* last_weight, const float* last_weight0,
                              const float* rgb_fg, const float* rgb_fg0, const float* target, int64_t n,
                              float* g_last_weight, float* g_last_weight0, float* g_rgb_fg, float* g_rgb_fg0,
                              float* loss2, void* stream);

/* The blend followed by to8b in one pass, for n rays: out_u8 (n,3) bytes = inerf_to8b(inerf_head_torso_blend(...)) bit for bit, and
 * out_rgb (n,3) = the fp32 blend, or NULL to skip it.  Replaces test_torso.py:523-524 on the rendered frame: a band of the composited
 * head + torso image leaves the GPU as 3n bytes.  Any alignment (16-byte aligned pointers take the vector path); n == 0 enqueues nothing. */
int inerf_head_torso_to8b(const float* rgb_head, const float* last_weight_torso, const float* rgb_fg_torso, int64_t n,
                          uint8_t* out_u8, float* out_rgb, void* stream);

/* ---- training-batch pixel sampler -------------------------------------------------------------
 * The pixel selection of the training sampler (audio_exp_nerf.py:141-187, data.HeadDataset.sample_pixels) and the batch built from
 * it (:189-191), on the device.  It draws from the same distribution as sample_pixels (an ordered k-subset per region, uniformly at
 * random, without replacement) but not the same numbers; the draw is fixed exactly by these rules:
 *   - pixel p = row * W + col; its keys are the words (x, y, z, w) of philox_at(rng_state, index = p, INERF_RNG_STREAM_PIXELS);
 *   - regions, from bounds[f] = {rr0, rr1, rc0, rc1, mr0, mr1, mc0, mc1} (inclusive int32) and the torso bitmask:
 *       R = rr0 <= row <= rr1 && rc0 <= col <= rc1   (face_rect: rr0 = fr[0], rr1 = fr[0] + fr[2], rc0 = fr[1], rc1 = fr[1] + fr[3])
 *       M = mr0 <= row <= mr1 && mc0 <= col <= mc1   (mouth: the row against the landmarks' x range, the column against their y range,
 *                                                      as the reference compares them; ceil of the lower and floor of the upper float
 *                                                      thresholds, so the integer tests equal its float64 ones)
 *       T = bit (p & 31) of torso_bits[f][p >> 5]   (the parsing pixel is pure red)
 *   - region r, its members and its key: 0 rect = R && !M, key x;  1 norect = !R, key x;  2 mouth = M, key y;  3 torso = T, key z
 *     (overlapping regions use different words, so their draws are independent);
 *   - selection: the k[r] members with the smallest (key << 32 | p), in ascending order of that value (ties in the key go to the lower
 *     pixel index);
 *   - output rows: rect, norect, mouth, torso, k[0] + k[1] + k[2] + k[3] = N_rand rows in all; the call writes the rows
 *     [first, first + count) only, so ranks that share rng_state and each take a band of N_rand emit disjoint parts of one batch.
 * Per output row: rays (count, 11) as inerf_get_rays_at writes them for that pixel and pose; target (count, 3) = the frame's bytes (BGR,
 * as stored) times fl(1 / 255), the fp32 bits of torch's CUDA `u8.float() / 255.0`; bc_rgb (count, 3) = bc_img at the pixel; coords
 * (count, 2) int64 (row, col), optional.
 * Every input is read from device memory (the frame index too), so a captured CUDA graph draws a fresh batch on every replay once the
 * offset of rng_state is advanced (inerf_rng_advance, not done here).  A frame index outside [0, n_frames) selects nothing and writes no
 * output; a region with fewer than k[r] members leaves its last rows unwritten -- the caller rules both out (the library cannot read
 * device data without a synchronise).
 * Limits: k[r] <= INERF_PIXEL_SAMPLER_MAX_K (INERF_E_UNSUPPORTED above: one CTA sorts each region in shared memory), H * W <=
 * INERF_PIXEL_SAMPLER_MAX_PIXELS (beyond it one of the 4096 histogram bins that bound the sort could overflow it). */
#define INERF_PIXEL_SAMPLER_MAX_K 4096
#define INERF_PIXEL_SAMPLER_MAX_PIXELS (1 << 22)

typedef struct InerfPixelSampleArgs {
    int32_t H, W, n_frames;
    int32_t k[4];                  /* region budgets: rect, norect, mouth, torso                                              */
    int32_t first, count;          /* the band of output rows                                                                 */
    float focal, cx, cy, near_, far_;
    const int64_t* frame_index;    /* device scalar                                                                           */
    const int32_t* bounds;         /* (n_frames, 8)                                                                           */
    const uint32_t* torso_bits;    /* (n_frames, ceil(H * W / 32))                                                            */
    const float* poses;            /* (n_frames, 3, 4) camera-to-world                                                        */
    const uint8_t* frames;         /* (n_frames, H, W, 3)                                                                     */
    const float* bc_img;           /* (H, W, 3) background                                                                    */
    const uint64_t* rng_state;     /* {seed, offset}                                                                          */
    float* rays;                   /* outputs, `count` rows each                                                              */
    float* target;
    float* bc_rgb;
    int64_t* coords;               /* NULL to skip                                                                            */
} InerfPixelSampleArgs;

/* Workspace of inerf_sample_train_pixels: the per-region key histograms, boundary bins and candidate buffers. */
int inerf_pixel_sampler_workspace_bytes(const InerfPixelSampleArgs* args, size_t* bytes);
/* workspace: 256-byte aligned, at least inerf_pixel_sampler_workspace_bytes.  Four kernels and one memset on `stream`; count == 0
 * enqueues nothing.  Every argument error is returned before any device work. */
int inerf_sample_train_pixels(const InerfPixelSampleArgs* args, void* workspace, size_t workspace_bytes, void* stream);

/* ---- image metrics ----------------------------------------------------------------------------------------------------------------
 * Scores B rendered frames against ground-truth frames, both uint8 (H, W, 3) as to8b writes them, for held-out evaluation (the scores of
 * the bytes a user sees in the video).  Row b of the batch is compared with gt_frames[frame_index[b]]; the index is read from device
 * memory, so the call may sit in a CUDA graph.  The results are exactly these:
 *   - sse[b] = {full, R, M}: the sum over the pixels of the region and over the 3 channels of (pred - gt)^2, exact in int64.  R and M are
 *     the inclusive boxes {r0, r1, c0, c1} = bounds[f][0..3] (face rect) and bounds[f][4..7] (mouth), as inerf_sample_train_pixels reads
 *     them; npix[b] = the number of frame pixels in the full frame, R and M.  When bounds is NULL only column 0 of sse and npix is written.
 *   - ssim_sum[b]: the sum over the 3 channels and over the (H - 10) x (W - 10) positions whose 11 x 11 window lies inside the frame of
 *       SSIM = ((2 mu_x mu_y + C1)(2 s_xy + C2)) / ((mu_x^2 + mu_y^2 + C1)(s_x^2 + s_y^2 + C2)),
 *     with mu, E[x^2], E[xy] weighted by the normalised 11-tap Gaussian (sigma 1.5) in both directions, biased moments (s_x^2 = E[x^2] -
 *     mu_x^2, s_xy = E[xy] - mu_x mu_y), C1 = (0.01 * 255)^2, C2 = (0.03 * 255)^2 (Wang et al. 2004; skimage's structural_similarity
 *     with gaussian_weights=True, sigma=1.5, use_sample_covariance=False, data_range=255, channel_axis=-1).  The mean SSIM is
 *     ssim_sum / (3 (H - 10)(W - 10)).  The moments are fp32 (each image shifted by a byte of its tile first); sse and npix are exact.
 * pred (B, H, W, 3), gt_frames (n_frames, H, W, 3), frame_index (B) int64, bounds (n_frames, 8) int32 or NULL; outputs sse, npix (B, 3)
 * int64 and ssim_sum (B) fp64.  A row whose frame index lies outside [0, n_frames) gets zeros in every output.
 * Work: two memsets of the accumulators, then one kernel of one CTA per 32 x 32 tile per row.  Every argument error is returned before
 * any device work: NULL pointers, B or n_frames < 0 (INERF_E_ARG); H or W < 11, H * W > INERF_IMAGE_METRICS_MAX_PIXELS (INERF_E_SHAPE).
 * B == 0 enqueues nothing. */
#define INERF_IMAGE_METRICS_MAX_PIXELS (1 << 24)
int inerf_image_metrics(const uint8_t* pred, const uint8_t* gt_frames, const int64_t* frame_index, const int32_t* bounds, int32_t B,
                        int32_t H, int32_t W, int32_t n_frames, int64_t* sse, int64_t* npix, double* ssim_sum, void* stream);

/* The squared error of B rendered frames over a per-frame pixel mask, e.g. the torso region the torso stage trains (its pixels are the
 * parsing map's pure red ones, the torso bitmask of inerf_sample_train_pixels).  Row b is compared with gt_frames[frame_index[b]] (index
 * read from device memory, so the call may sit in a CUDA graph):
 *   - sse[b] = the sum over the 3 channels and over the pixels p < H * W whose bit (p & 31) of bits[f][p >> 5] is set (p = row * W + col,
 *     f = frame_index[b]) of (pred - gt)^2, exact in int64;  npix[b] = the number of those pixels.
 * pred (B, H, W, 3) uint8, gt_frames (n_frames, H, W, 3) uint8, frame_index (B) int64, bits (n_frames, ceil(H * W / 32)) uint32 (the bits
 * past H * W in the last word are ignored); outputs sse, npix (B) int64.  A row whose frame index lies outside [0, n_frames) gets zeros.
 * Work: two memsets of the accumulators, then one kernel of one CTA per 1 024 pixels per row.  Every argument error is returned before any
 * device work, with inerf_image_metrics' codes and limits: NULL pointers, B or n_frames < 0 (INERF_E_ARG); H or W < 11, H * W >
 * INERF_IMAGE_METRICS_MAX_PIXELS (INERF_E_SHAPE).  B == 0 enqueues nothing. */
int inerf_masked_sse(const uint8_t* pred, const uint8_t* gt_frames, const int64_t* frame_index, const uint32_t* bits, int32_t B, int32_t H,
                     int32_t W, int32_t n_frames, int64_t* sse, int64_t* npix, void* stream);

/* LPIPS v0.1 with the AlexNet trunk (Zhang et al. 2018) of B rendered frames: out[b] is what lpips.LPIPS(net='alex', version='0.1')(in0,
 * in1) computes (normalize=False) for in0 = pred[b], in1 = gt_frames[frame_index[b]].  The frames are uint8 (H, W, 3) BGR as stored, so the
 * bytes of a pixel are read as B, G, R and fed to AlexNet as R, G, B.
 *   1. x = byte / 127.5 - 1 per channel (lpips' im2tensor), then the ScalingLayer (x - shift_c) / scale_c with shift = (-0.030, -0.088,
 *      -0.188), scale = (0.458, 0.448, 0.450) in R, G, B order.  Convolution zero padding applies to these scaled values.
 *   2. AlexNet features (torchvision layout): conv1 11 x 11 stride 4 pad 2, 3 -> 64, ReLU = f1; max pool 3 / 2; conv2 5 x 5 pad 2, 64 ->
 *      192, ReLU = f2; max pool 3 / 2; conv3 3 x 3 pad 1, 192 -> 384, ReLU = f3; conv4 3 x 3 pad 1, 384 -> 256, ReLU = f4; conv5 3 x 3
 *      pad 1, 256 -> 256, ReLU = f5.  (The final max pool is not used.)
 *   3. Per layer k and output position, each image's feature vector is normalised over the channels, f / (sqrt(sum_c f^2) + 1e-10); the
 *      squared difference of the two normalised vectors is dotted with lin_k (C_k weights, no bias); that is averaged over the layer's
 *      h_k x w_k positions.
 *   4. out[b] = the sum of the five layer means, added in layer order.
 * For 450 x 450 frames the maps are 111^2 (f1), 55^2 (f2) and 27^2 (f3 - f5); every map is non-empty for H, W >= 31.
 * params_host: host array of INERF_LPIPS_N_PARAMS device pointers to contiguous fp32, in this order: conv1.weight (64, 3, 11, 11),
 * conv1.bias (64), conv2.weight (192, 64, 5, 5), conv2.bias, conv3.weight (384, 192, 3, 3), conv3.bias, conv4.weight (256, 384, 3, 3),
 * conv4.bias, conv5.weight (256, 256, 3, 3), conv5.bias, lin0 (64), lin1 (192), lin2 (384), lin3 (256), lin4 (256) -- torchvision's
 * features.{0,3,6,8,10} and lpips' lin{0..4}.model.1.weight.  pred (B, H, W, 3), gt_frames (n_frames, H, W, 3), frame_index (B) int64, read
 * from device memory; out (B) fp32.  A row whose frame index lies outside [0, n_frames) gets 0.  The arithmetic is fp32 with every sum in
 * a fixed order: results are bit-identical from call to call and between eager calls and CUDA-graph replay.
 * workspace: device memory of at least inerf_lpips_workspace_bytes(B, H, W) bytes, 256-byte aligned (the fp32 feature maps of both images
 * of every row, 26.3 MB per row at 450 x 450, and the per-CTA partial sums).  Work: 13 kernels on `stream`, no allocation, no copy and no
 * synchronise, so the call may sit in a CUDA graph.  Every argument error is returned before any device work: NULL pointers, B or n_frames
 * < 0 (INERF_E_ARG); H or W < 31, H * W > INERF_IMAGE_METRICS_MAX_PIXELS, B > INERF_LPIPS_MAX_ROWS, a workspace smaller than needed
 * (INERF_E_SHAPE).  B == 0 enqueues nothing. */
#define INERF_LPIPS_N_PARAMS 15
#define INERF_LPIPS_MAX_ROWS 65535
int inerf_lpips_workspace_bytes(int32_t B, int32_t H, int32_t W, size_t* bytes);
int inerf_lpips(const float* const* params_host, const uint8_t* pred, const uint8_t* gt_frames, const int64_t* frame_index, int32_t B,
                int32_t H, int32_t W, int32_t n_frames, void* workspace, size_t workspace_bytes, float* out, void* stream);

/* ---- importance sampling -------------------------------------------------------------------- */

/* sample_pdf.  Replaces helper.py:269-313.
 * bins: (n, n_bins) with row stride bins_stride; weights: (n, n_bins-1) with row stride w_stride
 * (so weights[...,1:-1] of an (n,S) tensor is passed as w+1 with stride S).
 * u: n_imp floats shared by every ray when u_per_ray == 0 (torch.linspace(0,1,n_imp) for det=True),
 * else (n, n_imp) draws.  z_samples (n, n_imp); inds: NULL or (n, n_imp) int64 =
 * torch.searchsorted(cdf, u, right=True).
 * Optional fused tail of render_rays (audio_exp_nerf.py:347,364): when z_coarse != NULL (n, s1),
 * z_merged (n, s1+n_imp) = sort(cat(z_coarse, z_samples)) and z_std (n) = std(z_samples, unbiased=False). */
int inerf_sample_pdf(const float* bins, int bins_stride, const float* weights, int w_stride, int n, int n_bins,
                     int n_imp, const float* u, int u_per_ray, int policy, float* z_samples, int64_t* inds,
                     const float* z_coarse, int s1, float* z_merged, float* z_std, void* stream);

/* Fused form used by render_rays: bins = mid-points of z_coarse, weights = w_coarse[:,1:-1]
 * (audio_exp_nerf.py:342-347).  z_coarse, w_coarse: (n, s1). */
int inerf_importance_sample(const float* z_coarse, const float* w_coarse, int n, int s1, int n_imp,
                            const float* u, int u_per_ray, int policy, float* z_samples, int64_t* inds,
                            float* z_merged, float* z_std, void* stream);

/* inerf_importance_sample for the stochastic branch (perturb > 0, helper.py:282-283) with the draws made in the kernel: the ORDER
 * STATISTICS of n_imp iid U[0,1) per ray are generated directly (exponential spacings), so z_samples come out ascending and no sort
 * is needed; the CDF is a plain fp32 warp scan (bit-exactness against torch-CPU is only defined for det=True / supplied draws, which
 * stay with inerf_importance_sample).  z_samples may be NULL (the renderer only consumes z_merged and z_std). */
int inerf_importance_sample_rng(const float* z_coarse, const float* w_coarse, int n, int s1, int n_imp,
                                const uint64_t* rng_state, uint32_t stream_id, float* z_samples, float* z_merged,
                                float* z_std, void* stream);

/* ---- the whole inference render_rays in one call ------------------------------------------------------------------------------
 * Network.render_rays under torch.no_grad() (audio_exp_nerf.py:297-371; the torso variant train_torso.py:290-363 with rgb_map_fg !=
 * NULL): stratified depths -> coarse FaceNeRF -> raw2outputs -> sample_pdf + sort + std -> fine FaceNeRF -> raw2outputs, enqueued by
 * ONE entry point on one stream.  In the reference's configuration (64 + 128 samples, perturb > 0) that is FIVE launches per call
 * instead of ten, and neither the coarse weights nor the fine weights nor a tensor of draws reach HBM:
 *   1. set-up kernel: conditioning fold of BOTH nets + (optionally) the rays of pixels [first, first + n) + the jittered coarse depths;
 *   2. coarse FaceNeRF (inerf_mlp_fwd's kernel);
 *   3. compositor + importance sampler in one kernel: the weights go from the compositor's registers into the sampler's CDF scan;
 *   4. fine FaceNeRF;
 *   5. final compositor: maps + last_weight only (no (n, S) weights tensor unless asked for), the NaN / Inf flags of
 *      audio_exp_nerf.py:367-369 and the bump of the RNG offset.
 * Other shapes / perturb == 0 run the stand-alone kernels of this header inside the same call (deterministic depths keep the
 * bit-exact sample_pdf policy), so results are bit-identical to calling the stages one by one.
 * Needs n_importance > 0, an even n_samples >= 4 and an even n_samples + n_importance <= 256; raw_noise_std == 0. */
typedef struct InerfRenderNet {
    InerfNetDims dims;
    const float* const* params_host; /* INERF_N_PARAMS device pointers (host array)            */
    const void* packed;              /* inerf_mlp_pack blob for `mode` (NULL for INERF_MLP_FP32) */
    const float* aud;                /* conditioning vectors (device), NULL where the dim is 0  */
    const float* expr;
    const float* latent;
} InerfRenderNet;

/* bits of *nonfinite (the keys the reference scans, audio_exp_nerf.py:367-369) */
enum {
    INERF_NF_RGB_MAP = 1, INERF_NF_DISP_MAP = 2, INERF_NF_ACC_MAP = 4, INERF_NF_RGB0 = 8, INERF_NF_DISP0 = 16, INERF_NF_ACC0 = 32,
    INERF_NF_Z_STD = 64, INERF_NF_LAST_WEIGHT = 128
};

typedef struct InerfRenderArgs {
    int32_t mode;                    /* INERF_MLP_FP32 / _BF16 / _F16X2, both nets (not _F16X2_EMB: INERF_E_UNSUPPORTED) */
    int32_t n;                       /* rays                                                                               */
    int32_t n_samples, n_importance; /* args.N_samples, args.N_importance                                                  */
    int32_t perturb;                 /* 0: deterministic depths; 1: stratified jitter and importance draws made in-kernel  */
    int32_t lindisp, white_bkgd;
    /* rays: supplied (n, ray_stride >= 11) as inerf_pack_rays / inerf_get_rays write them, or -- gen_rays != 0 -- generated here for
     * the pixels [first, first + n) of the H x W frame (inerf_get_rays_range's arguments) into the workspace */
    const float* rays;
    int32_t ray_stride;
    int32_t gen_rays, H, W, first;
    float focal, cx, cy, near_, far_;
    const float* c2w;
    int32_t c2w_row_stride;
    const float* bc_rgb;             /* (n, 3)                                                                             */
    const float* t_vals;             /* torch.linspace(0, 1, n_samples) (host-generated table)                             */
    const float* u_vals;             /* torch.linspace(0, 1, n_importance); only read when perturb == 0                    */
    uint64_t* rng_state;             /* {seed, offset}; only used when perturb != 0; the offset is advanced by 1           */
    InerfRenderNet coarse, fine;
    /* outputs (device).  Required: rgb_map (n,3), disp_map, acc_map, depth_map, last_weight (n), disp0, acc0, z_std (n).
     * rgb0 (n,3): NULL = no coarse colour.  The coarse net then runs its density-only build in INERF_MLP_BF16 mode (the full net in the
     * others) and the coarse compositor reads sigma alone; every other output keeps its bits.  Not with the torso extras.
     * Optional (NULL to skip): weights (n, S) of the fine pass, z_vals (n, S) merged depths, and the torso extras rgb_map_fg (n,3),
     * rgb_map_fg0 (n,3), last_weight0 (n) -- the three are given together or not at all, and need rgb0. */
    float *rgb_map, *disp_map, *acc_map, *depth_map, *last_weight, *rgb0, *disp0, *acc0, *z_std;
    float *weights, *z_vals, *rgb_map_fg, *rgb_map_fg0, *last_weight0;
    int32_t* nonfinite;              /* NULL or a device int32: INERF_NF_* bits are OR-ed in (not cleared here)            */
    void* workspace;                 /* device scratch of inerf_render_workspace_bytes bytes, 256-byte aligned             */
    size_t workspace_bytes;
} InerfRenderArgs;

/* Scratch the call needs for these shapes (rays when generated, both conditioning buffers, coarse depths, raw of both passes -- the
 * coarse one a float per sample when rgb0 is NULL in INERF_MLP_BF16 mode -- merged depths, and the coarse weights / samples of the
 * deterministic path). */
int inerf_render_workspace_bytes(const InerfRenderArgs* args, size_t* bytes);
int inerf_render_rays_fused(const InerfRenderArgs* args, void* stream);
/* Measurement twin (the one entry point that SYNCHRONISES): the same call with a CUDA event between the stages; ms_host5 (HOST, 5 floats)
 * = device time of {set-up, coarse FaceNeRF, coarse raw2outputs + sampling, fine FaceNeRF, final raw2outputs}.  bench.py uses it for
 * the rooflines of the fused small kernels. */
int inerf_debug_render_stage_ms(const InerfRenderArgs* args, void* stream, float* ms_host5);

/* ---- FaceNeRF MLP --------------------------------------------------------------------------- */

/* Number of floats of the per-call conditioning buffer written by inerf_mlp_fold_cond. */
int inerf_mlp_cond_floats(const InerfNetDims* dims, size_t* n_floats);

/* Fold the per-call constant conditioning columns into biases (SURVEY.md Appendix B):
 *   b0'  = b0  + W0[:,63:]            . [aud | expr/3 | latent]
 *   b5'  = b5  + W5[:,63:63+cond]     . [aud | expr/3 | latent]
 *   bV0' = bV0 + WV0[:,283:283+expr]  . expr/3
 * Replaces the three einops.repeat + torch.cat of face_nerf.py:44-56,69 (and `expr * 1 / 3`, :49).
 * params_host: INERF_N_PARAMS device pointers (host array).  aud/expr/latent may be NULL when the
 * corresponding dim is 0.  cond: device buffer of inerf_mlp_cond_floats floats holding every bias
 * of the folded network: [b0'(W) b1..b4 b5' b6 b7 | bV0'(W/2) bV1 bV2 | alpha_b(1) rgb_b(3)], followed by the same biases as
 * bf16 (hi, lo) operand tiles for the tensor-core kernel (which adds them with one extra MMA per layer half). */
int inerf_mlp_fold_cond(const InerfNetDims* dims, const float* const* params_host, const float* aud,
                        const float* expr, const float* latent, float* cond, void* stream);

/* Bytes of the packed-weight blob for `mode` (0 for INERF_MLP_FP32, which reads nn.Linear layout). */
int inerf_mlp_packed_bytes(int mode, const InerfNetDims* dims, size_t* bytes);

/* Re-lay the per-point weights for `mode` (bf16, K-major 128B-swizzled UMMA tiles in MMA issue
 * order).  Re-run after every optimiser step. */
int inerf_mlp_pack(int mode, const InerfNetDims* dims, const float* const* params_host, void* packed,
                   void* stream);

/* run_network for one pass: points p = o + d*z, gamma_10(p), gamma_4(viewdir), FaceNeRF.
 * Replaces audio_exp_nerf.py:332 + :376-394 + face_nerf.py:40-80 (positional encoding fused into the
 * first-layer operand; no (P,90) tensor is materialised).
 * rays (n, ray_stride) as produced by inerf_get_rays/inerf_pack_rays; z (n, s); raw (n, s, 4). */
int inerf_mlp_fwd(int mode, const InerfNetDims* dims, const float* const* params_host, const void* packed,
                  const float* cond, const float* rays, int ray_stride, const float* z, int n, int s,
                  float* raw, void* stream);

/* ---- training (fp32 mode): forward that keeps activations + analytic backward ------------------------------- */

/* Buffer sizes for n_points = n*s points: acts (floats), deltas (floats), scratch (bytes, device). */
int inerf_mlp_train_sizes(const InerfNetDims* dims, int64_t n_points, size_t* acts_floats, size_t* deltas_floats,
                          size_t* scratch_bytes);

/* inerf_mlp_fwd (fused entry: rays/z) or inerf_mlp_fwd_embedded (x != NULL, p_embedded rows) in fp32 mode that also
 * stores every post-ReLU activation and both encodings in `acts` for inerf_mlp_bwd. */
int inerf_mlp_fwd_train(const InerfNetDims* dims, const float* const* params_host, const float* cond, const float* rays,
                        int ray_stride, const float* z, int n, int s, const float* x, int64_t p_embedded, float* raw,
                        float* acts, void* stream);

/* Backward of FaceNeRF: what torch.autograd computes for models/face_nerf.py:40-80 inside the reference's
 * loss.backward() (audio_exp_nerf.py:549).  d_raw (n_points,4).  grads_host: INERF_N_PARAMS device pointers (host array)
 * to ZERO-INITIALISED gradient tensors in nn.Linear layout; d_cond: zero-initialised [dim_aud+dim_expr+dim_latent] =
 * [d_aud | d_expr | d_latent].  deltas / scratch: workspaces sized by inerf_mlp_train_sizes. */
int inerf_mlp_bwd(const InerfNetDims* dims, const float* const* params_host, float* const* grads_host, const float* aud,
                  const float* expr, const float* latent, const float* acts, float* deltas, const float* d_raw,
                  int64_t n_points, float* d_cond, void* scratch, void* stream);

/* ---- training (bf16 tensor-core mode) ---------------------------------------------------------------------------------------
 * Same contract as the fp32 pair above, with bf16 operands on tcgen05: the forward keeps every post-ReLU activation as the 16 KB
 * shared-memory images of its own A operands plus one ReLU-mask bit per activation; the backward is a fused chain kernel
 * (delta_{l-1} = delta_l . W_l * mask, weights streamed TRANSPOSED, inerf_mlp_pack mode INERF_MLP_BF16_BWD), one long-K tcgen05 GEMM
 * per weight matrix for dW / db straight from those images, and the fp32 conditioning kernel.  The fused entry needs n*s points with
 * s >= 43; the embedded-row entry takes any number of rows. */
int inerf_mlp_train_sizes_bf16(const InerfNetDims* dims, int64_t n_points, size_t* acts_bytes, size_t* mask_bytes,
                               size_t* deltas_bytes, size_t* scratch_bytes);
int inerf_mlp_fwd_train_bf16(const InerfNetDims* dims, const float* const* params_host, const void* packed, const float* cond,
                             const float* rays, int ray_stride, const float* z, int n, int s, float* raw, void* acts, void* mask,
                             void* stream);
/* inerf_mlp_fwd_train_bf16 on embedded rows x (p, in_xyz+in_views), FaceNeRF.forward's input: packed is an INERF_MLP_BF16_EMB blob;
 * acts / mask are sized by inerf_mlp_train_sizes_bf16(dims, p, ...) and hold the same images, so inerf_mlp_bwd_bf16 (n_points = p)
 * is the backward.  Any p >= 0 (0 enqueues nothing); x, raw (p, 4), acts and mask 16-byte aligned. */
int inerf_mlp_fwd_train_bf16_embedded(const InerfNetDims* dims, const float* const* params_host, const void* packed, const float* cond,
                                      const float* x, int64_t p, float* raw, void* acts, void* mask, void* stream);
/* grads_host: ZERO-INITIALISED gradient tensors (nn.Linear layout, fp32); d_cond as in inerf_mlp_bwd. */
int inerf_mlp_bwd_bf16(const InerfNetDims* dims, const float* const* params_host, const void* packed_t, float* const* grads_host,
                       const float* aud, const float* expr, const float* latent, const void* acts, const void* mask, void* deltas,
                       const float* d_raw, int64_t n_points, float* d_cond, void* scratch, void* stream);

/* ---- per-frame conditioning nets -----------------------------------------------------------------------------------
 * AudioNet: DeepSpeech windows x (n, 16, 29) -> audio codes y (n, dim_aud).  Replaces models/audio_net.py:43-69 as called from
 * audio_exp_nerf.py:263,266.  params_host: 12 DEVICE pointers (host array) in state_dict order: encoder_conv.{0,2,4,6}.{weight,bias},
 * encoder_fc1.{0,2}.{weight,bias} (nn.Conv1d (out,in,3) / nn.Linear (out,in) layouts). */
int inerf_audio_net_fwd(const float* const* params_host, const float* x, int n, int dim_aud, float* y, void* stream);
/* AudioAttNet: attention over the smoothing window, x (seq_len = 8, dim_feat) -> y (dim_feat); the attention convolutions see the
 * first dim_att (32) channels.  Replaces models/audio_net.py:8-36 (audio_exp_nerf.py:264).  params_host: 12 device pointers:
 * attentionConvNet.{0,2,4,6,8}.{weight,bias}, attentionNet.0.{weight,bias}. */
int inerf_audio_att_fwd(const float* const* params_host, const float* x, int seq_len, int dim_feat, int dim_att, float* y, void* stream);

/* Backward of the two conditioning nets: what autograd computes for models/audio_net.py inside the reference's loss.backward()
 * (audio_exp_nerf.py:263-266 are in the graph; :493 optimises network.parameters(), these nets included).  The forward is recomputed
 * in shared memory.  grads_host: 12 DEVICE pointers (host array) to gradient tensors in the parameters' layouts, ACCUMULATED into
 * (zero them first).  inerf_audio_net_bwd: x (n,16,29), dy (n, dim_aud); the DeepSpeech features are data, so there is no dx.
 * inerf_audio_att_bwd: x (8, dim_feat), dy (dim_feat) -> dx (8, dim_feat), overwritten. */
int inerf_audio_net_bwd(const float* const* params_host, float* const* grads_host, const float* x, const float* dy, int n, int dim_aud,
                        void* stream);
int inerf_audio_att_bwd(const float* const* params_host, float* const* grads_host, const float* x, const float* dy, int seq_len,
                        int dim_feat, int dim_att, float* dx, void* stream);

/* FaceNeRF.forward on already-embedded inputs x (p, in_xyz+in_views) -- the reference module's own
 * call signature (face_nerf.py:40).  out (p, 4).  Any p >= 0 (0 enqueues nothing).
 * INERF_MLP_FP32: packed is ignored.  INERF_MLP_BF16: the tcgen05 kernel; packed must be an INERF_MLP_BF16_EMB blob (not the
 * INERF_MLP_BF16 blob of inerf_mlp_fwd) and x 16-byte aligned.  INERF_MLP_F16X2_EMB: the fp16x2 tcgen05 kernel at fp32-gate accuracy;
 * packed must be an INERF_MLP_F16X2_EMB blob and x 16-byte aligned.  INERF_MLP_F16X2: INERF_E_UNSUPPORTED (its blob is the fused
 * entry's; the two cannot be told apart). */
int inerf_mlp_fwd_embedded(int mode, const InerfNetDims* dims, const float* const* params_host,
                           const void* packed, const float* cond, const float* x, int64_t p, float* out,
                           void* stream);

#ifdef __cplusplus
}
#endif
#endif /* INERF_B200_H */
