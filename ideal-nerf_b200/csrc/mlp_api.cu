// C-ABI dispatch of the FaceNeRF MLP (include/inerf_b200.h): argument checks, then the launch of the mode's kernels -- fp32
// (mlp_fp32.cu, mlp_fp32_bwd.cu), bf16 (mlp_bf16.cu, mlp_bf16_bwd.cu, mlp_bf16_dw.cu) and fp16x2 (mlp_f16x2.cu).
#include "mlp_common.cuh"
#include "fold_cond.cuh"

using namespace inerf;

namespace {

int fill_args(MlpArgs& a, const InerfNetDims* dims, const float* const* params_host, const float* cond) {
    int rc = check_dims(dims);
    if (rc) return rc;
    if (!params_host || !cond) return fail(INERF_E_ARG, "mlp: NULL params/cond");
    for (int i = 0; i < INERF_N_PARAMS; ++i) {
        if (!params_host[i]) return fail(INERF_E_ARG, "mlp: NULL parameter pointer");
        a.w[i] = params_host[i];
    }
    a.cond = cond;
    a.cond_dim = dims->dim_aud + dims->dim_expr + dims->dim_latent;
    a.dim_expr = dims->dim_expr;
    return INERF_OK;
}

// The checks both backward entries share, after their own NULL-buffer check: every parameter / gradient pointer, d_cond when there are
// conditioning columns, and each conditioning vector of a non-zero dim.  `what` prefixes the messages.
int check_bwd_args(const char* what, const InerfNetDims* dims, const float* const* params_host, float* const* grads_host,
                   const float* aud, const float* expr, const float* latent, const float* d_cond) {
    for (int i = 0; i < INERF_N_PARAMS; ++i)
        if (!params_host[i] || !grads_host[i]) { set_error("%s: NULL parameter/gradient pointer", what); return INERF_E_ARG; }
    const int C = dims->dim_aud + dims->dim_expr + dims->dim_latent;
    if (C > 0 && !d_cond) { set_error("%s: d_cond is NULL", what); return INERF_E_ARG; }
    if ((dims->dim_aud > 0 && !aud) || (dims->dim_expr > 0 && !expr) || (dims->dim_latent > 0 && !latent)) {
        set_error("%s: conditioning vector missing for a non-zero dim", what);
        return INERF_E_ARG;
    }
    return INERF_OK;
}

}  // namespace

extern "C" int inerf_mlp_cond_floats(const InerfNetDims* dims, size_t* n_floats) {
    int rc = check_dims(dims);
    if (rc) return rc;
    if (!n_floats) return fail(INERF_E_ARG, "inerf_mlp_cond_floats: NULL");
    // the folded fp32 biases, then the same biases as operand tiles of the tensor-core kernels (16 x 4 KB + 6 x 2 KB per set): bf16
    // (hi, lo) for mlp_bf16.cu, fp16 (hi, mid, lo) for mlp_f16x2.cu
    *n_floats = (size_t)COND_FLOATS + 2 * BIAS_TILE_BYTES / sizeof(float);
    return INERF_OK;
}

extern "C" int inerf_mlp_fold_cond(const InerfNetDims* dims, const float* const* params_host, const float* aud,
                                   const float* expr, const float* latent, float* cond, void* stream) {
    int rc = check_dims(dims);
    if (rc) return rc;
    if (!params_host || !cond) return fail(INERF_E_ARG, "inerf_mlp_fold_cond: NULL pointer");
    if ((dims->dim_aud > 0 && !aud) || (dims->dim_expr > 0 && !expr) || (dims->dim_latent > 0 && !latent))
        return fail(INERF_E_ARG, "inerf_mlp_fold_cond: conditioning vector missing for a non-zero dim");
    FoldArgs f{};
    for (int i = 0; i < INERF_N_PARAMS; ++i) {
        if (!params_host[i]) return fail(INERF_E_ARG, "inerf_mlp_fold_cond: NULL parameter pointer");
        f.w[i] = params_host[i];
    }
    f.aud = aud; f.expr = expr; f.latent = latent;
    f.da = dims->dim_aud; f.de = dims->dim_expr; f.dl = dims->dim_latent;
    f.cond = cond;
    return mlp_fold_cond_launch(f, as_stream(stream));
}

extern "C" int inerf_mlp_packed_bytes(int mode, const InerfNetDims* dims, size_t* bytes) {
    int rc = check_dims(dims);
    if (rc) return rc;
    if (!bytes) return fail(INERF_E_ARG, "inerf_mlp_packed_bytes: NULL");
    switch (mode) {
        case INERF_MLP_FP32: *bytes = 0; return INERF_OK;
        case INERF_MLP_BF16: return mlp_bf16_packed_bytes(dims, bytes);
        case INERF_MLP_BF16_EMB: return mlp_bf16_packed_bytes(dims, bytes, true);
        case INERF_MLP_BF16_BWD: return mlp_bf16_bwd_packed_bytes(dims, bytes);
        case INERF_MLP_F16X2: return mlp_f16x2_packed_bytes(dims, bytes);
        case INERF_MLP_F16X2_EMB: return mlp_f16x2_packed_bytes(dims, bytes, true);
        default: return fail(INERF_E_UNSUPPORTED, "inerf_mlp_packed_bytes: unknown mode");
    }
}

extern "C" int inerf_mlp_pack(int mode, const InerfNetDims* dims, const float* const* params_host, void* packed,
                              void* stream) {
    int rc = check_dims(dims);
    if (rc) return rc;
    if (mode == INERF_MLP_FP32) return INERF_OK;
    if (mode < INERF_MLP_FP32 || mode > INERF_MLP_F16X2_EMB) return fail(INERF_E_UNSUPPORTED, "inerf_mlp_pack: unknown mode");
    if (!params_host || !packed) return fail(INERF_E_ARG, "inerf_mlp_pack: NULL pointer");
    const cudaStream_t st = as_stream(stream);
    switch (mode) {
        case INERF_MLP_BF16: return mlp_bf16_pack(dims, params_host, packed, st);
        case INERF_MLP_BF16_EMB: return mlp_bf16_pack(dims, params_host, packed, st, true);
        case INERF_MLP_BF16_BWD: return mlp_bf16_bwd_pack(dims, params_host, packed, st);
        case INERF_MLP_F16X2: return mlp_f16x2_pack(dims, params_host, packed, st);
        default: return mlp_f16x2_pack(dims, params_host, packed, st, true);      // INERF_MLP_F16X2_EMB
    }
}

extern "C" int inerf_mlp_fwd(int mode, const InerfNetDims* dims, const float* const* params_host, const void* packed,
                             const float* cond, const float* rays, int ray_stride, const float* z, int n, int s,
                             float* raw, void* stream) {
    MlpArgs a{};
    int rc = fill_args(a, dims, params_host, cond);
    if (rc) return rc;
    if (n < 0 || s <= 0 || ray_stride < 11) return fail(INERF_E_SHAPE, "inerf_mlp_fwd: bad n/s/ray_stride (rays need the viewdir columns)");
    if (n == 0) return INERF_OK;
    if (!rays || !z || !raw) return fail(INERF_E_ARG, "inerf_mlp_fwd: NULL pointer");
    if ((uintptr_t)raw & 15) return fail(INERF_E_ALIGN, "inerf_mlp_fwd: raw must be 16-byte aligned");
    a.rays = rays; a.ray_stride = ray_stride; a.z = z; a.s = s;
    a.P = (long long)n * s; a.out = raw; a.packed = packed;
    if (mode == INERF_MLP_FP32) return mlp_fp32_launch(a, false, as_stream(stream));
    if (mode == INERF_MLP_BF16) {
        if (!packed) return fail(INERF_E_ARG, "inerf_mlp_fwd: bf16 mode needs packed weights");
        return mlp_bf16_launch(a, false, as_stream(stream));
    }
    if (mode == INERF_MLP_F16X2) {
        if (!packed) return fail(INERF_E_ARG, "inerf_mlp_fwd: fp16x2 mode needs packed weights");
        return mlp_f16x2_launch(a, false, as_stream(stream));
    }
    if (mode == INERF_MLP_F16X2_EMB)
        return fail(INERF_E_UNSUPPORTED, "inerf_mlp_fwd: INERF_MLP_F16X2_EMB is the embedded-row mode of inerf_mlp_fwd_embedded; use INERF_MLP_F16X2");
    return fail(INERF_E_UNSUPPORTED, "inerf_mlp_fwd: unknown mode");
}

extern "C" int inerf_mlp_fwd_trace(int mode, const InerfNetDims* dims, const float* const* params_host, const void* packed,
                                   const float* cond, const float* rays, int ray_stride, const float* z, int n, int s,
                                   float* raw, float* trace, void* stream) {
    MlpArgs a{};
    int rc = fill_args(a, dims, params_host, cond);
    if (rc) return rc;
    if (mode != INERF_MLP_BF16) return fail(INERF_E_UNSUPPORTED, "inerf_mlp_fwd_trace: only the bf16 kernel has a trace build");
    if (n <= 0 || s <= 0 || ray_stride < 11) return fail(INERF_E_SHAPE, "inerf_mlp_fwd_trace: bad n/s/ray_stride");
    if (!rays || !z || !raw || !trace || !packed) return fail(INERF_E_ARG, "inerf_mlp_fwd_trace: NULL pointer");
    a.rays = rays; a.ray_stride = ray_stride; a.z = z; a.s = s;
    a.P = (long long)n * s; a.out = raw; a.packed = packed; a.trace = trace;
    return mlp_bf16_launch(a, false, as_stream(stream));
}

extern "C" int inerf_mlp_train_sizes(const InerfNetDims* dims, int64_t n_points, size_t* acts_floats, size_t* deltas_floats,
                                     size_t* scratch_bytes) {
    int rc = check_dims(dims);
    if (rc) return rc;
    if (n_points < 0 || !acts_floats || !deltas_floats || !scratch_bytes) return fail(INERF_E_ARG, "inerf_mlp_train_sizes: bad argument");
    const size_t p64 = (size_t)((n_points + 63) / 64) * 64;
    *acts_floats = p64 * SAVE_W;
    *deltas_floats = p64 * DELTA_W;
    *scratch_bytes = mlp_fp32_bwd_args_bytes();
    return INERF_OK;
}

extern "C" int inerf_mlp_fwd_train(const InerfNetDims* dims, const float* const* params_host, const float* cond,
                                   const float* rays, int ray_stride, const float* z, int n, int s, const float* x,
                                   int64_t p_embedded, float* raw, float* acts, void* stream) {
    MlpArgs a{};
    int rc = fill_args(a, dims, params_host, cond);
    if (rc) return rc;
    if (!raw || !acts) return fail(INERF_E_ARG, "inerf_mlp_fwd_train: NULL pointer");
    if (((uintptr_t)raw | (uintptr_t)acts) & 15) return fail(INERF_E_ALIGN, "inerf_mlp_fwd_train: raw/acts must be 16-byte aligned");
    a.out = raw; a.save = acts;
    if (x) {
        if (p_embedded <= 0) return p_embedded == 0 ? INERF_OK : fail(INERF_E_SHAPE, "inerf_mlp_fwd_train: p < 0");
        a.x = x; a.P = p_embedded; a.s = 1;
        return mlp_fp32_launch(a, true, as_stream(stream));
    }
    if (n < 0 || s <= 0 || ray_stride < 11) return fail(INERF_E_SHAPE, "inerf_mlp_fwd_train: bad n/s/ray_stride");
    if (n == 0) return INERF_OK;
    if (!rays || !z) return fail(INERF_E_ARG, "inerf_mlp_fwd_train: NULL pointer");
    a.rays = rays; a.ray_stride = ray_stride; a.z = z; a.s = s; a.P = (long long)n * s;
    return mlp_fp32_launch(a, false, as_stream(stream));
}

extern "C" int inerf_mlp_bwd(const InerfNetDims* dims, const float* const* params_host, float* const* grads_host,
                             const float* aud, const float* expr, const float* latent, const float* acts, float* deltas,
                             const float* d_raw, int64_t n_points, float* d_cond, void* scratch, void* stream) {
    int rc = check_dims(dims);
    if (rc) return rc;
    if (n_points < 0) return fail(INERF_E_SHAPE, "inerf_mlp_bwd: n_points < 0");
    if (n_points == 0) return INERF_OK;
    if (!params_host || !grads_host || !acts || !deltas || !d_raw || !scratch) return fail(INERF_E_ARG, "inerf_mlp_bwd: NULL pointer");
    if ((rc = check_bwd_args("inerf_mlp_bwd", dims, params_host, grads_host, aud, expr, latent, d_cond))) return rc;
    if (((uintptr_t)acts | (uintptr_t)deltas | (uintptr_t)d_raw) & 15) return fail(INERF_E_ALIGN, "inerf_mlp_bwd: acts/deltas/d_raw must be 16-byte aligned");
    return mlp_fp32_bwd_launch(dims, params_host, grads_host, aud, expr, latent, acts, deltas, d_raw, n_points, d_cond, scratch,
                               as_stream(stream));
}

extern "C" int inerf_debug_hang_info(int32_t* out8) {
    if (!out8) return fail(INERF_E_ARG, "inerf_debug_hang_info: NULL");
    return mlp_bf16_hang_info(out8);
}

extern "C" int inerf_mlp_fwd_embedded(int mode, const InerfNetDims* dims, const float* const* params_host,
                                      const void* packed, const float* cond, const float* x, int64_t p, float* out,
                                      void* stream) {
    MlpArgs a{};
    int rc = fill_args(a, dims, params_host, cond);
    if (rc) return rc;
    if (p < 0) return fail(INERF_E_SHAPE, "inerf_mlp_fwd_embedded: p < 0");
    if (p == 0) return INERF_OK;
    if (!x || !out) return fail(INERF_E_ARG, "inerf_mlp_fwd_embedded: NULL pointer");
    if ((uintptr_t)out & 15) return fail(INERF_E_ALIGN, "inerf_mlp_fwd_embedded: out must be 16-byte aligned");
    a.x = x; a.P = p; a.out = out; a.packed = packed; a.s = 1;
    if (mode == INERF_MLP_FP32) return mlp_fp32_launch(a, true, as_stream(stream));
    if (mode == INERF_MLP_BF16) {
        if (!packed) return fail(INERF_E_ARG, "inerf_mlp_fwd_embedded: bf16 mode needs packed weights (INERF_MLP_BF16_EMB)");
        return mlp_bf16_launch(a, true, as_stream(stream));
    }
    if (mode == INERF_MLP_F16X2_EMB) {
        if (!packed) return fail(INERF_E_ARG, "inerf_mlp_fwd_embedded: fp16x2 mode needs packed weights (INERF_MLP_F16X2_EMB)");
        return mlp_f16x2_launch(a, true, as_stream(stream));
    }
    if (mode == INERF_MLP_F16X2)      // the two fp16x2 blobs cannot be told apart: embedded rows take the mode of their own blob
        return fail(INERF_E_UNSUPPORTED, "inerf_mlp_fwd_embedded: fp16x2 on embedded rows is mode INERF_MLP_F16X2_EMB, with that mode's packed blob");
    return fail(INERF_E_UNSUPPORTED, "inerf_mlp_fwd_embedded: unknown mode");
}

// ---- training, bf16 tensor-core mode -----------------------------------------------------------------------------------------

extern "C" int inerf_mlp_train_sizes_bf16(const InerfNetDims* dims, int64_t n_points, size_t* acts_bytes, size_t* mask_bytes,
                                          size_t* deltas_bytes, size_t* scratch_bytes) {
    int rc = check_dims(dims);
    if (rc) return rc;
    if (n_points < 0 || !acts_bytes || !mask_bytes || !deltas_bytes || !scratch_bytes) return fail(INERF_E_ARG, "inerf_mlp_train_sizes_bf16: bad argument");
    const size_t n_tiles = (size_t)((n_points + 255) / 256) * 2;          // 128-point tiles, two per kernel iteration
    *acts_bytes = n_tiles * TRAIN_IMGS * 16384;
    *deltas_bytes = n_tiles * TRAIN_IMGS * 16384;
    *mask_bytes = n_tiles * TRAIN_MASK_WORDS * 128 * sizeof(uint32_t);
    *scratch_bytes = mlp_bf16_dw_scratch_bytes();
    return INERF_OK;
}

extern "C" int inerf_mlp_fwd_train_bf16(const InerfNetDims* dims, const float* const* params_host, const void* packed, const float* cond,
                                        const float* rays, int ray_stride, const float* z, int n, int s, float* raw, void* acts,
                                        void* mask, void* stream) {
    MlpArgs a{};
    int rc = fill_args(a, dims, params_host, cond);
    if (rc) return rc;
    if (n < 0 || s <= 0 || ray_stride < 11) return fail(INERF_E_SHAPE, "inerf_mlp_fwd_train_bf16: bad n/s/ray_stride");
    if (n == 0) return INERF_OK;
    if (!rays || !z || !raw || !packed || !acts || !mask) return fail(INERF_E_ARG, "inerf_mlp_fwd_train_bf16: NULL pointer");
    if (((uintptr_t)raw | (uintptr_t)acts | (uintptr_t)mask) & 15) return fail(INERF_E_ALIGN, "inerf_mlp_fwd_train_bf16: raw/acts/mask must be 16-byte aligned");
    a.rays = rays; a.ray_stride = ray_stride; a.z = z; a.s = s; a.P = (long long)n * s; a.out = raw; a.packed = packed;
    a.save_img = reinterpret_cast<uint8_t*>(acts); a.save_mask = reinterpret_cast<uint32_t*>(mask);
    return mlp_bf16_launch(a, false, as_stream(stream));
}

extern "C" int inerf_mlp_fwd_train_bf16_embedded(const InerfNetDims* dims, const float* const* params_host, const void* packed,
                                                 const float* cond, const float* x, int64_t p, float* raw, void* acts, void* mask,
                                                 void* stream) {
    MlpArgs a{};
    int rc = fill_args(a, dims, params_host, cond);
    if (rc) return rc;
    if (p < 0) return fail(INERF_E_SHAPE, "inerf_mlp_fwd_train_bf16_embedded: p < 0");
    if (p == 0) return INERF_OK;
    if (!x || !raw || !packed || !acts || !mask) return fail(INERF_E_ARG, "inerf_mlp_fwd_train_bf16_embedded: NULL pointer");
    if (((uintptr_t)x | (uintptr_t)raw | (uintptr_t)acts | (uintptr_t)mask) & 15)
        return fail(INERF_E_ALIGN, "inerf_mlp_fwd_train_bf16_embedded: x/raw/acts/mask must be 16-byte aligned");
    a.x = x; a.P = p; a.s = 1; a.out = raw; a.packed = packed;
    a.save_img = reinterpret_cast<uint8_t*>(acts); a.save_mask = reinterpret_cast<uint32_t*>(mask);
    return mlp_bf16_launch(a, true, as_stream(stream));
}

extern "C" int inerf_mlp_bwd_bf16(const InerfNetDims* dims, const float* const* params_host, const void* packed_t,
                                  float* const* grads_host, const float* aud, const float* expr, const float* latent, const void* acts,
                                  const void* mask, void* deltas, const float* d_raw, int64_t n_points, float* d_cond, void* scratch,
                                  void* stream) {
    int rc = check_dims(dims);
    if (rc) return rc;
    if (n_points < 0) return fail(INERF_E_SHAPE, "inerf_mlp_bwd_bf16: n_points < 0");
    if (n_points == 0) return INERF_OK;
    if (!params_host || !grads_host || !packed_t || !acts || !mask || !deltas || !d_raw || !scratch) return fail(INERF_E_ARG, "inerf_mlp_bwd_bf16: NULL pointer");
    if ((rc = check_bwd_args("inerf_mlp_bwd_bf16", dims, params_host, grads_host, aud, expr, latent, d_cond))) return rc;
    if (((uintptr_t)acts | (uintptr_t)deltas | (uintptr_t)d_raw | (uintptr_t)packed_t | (uintptr_t)mask) & 15)
        return fail(INERF_E_ALIGN, "inerf_mlp_bwd_bf16: buffers must be 16-byte aligned");
    cudaStream_t st = as_stream(stream);
    rc = mlp_bf16_bwd_chain_launch(dims, params_host, packed_t, reinterpret_cast<const uint32_t*>(mask), d_raw,
                                   reinterpret_cast<uint8_t*>(deltas), n_points, st);
    if (rc) return rc;
    const long long n_tiles = ((n_points + 255) / 256) * 2;
    rc = mlp_bf16_dw_launch(dims, grads_host, reinterpret_cast<const uint8_t*>(deltas), reinterpret_cast<const uint8_t*>(acts), n_tiles,
                            scratch, st);
    if (rc) return rc;
    if (dims->dim_aud + dims->dim_expr + dims->dim_latent > 0) rc = mlp_bwd_cond_launch(dims, params_host, grads_host, aud, expr, latent, d_cond, st);
    return rc;
}
