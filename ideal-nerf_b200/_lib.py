"""ctypes binding of libinerf_b200.so (the C ABI declared in include/inerf_b200.h) and its builder.

The library is the product: there is no Python / PyTorch / CPU fallback.  ``lib()`` raises if the
shared object has not been built, and every entry point raises when the current device is not
sm_100 -- nothing here routes to ``oracle/``.
"""
import ctypes
import os
import shutil
import subprocess

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
REPO_ROOT = os.path.dirname(PKG_DIR)
CSRC = os.path.join(PKG_DIR, "csrc")
SO_PATH = os.environ.get("INERF_SO") or os.path.join(PKG_DIR, "libinerf_b200.so")     # INERF_SO: profiling builds only
SOURCES = ["api.cu", "rays.cu", "composite.cu", "sample_pdf.cu", "mlp_api.cu", "mlp_fp32.cu", "mlp_fp32_bwd.cu", "mlp_bf16.cu", "mlp_bf16_bwd.cu",
           "mlp_bf16_dw.cu", "mlp_f16x2.cu", "audio_net.cu", "render_fused.cu", "pixel_sampler.cu", "image_metrics.cu",
           "lpips.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "--shared"]

INERF_MLP_FP32, INERF_MLP_BF16, INERF_MLP_BF16_BWD, INERF_MLP_F16X2, INERF_MLP_BF16_EMB, INERF_MLP_F16X2_EMB = 0, 1, 2, 3, 4, 5
INERF_PDF_EXACT_TORCH_CPU, INERF_PDF_FAST = 0, 1
N_PARAMS = 26

c_f32p = ctypes.c_void_p     # device pointers travel as opaque addresses
c_stream = ctypes.c_void_p


class InerfNetDims(ctypes.Structure):
    _fields_ = [("dim_aud", ctypes.c_int32), ("dim_expr", ctypes.c_int32), ("dim_latent", ctypes.c_int32),
                ("width", ctypes.c_int32), ("depth", ctypes.c_int32), ("in_xyz", ctypes.c_int32),
                ("in_views", ctypes.c_int32)]


ParamArray = ctypes.c_void_p * N_PARAMS


class InerfRenderNet(ctypes.Structure):
    """One FaceNeRF as inerf_render_rays_fused takes it (include/inerf_b200.h)."""
    _fields_ = [("dims", InerfNetDims), ("params_host", ctypes.POINTER(ctypes.c_void_p)), ("packed", ctypes.c_void_p),
                ("aud", ctypes.c_void_p), ("expr", ctypes.c_void_p), ("latent", ctypes.c_void_p)]


class InerfRenderArgs(ctypes.Structure):
    _fields_ = ([(k, ctypes.c_int32) for k in ("mode", "n", "n_samples", "n_importance", "perturb", "lindisp", "white_bkgd")] +
                [("rays", ctypes.c_void_p), ("ray_stride", ctypes.c_int32)] +
                [(k, ctypes.c_int32) for k in ("gen_rays", "H", "W", "first")] +
                [(k, ctypes.c_float) for k in ("focal", "cx", "cy", "near_", "far_")] +
                [("c2w", ctypes.c_void_p), ("c2w_row_stride", ctypes.c_int32), ("bc_rgb", ctypes.c_void_p), ("t_vals", ctypes.c_void_p),
                 ("u_vals", ctypes.c_void_p), ("rng_state", ctypes.c_void_p), ("coarse", InerfRenderNet), ("fine", InerfRenderNet)] +
                [(k, ctypes.c_void_p) for k in ("rgb_map", "disp_map", "acc_map", "depth_map", "last_weight", "rgb0", "disp0", "acc0", "z_std",
                                                "weights", "z_vals", "rgb_map_fg", "rgb_map_fg0", "last_weight0", "nonfinite", "workspace")] +
                [("workspace_bytes", ctypes.c_size_t)])


class InerfPixelSampleArgs(ctypes.Structure):
    _fields_ = ([(k, ctypes.c_int32) for k in ("H", "W", "n_frames")] + [("k", ctypes.c_int32 * 4)] +
                [(k, ctypes.c_int32) for k in ("first", "count")] + [(k, ctypes.c_float) for k in ("focal", "cx", "cy", "near_", "far_")] +
                [(k, ctypes.c_void_p) for k in ("frame_index", "bounds", "torso_bits", "poses", "frames", "bc_img", "rng_state", "rays", "target",
                                                "bc_rgb", "coords")])


INERF_PIXEL_SAMPLER_MAX_K = 4096
INERF_PIXEL_SAMPLER_MAX_PIXELS = 1 << 22
INERF_IMAGE_METRICS_MAX_PIXELS = 1 << 24
INERF_LPIPS_N_PARAMS = 15
INERF_LPIPS_MAX_ROWS = 65535

NF_BITS = {"rgb_map": 1, "disp_map": 2, "acc_map": 4, "rgb0": 8, "disp0": 16, "acc0": 32, "z_std": 64, "last_weight": 128}     # INERF_NF_*

_I, _F, _P, _L, _SZP = ctypes.c_int, ctypes.c_float, ctypes.c_void_p, ctypes.c_int64, ctypes.POINTER(ctypes.c_size_t)
_DIMS = ctypes.POINTER(InerfNetDims)
_PARAMS = ctypes.POINTER(ctypes.c_void_p)

# name -> (restype, argtypes); must list every symbol include/inerf_b200.h declares
SIGNATURES = {
    "inerf_version": (_I, []),
    "inerf_last_error": (ctypes.c_char_p, []),
    "inerf_device_check": (_I, []),
    "inerf_sizeof": (ctypes.c_size_t, [_I]),
    "inerf_get_rays": (_I, [_I, _I, _F, _F, _F, _P, _I, _F, _F, _P, _P]),
    "inerf_get_rays_at": (_I, [_P, _I, _F, _F, _F, _P, _I, _F, _F, _P, _P]),
    "inerf_get_rays_range": (_I, [_I, _I, _F, _F, _F, _P, _I, _F, _F, _I, _I, _P, _P]),
    "inerf_rng_advance": (_I, [_P, ctypes.c_uint64, _P]),
    "inerf_sample_coarse_rng": (_I, [_P, _I, _I, _I, _P, _P, _I, _P, _P]),
    "inerf_flag_nonfinite": (_I, [_PARAMS, ctypes.POINTER(ctypes.c_int64), _I, _P, _P]),
    "inerf_importance_sample_rng": (_I, [_P, _P, _I, _I, _I, _P, ctypes.c_uint32, _P, _P, _P, _P]),
    "inerf_pack_rays": (_I, [_P, _P, _I, _F, _F, _P, _P]),
    "inerf_posenc": (_I, [_P, _L, _I, _I, _P, _P]),
    "inerf_to8b": (_I, [_P, _L, _P, _P]),
    "inerf_sample_coarse": (_I, [_P, _I, _I, _I, _P, _P, _I, _P, _P]),
    "inerf_composite_fwd": (_I, [_P, _P, _P, _I, _P, _P, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P]),
    "inerf_composite_bwd": (_I, [_P, _P, _P, _I, _P, _P, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P]),
    "inerf_mse_pair": (_I, [_P, _P, _P, _L, _P, _P, _P, _P]),
    "inerf_head_torso_blend": (_I, [_P, _P, _P, _I, _P, _P]),
    "inerf_head_torso_mse_pair": (_I, [_P, _P, _P, _P, _P, _P, _P, _L, _P, _P, _P, _P, _P, _P]),
    "inerf_head_torso_to8b": (_I, [_P, _P, _P, _L, _P, _P, _P]),
    "inerf_sample_pdf": (_I, [_P, _I, _P, _I, _I, _I, _I, _P, _I, _I, _P, _P, _P, _I, _P, _P, _P]),
    "inerf_importance_sample": (_I, [_P, _P, _I, _I, _I, _P, _I, _I, _P, _P, _P, _P, _P]),
    "inerf_render_workspace_bytes": (_I, [ctypes.POINTER(InerfRenderArgs), _SZP]),
    "inerf_render_rays_fused": (_I, [ctypes.POINTER(InerfRenderArgs), _P]),
    "inerf_debug_render_stage_ms": (_I, [ctypes.POINTER(InerfRenderArgs), _P, ctypes.POINTER(ctypes.c_float)]),
    "inerf_mlp_cond_floats": (_I, [_DIMS, _SZP]),
    "inerf_mlp_fold_cond": (_I, [_DIMS, _PARAMS, _P, _P, _P, _P, _P]),
    "inerf_mlp_packed_bytes": (_I, [_I, _DIMS, _SZP]),
    "inerf_mlp_pack": (_I, [_I, _DIMS, _PARAMS, _P, _P]),
    "inerf_mlp_fwd": (_I, [_I, _DIMS, _PARAMS, _P, _P, _P, _I, _P, _I, _I, _P, _P]),
    "inerf_mlp_fwd_trace": (_I, [_I, _DIMS, _PARAMS, _P, _P, _P, _I, _P, _I, _I, _P, _P, _P]),
    "inerf_mlp_train_sizes": (_I, [_DIMS, _L, _SZP, _SZP, _SZP]),
    "inerf_mlp_fwd_train": (_I, [_DIMS, _PARAMS, _P, _P, _I, _P, _I, _I, _P, _L, _P, _P, _P]),
    "inerf_mlp_bwd": (_I, [_DIMS, _PARAMS, _PARAMS, _P, _P, _P, _P, _P, _P, _L, _P, _P, _P]),
    "inerf_mlp_train_sizes_bf16": (_I, [_DIMS, _L, _SZP, _SZP, _SZP, _SZP]),
    "inerf_mlp_fwd_train_bf16": (_I, [_DIMS, _PARAMS, _P, _P, _P, _I, _P, _I, _I, _P, _P, _P, _P]),
    "inerf_mlp_fwd_train_bf16_embedded": (_I, [_DIMS, _PARAMS, _P, _P, _P, _L, _P, _P, _P, _P]),
    "inerf_mlp_bwd_bf16": (_I, [_DIMS, _PARAMS, _P, _PARAMS, _P, _P, _P, _P, _P, _P, _P, _L, _P, _P, _P]),
    "inerf_audio_net_fwd": (_I, [_PARAMS, _P, _I, _I, _P, _P]),
    "inerf_audio_att_fwd": (_I, [_PARAMS, _P, _I, _I, _I, _P, _P]),
    "inerf_audio_net_bwd": (_I, [_PARAMS, _PARAMS, _P, _P, _I, _I, _P]),
    "inerf_audio_att_bwd": (_I, [_PARAMS, _PARAMS, _P, _P, _I, _I, _I, _P, _P]),
    "inerf_debug_hang_info": (_I, [ctypes.POINTER(ctypes.c_int32)]),
    "inerf_mlp_fwd_embedded": (_I, [_I, _DIMS, _PARAMS, _P, _P, _P, _L, _P, _P]),
    "inerf_pixel_sampler_workspace_bytes": (_I, [ctypes.POINTER(InerfPixelSampleArgs), _SZP]),
    "inerf_sample_train_pixels": (_I, [ctypes.POINTER(InerfPixelSampleArgs), _P, ctypes.c_size_t, _P]),
    "inerf_image_metrics": (_I, [_P, _P, _P, _P, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, _P, _P, _P, _P]),
    "inerf_masked_sse": (_I, [_P, _P, _P, _P, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, _P, _P, _P]),
    "inerf_lpips_workspace_bytes": (_I, [ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, _SZP]),
    "inerf_lpips": (_I, [_PARAMS, _P, _P, _P, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, _P, ctypes.c_size_t, _P, _P]),
}

_lib = None


def _stale():
    if not os.path.exists(SO_PATH):
        return True
    t = os.path.getmtime(SO_PATH)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(REPO_ROOT, "include", "inerf_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """Compile csrc/*.cu for sm_100a into ideal-nerf_b200/libinerf_b200.so (nvcc cross-compiles without a GPU).  One object per source,
    compiled in parallel and cached under build/obj by (source, header) modification time, then one device link."""
    if not force and not _stale():
        return SO_PATH
    from concurrent.futures import ThreadPoolExecutor
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: cannot build libinerf_b200.so")
    extra = os.environ.get("INERF_EXTRA_NVCC", "").split()
    objdir = os.path.join(REPO_ROOT, "build", "obj" + ("_" + str(abs(hash(tuple(extra))) % 10 ** 8) if extra else ""))
    os.makedirs(objdir, exist_ok=True)
    hdrs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))] + [os.path.join(REPO_ROOT, "include", "inerf_b200.h")]
    t_hdr = max(os.path.getmtime(h) for h in hdrs)
    flags = [f for f in NVCC_FLAGS if f != "--shared"]

    def compile_one(src):
        obj = os.path.join(objdir, src[:-3] + ".o")
        spath = os.path.join(CSRC, src)
        if not force and os.path.exists(obj) and os.path.getmtime(obj) > max(t_hdr, os.path.getmtime(spath)):
            return obj, ""
        r = subprocess.run([nvcc] + flags + extra + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", obj, spath],
                           cwd=CSRC, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n" + r.stdout + r.stderr)
        return obj, r.stderr

    with ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 4)) as ex:
        res = list(ex.map(compile_one, SOURCES))
    r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "--shared", "-Xcompiler", "-fPIC", "-o", SO_PATH + ".tmp"] + [o for o, _ in res],
                       capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc link failed:\n" + r.stdout + r.stderr)
    os.replace(SO_PATH + ".tmp", SO_PATH)
    if verbose:
        print("".join(e for _, e in res))
    return SO_PATH


def lib():
    """The loaded C-ABI library.  Fails loudly when it is missing -- there is no fallback path."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise RuntimeError(f"{SO_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(nvcc, sm_100a).  ideal-nerf_b200 has no CPU or PyTorch fallback.")
        L = ctypes.CDLL(SO_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)           # AttributeError here = header/library mismatch
            fn.restype, fn.argtypes = res, args
        for which, struct in ((0, InerfNetDims), (1, InerfRenderNet), (2, InerfRenderArgs), (4, InerfPixelSampleArgs)):      # the ctypes mirrors must match the header
            if L.inerf_sizeof(which) != ctypes.sizeof(struct):
                raise RuntimeError(f"{struct.__name__}: ctypes layout ({ctypes.sizeof(struct)} B) differs from the library's "
                                   f"({L.inerf_sizeof(which)} B); rebuild libinerf_b200.so")
        _lib = L
    return _lib


def check(rc, what):
    if rc != 0:
        msg = lib().inerf_last_error().decode("utf-8", "replace")
        kind = "CUDA error" if rc > 0 else "argument error"
        raise RuntimeError(f"{what}: {kind} {rc}: {msg}")
