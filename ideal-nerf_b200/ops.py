"""Tensor-level wrappers over the C ABI (include/inerf_b200.h) + autograd Functions.

PyTorch supplies device memory, streams and autograd bookkeeping only; every op below is one
hand-written CUDA kernel launched through ctypes on the current stream.
"""
import ctypes
import os

import torch

from . import _lib
from ._lib import InerfNetDims, ParamArray, check

_tables = {}

# ---- launch accounting (bench.py reads these; one entry per C-ABI kernel launch) -----------------
LAUNCHES = {"count": 0}
# inference render_rays through the single fused entry point (inerf_render_rays_fused); INERF_FUSED_RENDER=0 keeps the stage-by-stage calls
FUSED_RENDER = os.environ.get("INERF_FUSED_RENDER", "1") != "0"
_timing = None          # None, or dict name -> list of (start_event, end_event)


class kernel_timing:
    """Context manager: record a CUDA-event pair around every kernel launch, on the launching stream."""

    def __enter__(self):
        global _timing
        _timing = {}
        return self

    def __exit__(self, *exc):
        global _timing
        self.events, _timing = _timing, None
        return False

    def summary(self):
        """name -> (launches, total_ms).  Call after a torch.cuda.synchronize()."""
        return {k: (len(v), sum(a.elapsed_time(b) for a, b in v)) for k, v in self.events.items()}


def call(name, fn, *args, launches=1):
    """Launch one C-ABI entry point: count its kernel launches, optionally bracket it with events, raise on error."""
    LAUNCHES["count"] += launches
    if _timing is None:
        check(fn(*args), name)
        return
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    check(fn(*args), name)
    b.record()
    _timing.setdefault(name, []).append((a, b))


def _need_cuda(t, name):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError(f"ideal-nerf_b200: `{name}` must be a CUDA tensor (there is no CPU path)")


def f32c(t, name="tensor"):
    _need_cuda(t, name)
    if t.dtype != torch.float32:
        t = t.float()
    return t if t.is_contiguous() else t.contiguous()


def ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def linspace_table(steps, device):
    """torch.linspace(0,1,steps) evaluated on the CPU (the reference's bits, SURVEY.md 7-1), cached per device."""
    key = (int(steps), str(device))
    if key not in _tables:
        _tables[key] = torch.linspace(0., 1., steps=int(steps)).to(device)
    return _tables[key]


# ------------------------------------------------------------------------------------------------
# rays / encoding / coarse depths
# ------------------------------------------------------------------------------------------------

def get_rays_packed(H, W, focal, c2w, near, far, cx=None, cy=None):
    """(H*W, 11) packed rays for a full frame.  helper.py:228-243 + audio_exp_nerf.py:409-427."""
    c2w = f32c(c2w, "c2w")
    if c2w.dim() != 2 or c2w.shape[0] < 3 or c2w.shape[1] != 4:
        raise ValueError("c2w must be (3,4) or (4,4)")
    cx = W * .5 if cx is None else cx
    cy = H * .5 if cy is None else cy
    rays = torch.empty((H * W, 11), device=c2w.device, dtype=torch.float32)
    with torch.cuda.device(c2w.device):
        call("inerf_get_rays", _lib.lib().inerf_get_rays, H, W, float(focal), float(cx), float(cy), ptr(c2w), 4, float(near), float(far),
                                        ptr(rays), stream())
    return rays


def get_rays_range(H, W, focal, c2w, near, far, first, count, cx=None, cy=None):
    """(count, 11) packed rays of the pixels [first, first + count) of the frame: get_rays_packed(...)[first:first + count] without
    generating the rest of the frame (one rank's band when a frame's rays are sharded over several GPUs)."""
    c2w = f32c(c2w, "c2w")
    if c2w.dim() != 2 or c2w.shape[0] < 3 or c2w.shape[1] != 4:
        raise ValueError("c2w must be (3,4) or (4,4)")
    cx = W * .5 if cx is None else cx
    cy = H * .5 if cy is None else cy
    rays = torch.empty((count, 11), device=c2w.device, dtype=torch.float32)
    with torch.cuda.device(c2w.device):
        call("inerf_get_rays_range", _lib.lib().inerf_get_rays_range, H, W, float(focal), float(cx), float(cy), ptr(c2w), 4, float(near),
             float(far), int(first), int(count), ptr(rays), stream())
    return rays


def get_rays_at(coords, focal, c2w, near, far, cx, cy):
    """(n, 11) packed rays of the selected pixels; coords (n, 2) int64 = (row, col).  Same bits as get_rays_packed(...)[row * W + col]."""
    _need_cuda(coords, "coords")
    coords = coords.to(torch.int64).contiguous()
    c2w = f32c(c2w, "c2w")
    n = coords.shape[0]
    rays = torch.empty((n, 11), device=c2w.device, dtype=torch.float32)
    with torch.cuda.device(c2w.device):
        call("inerf_get_rays_at", _lib.lib().inerf_get_rays_at, ptr(coords), n, float(focal), float(cx), float(cy), ptr(c2w), c2w.stride(0),
             float(near), float(far), ptr(rays), stream())
    return rays


def pack_rays(rays_o, rays_d, near, far):
    rays_o = f32c(rays_o.reshape(-1, 3), "rays_o")
    rays_d = f32c(rays_d.reshape(-1, 3), "rays_d")
    n = rays_o.shape[0]
    rays = torch.empty((n, 11), device=rays_o.device, dtype=torch.float32)
    with torch.cuda.device(rays.device):
        call("inerf_pack_rays", _lib.lib().inerf_pack_rays, ptr(rays_o), ptr(rays_d), n, float(near), float(far), ptr(rays), stream())
    return rays


def posenc(x, n_freqs):
    x = f32c(x, "x")
    dims = x.shape[-1]
    flat = x.reshape(-1, dims)
    out = torch.empty((flat.shape[0], dims * (1 + 2 * n_freqs)), device=x.device, dtype=torch.float32)
    with torch.cuda.device(x.device):
        call("inerf_posenc", _lib.lib().inerf_posenc, ptr(flat), flat.shape[0], dims, n_freqs, ptr(out), stream())
    return out.reshape(*x.shape[:-1], out.shape[-1])


def to8b(x):
    """(255 * clip(x, 0, 1)).astype(uint8) on the device (helper.py:154)."""
    x = f32c(x, "x")
    out = torch.empty(x.shape, device=x.device, dtype=torch.uint8)
    with torch.cuda.device(x.device):
        call("inerf_to8b", _lib.lib().inerf_to8b, ptr(x), x.numel(), ptr(out), stream())
    return out


def sample_coarse(rays, n_samples, t_rand=None, lindisp=False):
    rays = f32c(rays, "rays")
    n = rays.shape[0]
    t_vals = linspace_table(n_samples, rays.device)
    if t_rand is not None:
        t_rand = f32c(t_rand, "t_rand")
        assert t_rand.shape == (n, n_samples)
    z = torch.empty((n, n_samples), device=rays.device, dtype=torch.float32)
    with torch.cuda.device(rays.device):
        call("inerf_sample_coarse", _lib.lib().inerf_sample_coarse, ptr(rays), n, rays.shape[1], n_samples, ptr(t_vals), ptr(t_rand),
                                             int(bool(lindisp)), ptr(z), stream())
    return z


# ------------------------------------------------------------------------------------------------
# in-kernel random draws (perturb > 0): Philox state per device, {seed, offset} in device memory
# ------------------------------------------------------------------------------------------------
RNG_STREAM_COARSE, RNG_STREAM_PDF, RNG_STREAM_PIXELS = 1, 2, 3
_rng_states = {}


def rng_state(device):
    """The (2,) int64 device tensor {seed, offset} the *_rng kernels read.  Seeded from torch's generator on first use
    (torch.manual_seed before the first stochastic render makes a run reproducible); `seed_rng` re-seeds explicitly."""
    key = torch.device(device).index if torch.device(device).index is not None else torch.cuda.current_device()
    st = _rng_states.get(key)
    if st is None:
        st = torch.tensor([torch.initial_seed() & 0x7FFFFFFFFFFFFFFF, 0], dtype=torch.int64, device=torch.device("cuda", key))
        _rng_states[key] = st
    return st


def seed_rng(seed, device=None, offset=0):
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    rng_state(dev).copy_(torch.tensor([int(seed) & 0x7FFFFFFFFFFFFFFF, int(offset)], dtype=torch.int64))


def rng_advance(state, increment=1):
    """offset += increment on the device (one tiny launch; graph-capturable): the next stochastic call draws fresh numbers."""
    with torch.cuda.device(state.device):
        call("inerf_rng_advance", _lib.lib().inerf_rng_advance, ptr(state), int(increment), stream())


def sample_coarse_rng(rays, n_samples, state=None, lindisp=False, advance=True):
    """Stratified depths with the jitter drawn in the kernel (audio_exp_nerf.py:321-328 without the torch.rand tensor)."""
    rays = f32c(rays, "rays")
    n = rays.shape[0]
    state = rng_state(rays.device) if state is None else state
    t_vals = linspace_table(n_samples, rays.device)
    z = torch.empty((n, n_samples), device=rays.device, dtype=torch.float32)
    with torch.cuda.device(rays.device):
        call("inerf_sample_coarse_rng", _lib.lib().inerf_sample_coarse_rng, ptr(rays), n, rays.shape[1], n_samples, ptr(t_vals), ptr(state),
             int(bool(lindisp)), ptr(z), stream())
    if advance:
        rng_advance(state)
    return z


def importance_sample_rng(z_coarse, w_coarse, n_importance, state=None, stream_id=RNG_STREAM_PDF, want_samples=False, advance=True):
    """importance_sample for perturb > 0 with u ~ U[0,1) drawn in the kernel as sorted order statistics (helper.py:282-283 without the
    torch.rand tensor and without a sort).  Returns (z_samples|None, z_merged, z_std)."""
    z_coarse, w_coarse = f32c(z_coarse.detach(), "z_vals"), f32c(w_coarse.detach(), "weights")
    n, s1 = z_coarse.shape
    dev = z_coarse.device
    state = rng_state(dev) if state is None else state
    zs = torch.empty((n, n_importance), device=dev) if want_samples else None
    zm = torch.empty((n, s1 + n_importance), device=dev)
    zstd = torch.empty((n,), device=dev)
    with torch.cuda.device(dev):
        call("inerf_importance_sample_rng", _lib.lib().inerf_importance_sample_rng, ptr(z_coarse), ptr(w_coarse), n, s1, n_importance,
             ptr(state), int(stream_id), ptr(zs), ptr(zm), ptr(zstd), stream())
    if advance:
        rng_advance(state)
    return zs, zm, zstd


def sample_train_pixels(frame_index, budgets, bounds, torso_bits, poses, frames, bc_img, focal, cx, cy, near, far, first=0, count=None,
                        state=None, want_coords=False, advance=True):
    """The training batch of frame `frame_index` (int64 device scalar) drawn on the device (include/inerf_b200.h, inerf_sample_train_pixels):
    budgets = (rect, norect, mouth, torso) rows; bounds (F, 8) int32, torso_bits (F, ceil(H*W/32)) int32 / uint32 bits, poses (F, 3, 4)
    fp32, frames (F, H, W, 3) uint8, bc_img (H, W, 3) fp32.  Returns (rays (count, 11), target (count, 3), bc_rgb (count, 3),
    coords (count, 2) int64 or None) for the rows [first, first + count) of the N_rand = sum(budgets) rows.  Draws from `state` (default:
    the device's Philox state), whose offset is advanced afterwards when `advance`."""
    dev = frames.device
    for t, name, dt in ((frame_index, "frame_index", torch.int64), (bounds, "bounds", torch.int32), (torso_bits, "torso_bits", torch.int32),
                        (poses, "poses", torch.float32), (frames, "frames", torch.uint8), (bc_img, "bc_img", torch.float32)):
        _need_cuda(t, name)
        if t.dtype != dt or not t.is_contiguous() or t.device != dev:
            raise ValueError(f"sample_train_pixels: `{name}` must be a contiguous {dt} tensor on {dev}")
    F, H, W = frames.shape[0], frames.shape[1], frames.shape[2]
    n_rand = sum(int(k) for k in budgets)
    count = n_rand - int(first) if count is None else int(count)
    state = rng_state(dev) if state is None else state
    rays = torch.empty((count, 11), device=dev, dtype=torch.float32)
    target = torch.empty((count, 3), device=dev, dtype=torch.float32)
    bc_rgb = torch.empty((count, 3), device=dev, dtype=torch.float32)
    coords = torch.empty((count, 2), device=dev, dtype=torch.int64) if want_coords else None
    a = _lib.InerfPixelSampleArgs(H=H, W=W, n_frames=F, k=(ctypes.c_int32 * 4)(*[int(k) for k in budgets]), first=int(first), count=count,
                                  focal=float(focal), cx=float(cx), cy=float(cy), near_=float(near), far_=float(far),
                                  frame_index=frame_index.data_ptr(), bounds=bounds.data_ptr(), torso_bits=torso_bits.data_ptr(),
                                  poses=poses.data_ptr(), frames=frames.data_ptr(), bc_img=bc_img.data_ptr(), rng_state=state.data_ptr(),
                                  rays=rays.data_ptr(), target=target.data_ptr(), bc_rgb=bc_rgb.data_ptr(),
                                  coords=coords.data_ptr() if want_coords else None)
    L = _lib.lib()
    nbytes = ctypes.c_size_t(0)
    check(L.inerf_pixel_sampler_workspace_bytes(ctypes.byref(a), ctypes.byref(nbytes)), "inerf_pixel_sampler_workspace_bytes")
    ws = torch.empty((nbytes.value,), device=dev, dtype=torch.uint8)
    with torch.cuda.device(dev):
        call("inerf_sample_train_pixels", L.inerf_sample_train_pixels, ctypes.byref(a), ptr(ws), nbytes.value, stream(), launches=4)
    if advance:
        rng_advance(state)
    return rays, target, bc_rgb, coords


def image_metrics(pred_u8, gt_frames, frame_index, bounds=None):
    """Scores of rendered frames against ground truth on the device (include/inerf_b200.h, inerf_image_metrics): pred_u8 (B, H, W, 3)
    uint8, gt_frames (F, H, W, 3) uint8 (e.g. DeviceHeadDataset.frames), frame_index (B,) int64 device tensor selecting each row's ground
    truth, bounds (F, 8) int32 face-rect / mouth boxes (DeviceHeadDataset.bounds) or None.  Returns device tensors {sse (B, 3) int64,
    npix (B, 3) int64: full frame, face rect, mouth box (0 without bounds); ssim (B,) float64: the mean SSIM over the channels and the
    (H - 10) x (W - 10) positions whose window lies inside the frame}.  A row whose index is outside [0, F) scores 0 everywhere.
    One kernel and no host synchronise: the call may be captured in a CUDA graph."""
    dev = gt_frames.device
    for t, name, dt in ((pred_u8, "pred_u8", torch.uint8), (gt_frames, "gt_frames", torch.uint8), (frame_index, "frame_index", torch.int64),
                        (bounds, "bounds", torch.int32)):
        if t is None:
            continue
        _need_cuda(t, name)
        if t.dtype != dt or not t.is_contiguous() or t.device != dev:
            raise ValueError(f"image_metrics: `{name}` must be a contiguous {dt} tensor on {dev}")
    if gt_frames.dim() != 4 or gt_frames.shape[3] != 3 or pred_u8.dim() != 4 or pred_u8.shape[1:] != gt_frames.shape[1:]:
        raise ValueError(f"image_metrics: pred_u8 {tuple(pred_u8.shape)} and gt_frames {tuple(gt_frames.shape)} must be (B, H, W, 3) and "
                         "(F, H, W, 3)")
    B, F, H, W = pred_u8.shape[0], gt_frames.shape[0], gt_frames.shape[1], gt_frames.shape[2]
    if frame_index.shape != (B,):
        raise ValueError(f"image_metrics: frame_index {tuple(frame_index.shape)} must be ({B},)")
    if bounds is not None and bounds.shape != (F, 8):
        raise ValueError(f"image_metrics: bounds {tuple(bounds.shape)} must be ({F}, 8)")
    new = torch.empty if bounds is not None else torch.zeros           # without bounds the kernel writes column 0 only
    sse, npix = new((B, 3), device=dev, dtype=torch.int64), new((B, 3), device=dev, dtype=torch.int64)
    ssim_sum = torch.empty((B,), device=dev, dtype=torch.float64)
    with torch.cuda.device(dev):
        call("inerf_image_metrics", _lib.lib().inerf_image_metrics, ptr(pred_u8), ptr(gt_frames), ptr(frame_index), ptr(bounds), B, H, W, F,
             ptr(sse), ptr(npix), ptr(ssim_sum), stream())
    return {"sse": sse, "npix": npix, "ssim": ssim_sum / (3 * (H - 10) * (W - 10))}


def masked_sse(pred_u8, gt_frames, frame_index, bits):
    """Squared error of rendered frames over a per-frame pixel mask on the device (include/inerf_b200.h, inerf_masked_sse): pred_u8
    (B, H, W, 3) uint8, gt_frames (F, H, W, 3) uint8, frame_index (B,) int64 device tensor, bits (F, ceil(H*W/32)) int32 holding the uint32
    words of data.torso_bits (e.g. DeviceTorsoDataset.torso_bits).  Returns device tensors (sse (B,) int64 over the 3 channels of the masked
    pixels, npix (B,) int64 masked pixels); a row whose index is outside [0, F) gets zeros.  One kernel and no host synchronise: the call
    may be captured in a CUDA graph."""
    dev = gt_frames.device
    for t, name, dt in ((pred_u8, "pred_u8", torch.uint8), (gt_frames, "gt_frames", torch.uint8), (frame_index, "frame_index", torch.int64),
                        (bits, "bits", torch.int32)):
        _need_cuda(t, name)
        if t.dtype != dt or not t.is_contiguous() or t.device != dev:
            raise ValueError(f"masked_sse: `{name}` must be a contiguous {dt} tensor on {dev}")
    if gt_frames.dim() != 4 or gt_frames.shape[3] != 3 or pred_u8.dim() != 4 or pred_u8.shape[1:] != gt_frames.shape[1:]:
        raise ValueError(f"masked_sse: pred_u8 {tuple(pred_u8.shape)} and gt_frames {tuple(gt_frames.shape)} must be (B, H, W, 3) and "
                         "(F, H, W, 3)")
    B, F, H, W = pred_u8.shape[0], gt_frames.shape[0], gt_frames.shape[1], gt_frames.shape[2]
    if frame_index.shape != (B,):
        raise ValueError(f"masked_sse: frame_index {tuple(frame_index.shape)} must be ({B},)")
    if bits.shape != (F, (H * W + 31) // 32):
        raise ValueError(f"masked_sse: bits {tuple(bits.shape)} must be ({F}, {(H * W + 31) // 32})")
    sse, npix = torch.empty((B,), device=dev, dtype=torch.int64), torch.empty((B,), device=dev, dtype=torch.int64)
    with torch.cuda.device(dev):
        call("inerf_masked_sse", _lib.lib().inerf_masked_sse, ptr(pred_u8), ptr(gt_frames), ptr(frame_index), ptr(bits), B, H, W, F, ptr(sse),
             ptr(npix), stream())
    return sse, npix


# inerf_lpips' 15 parameters in ABI order: conv1..conv5 (weight, bias), then lin0..lin4
LPIPS_CHANNELS = (64, 192, 384, 256, 256)
LPIPS_SHAPES = ([s for cout, cin, k in zip(LPIPS_CHANNELS, (3, 64, 192, 384, 256), (11, 5, 3, 3, 3)) for s in ((cout, cin, k, k), (cout,))] +
                [(c,) for c in LPIPS_CHANNELS])


def lpips(pred_u8, gt_frames, frame_index, weights):
    """LPIPS v0.1 (AlexNet trunk) of rendered frames against ground truth on the device (include/inerf_b200.h, inerf_lpips): pred_u8
    (B, H, W, 3) uint8, gt_frames (F, H, W, 3) uint8 (BGR as stored, e.g. DeviceHeadDataset.frames), frame_index (B,) int64 device tensor
    selecting each row's ground truth, weights the 15 fp32 device tensors of evaluate.load_lpips.  Returns (B,) float32 on the device,
    what lpips.LPIPS(net='alex')(pred, gt) gives each row; a row whose index is outside [0, F) gets 0.  Frames need H, W >= 31.  One C
    call, no host synchronise: the call may be captured in a CUDA graph (its workspace is allocated here, before the launches)."""
    dev = gt_frames.device
    for t, name, dt in ((pred_u8, "pred_u8", torch.uint8), (gt_frames, "gt_frames", torch.uint8), (frame_index, "frame_index", torch.int64)):
        _need_cuda(t, name)
        if t.dtype != dt or not t.is_contiguous() or t.device != dev:
            raise ValueError(f"lpips: `{name}` must be a contiguous {dt} tensor on {dev}")
    if gt_frames.dim() != 4 or gt_frames.shape[3] != 3 or pred_u8.dim() != 4 or pred_u8.shape[1:] != gt_frames.shape[1:]:
        raise ValueError(f"lpips: pred_u8 {tuple(pred_u8.shape)} and gt_frames {tuple(gt_frames.shape)} must be (B, H, W, 3) and "
                         "(F, H, W, 3)")
    B, F, H, W = pred_u8.shape[0], gt_frames.shape[0], gt_frames.shape[1], gt_frames.shape[2]
    if frame_index.shape != (B,):
        raise ValueError(f"lpips: frame_index {tuple(frame_index.shape)} must be ({B},)")
    if len(weights) != len(LPIPS_SHAPES):
        raise ValueError(f"lpips: {len(weights)} weight tensors, need {len(LPIPS_SHAPES)} (evaluate.load_lpips)")
    for i, (t, shape) in enumerate(zip(weights, LPIPS_SHAPES)):
        _need_cuda(t, f"weights[{i}]")
        if t.dtype != torch.float32 or not t.is_contiguous() or t.device != dev or tuple(t.shape) != shape:
            raise ValueError(f"lpips: weights[{i}] must be a contiguous float32 {shape} tensor on {dev}, got {t.dtype} "
                             f"{tuple(t.shape)} on {t.device}")
    L = _lib.lib()
    out = torch.empty((B,), device=dev, dtype=torch.float32)
    if B == 0:
        return out
    nbytes = ctypes.c_size_t(0)
    check(L.inerf_lpips_workspace_bytes(B, H, W, ctypes.byref(nbytes)), "inerf_lpips_workspace_bytes")
    ws = torch.empty((nbytes.value,), device=dev, dtype=torch.uint8)
    params = (ctypes.c_void_p * len(weights))(*[t.data_ptr() for t in weights])
    with torch.cuda.device(dev):
        call("inerf_lpips", L.inerf_lpips, params, ptr(pred_u8), ptr(gt_frames), ptr(frame_index), B, H, W, F, ptr(ws), nbytes.value,
             ptr(out), stream(), launches=13)
    return out


def flag_nonfinite(tensors, flags):
    """OR bit i into the int32 device scalar `flags` when tensors[i] holds a NaN / Inf; ONE launch, no host synchronisation."""
    tensors = [f32c(t, "tensor") for t in tensors]
    k = len(tensors)
    xs = (ctypes.c_void_p * k)(*[t.data_ptr() for t in tensors])
    ns = (ctypes.c_int64 * k)(*[t.numel() for t in tensors])
    with torch.cuda.device(flags.device):
        call("inerf_flag_nonfinite", _lib.lib().inerf_flag_nonfinite, xs, ns, k, ptr(flags), stream())
    return flags


# ------------------------------------------------------------------------------------------------
# compositing
# ------------------------------------------------------------------------------------------------

def _dir_view(rays_d):
    """(pointer tensor, stride) for ray directions given either an (n,3) tensor or a column view of packed rays."""
    _need_cuda(rays_d, "rays_d")
    if rays_d.dtype == torch.float32 and rays_d.dim() == 2 and rays_d.shape[1] == 3 and rays_d.stride(1) == 1 \
            and rays_d.stride(0) >= 3:
        return rays_d, rays_d.stride(0)
    d = f32c(rays_d.reshape(-1, 3), "rays_d")
    return d, 3


class _Composite(torch.autograd.Function):
    @staticmethod
    def forward(ctx, raw, z, rays_d, bc_rgb, noise, white_bkgd, with_fg):
        raw, z, bc_rgb = f32c(raw, "raw"), f32c(z, "z_vals"), f32c(bc_rgb, "bc_rgb")
        n, s = z.shape
        assert raw.shape == (n, s, 4), f"raw {tuple(raw.shape)} vs z {tuple(z.shape)}"
        d, ds = _dir_view(rays_d)
        noise = f32c(noise, "noise") if noise is not None else None
        dev = raw.device
        rgb = torch.empty((n, 3), device=dev); disp = torch.empty((n,), device=dev)
        acc = torch.empty((n,), device=dev); depth = torch.empty((n,), device=dev)
        weights = torch.empty((n, s), device=dev)
        fg = torch.empty((n, 3), device=dev) if with_fg else None
        with torch.cuda.device(dev):
            call("inerf_composite_fwd", _lib.lib().inerf_composite_fwd, ptr(raw), ptr(z), ptr(d), ds, ptr(bc_rgb), ptr(noise), n, s,
                                                 int(bool(white_bkgd)), ptr(rgb), ptr(disp), ptr(acc), ptr(depth),
                                                 ptr(weights), ptr(fg), stream())
        ctx.save_for_backward(raw, z, d, bc_rgb, noise)
        ctx.meta = (ds, int(bool(white_bkgd)), with_fg)
        ctx.set_materialize_grads(False)
        if with_fg:
            return rgb, disp, acc, weights, depth, fg
        return rgb, disp, acc, weights, depth

    @staticmethod
    def backward(ctx, g_rgb, g_disp, g_acc, g_w, g_depth, g_fg=None):
        raw, z, d, bc_rgb, noise = ctx.saved_tensors
        ds, white, with_fg = ctx.meta
        n, s = z.shape
        gs = [None if g is None else f32c(g, "grad") for g in (g_rgb, g_disp, g_acc, g_depth, g_w, g_fg)]
        d_raw = torch.empty_like(raw)
        with torch.cuda.device(raw.device):
            call("inerf_composite_bwd", _lib.lib().inerf_composite_bwd, ptr(raw), ptr(z), ptr(d), ds, ptr(bc_rgb), ptr(noise), n, s, white,
                                                 ptr(gs[0]), ptr(gs[1]), ptr(gs[2]), ptr(gs[3]), ptr(gs[4]), ptr(gs[5]),
                                                 ptr(d_raw), stream())
        return d_raw, None, None, None, None, None, None


def composite(raw, z, rays_d, bc_rgb, noise=None, white_bkgd=False, with_fg=False):
    """raw2outputs.  Returns (rgb_map, disp_map, acc_map, weights, depth_map[, rgb_map_fg])."""
    if z.shape[0] == 0:
        n, s = z.shape
        e = raw.new_zeros
        out = (e((0, 3)), e((0,)), e((0,)), e((0, s)), e((0,)))
        return out + (e((0, 3)),) if with_fg else out
    return _Composite.apply(raw, z, rays_d, bc_rgb, noise, white_bkgd, with_fg)


class _MsePair(torch.autograd.Function):
    """img_loss + img_loss0 (audio_exp_nerf.py:540-546): one kernel computes both means and both gradients."""

    @staticmethod
    def forward(ctx, rgb, rgb0, target):
        a, b, t = f32c(rgb, "rgb"), f32c(rgb0, "rgb0"), f32c(target, "target")
        assert a.shape == b.shape == t.shape
        ga, gb = torch.empty_like(a), torch.empty_like(b)
        loss2 = torch.empty((2,), device=a.device)
        with torch.cuda.device(a.device):
            call("inerf_mse_pair", _lib.lib().inerf_mse_pair, ptr(a), ptr(b), ptr(t), a.numel(), ptr(ga), ptr(gb), ptr(loss2), stream())
        ctx.save_for_backward(ga, gb)
        return loss2

    @staticmethod
    def backward(ctx, g):
        ga, gb = ctx.saved_tensors
        return ga * g[0], gb * g[1], None


def mse_pair(rgb, rgb0, target):
    """(F.mse_loss(rgb, target), F.mse_loss(rgb0, target)) as a 2-vector, differentiable in rgb and rgb0."""
    return _MsePair.apply(rgb, rgb0, target)


class _Blend(torch.autograd.Function):
    @staticmethod
    def forward(ctx, rgb_head, lw, fg):
        a, b, c = f32c(rgb_head, "rgb_head"), f32c(lw, "last_weight"), f32c(fg, "rgb_fg")
        shape = a.shape
        a2, c2 = a.reshape(-1, 3), c.reshape(-1, 3)
        out = torch.empty_like(a2)
        with torch.cuda.device(a.device):
            call("inerf_head_torso_blend", _lib.lib().inerf_head_torso_blend, ptr(a2), ptr(b.reshape(-1)), ptr(c2), a2.shape[0], ptr(out),
                                                    stream())
        ctx.save_for_backward(a, b)
        return out.reshape(shape)

    @staticmethod
    def backward(ctx, g):
        a, b = ctx.saved_tensors                 # three-term product rule of a 3-float-per-ray blend
        return g * b[..., None], (g * a).sum(-1), g


def head_torso_blend(rgb_head, last_weight_torso, rgb_fg_torso):
    """rgb_head * last_weight_torso[..., None] + rgb_fg_torso   (train_torso.py:269-270)."""
    return _Blend.apply(rgb_head, last_weight_torso, rgb_fg_torso)


class _HeadTorsoMsePair(torch.autograd.Function):
    """img_loss + img_loss0 of the torso stage: both composites, both losses and the gradients reaching the torso pair in one kernel."""

    @staticmethod
    def forward(ctx, rgb_head, rgb_head0, lw, lw0, fg, fg0, target):
        h, h0 = f32c(rgb_head, "rgb_head"), f32c(rgb_head0, "rgb_head0")
        w, w0 = f32c(lw, "last_weight"), f32c(lw0, "last_weight0")
        f, f0, t = f32c(fg, "rgb_fg"), f32c(fg0, "rgb_fg0"), f32c(target, "target")
        n = w.numel()
        if not (h.numel() == h0.numel() == f.numel() == f0.numel() == t.numel() == 3 * n and w0.numel() == n):
            raise ValueError(f"head_torso_mse_pair: rgb_head {tuple(h.shape)}, rgb_head0 {tuple(h0.shape)}, last_weight {tuple(w.shape)}, "
                             f"last_weight0 {tuple(w0.shape)}, rgb_fg {tuple(f.shape)}, rgb_fg0 {tuple(f0.shape)}, target {tuple(t.shape)} "
                             "are not (n,3) x 2, (n) x 2, (n,3) x 3")
        g_w, g_w0, g_f, g_f0 = torch.empty_like(w), torch.empty_like(w0), torch.empty_like(f), torch.empty_like(f0)
        loss2 = torch.empty((2,), device=w.device)
        with torch.cuda.device(w.device):
            call("inerf_head_torso_mse_pair", _lib.lib().inerf_head_torso_mse_pair, ptr(h), ptr(h0), ptr(w), ptr(w0), ptr(f), ptr(f0), ptr(t),
                 n, ptr(g_w), ptr(g_w0), ptr(g_f), ptr(g_f0), ptr(loss2), stream())
        ctx.save_for_backward(g_w, g_w0, g_f, g_f0)
        ctx.shapes = (lw.shape, lw0.shape, fg.shape, fg0.shape)
        return loss2

    @staticmethod
    def backward(ctx, g):
        g_w, g_w0, g_f, g_f0 = ctx.saved_tensors
        s = ctx.shapes
        return (None, None, (g_w * g[0]).view(s[0]), (g_w0 * g[1]).view(s[1]), (g_f * g[0]).view(s[2]), (g_f0 * g[1]).view(s[3]), None)


def head_torso_mse_pair(rgb_head, rgb_head0, last_weight, last_weight0, rgb_fg, rgb_fg0, target):
    """(F.mse_loss(head_torso_blend(rgb_head, last_weight, rgb_fg), target), the same for the coarse set) as a 2-vector, differentiable
    in last_weight, last_weight0, rgb_fg and rgb_fg0 (train_torso.py:269-271).  The head is frozen in the torso stage and the kernel
    computes no gradient for it, so a head image that requires grad raises instead of silently losing its gradient."""
    if (isinstance(rgb_head, torch.Tensor) and rgb_head.requires_grad) or (isinstance(rgb_head0, torch.Tensor) and rgb_head0.requires_grad):
        raise ValueError("head_torso_mse_pair: rgb_head / rgb_head0 require grad, but no gradient w.r.t. the head image is computed; "
                         "render the head pair under torch.no_grad() or pass .detach()")
    return _HeadTorsoMsePair.apply(rgb_head, rgb_head0, last_weight, last_weight0, rgb_fg, rgb_fg0, target)


def head_torso_to8b(rgb_head, last_weight_torso, rgb_fg_torso, out=None, out_rgb=None):
    """to8b(head_torso_blend(...)) in one kernel (test_torso.py:523-524), no autograd: (n, 3) uint8 for n rays, written into `out` when
    given.  out_rgb: None, or a contiguous float32 tensor of 3n values that receives the fp32 blend."""
    a, b, c = f32c(rgb_head.detach(), "rgb_head"), f32c(last_weight_torso.detach(), "last_weight"), f32c(rgb_fg_torso.detach(), "rgb_fg")
    n = a.numel() // 3
    if a.numel() != 3 * n or b.numel() != n or c.numel() != 3 * n:
        raise ValueError(f"head_torso_to8b: rgb_head {tuple(a.shape)}, last_weight {tuple(b.shape)}, rgb_fg {tuple(c.shape)} are not "
                         "(n,3), (n), (n,3)")
    if out is None:
        out = torch.empty((n, 3), device=a.device, dtype=torch.uint8)
    for t, dt, name in ((out, torch.uint8, "out"), (out_rgb, torch.float32, "out_rgb")):
        if t is not None:
            _need_cuda(t, name)
            if t.dtype != dt or t.numel() != 3 * n or not t.is_contiguous():
                raise ValueError(f"head_torso_to8b: `{name}` must be a contiguous {dt} tensor of {3 * n} values")
    with torch.cuda.device(a.device):
        call("inerf_head_torso_to8b", _lib.lib().inerf_head_torso_to8b, ptr(a), ptr(b), ptr(c), n, ptr(out), ptr(out_rgb), stream())
    return out


# ------------------------------------------------------------------------------------------------
# importance sampling
# ------------------------------------------------------------------------------------------------

def sample_pdf_raw(bins, weights, u, policy=_lib.INERF_PDF_EXACT_TORCH_CPU, want_inds=False):
    """helper.py:269-313.  u: (n_imp,) shared table or (n, n_imp) draws.  Returns (samples, inds|None)."""
    bins, weights, u = f32c(bins, "bins"), f32c(weights, "weights"), f32c(u, "u")
    n, nb = bins.shape
    assert weights.shape == (n, nb - 1), "weights must be (n, n_bins-1)"
    per_ray = int(u.dim() == 2)
    n_imp = u.shape[-1]
    zs = torch.empty((n, n_imp), device=bins.device)
    inds = torch.empty((n, n_imp), device=bins.device, dtype=torch.int64) if want_inds else None
    with torch.cuda.device(bins.device):
        call("inerf_sample_pdf", _lib.lib().inerf_sample_pdf, ptr(bins), nb, ptr(weights), nb - 1, n, nb, n_imp, ptr(u), per_ray, policy,
                                          ptr(zs), ptr(inds), None, 0, None, None, stream())
    return zs, inds


def importance_sample(z_coarse, w_coarse, u, policy=_lib.INERF_PDF_EXACT_TORCH_CPU, want_inds=False):
    """Fused z_mid / weights[...,1:-1] / sample_pdf / sort(cat) / std of audio_exp_nerf.py:342-347,364.

    Returns (z_samples, z_merged, z_std, inds|None); nothing here is differentiable (the reference detaches)."""
    z_coarse, w_coarse, u = f32c(z_coarse.detach(), "z_vals"), f32c(w_coarse.detach(), "weights"), f32c(u, "u")
    n, s1 = z_coarse.shape
    per_ray = int(u.dim() == 2)
    n_imp = u.shape[-1]
    dev = z_coarse.device
    zs = torch.empty((n, n_imp), device=dev)
    zm = torch.empty((n, s1 + n_imp), device=dev)
    zstd = torch.empty((n,), device=dev)
    inds = torch.empty((n, n_imp), device=dev, dtype=torch.int64) if want_inds else None
    with torch.cuda.device(dev):
        call("inerf_importance_sample", _lib.lib().inerf_importance_sample, ptr(z_coarse), ptr(w_coarse), n, s1, n_imp, ptr(u), per_ray, policy,
                                                 ptr(zs), ptr(inds), ptr(zm), ptr(zstd), stream())
    return zs, zm, zstd, inds


# ------------------------------------------------------------------------------------------------
# the whole inference render_rays in one C call
# ------------------------------------------------------------------------------------------------

def _render_net(net, aud, expr, latent, keep):
    """InerfRenderNet of one FaceNeRF module; `keep` collects every object whose memory the struct points into."""
    params = [p.detach() for p in net._prep(aud, expr, latent)]
    packed = net.packed_weights(net.kernel_params())
    arr = param_array(params)
    f = lambda t, d: f32c(t.detach(), "conditioning").reshape(-1) if d > 0 else None
    a, e, l = f(aud, net.dim_aud), f(expr, net.dim_expr), f(latent, net.dim_latent)
    keep += [params, packed, arr, a, e, l]
    r = _lib.InerfRenderNet()
    r.dims = net._dims
    r.params_host = ctypes.cast(arr, ctypes.POINTER(ctypes.c_void_p))
    r.packed = packed.data_ptr() if packed is not None else None
    r.aud, r.expr, r.latent = (t.data_ptr() if t is not None else None for t in (a, e, l))
    return r


def render_rays_fused(net_coarse, net_fine, cond_coarse, cond_fine, bc_rgb, n_samples, n_importance, perturb, rays=None, gen=None,
                      lindisp=False, white_bkgd=False, with_fg=False, want_weights=False, want_z=False, check_numerics=False, state=None,
                      stage_ms=None):
    """Network.render_rays under no_grad as ONE C call (inerf_render_rays_fused): five kernel launches in the reference's
    configuration (set-up, coarse FaceNeRF, compositor + sampler, fine FaceNeRF, final compositor).  rays: packed (n, 11), or
    gen = dict(H, W, focal, cx, cy, near, far, c2w, first, count) to generate the rays of pixels [first, first + count) on the fly.
    cond_*: (aud, expr, latent) of each net.  Returns the render_rays dict (plus '_nonfinite' bits when check_numerics)."""
    mode = net_coarse._mode()
    bc_rgb = f32c(bc_rgb, "bc_rgb")
    dev = bc_rgb.device
    keep = []
    a = _lib.InerfRenderArgs()
    a.mode, a.n_samples, a.n_importance = mode, int(n_samples), int(n_importance)
    a.perturb, a.lindisp, a.white_bkgd = int(perturb > 0.), int(bool(lindisp)), int(bool(white_bkgd))
    if gen is not None:
        c2w = f32c(gen["c2w"], "c2w")
        n = int(gen["count"])
        a.gen_rays, a.H, a.W, a.first = 1, int(gen["H"]), int(gen["W"]), int(gen["first"])
        a.focal, a.cx, a.cy, a.near_, a.far_ = float(gen["focal"]), float(gen["cx"]), float(gen["cy"]), float(gen["near"]), float(gen["far"])
        a.c2w, a.c2w_row_stride = c2w.data_ptr(), c2w.stride(0)
        keep.append(c2w)
    else:
        rays = f32c(rays, "rays")
        n = rays.shape[0]
        a.rays, a.ray_stride = rays.data_ptr(), rays.shape[1]
    a.n = n
    assert bc_rgb.shape == (n, 3), f"bc_rgb {tuple(bc_rgb.shape)} for {n} rays"
    a.bc_rgb = bc_rgb.data_ptr()
    t_vals, u_vals = linspace_table(n_samples, dev), linspace_table(n_importance, dev)
    a.t_vals, a.u_vals = t_vals.data_ptr(), u_vals.data_ptr()
    if a.perturb:
        state = rng_state(dev) if state is None else state
        a.rng_state = state.data_ptr()
    a.coarse = _render_net(net_coarse, *cond_coarse, keep)
    a.fine = _render_net(net_fine, *cond_fine, keep)
    stot = n_samples + n_importance
    out = torch.empty((n * (13 + (7 if with_fg else 0)),), device=dev)
    cuts = [("rgb_map", 3), ("disp_map", 1), ("acc_map", 1), ("depth_map", 1), ("last_weight", 1), ("rgb0", 3), ("disp0", 1), ("acc0", 1),
            ("z_std", 1)] + ([("rgb_map_fg", 3), ("rgb_map_fg0", 3), ("last_weight0", 1)] if with_fg else [])
    ret, o = {}, 0
    for k, w in cuts:
        ret[k] = out[o:o + n * w].view(n, 3) if w == 3 else out[o:o + n]
        setattr(a, k, ret[k].data_ptr())
        o += n * w
    if want_weights:
        ret["_weights"] = torch.empty((n, stot), device=dev)
        a.weights = ret["_weights"].data_ptr()
    if want_z:
        ret["_z_vals"] = torch.empty((n, stot), device=dev)
        a.z_vals = ret["_z_vals"].data_ptr()
    flag = None
    if check_numerics:
        flag = torch.zeros((1,), dtype=torch.int32, device=dev)
        a.nonfinite = flag.data_ptr()
    nb = ctypes.c_size_t()
    check(_lib.lib().inerf_render_workspace_bytes(ctypes.byref(a), ctypes.byref(nb)), "inerf_render_workspace_bytes")
    ws = torch.empty((max(nb.value, 1),), device=dev, dtype=torch.uint8)
    a.workspace, a.workspace_bytes = ws.data_ptr(), nb.value
    if n > 0:
        with torch.cuda.device(dev):
            fast = a.perturb and n_samples == 64 and n_importance == 128 and not lindisp
            if stage_ms is not None:      # measurement: device time of the five stages (synchronises), appended to the caller's list
                ms = (ctypes.c_float * 5)()
                call("inerf_render_rays_fused", _lib.lib().inerf_debug_render_stage_ms, ctypes.byref(a), stream(), ms, launches=5 if fast else 7)
                stage_ms.append([float(v) for v in ms])
            else:
                call("inerf_render_rays_fused", _lib.lib().inerf_render_rays_fused, ctypes.byref(a), stream(), launches=5 if fast else 7)
    ret["_depth_map"] = ret.pop("depth_map")
    if flag is not None:
        bits = int(flag.item())
        ret["_nonfinite"] = [k for k, b in _lib.NF_BITS.items() if bits & b]
    return ret


# ------------------------------------------------------------------------------------------------
# FaceNeRF MLP
# ------------------------------------------------------------------------------------------------

def zero_grads_like(params):
    """Zero gradient tensors for `params` as views of ONE flat buffer (a single memset instead of 26 fill kernels; the flat
    buffer is what a data-parallel all-reduce sends).  Returns (views, flat)."""
    sizes = [(p.numel() + 3) // 4 * 4 for p in params]                 # 16-byte aligned starts
    flat = torch.zeros((sum(sizes),), device=params[0].device, dtype=torch.float32)
    views, o = [], 0
    for p, n in zip(params, sizes):
        views.append(flat[o:o + p.numel()].view(p.shape))
        o += n
    return views, flat


def net_dims(dim_aud, dim_expr, dim_latent):
    return InerfNetDims(int(dim_aud), int(dim_expr), int(dim_latent), 256, 8, 63, 27)


def param_array(params):
    """ctypes array of the 26 device pointers in include/inerf_b200.h order (tensors must stay alive)."""
    assert len(params) == _lib.N_PARAMS
    arr = ParamArray()
    for i, p in enumerate(params):
        _need_cuda(p, "parameter")
        assert p.dtype == torch.float32 and p.is_contiguous()
        arr[i] = p.data_ptr()
    return arr


def fold_cond(dims, params, aud, expr, latent):
    n = ctypes.c_size_t()
    check(_lib.lib().inerf_mlp_cond_floats(ctypes.byref(dims), ctypes.byref(n)), "inerf_mlp_cond_floats")
    dev = params[0].device
    cond = torch.empty((n.value,), device=dev)
    aud = f32c(aud, "aud") if dims.dim_aud > 0 else None
    expr = f32c(expr, "expr") if dims.dim_expr > 0 else None
    latent = f32c(latent, "latent_code") if dims.dim_latent > 0 else None
    arr = param_array(params)
    with torch.cuda.device(dev):
        call("inerf_mlp_fold_cond", _lib.lib().inerf_mlp_fold_cond, ctypes.byref(dims), arr, ptr(aud), ptr(expr), ptr(latent), ptr(cond),
                                             stream())
    return cond


def pack_weights(mode, dims, params, out=None):
    """The packed weight blob of `mode` (None when the mode has none), written into `out` when given (a uint8 tensor of exactly that
    size), else into a new tensor."""
    nb = ctypes.c_size_t()
    check(_lib.lib().inerf_mlp_packed_bytes(mode, ctypes.byref(dims), ctypes.byref(nb)), "inerf_mlp_packed_bytes")
    if nb.value == 0:
        return None
    dev = params[0].device
    if out is not None:
        _need_cuda(out, "out")
        if out.dtype != torch.uint8 or out.numel() != nb.value or not out.is_contiguous() or out.device != dev:
            raise ValueError(f"pack_weights: `out` must be a contiguous uint8 tensor of {nb.value} bytes on {dev}")
    packed = torch.empty((nb.value,), device=dev, dtype=torch.uint8) if out is None else out
    arr = param_array(params)
    with torch.cuda.device(dev):
        call("inerf_mlp_pack", _lib.lib().inerf_mlp_pack, mode, ctypes.byref(dims), arr, ptr(packed), stream())
    return packed


def mlp_fwd(mode, dims, params, packed, cond, rays, z):
    """run_network for one pass (points, gamma(p), gamma(v), FaceNeRF).  rays (n,11), z (n,s) -> raw (n,s,4)."""
    rays, z = f32c(rays, "rays"), f32c(z, "z_vals")
    n, s = z.shape
    raw = torch.empty((n, s, 4), device=z.device)
    arr = param_array(params)
    with torch.cuda.device(z.device):
        call("inerf_mlp_fwd", _lib.lib().inerf_mlp_fwd, mode, ctypes.byref(dims), arr, ptr(packed), ptr(cond), ptr(rays), rays.shape[1],
                                       ptr(z), n, s, ptr(raw), stream())
    return raw


def mlp_fwd_train(dims, params, cond, rays=None, z=None, x=None):
    """fp32 forward that keeps the activations for mlp_bwd.  Returns (raw, acts, n_points)."""
    if x is None:
        rays, z = f32c(rays, "rays"), f32c(z, "z_vals")
        n, s = z.shape
        n_points, dev, out_shape = n * s, z.device, (n, s, 4)
    else:
        x = f32c(x, "x")
        n, s, n_points, dev, out_shape = 0, 1, x.shape[0], x.device, (x.shape[0], 4)
    sizes = [ctypes.c_size_t() for _ in range(3)]
    check(_lib.lib().inerf_mlp_train_sizes(ctypes.byref(dims), n_points, *[ctypes.byref(v) for v in sizes]), "inerf_mlp_train_sizes")
    raw = torch.empty(out_shape, device=dev)
    acts = torch.empty((sizes[0].value,), device=dev)
    arr = param_array(params)
    with torch.cuda.device(dev):
        call("inerf_mlp_fwd_train", _lib.lib().inerf_mlp_fwd_train, ctypes.byref(dims), arr, ptr(cond), ptr(rays),
             rays.shape[1] if rays is not None else 11, ptr(z), n, s, ptr(x), n_points if x is not None else 0, ptr(raw),
             ptr(acts), stream())
    return raw, acts, n_points


def mlp_bwd(dims, params, aud, expr, latent, acts, d_raw, n_points):
    """Analytic backward of FaceNeRF (fp32).  Returns (grads[26] in nn.Linear layout, d_cond [aud|expr|latent])."""
    dev = acts.device
    sizes = [ctypes.c_size_t() for _ in range(3)]
    check(_lib.lib().inerf_mlp_train_sizes(ctypes.byref(dims), n_points, *[ctypes.byref(v) for v in sizes]), "inerf_mlp_train_sizes")
    deltas = torch.empty((sizes[1].value,), device=dev)
    scratch = torch.empty((sizes[2].value,), device=dev, dtype=torch.uint8)
    grads, _ = zero_grads_like(params)
    d_cond = torch.zeros((max(1, dims.dim_aud + dims.dim_expr + dims.dim_latent),), device=dev)
    d_raw = f32c(d_raw, "d_raw").reshape(-1, 4)
    parr, garr = param_array(params), param_array(grads)
    with torch.cuda.device(dev):
        call("inerf_mlp_bwd", _lib.lib().inerf_mlp_bwd, ctypes.byref(dims), parr, garr, ptr(aud), ptr(expr), ptr(latent),
             ptr(acts), ptr(deltas), ptr(d_raw), n_points, ptr(d_cond), ptr(scratch), stream())
    return grads, d_cond


def _train_sizes_bf16(dims, n_points):
    sizes = [ctypes.c_size_t() for _ in range(4)]
    check(_lib.lib().inerf_mlp_train_sizes_bf16(ctypes.byref(dims), n_points, *[ctypes.byref(v) for v in sizes]), "inerf_mlp_train_sizes_bf16")
    return [v.value for v in sizes]          # acts, mask, deltas, scratch (bytes)


def mlp_fwd_train_bf16(dims, params, packed, cond, rays=None, z=None, x=None):
    """bf16 tensor-core forward that keeps the activation images + ReLU masks for mlp_bwd_bf16.  Returns (raw, acts, mask, n_points).
    rays (n,11) / z (n,s) with the INERF_MLP_BF16 blob, or embedded rows x (P, 90) with the INERF_MLP_BF16_EMB blob."""
    if x is None:
        rays, z = f32c(rays, "rays"), f32c(z, "z_vals")
        n, s = z.shape
        n_points, dev, out_shape = n * s, z.device, (n, s, 4)
    else:
        x = _rows90(x)
        n_points, dev, out_shape = x.shape[0], x.device, (x.shape[0], 4)
    acts_b, mask_b, _, _ = _train_sizes_bf16(dims, n_points)
    raw = torch.empty(out_shape, device=dev)
    acts = torch.empty((acts_b,), device=dev, dtype=torch.uint8)
    mask = torch.empty((mask_b,), device=dev, dtype=torch.uint8)
    arr = param_array(params)
    with torch.cuda.device(dev):
        if x is None:
            call("inerf_mlp_fwd_train", _lib.lib().inerf_mlp_fwd_train_bf16, ctypes.byref(dims), arr, ptr(packed), ptr(cond), ptr(rays),
                 rays.shape[1], ptr(z), n, s, ptr(raw), ptr(acts), ptr(mask), stream())
        else:
            call("inerf_mlp_fwd_train_bf16_embedded", _lib.lib().inerf_mlp_fwd_train_bf16_embedded, ctypes.byref(dims), arr, ptr(packed),
                 ptr(cond), ptr(x), n_points, ptr(raw), ptr(acts), ptr(mask), stream())
    return raw, acts, mask, n_points


def mlp_bwd_bf16(dims, params, packed_t, aud, expr, latent, acts, mask, d_raw, n_points, keep_deltas=False):
    """bf16 tensor-core backward of FaceNeRF.  Returns (grads[26] fp32 in nn.Linear layout, d_cond [aud|expr|latent])."""
    dev = acts.device
    _, _, deltas_b, scratch_b = _train_sizes_bf16(dims, n_points)
    deltas = torch.empty((deltas_b,), device=dev, dtype=torch.uint8)
    scratch = torch.empty((scratch_b,), device=dev, dtype=torch.uint8)
    grads, _ = zero_grads_like(params)
    d_cond = torch.zeros((max(1, dims.dim_aud + dims.dim_expr + dims.dim_latent),), device=dev)
    d_raw = f32c(d_raw, "d_raw").reshape(-1, 4)
    parr, garr = param_array(params), param_array(grads)
    with torch.cuda.device(dev):
        call("inerf_mlp_bwd", _lib.lib().inerf_mlp_bwd_bf16, ctypes.byref(dims), parr, ptr(packed_t), garr, ptr(aud), ptr(expr), ptr(latent),
             ptr(acts), ptr(mask), ptr(deltas), ptr(d_raw), n_points, ptr(d_cond), ptr(scratch), stream())
    if keep_deltas:
        mlp_bwd_bf16.deltas = deltas
    return grads, d_cond


def decode_images(buf, n_tiles, n_imgs=40):
    """Test helper: [n_tiles][n_imgs] 16 KB images (128 rows x 64 bf16, 128-byte swizzle) -> float tensor (n_tiles, n_imgs, 128, 64)."""
    b = buf[: n_tiles * n_imgs * 16384].view(torch.bfloat16).reshape(n_tiles, n_imgs, 128, 8, 8)      # row, 16-byte chunk, element
    r = torch.arange(128, device=buf.device) & 7
    idx = (torch.arange(8, device=buf.device)[None, :] ^ r[:, None])                                    # logical chunk c lives at c ^ (row & 7)
    out = torch.gather(b, 3, idx[None, None, :, :, None].expand(n_tiles, n_imgs, 128, 8, 8))
    return out.reshape(n_tiles, n_imgs, 128, 64).float()


def mlp_fwd_trace(mode, dims, params, packed, cond, rays, z):
    """bf16 kernel with the per-layer activation trace of the first 256 points: returns (raw, trace[11,256,256])."""
    rays, z = f32c(rays, "rays"), f32c(z, "z_vals")
    n, s = z.shape
    raw = torch.empty((n, s, 4), device=z.device)
    trace = torch.zeros((11 * 256 * 256 + 148 * 8 * 2 + 148 * 16,), device=z.device)     # activations + per-CTA issuer / epilogue timing
    arr = param_array(params)
    with torch.cuda.device(z.device):
        call("inerf_mlp_fwd_trace", _lib.lib().inerf_mlp_fwd_trace, mode, ctypes.byref(dims), arr, ptr(packed), ptr(cond),
             ptr(rays), rays.shape[1], ptr(z), n, s, ptr(raw), ptr(trace), stream())
    mlp_fwd_trace.timing = trace[11 * 256 * 256:11 * 256 * 256 + 148 * 16].reshape(-1, 8)
    mlp_fwd_trace.layer_waits = trace[11 * 256 * 256 + 148 * 16:].reshape(148, 16)
    return raw, trace[:11 * 256 * 256].reshape(11, 256, 256)


def _rows90(x):
    """x as the embedded-row kernels read it: contiguous fp32 (P, 90), 16-byte aligned as the bf16 kernel needs (a row slice may start off
    alignment)."""
    x = f32c(x, "x")
    assert x.dim() == 2 and x.shape[1] == 90, "x must be (P, 63+27)"
    return x if x.data_ptr() % 16 == 0 else x.clone()


def mlp_fwd_embedded(mode, dims, params, packed, cond, x):
    """FaceNeRF.forward on embedded rows x (P, 90) -> (P, 4).  bf16 mode takes the INERF_MLP_BF16_EMB blob; fp16x2 runs as mode
    INERF_MLP_F16X2_EMB with that mode's blob."""
    x = _rows90(x)
    out = torch.empty((x.shape[0], 4), device=x.device)
    arr = param_array(params)
    with torch.cuda.device(x.device):
        call("inerf_mlp_fwd_embedded", _lib.lib().inerf_mlp_fwd_embedded, mode, ctypes.byref(dims), arr, ptr(packed), ptr(cond), ptr(x),
                                                x.shape[0], ptr(out), stream())
    return out
