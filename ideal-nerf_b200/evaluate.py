"""Held-out evaluation: render the frames of a split and score them against the dataset's frames on the device.

The reference's eval loop (eval_aud_exp_nerf.py:485-495) only writes a video.  evaluate_split renders frame i of a DeviceHeadDataset
from (poses[i], codes[i], exprs[i]) through the video drivers of frame.py and, on rank 0, scores the uint8 bytes of each rendered frame
against dataset.frames[i] with one kernel (ops.image_metrics, inerf_image_metrics) before they are copied to the host: PSNR over the full
frame, the face rectangle and the mouth box, and SSIM.  Frames are compared as stored (BGR, the channel order the model is trained in).
With LPIPS weights (load_lpips: the user's copies of torchvision's AlexNet and lpips' v0.1 linear heads) each frame also gets its LPIPS
(ops.lpips, inerf_lpips), which reads the BGR bytes and feeds AlexNet RGB.

The split is loaded as DeviceHeadDataset(data_dir, aud_file, "val", args) with zero training budgets (args.N_rand = args.mouth_rays =
args.torso_rays = 0): evaluation never draws a batch, and held-out frames need not hold the pixels the training budgets ask for, which the
dataset checks at construction.
"""
import math
import os

import numpy as np
import torch

from . import ops
from .data import DeviceTorsoDataset
from .frame import HeadTorsoFrameRenderer, render_head_torso_video, render_video


def psnr(sse, npix):
    """PSNR in dB of uint8 images from their exact squared error over 3 channels: 10 log10(255^2 * 3 * npix / sse), inf where sse == 0.
    sse, npix: int64 tensors or arrays of the same shape (ops.image_metrics' sse / npix).  Returns float64 of that shape, on sse's
    device."""
    sse = torch.as_tensor(sse)
    npix = torch.as_tensor(npix, device=sse.device)
    s, n = sse.double(), npix.double()
    return torch.where(sse == 0, torch.full_like(s, math.inf), 10. * torch.log10(255. ** 2 * 3. * n / s))


@torch.no_grad()
def audio_codes(network, dataset):
    """(F, dim_aud) audio codes of the dataset's frames: row i is network.audio_feature(dataset.auds, i, len(dataset)) (AudioNet over the
    smoothing window, then AudioAttNet), the code the eval loop conditions frame i on."""
    return torch.stack([network.audio_feature(dataset.auds, i, len(dataset)) for i in range(len(dataset))])


def _state_dict(src, what):
    if isinstance(src, (str, os.PathLike)):
        return torch.load(src, map_location="cpu", weights_only=True)
    if not isinstance(src, dict):
        raise ValueError(f"load_lpips: `{what}` must be a path or a state dict")
    return src


def load_lpips(alexnet, lin, device="cuda"):
    """The weights ops.lpips and evaluate_split(lpips=...) take, from user-supplied files (or their already-loaded state dicts):
    alexnet, torchvision's AlexNet (alexnet-owt-7be5be79.pth: features.{0,3,6,8,10}.{weight,bias}; classifier.* is ignored); lin, the
    lpips package's v0.1 heads (weights/v0.1/alex.pth: lin{0..4}.model.1.weight, (1, C, 1, 1)).  Returns the 15 contiguous float32
    tensors on `device` in inerf_lpips' order: conv1..conv5 (weight, bias), then lin0..lin4 as (C,).  A missing key or a wrong shape
    raises ValueError naming it."""
    alexnet, lin = _state_dict(alexnet, "alexnet"), _state_dict(lin, "lin")
    keys = [(alexnet, f"features.{i}.{p}") for i in (0, 3, 6, 8, 10) for p in ("weight", "bias")]
    keys += [(lin, f"lin{k}.model.1.weight") for k in range(5)]
    out = []
    for (sd, key), shape in zip(keys, ops.LPIPS_SHAPES):
        if key not in sd:
            raise ValueError(f"load_lpips: missing key {key}")
        t = torch.as_tensor(sd[key])
        want = (1, shape[0], 1, 1) if key.startswith("lin") else shape
        if tuple(t.shape) != want:
            raise ValueError(f"load_lpips: {key} has shape {tuple(t.shape)}, expected {want}")
        out.append(t.detach().reshape(shape).to(device=device, dtype=torch.float32).contiguous())
    return out


@torch.no_grad()
def evaluate_split(renderer, dataset, latent, codes, perturb=0., keep_video=True, lpips=None):
    """Render every frame of `dataset` (a DeviceHeadDataset of the split) and score it against the frame it holds out.

    renderer: frame.FrameRenderer (head) or frame.HeadTorsoFrameRenderer (head + torso) of a network whose H, W and focal are the
    dataset's; frame i is rendered from (dataset.poses[i], codes[i], dataset.exprs[i]) with background dataset.bc_img, through
    render_video / render_head_torso_video, so several ranks work as they do there.  codes: (F, dim_aud), e.g. audio_codes(network,
    dataset).  No host synchronise until the last frame.

    Returns, on rank 0, a dict of host values: psnr (F, 3) float64 (full frame, face rect, mouth box), ssim (F,) float64, their means over
    the frames mean_psnr (3,) and mean_ssim, the exact sse / npix (F, 3) int64 behind the PSNR, and video (F, H, W, 3) uint8 (the rendered
    bytes, the frames' channel order) when keep_video, else None.  Other ranks return None.

    When dataset is a data.DeviceTorsoDataset (render it with HeadTorsoFrameRenderer(torso_net, dataset.torso_pose)), each frame is also
    scored over its torso pixels (dataset.torso_bits, ops.masked_sse), the region the torso stage trains -- the head pair is frozen there,
    so the face rect and mouth box measure the head, and the full frame is mostly background.  Extra keys: sse_torso, npix_torso (F,)
    int64, psnr_torso (F,) float64 and mean_psnr_torso.

    lpips: None, or the weights of load_lpips.  Then each frame is also scored with LPIPS v0.1 (AlexNet) over the full frame (ops.lpips,
    on the same bytes), and the dict gains lpips (F,) float64 and mean_lpips.  Without it the dict is what it was without the option."""
    n = len(dataset)
    if codes.shape[0] != n:
        raise ValueError(f"evaluate_split: {codes.shape[0]} audio codes for {n} frames")
    dev = dataset.frames.device
    index = torch.arange(n, dtype=torch.int64, device=dev)
    frames = [(dataset.poses[i], codes[i], dataset.exprs[i]) for i in range(n)]
    torso = isinstance(dataset, DeviceTorsoDataset)
    scores, torso_scores, lpips_scores = [], [], []

    def on_frame(i, img):
        scores.append(ops.image_metrics(img[None], dataset.frames, index[i:i + 1], dataset.bounds))
        if torso:
            torso_scores.append(ops.masked_sse(img[None], dataset.frames, index[i:i + 1], dataset.torso_bits))
        if lpips is not None:
            lpips_scores.append(ops.lpips(img[None], dataset.frames, index[i:i + 1], lpips))

    drive = render_head_torso_video if isinstance(renderer, HeadTorsoFrameRenderer) else render_video
    video = drive(renderer, frames, latent, dataset.bc_img, perturb, on_frame=on_frame)
    if renderer.rank != 0:
        return None
    sse = torch.cat([s["sse"] for s in scores]).cpu().numpy()
    npix = torch.cat([s["npix"] for s in scores]).cpu().numpy()
    ssim = torch.cat([s["ssim"] for s in scores]).cpu().numpy()
    p = psnr(sse, npix).numpy()
    res = {"psnr": p, "ssim": ssim, "mean_psnr": p.mean(0), "mean_ssim": float(ssim.mean()), "sse": sse, "npix": npix,
           "video": video.numpy() if keep_video else None}
    if torso:
        sse_t = torch.cat([s for s, _ in torso_scores]).cpu().numpy()
        npix_t = torch.cat([c for _, c in torso_scores]).cpu().numpy()
        p_t = psnr(sse_t, npix_t).numpy()
        res.update(sse_torso=sse_t, npix_torso=npix_t, psnr_torso=p_t, mean_psnr_torso=float(p_t.mean()))
    if lpips is not None:
        lp = torch.cat(lpips_scores).cpu().numpy().astype(np.float64)
        res.update(lpips=lp, mean_lpips=float(lp.mean()))
    return res
