"""Seeded synthetic inputs of the shapes BASELINE.json names (SURVEY.md 8d): camera, background,
audio / expression / latent codes, random-init FaceNeRF weights with the normalised-density preset.

Used by bench.py and __graft_entry__.smoke(); write_head_subject writes a small subject on disk for the dataset classes.
The tensors follow the same generator sequence as the test oracle's synthetic_frame so both arms of
the benchmark see the same data, but nothing here imports the test infrastructure.
"""
import torch

from . import ops

NEAR = 0.5772005200386048   # NeRFs/HeadNeRF/configs/audio_expr_nerf/may/paper_model/torso_bg.txt:11-12
FAR = 1.1772005200386046
TORSO_RGB = (40, 150, 90)   # the torso colour of write_head_subject's com_imgs


def camera():
    c2w = torch.eye(4)
    c2w[2, 3] = 0.7772
    return dict(H=450, W=450, focal=1200., cx=225., cy=225., c2w=c2w)


def frame_inputs(seed=0):
    """Host tensors of one frame: pose (4,4), bc_rgb (H*W,3), aud (64), expr (76), latent (32)."""
    cam = camera()
    g = torch.Generator().manual_seed(seed)
    bc = torch.rand(cam["H"] * cam["W"], 3, generator=g)
    aud = torch.randn(64, generator=g)
    expr = torch.randn(76, generator=g)
    return dict(pose=cam["c2w"], bc_rgb=bc, aud=aud, expr=expr, latent=torch.ones(32))


def video_codes(n_frames, seed=0, sigma=0.1):
    """Seeded Gaussian random walk of audio/expression codes for an n_frames eval video (config 5)."""
    g = torch.Generator().manual_seed(seed + 17)
    aud = torch.cumsum(torch.randn(n_frames, 64, generator=g) * sigma, 0)
    expr = torch.cumsum(torch.randn(n_frames, 76, generator=g) * sigma, 0)
    return aud, expr


@torch.no_grad()
def normalise_density_(net, rays, aud, expr, latent, n_samples=64, target_std=8.0):
    """SURVEY.md 7-7 preset, in place: rescale alpha_linear so raw sigma on the coarse samples is ~N(0.01, 8^2).
    Random-init FaceNeRF gives sigma ~ -0.3 +- 0.1 => every ray would be pure background."""
    mode, net.mlp_mode = net.mlp_mode, "fp32"
    z = ops.sample_coarse(rays, n_samples)
    s = net.query(rays, z, aud, expr, latent)[..., 3]
    net.mlp_mode = mode
    k = target_std / float(s.std())
    net.alpha_linear.weight.mul_(k)
    net.alpha_linear.bias.copy_((net.alpha_linear.bias - float(s.mean())) * k + 0.01)
    return net


def write_head_subject(d, H=450, W=450, n_frames=64, seed=0, torso_rows=40, constant_rgb=None, n_aud=None, val_frames=0, com_imgs=False):
    """A seeded synthetic subject in the reference's on-disk layout (data.py): random JPEG frames (or one constant colour), parsing maps
    whose last `torso_rows` rows are torso, landmarks that give a mouth box near the centre, a face rectangle, bc.jpg, aud.npy and
    transforms_exp_train.json.  With val_frames > 0 it also writes transforms_exp_val.json: `val_frames` held-out frames (img_id n_frames + j, aud_id
    the train audio's length + j, poses continuing the train path) whose DeepSpeech windows are appended to aud.npy; every train file is the same as
    with val_frames = 0 except that longer aud.npy.  With com_imgs it also writes com_imgs/<img_id>.jpg, the torso stage's targets
    (gt_dirs = com_imgs): each frame's head image with its last `torso_rows` rows painted TORSO_RGB (no draw from the generator, so every
    other file keeps its bytes).  Returns the args a HeadDataset needs for it (gt_dirs = head_imgs)."""
    import json
    import os

    import numpy as np
    from PIL import Image
    for sub in ("head_imgs", "ori_imgs", "parsing") + (("com_imgs",) if com_imgs else ()):
        os.makedirs(os.path.join(d, sub), exist_ok=True)
    rng = np.random.RandomState(seed)

    def frame(i, aud_id):
        img = np.empty((H, W, 3), np.uint8)
        img[:] = constant_rgb if constant_rgb is not None else rng.randint(0, 255, (H, W, 3), dtype=np.uint8)
        Image.fromarray(img).save(os.path.join(d, "head_imgs", f"{i}.jpg"), quality=95)
        if com_imgs:
            img[H - torso_rows:] = TORSO_RGB
            Image.fromarray(img).save(os.path.join(d, "com_imgs", f"{i}.jpg"), quality=95)
        parse = np.zeros((H, W, 3), np.uint8)
        parse[H - torso_rows:, :, 0] = 255
        Image.fromarray(parse).save(os.path.join(d, "parsing", f"{i}.png"))
        lms = rng.rand(68, 2) * 10 + H * 0.3
        lms[48:] = rng.rand(20, 2) * 0.1 * min(H, W) + np.array([H * 0.55, W * 0.45])
        np.savetxt(os.path.join(d, "ori_imgs", f"{i}.lms"), lms)
        pose = np.eye(4)
        pose[:3, 3] = [0.001 * i, -0.002, 0.7772]
        return {"img_id": i, "aud_id": aud_id, "transform_matrix": pose.tolist(),
                "face_rect": [H // 8, W // 8, H * 5 // 8, W * 3 // 4], "exp": rng.randn(76).tolist()}

    def transforms(mode, frames):
        with open(os.path.join(d, f"transforms_exp_{mode}.json"), "w") as fp:
            json.dump({"focal_len": 1200.0 * W / 450, "cx": W / 2, "cy": H / 2, "frames": frames}, fp)

    transforms("train", [frame(i, i) for i in range(n_frames)])
    aud = rng.randn(n_aud or n_frames, 16, 29).astype(np.float32)
    np.save(os.path.join(d, "aud.npy"), aud)
    Image.fromarray(rng.randint(0, 255, (H, W, 3), dtype=np.uint8)).save(os.path.join(d, "bc.jpg"), quality=95)
    if val_frames > 0:                      # drawn after every train file, so those keep their bytes
        n_aud_train = aud.shape[0]
        transforms("val", [frame(n_frames + j, n_aud_train + j) for j in range(val_frames)])
        np.save(os.path.join(d, "aud.npy"), np.concatenate([aud, rng.randn(val_frames, 16, 29).astype(np.float32)]))
