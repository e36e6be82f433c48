"""Dataset formats of the reference's HeadNeRF training script (NeRFs/HeadNeRF/train/audio_exp_nerf.py:45-196, class GetData), written by
data_util/process_data.py:253-288:

    <data_dir>/transforms_exp_{train,val}.json   {"focal_len", "cx", "cy", "frames": [{"img_id", "aud_id", "transform_matrix" 4x4,
                                                  "face_rect" [x, y, w, h], "exp" [76 or 79]}]}
    <data_dir>/<aud_file> (aud.npy)               (T, 16, 29) DeepSpeech windows
    <data_dir>/bc.jpg                             background, RGB
    <data_dir>/<gt_dirs>/<img_id>.jpg             target frames (the reference reads them with cv2: BGR channel order)
    <data_dir>/ori_imgs/<img_id>.lms              68 x 2 landmarks; rows 48.. are the mouth
    <data_dir>/parsing/<img_id>.png               face parsing; pure red = torso

HeadDataset is host side (json / numpy / PIL), except that the N_rand training rays are generated on the device for the SELECTED pixels
(ops.get_rays_at) instead of building the 450 x 450 ray grid per sample and indexing it (:123-139,189-191).  DeviceHeadDataset decodes
every frame once and draws each batch on the device (ops.sample_train_pixels): no host work per step.  DeviceTorsoDataset does the same
for the torso stage: the head batch plus the torso rays of the same pixels and the frozen head's per-frame codes."""
import json
import os

import numpy as np
import torch

from . import _lib, ops


def _imread_rgb(path):
    from PIL import Image
    return np.asarray(Image.open(path).convert("RGB"))


class HeadDataset(torch.utils.data.Dataset):
    """GetData (audio_exp_nerf.py:45).  __getitem__ returns the reference's tuple
    (batch_rays (2, N_rand, 3), target_s (N_rand, 3), bc_rgb, auds (T, 16, 29), raw_img, pose (3, 4), exp, index) with device tensors."""

    def __init__(self, data_dir, aud_file, mode, args, skip=1, device="cuda"):
        self.data_dir, self.aud_file, self.mode, self.args, self.device = data_dir, aud_file, mode, args, torch.device(device)
        with open(os.path.join(data_dir, f"transforms_exp_{mode}.json")) as fp:
            self.meta = json.load(fp)
        self.aud_features = np.load(os.path.join(data_dir, aud_file))
        self.background_img = torch.tensor(_imread_rgb(os.path.join(data_dir, "bc.jpg")) / 255.0).to(self.device)
        self.focal, self.cx, self.cy = float(self.meta["focal_len"]), float(self.meta["cx"]), float(self.meta["cy"])
        self.H, self.W = int(self.cy * 2), int(self.cx * 2)
        self.skip = 1 if mode == "train" else getattr(args, "testskip", 1)
        self.all_imgs, self.all_parse_imgs, self.all_landmarks = [], [], []
        self.all_poses, self.all_face_rects, self.all_exprs, auds = [], [], [], []
        for frame in self.meta["frames"][::skip]:
            iid = str(frame["img_id"])
            self.all_imgs.append(os.path.join(data_dir, args.gt_dirs, iid + ".jpg"))
            self.all_landmarks.append(os.path.join(data_dir, "ori_imgs", iid + ".lms"))
            self.all_parse_imgs.append(os.path.join(data_dir, "parsing", iid + ".png"))
            self.all_poses.append(np.array(frame["transform_matrix"]))
            auds.append(self.aud_features[min(frame["aud_id"], self.aud_features.shape[0] - 1)])
            self.all_face_rects.append(np.array(frame["face_rect"], dtype=np.int32))
            self.all_exprs.append(frame["exp"])
        self.data_size = len(self.all_imgs)
        self.auds = torch.tensor(np.asarray(auds), dtype=torch.float).to(self.device)

    def __len__(self):
        return self.data_size

    def sample_pixels(self, face_rect, landmark, parse_img):
        """The pixel selection of sample_rays (:141-187), same region tests and the same order of np.random.choice draws
        (mouth, torso, face rectangle, outside), returned as (N_rand, 2) int64 (row, col) in the reference's concatenation order
        (rect, norect, mouth, torso).  NB the reference compares the ROW coordinate with the x ranges (coords[:, 0] is the row)."""
        a, H, W = self.args, self.H, self.W
        lm = landmark[48:]
        max_x, min_x = np.max(lm[:, 0]) + 20, np.min(lm[:, 0]) - 20
        max_y, min_y = np.max(lm[:, 1]) + 20, np.min(lm[:, 1]) - 20
        rr, cc = np.meshgrid(np.arange(H), np.arange(W), indexing="ij")
        coords = np.stack([rr, cc], -1).reshape(-1, 2)
        mouth = (coords[:, 0] >= min_x) & (coords[:, 0] <= max_x) & (coords[:, 1] >= min_y) & (coords[:, 1] <= max_y)
        rect = (coords[:, 0] >= face_rect[0]) & (coords[:, 0] <= face_rect[0] + face_rect[2]) & \
               (coords[:, 1] >= face_rect[1]) & (coords[:, 1] <= face_rect[1] + face_rect[3])
        torso = ((parse_img[:, :, 0] == 255) & (parse_img[:, :, 1] == 0) & (parse_img[:, :, 2] == 0)).reshape(-1)
        c_mouth, c_rect, c_norect, c_torso = coords[mouth], coords[rect & ~mouth], coords[~rect], coords[torso]
        mouth_num, torso_num = a.mouth_rays, a.torso_rays
        sample_num = a.N_rand - mouth_num - torso_num
        rect_num = int(sample_num * a.sample_rate)
        norect_num = sample_num - rect_num
        s_mouth = c_mouth[np.random.choice(c_mouth.shape[0], size=[mouth_num], replace=False)]
        s_torso = c_torso[np.random.choice(c_torso.shape[0], size=[torso_num], replace=False)]
        s_rect = c_rect[np.random.choice(c_rect.shape[0], size=[rect_num], replace=False)]
        s_norect = c_norect[np.random.choice(c_norect.shape[0], size=[norect_num], replace=False)]
        return np.concatenate([s_rect, s_norect, s_mouth, s_torso], 0).astype(np.int64)

    def __getitem__(self, index):
        if index is None:
            index = np.random.choice(self.data_size)
        raw_img = torch.tensor(_imread_rgb(self.all_imgs[index])[:, :, ::-1].copy())            # cv2.imread order: BGR
        self.H, self.W = raw_img.shape[0], raw_img.shape[1]
        target = raw_img.to(self.device).float() / 255.0
        parse = _imread_rgb(self.all_parse_imgs[index])
        pose = self.all_poses[index][:3, :4]
        sel = torch.from_numpy(self.sample_pixels(self.all_face_rects[index], np.loadtxt(self.all_landmarks[index]), parse)).to(self.device)
        rays = ops.get_rays_at(sel, self.focal, torch.tensor(pose, dtype=torch.float32, device=self.device), 0.0, 1.0, self.cx, self.cy)
        batch_rays = torch.stack([rays[:, 0:3], rays[:, 3:6]], 0)
        target_s = target[sel[:, 0], sel[:, 1]]
        bc_rgb = self.background_img[sel[:, 0], sel[:, 1]] if self.mode == "train" else self.background_img
        exp = torch.tensor(self.all_exprs[index], dtype=torch.float32)
        return batch_rays, target_s, bc_rgb, self.auds, raw_img, pose, exp, index


# ---- the device-resident dataset -------------------------------------------------------------------------------------------------
REGIONS = ("rect", "norect", "mouth", "torso")          # the output order of sample_pixels and of inerf_sample_train_pixels


def region_budgets(args):
    """(rect, norect, mouth, torso) rows of sample_pixels: mouth_rays, torso_rays, int((N_rand - mouth - torso) * sample_rate), the rest."""
    mouth, torso = int(args.mouth_rays), int(args.torso_rays)
    sample_num = int(args.N_rand) - mouth - torso
    rect = int(sample_num * args.sample_rate)
    k = (rect, sample_num - rect, mouth, torso)
    if min(k) < 0:
        raise ValueError(f"negative region budget {dict(zip(REGIONS, k))} from N_rand={args.N_rand}, mouth_rays={args.mouth_rays}, "
                         f"torso_rays={args.torso_rays}, sample_rate={args.sample_rate}")
    return k


def _lower(v, n):
    """Smallest integer i in [0, n] with i >= v (n: none of 0..n-1 qualifies)."""
    return n if np.isnan(v) else int(np.clip(np.ceil(v), 0, n))


def _upper(v, n):
    """Largest integer i in [-1, n-1] with i <= v (-1: none of 0..n-1 qualifies)."""
    return -1 if np.isnan(v) else int(np.clip(np.floor(v), -1, n - 1))


def region_bounds(face_rect, landmark, H, W):
    """int32 (8,) = inclusive (row lo, row hi, col lo, col hi) of the face rectangle, then of the mouth box, such that integer tests on
    (row, col) select exactly the pixels of sample_pixels' predicates (the mouth's row against the landmarks' x range and its column
    against their y range, as the reference compares them; float thresholds rounded inwards)."""
    lm = np.asarray(landmark, dtype=np.float64)[48:]
    fr = [int(v) for v in face_rect]
    mr0, mr1 = np.min(lm[:, 0]) - 20, np.max(lm[:, 0]) + 20
    mc0, mc1 = np.min(lm[:, 1]) - 20, np.max(lm[:, 1]) + 20
    return np.array([_lower(fr[0], H), _upper(fr[0] + fr[2], H), _lower(fr[1], W), _upper(fr[1] + fr[3], W),
                     _lower(mr0, H), _upper(mr1, H), _lower(mc0, W), _upper(mc1, W)], dtype=np.int32)


def torso_bits(parse_img):
    """uint32 (ceil(H*W/32),): bit p & 31 of word p >> 5 is set where parsing pixel p = row * W + col is pure red (255, 0, 0)."""
    t = ((parse_img[:, :, 0] == 255) & (parse_img[:, :, 1] == 0) & (parse_img[:, :, 2] == 0)).reshape(-1)
    t = np.concatenate([t, np.zeros((-t.size) % 32, bool)])
    return (t.reshape(-1, 32).astype(np.uint64) << np.arange(32, dtype=np.uint64)).sum(1).astype(np.uint32)


def region_sizes(bounds, n_torso, H, W):
    """Members of (rect, norect, mouth, torso) of each frame: bounds (F, 8) as region_bounds, n_torso (F,) -> int64 (F, 4)."""
    b = np.asarray(bounds, dtype=np.int64)

    def area(r0, r1, c0, c1):
        return np.maximum(r1 - r0 + 1, 0) * np.maximum(c1 - c0 + 1, 0)

    rect = area(b[:, 0], b[:, 1], b[:, 2], b[:, 3])
    mouth = area(b[:, 4], b[:, 5], b[:, 6], b[:, 7])
    both = area(np.maximum(b[:, 0], b[:, 4]), np.minimum(b[:, 1], b[:, 5]), np.maximum(b[:, 2], b[:, 6]), np.minimum(b[:, 3], b[:, 7]))
    return np.stack([rect - both, H * W - rect, mouth, np.asarray(n_torso, dtype=np.int64)], 1)


def check_region_sizes(sizes, budgets, names=None):
    """ValueError naming the first frame and region with fewer members than its budget (np.random.choice(replace=False) would raise there
    in the middle of training)."""
    short = np.argwhere(np.asarray(sizes) < np.asarray(budgets)[None, :])
    if len(short):
        f, r = (int(v) for v in short[0])
        name = names[f] if names is not None else str(f)
        raise ValueError(f"frame {f} ({name}): region '{REGIONS[r]}' has {int(sizes[f][r])} pixels, fewer than its budget of {budgets[r]} rays")


class DeviceHeadDataset(HeadDataset):
    """HeadDataset with every frame decoded once and kept on the device (BGR uint8), and each training batch drawn there.

    sample(index) draws the batch with the region budgets of sample_pixels -- from the same distribution, not the same numbers: the draw
    is the Philox contract of inerf_sample_train_pixels (include/inerf_b200.h) -- and builds rays, targets, bc_rgb, the audio window, the
    expression and the pose without a host synchronise, so `index` may be an int64 device tensor and the call may sit in a CUDA graph.
    Memory: F * H * W * 3 bytes of frames (5 000 frames of 450 x 450: 3.0 GB) plus small per-frame tables."""

    def __init__(self, data_dir, aud_file, mode, args, skip=1, device="cuda"):
        super().__init__(data_dir, aud_file, mode, args, skip, device)
        self.budgets = region_budgets(args)
        imgs = [_imread_rgb(p)[:, :, ::-1] for p in self.all_imgs]              # cv2.imread order: BGR
        shapes = {im.shape for im in imgs}
        if len(shapes) != 1:
            raise ValueError(f"frames differ in size: {sorted(shapes)}")
        H, W = imgs[0].shape[:2]
        if tuple(self.background_img.shape[:2]) != (H, W):
            raise ValueError(f"bc.jpg is {tuple(self.background_img.shape[:2])}, the frames are {(H, W)}")
        if H * W > _lib.INERF_PIXEL_SAMPLER_MAX_PIXELS:
            raise ValueError(f"{H} x {W} frames exceed the sampler's {_lib.INERF_PIXEL_SAMPLER_MAX_PIXELS} pixels")
        self.H, self.W = H, W
        bounds, bits, n_torso = [], [], []
        for rect, lms, parse in zip(self.all_face_rects, self.all_landmarks, self.all_parse_imgs):
            bounds.append(region_bounds(rect, np.loadtxt(lms), H, W))
            b = torso_bits(_imread_rgb(parse))
            bits.append(b)
            n_torso.append(int(np.unpackbits(b.view(np.uint8)).sum()))
        check_region_sizes(region_sizes(np.stack(bounds), n_torso, H, W), self.budgets, [os.path.basename(p) for p in self.all_imgs])
        dev = self.device
        self.frames = torch.from_numpy(np.ascontiguousarray(np.stack(imgs))).to(dev)
        self.bounds = torch.from_numpy(np.stack(bounds)).to(dev)
        self.torso_bits = torch.from_numpy(np.stack(bits).view(np.int32)).to(dev)
        self.poses = torch.tensor(np.stack(self.all_poses)[:, :3, :4], dtype=torch.float32, device=dev)
        self.exprs = torch.tensor(np.asarray(self.all_exprs), dtype=torch.float32, device=dev)
        self.bc_img = self.background_img.float().contiguous()
        half = int(getattr(args, "smo_size", 8) / 2)
        pad = torch.zeros((half,) + tuple(self.auds.shape[1:]), dtype=self.auds.dtype, device=dev)
        self.auds_padded = torch.cat([pad, self.auds, pad], 0)
        self._win = torch.arange(2 * half, dtype=torch.int64, device=dev)
        self._index = torch.zeros((), dtype=torch.int64, device=dev)

    def _draw(self, index, rank, world, want_coords):
        """(idx (1,) int64 device tensor, ops.sample_train_pixels' (rays, target, bc_rgb, coords)) of rows frame.band(N_rand, rank, world)
        of frame `index`'s batch."""
        from .frame import band
        if torch.is_tensor(index):
            idx = index.reshape(())
            if idx.dtype != torch.int64 or idx.device != self.frames.device:
                raise ValueError(f"a tensor index must be an int64 scalar on {self.frames.device}")
        else:
            if not 0 <= int(index) < self.data_size:
                raise IndexError(f"frame {index} outside [0, {self.data_size})")
            idx = self._index.fill_(int(index))
        lo, hi = band(sum(self.budgets), rank, world)
        batch = ops.sample_train_pixels(idx, self.budgets, self.bounds, self.torso_bits, self.poses, self.frames, self.bc_img, self.focal,
                                        self.cx, self.cy, self.args.near, self.args.far, first=lo, count=hi - lo, want_coords=want_coords)
        return idx.reshape(1), batch

    def sample(self, index, rank=0, world=1):
        """The training batch of frame `index` (host int or int64 device scalar), rows frame.band(N_rand, rank, world) of it: a dict with
        rays (n, 11) packed with args.near / args.far, target (n, 3), bc_rgb (n, 3), aud_window (smo_size, 16, 29) =
        Network.audio_window(auds, index, len(self)), expr, pose (3, 4).  Advances the Philox offset by one."""
        i1, (rays, target, bc_rgb, _) = self._draw(index, rank, world, False)
        return {"rays": rays, "target": target, "bc_rgb": bc_rgb, "aud_window": self.auds_padded.index_select(0, i1 + self._win),
                "expr": self.exprs.index_select(0, i1)[0], "pose": self.poses.index_select(0, i1)[0]}

    def __getitem__(self, index):
        """HeadDataset's tuple (batch_rays (2, N_rand, 3), target_s, bc_rgb, auds, raw_img, pose, exp, index) built from sample(): raw_img
        is the device frame (BGR uint8), bc_rgb fp32."""
        if index is None:
            index = np.random.choice(self.data_size)
        b = DeviceHeadDataset.sample(self, index)
        rays = b["rays"]
        batch_rays = torch.stack([rays[:, 0:3], rays[:, 3:6]], 0)
        return batch_rays, b["target"], b["bc_rgb"], self.auds, self.frames[index], self.all_poses[index][:3, :4], b["expr"], index


class DeviceTorsoDataset(DeviceHeadDataset):
    """The torso stage's batches (NeRFs/TorsoNeRF/train_torso.py) drawn on the device: DeviceHeadDataset's files, checks and region
    budgets, with targets from args.gt_dirs (for this stage the composited head + torso frames, conventionally com_imgs), plus what
    train.TorsoTrainStep takes besides the head batch.

    The pixels are drawn with the head stage's region machinery (face rect, mouth box, torso mask and their budgets) on the gt_dirs frames.
    The reference's train_torso.py loader was not available when this was written, so that it samples the same regions is not verified.

    aud_codes: (F, args.dim_aud), row i = the frozen head's audio code of frame i, computed once, e.g. evaluate.audio_codes(head_network,
    HeadDataset(...)) after checkpoint.load_head_checkpoint (the torso stage trains no audio net).  latent_codes: (F, 32), as
    checkpoint.load_head_into_torso returns them; required for mode "train", optional otherwise (sample() then raises).  torso_pose: the
    fixed camera of the torso pair, (3, 4) or (4, 4); default: the transform_matrix of the first frame of transforms_exp_train.json, for
    every mode (the frame-0 camera of frame.HeadTorsoFrameRenderer: a val split is rendered from the camera the torso was trained with).
    Kept as torso_pose (3, 4) fp32 on the device.  A table of the wrong shape raises ValueError here, naming it.

    sample(index, rank=0, world=1) returns a dict keyed by TorsoTrainStep's parameters, so step(**ds.sample(i)) runs one iteration:
    rays_head, target, bc_rgb are DeviceHeadDataset.sample's rays, target and bc_rgb for the same Philox state (one draw; the offset advances
    once); rays_torso are the rays of the same pixels from torso_pose (ops.get_rays_at on the sampler's coordinates, the bits the sampler
    writes for a pose); aud_feature, pose (3, 4), expr, latent_code are row `index` of the tables.  No host synchronise: `index` may be an
    int64 device scalar and the call may sit in a CUDA graph.  __getitem__ keeps DeviceHeadDataset's tuple."""

    def __init__(self, data_dir, aud_file, mode, args, aud_codes, latent_codes=None, torso_pose=None, skip=1, device="cuda"):
        super().__init__(data_dir, aud_file, mode, args, skip, device)
        if torso_pose is None:
            with open(os.path.join(data_dir, "transforms_exp_train.json")) as fp:
                torso_pose = json.load(fp)["frames"][0]["transform_matrix"]
        pose = torch.as_tensor(torso_pose).detach()
        if tuple(pose.shape) not in ((3, 4), (4, 4)):
            raise ValueError(f"torso_pose is {tuple(pose.shape)}, not (3, 4) or (4, 4)")
        self.torso_pose = pose[:3].to(self.device, torch.float32).contiguous()
        self.aud_codes = self._table("aud_codes", aud_codes, int(args.dim_aud))
        if latent_codes is None and mode == "train":
            raise ValueError("latent_codes: the train split needs the head's (F, 32) latent codes")
        self.latent_codes = None if latent_codes is None else self._table("latent_codes", latent_codes, 32)

    def _table(self, name, t, width):
        t = torch.as_tensor(t).detach()
        if tuple(t.shape) != (self.data_size, width):
            raise ValueError(f"{name} is {tuple(t.shape)}, this split needs ({self.data_size}, {width})")
        return t.to(self.device, torch.float32).contiguous()

    def sample(self, index, rank=0, world=1):
        """The torso batch of frame `index` (host int or int64 device scalar), rows frame.band(N_rand, rank, world) of it: {rays_head,
        rays_torso (n, 11), bc_rgb, target (n, 3), aud_feature (dim_aud,), pose (3, 4), expr, latent_code (32,)}.  Advances the Philox
        offset by one."""
        if self.latent_codes is None:
            raise ValueError("DeviceTorsoDataset.sample needs latent_codes (given none for this split)")
        i1, (rays, target, bc_rgb, coords) = self._draw(index, rank, world, True)
        rays_torso = ops.get_rays_at(coords, self.focal, self.torso_pose, self.args.near, self.args.far, self.cx, self.cy)
        return {"rays_head": rays, "rays_torso": rays_torso, "bc_rgb": bc_rgb, "target": target,
                "aud_feature": self.aud_codes.index_select(0, i1)[0], "pose": self.poses.index_select(0, i1)[0],
                "expr": self.exprs.index_select(0, i1)[0], "latent_code": self.latent_codes.index_select(0, i1)[0]}
