"""Train a talking head from a dataset directory: the head stage of NeRFs/HeadNeRF/train/audio_exp_nerf.py:451-593 (fit_head) and the
torso stage of NeRFs/TorsoNeRF/train_torso.py (fit_torso), on one GPU or data parallel over NCCL.

    python -m ideal_nerf_b200.fit --config subject.txt [--stage head] [reference flags]
    python -m ideal_nerf_b200.fit --config subject_torso.txt --stage torso --head_ckpt <basedir>/<head expname>/head.tar
    torchrun --nproc_per_node N -m ideal_nerf_b200.fit --config subject.txt           # one process per GPU, NCCL

Flags and --config files are helper.config_parser's (the reference's names and defaults), plus --stage, --head_ckpt and --seed.
Each step is the existing device path: DeviceHeadDataset / DeviceTorsoDataset.sample draws the batch, TrainStep / TorsoTrainStep
(cuda_graph=True) replays the iteration as one CUDA graph.  Per step the host issues the draw and the replay and nothing else; it
synchronises with the device only on boundary steps (see Fit.run):

* log, every i_print steps and at the end: every step wrote its losses, the PSNR of img_loss and the learning rate into the step's
  device log ring (log_rows = i_print); rank 0 copies the ring to the host once and appends one JSON line per step to
  <basedir>/<expname>/log.jsonl with the reference's TensorBoard scalar names (train/loss, train/psnr, train/learning_rate and, for
  the head, train/latent_code_loss).
* save, every i_weights steps and at the end: rank 0 writes the checkpoint under the reference's name -- head.tar for the head
  (audio_exp_nerf.py:584-591), {global_step:06d}_torso.tar for the torso (train_torso.py:565-572) -- through a temporary file.
* validate, every i_testset steps: evaluate_split on the val split (zero training budgets, keep_video=False, perturb = 0), one line
  with val/psnr, val/psnr_face, val/psnr_mouth, val/ssim (and val/psnr_torso for the torso stage).
* image, every i_img steps: frame 0 of the val split rendered and written as val_{global_step:06d}.png (the stand-in for the
  reference's TensorBoard image).
Validation and the image render in eval() mode and switch back to train() afterwards: both switches drop the FaceNeRFs' packed-weight
caches, which the graph's in-place Adam updates do not invalidate (FaceNeRF.invalidate_packed).

Frame order: N_iters epochs over the train frames, each epoch a permutation of them from numpy's generator seeded with (seed, epoch) --
the same on every rank, uploaded once per epoch.  Whether the reference's DataLoader (audio_exp_nerf.py:466-474) shuffles is not
recorded, and its loop (:529-530) was not at hand when this was written: that it visits the frames in a permutation per epoch is not
verified.

Randomness: the in-kernel Philox stream is re-seeded with (seed, 64 * global_step) at start-up and after every boundary step, so that
all ranks draw alike (complementary bands of one batch) and a run resumed from a checkpoint of a boundary step draws what the
uninterrupted run drew.

Resume: unless --no_reload, the naturally sorted last checkpoint of <basedir>/<expname> (any *.tar for the head, as :516-525; the
*_torso.tar files for the torso) is loaded through TrainStep.load / TorsoTrainStep.load -- weights, latent codes, Adam state,
learning rate, global_step -- before the first step; else --ft_path starts the head from checkpoint.load_finetune_checkpoint
(:498-514)."""
import copy
import json
import os
import re

import numpy as np
import torch
import torch.distributed as dist

from . import checkpoint, ops
from .data import DeviceHeadDataset, DeviceTorsoDataset, HeadDataset
from .evaluate import audio_codes, evaluate_split
from .frame import FrameRenderer, HeadTorsoFrameRenderer
from .helper import config_parser
from .render import Network, TorsoNetwork, init_weights
from .train import TorsoTrainStep, TrainStep

RNG_STRIDE = 64          # Philox offsets per global step; a step uses at most 3 (the draw, one per render pass)
HEAD_CKPT = "head.tar"
SCALARS = {"loss": "train/loss", "psnr": "train/psnr", "lr": "train/learning_rate", "latent_code_loss": "train/latent_code_loss"}


def fit_parser():
    """helper.config_parser plus the trainer's own flags."""
    p = config_parser()
    p.add_argument("--stage", choices=("head", "torso"), default="head")
    p.add_argument("--head_ckpt", type=str, default=None, help="torso stage: the head.tar the torso is trained under")
    p.add_argument("--seed", type=int, default=0, help="weights, frame order and Philox stream")
    return p


def run_dir(args):
    return os.path.join(args.basedir, args.expname)


def _natural_key(name):
    return [int(t) if t.isdigit() else t for t in re.split(r"(\d+)", name)]


def latest_checkpoint(d, suffix=".tar"):
    """The naturally sorted last file of directory d ending in `suffix` (audio_exp_nerf.py:516-525), or None."""
    if not os.path.isdir(d):
        return None
    names = sorted((f for f in os.listdir(d) if f.endswith(suffix)), key=_natural_key)
    return os.path.join(d, names[-1]) if names else None


def checkpoint_name(stage, global_step):
    return HEAD_CKPT if stage == "head" else f"{int(global_step):06d}_torso.tar"


def epoch_order(seed, epoch, n):
    """The frame permutation of `epoch`: int64 (n,), a function of (seed, epoch) only."""
    return np.random.default_rng([int(seed), int(epoch)]).permutation(n).astype(np.int64)


def events(global_step, args, total):
    """What happens after the step that brings the count to `global_step` (1-based) in a run of `total` steps."""
    s = int(global_step)

    def every(n):
        return int(n) > 0 and s % int(n) == 0

    return {"log": every(args.i_print) or s == total, "save": every(args.i_weights) or s == total,
            "val": every(args.i_testset), "img": every(args.i_img)}


def _val_args(args):
    a = copy.copy(args)
    a.N_rand = a.mouth_rays = a.torso_rays = 0          # evaluation never draws a batch (evaluate.py)
    return a


def _has_split(args, mode):
    return os.path.isfile(os.path.join(args.datadir, f"transforms_exp_{mode}.json"))


class Fit:
    """The loop shared by the two stages.  Subclasses build self.step (TrainStep / TorsoTrainStep with cuda_graph=True and
    log_rows = i_print), self.ds (the train split), self.val (the val split or None), self.renderer, and define _call(idx, g),
    _val_codes(g), _latent(); run() then trains to N_iters epochs."""
    stage = None

    def _setup(self, args, rank, world, group):
        if int(args.i_print) < 1:
            raise ValueError(f"i_print must be >= 1 (the log ring holds i_print steps), got {args.i_print}")
        self.args, self.rank, self.world, self.group = args, rank, world, group
        self.seed = int(getattr(args, "seed", 0))                         # helper.config_parser has no --seed; fit_parser adds it
        self.dev = torch.device("cuda", torch.cuda.current_device())
        self.dir = run_dir(args)
        if rank == 0:
            os.makedirs(self.dir, exist_ok=True)
        self.log_path = os.path.join(self.dir, "log.jsonl")

    def _start(self, suffix):
        """Resumes from the latest checkpoint unless --no_reload (self.resumed: its path or None), then seeds the Philox stream for the
        first step."""
        self.resumed = None if self.args.no_reload else latest_checkpoint(self.dir, suffix)
        if self.resumed is not None:
            self.step.load(self.resumed, map_location=self.dev)
        self._order, self._epoch, self._logged = None, -1, self.step.global_step
        ops.seed_rng(self.seed, self.dev, RNG_STRIDE * self.step.global_step)

    @property
    def total(self):
        return int(self.args.N_iters) * len(self.ds)

    def run(self, stop=None):
        """Train up to global_step = stop (default: N_iters epochs).  Between boundary steps nothing here synchronises with the device:
        the frame index is a device scalar, the epoch's permutation goes up once through pinned memory, and the losses stay in the step's
        log ring."""
        a, n = self.args, len(self.ds)
        stop = self.total if stop is None else min(int(stop), self.total)
        g = self.step.global_step
        while g < stop:
            if g // n != self._epoch:
                self._epoch = g // n
                self._order = torch.from_numpy(epoch_order(self.seed, self._epoch, n)).pin_memory().to(self.dev, non_blocking=True)
            self._call(self._order[g % n], g)
            g += 1
            ev = events(g, a, self.total)
            if not any(ev.values()):
                continue
            if ev["log"]:
                self._flush_log(g)
            if ev["save"] and self.rank == 0:
                path = os.path.join(self.dir, checkpoint_name(self.stage, g))
                self.step.save(path + ".tmp")
                os.replace(path + ".tmp", path)
            if self.val is not None and (ev["val"] or ev["img"]):
                self._validate(g, ev["val"], ev["img"])
            ops.seed_rng(self.seed, self.dev, RNG_STRIDE * g)
        return self

    def _append(self, lines):
        with open(self.log_path, "a") as fp:
            for d in lines:
                fp.write(json.dumps(d) + "\n")

    def _flush_log(self, g):
        """Rank 0: one line per step since the last flush, from one host copy of the log ring."""
        if self.rank != 0:
            return
        ring = self.step.log_ring.cpu().numpy().astype(np.float64)
        cols = type(self.step).LOG_COLUMNS
        lines = []
        for j in range(self._logged, g):
            row = dict(zip(cols, ring[j % ring.shape[0]].tolist()))
            lines.append({"step": j + 1, **{SCALARS[c]: row[c] for c in cols if c in SCALARS}})
        self._logged = g
        self._append(lines)

    @torch.no_grad()
    def _validate(self, g, score, image):
        net = self.step.net
        net.eval()
        codes = self._val_codes(g)
        latent = self._latent()
        if score:
            res = evaluate_split(self.renderer, self.val, latent, codes, keep_video=False)
            if self.rank == 0:
                p = res["mean_psnr"]
                line = {"step": g, "val/psnr": float(p[0]), "val/psnr_face": float(p[1]), "val/psnr_mouth": float(p[2]),
                        "val/ssim": float(res["mean_ssim"])}
                if "mean_psnr_torso" in res:
                    line["val/psnr_torso"] = float(res["mean_psnr_torso"])
                self._append([line])
        if image:
            v = self.val
            rgb = self.renderer.render_frame(v.poses[0], codes[0], v.exprs[0], latent, v.bc_img, 0.)
            if self.rank == 0:
                from PIL import Image
                img = ops.to8b(rgb).reshape(v.H, v.W, 3).cpu().numpy()[:, :, ::-1]          # the frames are BGR
                Image.fromarray(np.ascontiguousarray(img)).save(os.path.join(self.dir, f"val_{g:06d}.png"))
        net.train()


class HeadFit(Fit):
    """fit_head's state: network, latent codes, datasets, the graph step and the loop position.

    Audio phases (Network.audio_feature, audio_exp_nerf.py:241-266): a step with global_step < nosmo_iters conditions on AudioNet of the
    frame's own DeepSpeech features (TrainStep(smooth=False): row smo_size // 2 of the sampled window), so AudioNet trains and
    AudioAttNet does not; from nosmo_iters on, the smoothing window through AudioNet and AudioAttNet.  TrainStep holds one captured graph per phase (max_graphs=2);
    the switch costs one eager step and one capture.  AudioAttNet's Adam moments stay zero in the first phase, but the flat Adam's step
    count is shared, so its first updates use the bias correction of step nosmo_iters where the reference's per-parameter Adam starts
    AudioAttNet at step 1."""
    stage = "head"

    def __init__(self, args, rank=0, world=1, group=None):
        self._setup(args, rank, world, group)
        dev = self.dev
        self.ds = DeviceHeadDataset(args.datadir, args.aud_file, "train", args, device=dev)
        self.val = None
        if (int(args.i_testset) > 0 or int(args.i_img) > 0) and _has_split(args, "val"):
            self.val = DeviceHeadDataset(args.datadir, args.aud_file, "val", _val_args(args), device=dev)
        torch.manual_seed(self.seed)
        net = Network(self.ds.H, self.ds.W, self.ds.focal, args.near, args.far, args.chunk, None, args.N_samples, args.N_importance,
                      args=args)
        net.apply(init_weights)
        net = net.to(dev).train()
        latent = torch.ones(len(self.ds), 32, device=dev)
        self.step = TrainStep(net, latent, args, world, group, cuda_graph=True, max_graphs=2, log_rows=int(args.i_print))
        self._start(".tar")
        if self.resumed is None and args.ft_path not in (None, "None"):
            checkpoint.load_finetune_checkpoint(args.ft_path, net, map_location=dev)
            for m in (net.face_nerf_coarse, net.face_nerf_fine):
                m.invalidate_packed()
        self.renderer = FrameRenderer(net, rank, world, group)

    def _call(self, idx, g):
        b = self.ds.sample(idx, self.rank, self.world)
        self.step(b["rays"], b["bc_rgb"], b["target"], None, b["expr"], idx, aud_window=b["aud_window"],
                  smooth=g >= int(self.args.nosmo_iters))

    def _val_codes(self, g):
        """The val frames' audio codes in the phase of step g (Network.audio_feature(auds, i, F, g))."""
        v, net = self.val, self.step.net
        return torch.stack([net.audio_feature(v.auds, i, len(v), g).reshape(-1) for i in range(len(v))])

    def _latent(self):
        # the held-out frames have no latent code of their own; which row the reference's validation render (:568-582) conditions on
        # was not re-read: row 0
        return self.step.latent_codes.detach()[0]


class TorsoFit(Fit):
    """fit_torso's state.  The torso network's head pair comes from `head_tar` (checkpoint.load_head_into_torso), and so do the latent
    codes; each frame's audio code is the head's smoothed code (evaluate.audio_codes, AudioNet then AudioAttNet), computed once.  Only the
    torso pair trains (TorsoTrainStep).  What TorsoTrainStep documents as unverified carries over: the reference's train_torso.py was not
    at hand, so that its loss and learning-rate schedule are the composites' MSE and audio_exp_nerf.py:554-558's, that its loader samples
    DeviceTorsoDataset's regions, and that its {:06d}_torso.tar has TorsoTrainStep.save's layout are not verified."""
    stage = "torso"

    def __init__(self, args, head_tar, rank=0, world=1, group=None):
        self._setup(args, rank, world, group)
        dev = self.dev
        meta = HeadDataset(args.datadir, args.aud_file, "train", args, device=dev)          # metadata and audio only
        head = Network(meta.H, meta.W, meta.focal, args.near, args.far, args.chunk, None, args.N_samples, args.N_importance,
                       args=args).to(dev)
        checkpoint.load_head_checkpoint(head_tar, head, map_location=dev)
        codes = audio_codes(head, meta)
        torch.manual_seed(self.seed)
        tnet = TorsoNetwork(meta.H, meta.W, meta.focal, args.near, args.far, args.chunk, args.N_samples, args.N_importance, args=args,
                            dim_expr=args.dim_expr)
        tnet.apply(init_weights)
        tnet = tnet.to(dev)
        latent = checkpoint.load_head_into_torso(head_tar, tnet, map_location=dev)
        if latent is None:
            raise ValueError(f"{head_tar} has no latent codes: not a head.tar")
        self.head_latent = latent.to(dev)
        self.ds = DeviceTorsoDataset(args.datadir, args.aud_file, "train", args, codes, self.head_latent, device=dev)
        self.val = None
        if (int(args.i_testset) > 0 or int(args.i_img) > 0) and _has_split(args, "val"):
            va = _val_args(args)
            self._val_code_table = audio_codes(head, HeadDataset(args.datadir, args.aud_file, "val", va, device=dev))
            self.val = DeviceTorsoDataset(args.datadir, args.aud_file, "val", va, self._val_code_table, device=dev)
        del head
        self.step = TorsoTrainStep(tnet.train(), args, world, group, cuda_graph=True, log_rows=int(args.i_print))
        self._start("_torso.tar")
        self.renderer = HeadTorsoFrameRenderer(tnet, self.ds.torso_pose, rank, world, group)

    def _call(self, idx, g):
        self.step(**self.ds.sample(idx, self.rank, self.world))

    def _val_codes(self, g):
        return self._val_code_table

    def _latent(self):
        return self.head_latent[0]


def fit_head(args, rank=0, world=1, group=None):
    """Train the head stage to N_iters epochs (resuming first, see the module docstring); returns the HeadFit."""
    return HeadFit(args, rank, world, group).run()


def fit_torso(args, head_tar, rank=0, world=1, group=None):
    """Train the torso stage under the head of `head_tar` to N_iters epochs; returns the TorsoFit."""
    return TorsoFit(args, head_tar, rank, world, group).run()


def main(argv=None):
    args = fit_parser().parse_args(argv)
    if not args.basedir or not args.expname:
        raise SystemExit("--basedir and --expname name the run directory")
    if args.stage == "torso" and not args.head_ckpt:
        raise SystemExit("--stage torso needs --head_ckpt, the head.tar of the head stage")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    try:
        if args.stage == "head":
            fit_head(args, rank, world)
        else:
            fit_torso(args, args.head_ckpt, rank, world)
    finally:
        if world > 1:
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
