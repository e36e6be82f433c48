"""Head + torso talking-head video (test_torso.py:516-531) through frame.render_head_torso_video: fps and frame latency.

    python profiles/head_torso_video.py [--frames 200] [--out FILE]                  # one GPU
    torchrun --nproc-per-node N profiles/head_torso_video.py [--frames 200]          # rays of every frame sharded over N GPUs

450 x 450 frames, 64 + 128 samples per ray for both the head pair and the torso pair, perturb = 0, bf16 tensor-core MLP mode; the four
FaceNeRFs are random-init with the normalised-density preset (the torso neither empty nor opaque), the torso rays come from the frame-0
camera, and every frame has its own head pose and audio / expression codes (a seeded random walk).  Reported:
  * render_head_torso_video over --frames frames: blend + to8b in one kernel per band, uint8 band all-gather, one pinned host array;
    the time runs from the first launch to the end of the last host copy (device events, max over ranks); measured twice;
  * render_video (the fp32 driver: fp32 band gather, to8b on rank 0) on the same renderer and frames, for comparison;
  * render_video(FrameRenderer(net)) -- the head pair alone on the same frames -- the single-model frame the composite costs ~2x of;
  * frame latency: one frame rendered, gathered and copied to the host with a synchronise, median of 10 after 2 warm-up frames;
  * a checksum of the video bytes: equal at every GPU count when the sharded frames are bit-identical.
"""
import argparse
import math
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402
import ideal_nerf_b200 as M  # noqa: E402
from ideal_nerf_b200 import ops, synthetic as S  # noqa: E402
from ideal_nerf_b200.frame import FrameRenderer, HeadTorsoFrameRenderer, render_head_torso_video, render_video  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--frames", type=int, default=200)
ap.add_argument("--out", default=None, help="also write the report to this file (rank 0)")
args = ap.parse_args()

world = int(os.environ.get("WORLD_SIZE", "1"))
rank = int(os.environ.get("RANK", "0"))
local = int(os.environ.get("LOCAL_RANK", "0"))
assert torch.cuda.is_available(), "needs a GPU"
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
if world > 1:
    dist.init_process_group("nccl", device_id=dev)
lines = []


def say(s):
    if rank == 0:
        print(s, flush=True)
        lines.append(s)


def barrier():
    if world > 1:
        dist.barrier()


def max_over_ranks(x):
    t = torch.tensor([x], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


if rank == 0:
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:          # the measurement stands without it, but says so
        smi = f"nvidia-smi unavailable ({e})"
    say(f"card: {torch.cuda.get_device_name(dev)}; nvidia-smi name, power limit, max SM clock: {smi}; GPUs: {world}")

H = W = 450
cam, fr = S.camera(), S.frame_inputs(0)
T = args.frames
torch.manual_seed(1234)                                          # the same weights on every rank
net = M.TorsoNetwork(H, W, cam["focal"], S.NEAR, S.FAR, 1 << 20, 64, 128,
                     args=M.default_args(dim_aud=64, dim_expr=79, perturb=0., mlp_mode="bf16", N_samples=64, N_importance=128))
net.apply(M.init_weights)
net = net.to(dev).eval()
g = torch.Generator().manual_seed(17)
auds = torch.cumsum(torch.randn(T, 64, generator=g) * 0.1, 0).to(dev)
exprs = torch.cumsum(torch.randn(T, 79, generator=g) * 0.1, 0).to(dev)


def pose(i):
    """Head pose of frame i: the camera turned about y by up to 0.05 rad and shifted sideways by up to 1 cm."""
    p = cam["c2w"].clone()
    a = 0.05 * math.sin(2 * math.pi * i / 100)
    p[:3, :3] = torch.tensor([[math.cos(a), 0., math.sin(a)], [0., 1., 0.], [-math.sin(a), 0., math.cos(a)]])
    p[0, 3] += 0.01 * math.sin(2 * math.pi * i / 70)
    return p.to(dev)


pose0 = cam["c2w"].to(dev)                                        # frame-0 camera of the torso rays (train_torso.py:132-134)
lat, bc = fr["latent"].to(dev), fr["bc_rgb"].to(dev)
frames = [(pose(i), auds[i], exprs[i]) for i in range(T)]
with torch.no_grad():
    rays_h = ops.get_rays_packed(H, W, cam["focal"], frames[0][0], S.NEAR, S.FAR)[::197].contiguous()
    rays_t = ops.get_rays_packed(H, W, cam["focal"], pose0, S.NEAR, S.FAR)[::197].contiguous()
    for fn in (net.face_nerf_coarse, net.face_nerf_fine):
        S.normalise_density_(fn, rays_h, auds[0], exprs[0], lat)
    sig = net.torso_signal(auds[0], frames[0][0])
    for fn in (net.torso_coarse_nerf, net.torso_fine_nerf):
        S.normalise_density_(fn, rays_t, sig, None, None)

with torch.no_grad():
    lw0 = float(HeadTorsoFrameRenderer(net, pose0).render_passes(*frames[0], lat, bc)[1]["last_weight"].mean())
say(f"torso mean last_weight of frame 0: {lw0:.3f} (the preset is neither empty nor opaque)")
renderer = HeadTorsoFrameRenderer(net, pose0, rank, world)
head_only = FrameRenderer(net, rank, world)


def timed_video(fn, r):
    with torch.no_grad():
        fn(r, frames[:4], lat, bc)                                # warm-up: every kernel, the gather buffers, the pinned allocator
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        vid = fn(r, frames, lat, bc)
        e1.record()
        torch.cuda.synchronize()
        barrier()
    return max_over_ranks(e0.elapsed_time(e1)), vid


def report(name, ms):
    say(f"{name:62s} {T} frames {ms:9.1f} ms  {T / (ms * 1e-3):7.2f} fps  {ms / T:7.2f} ms/frame")


ms_a, vid = timed_video(render_head_torso_video, renderer)
report("render_head_torso_video (uint8 band gather)", ms_a)
ms_b, vid32 = timed_video(render_video, renderer)
report("render_video(HeadTorsoFrameRenderer) (fp32 band gather)", ms_b)
ms_h, _ = timed_video(render_video, head_only)
report("render_video(FrameRenderer) -- head pair alone", ms_h)
ms_a2, _ = timed_video(render_head_torso_video, renderer)
report("render_head_torso_video, again", ms_a2)

one = torch.empty((H, W, 3), dtype=torch.uint8).pin_memory()
lat_ms = []
with torch.no_grad():
    for i in range(12):
        barrier()
        t0 = time.perf_counter()
        u8, _ = renderer.render_band_u8(*frames[i], lat, bc)
        img = renderer.gather_image(u8, H * W)
        if rank == 0:
            one.copy_(img.reshape(H, W, 3), non_blocking=True)
        torch.cuda.synchronize()
        lat_ms.append((time.perf_counter() - t0) * 1e3)
lat_med = max_over_ranks(sorted(lat_ms[2:])[len(lat_ms[2:]) // 2])
say(f"frame latency (render -> uint8 gather -> pinned host copy, synchronised): median {lat_med:.2f} ms over 10 frames")

if rank == 0:
    same = bool(torch.equal(vid, vid32))
    say(f"composite / head-alone time per frame: {ms_a / ms_h:.2f}; uint8 video == fp32-gather video: {same}")
    say(f"video checksum (sum of all bytes): {int(vid.to(torch.int64).sum())}")
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")
if world > 1:
    dist.destroy_process_group()
