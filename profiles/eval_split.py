"""Cost of scoring a held-out split on the device, and the bf16 / fp16x2 render parity on its frames (results: profiles/r08_eval_split.txt).

Writes a synthetic 450 x 450 subject with a 200-frame val split, loads it as an evaluation dataset (zero training budgets), builds a
HeadNeRF with the normalised-density preset (synthetic.normalise_density_) in bf16 mode and, in one process, with perturb = 0:
  (a) render_video alone on the split's 200 frames, and evaluate_split on the same frames (render + score + host copy), alternated
      twice: frames / s of each (wall time of the whole call, which ends in a synchronise);
  (b) the kernel alone (ops.image_metrics of one 450^2 frame, with boxes) with CUDA events over 2 000 back-to-back calls, and one call
      scoring all 200 frames at once;
  (c) the host time of the numpy float64 oracle (oracle/image_metrics_ref.py) per frame, over 5 frames;
  (d) the same split rendered in fp16x2 mode (the fp32-gate tensor-core mode) and the bf16 video scored against it: PSNR and SSIM.
    python profiles/eval_split.py [--frames 200] [--out profiles/r08_eval_split.txt]"""
import argparse
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import ideal_nerf_b200 as M  # noqa: E402
from ideal_nerf_b200 import synthetic as S  # noqa: E402
from ideal_nerf_b200.data import DeviceHeadDataset  # noqa: E402
from ideal_nerf_b200.evaluate import audio_codes, evaluate_split, psnr  # noqa: E402
from ideal_nerf_b200.frame import FrameRenderer, render_video  # noqa: E402
from oracle import image_metrics_ref as IM  # noqa: E402

p = argparse.ArgumentParser()
p.add_argument("--frames", type=int, default=200)
p.add_argument("--out", default=None)
args = p.parse_args()
assert torch.cuda.is_available(), "this measurement needs a GPU"
dev = torch.device("cuda:0")
lines = []


def log(s):
    print(s, flush=True)
    lines.append(s)


smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
log(f"# card: {torch.cuda.get_device_name(0)}; nvidia-smi name, power limit, max SM clock: {smi.stdout.strip() or 'n/a'}")
tmp = tempfile.mkdtemp()
t0 = time.perf_counter()
S.write_head_subject(tmp, 450, 450, n_frames=1, seed=0, torso_rows=40, val_frames=args.frames)
a = M.default_args(N_rand=0, mouth_rays=0, torso_rays=0, gt_dirs="head_imgs", near=S.NEAR, far=S.FAR, dim_aud=64, dim_expr=76, perturb=0.,
                   mlp_mode="bf16")
ds = DeviceHeadDataset(tmp, "aud.npy", "val", a)
F = len(ds)
log(f"# subject: {F} val frames of {ds.H} x {ds.W}, written and loaded in {time.perf_counter() - t0:.1f} s; bf16 mode, perturb 0, "
    "64 + 128 samples")
torch.manual_seed(4321)
net = M.Network(ds.H, ds.W, ds.focal, S.NEAR, S.FAR, 8192, None, 64, 128, args=a)
net.apply(M.init_weights)
net = net.to(dev).eval()
latent = torch.ones(32, device=dev)
codes = audio_codes(net, ds)
rays = M.ops.get_rays_packed(ds.H, ds.W, ds.focal, ds.poses[0], S.NEAR, S.FAR)[::97].contiguous()
for fn in (net.face_nerf_coarse, net.face_nerf_fine):
    S.normalise_density_(fn, rays, codes[0], ds.exprs[0], latent)
frames = [(ds.poses[i], codes[i], ds.exprs[i]) for i in range(F)]
r = FrameRenderer(net)


def wall(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


with torch.no_grad():
    render_video(r, frames[:4], latent, ds.bc_img)                                    # warm-up: modules, blobs, pinned buffers
    evaluate_split(r, ds, latent, codes, keep_video=False)
    t_r, t_e = [], []
    for _ in range(2):
        t, vid_bf16 = wall(lambda: render_video(r, frames, latent, ds.bc_img))
        t_r.append(t)
        t, res = wall(lambda: evaluate_split(r, ds, latent, codes))
        t_e.append(t)
assert np.array_equal(res["video"], vid_bf16.numpy()), "evaluate_split's video differs from render_video's"
log(f"(a) render_video alone:   {F / min(t_r):7.2f} frames/s ({min(t_r) / F * 1e3:.2f} ms / frame; runs {', '.join(f'{t:.2f}' for t in t_r)} s)")
log(f"    evaluate_split:       {F / min(t_e):7.2f} frames/s ({min(t_e) / F * 1e3:.2f} ms / frame; runs {', '.join(f'{t:.2f}' for t in t_e)} s)"
    f"  -> scoring adds {(min(t_e) - min(t_r)) / F * 1e3:+.2f} ms / frame ({(min(t_e) / min(t_r) - 1) * 100:+.1f} %)")
log(f"    scores against the (random-JPEG) ground truth: mean PSNR full / face / mouth {np.round(res['mean_psnr'], 3).tolist()} dB, "
    f"mean SSIM {res['mean_ssim']:.5f}")

# (b) the kernel alone
vid_dev = torch.from_numpy(vid_bf16.numpy()).to(dev)
idx = torch.arange(F, dtype=torch.int64, device=dev)
one, i0 = vid_dev[:1], idx[:1]
for _ in range(50):
    M.ops.image_metrics(one, ds.frames, i0, ds.bounds)
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
n = 2000
e0.record()
for _ in range(n):
    M.ops.image_metrics(one, ds.frames, i0, ds.bounds)
e1.record()
torch.cuda.synchronize()
per = e0.elapsed_time(e1) / n
side = torch.cuda.Stream()                                                            # the same call, 100 times in one CUDA graph:
side.wait_stream(torch.cuda.current_stream())                                        # device time without the Python enqueue
with torch.cuda.stream(side):
    M.ops.image_metrics(one, ds.frames, i0, ds.bounds)
torch.cuda.current_stream().wait_stream(side)
g = torch.cuda.CUDAGraph()
with torch.cuda.graph(g):
    for _ in range(100):
        M.ops.image_metrics(one, ds.frames, i0, ds.bounds)
g.replay()
torch.cuda.synchronize()
e0.record()
for _ in range(20):
    g.replay()
e1.record()
torch.cuda.synchronize()
per_graph = e0.elapsed_time(e1) / 2000
e0.record()
for _ in range(10):
    M.ops.image_metrics(vid_dev, ds.frames, idx, ds.bounds)
e1.record()
torch.cuda.synchronize()
batch = e0.elapsed_time(e1) / 10
log(f"(b) ops.image_metrics, one 450^2 frame with boxes (2 memsets + 1 kernel + the SSIM division): {per * 1e3:.1f} us per call issued "
    f"back to back from Python (CUDA events over {n} calls: the host enqueue bounds it), {per_graph * 1e3:.1f} us per call replayed from a "
    f"CUDA graph (2 000 calls); all {F} frames in one call: {batch:.3f} ms ({batch / F * 1e3:.1f} us / frame, "
    f"{2 * F * ds.H * ds.W * 3 / (batch * 1e-3) / 1e9:.0f} GB/s of frame bytes read)")

# (c) the numpy oracle on the host
gt_host, b_host = ds.frames.cpu().numpy(), ds.bounds.cpu().numpy()
vid_host = vid_bf16.numpy()
t0 = time.perf_counter()
sse, npix, ssim_sum = IM.image_metrics(vid_host[:5], gt_host, np.arange(5), b_host)
t_host = (time.perf_counter() - t0) / 5
assert np.array_equal(sse, res["sse"][:5]) and np.array_equal(npix, res["npix"][:5])
err = np.abs(ssim_sum / (3 * 440 * 440) - res["ssim"][:5]).max()
log(f"(c) numpy float64 oracle on the host: {t_host * 1e3:.1f} ms per frame (5 frames; one CPU thread of the GPU host); kernel vs oracle: "
    f"SSE / npix equal, SSIM max |diff| {err:.2e}")

# (d) bf16 against fp16x2 on the split's frames
net.set_mlp_mode("fp16x2")
with torch.no_grad():
    vid_f16 = render_video(r, frames, latent, ds.bc_img)
ref = torch.from_numpy(vid_f16.numpy()).to(dev)
s = M.ops.image_metrics(vid_dev, ref, idx)
pp = psnr(s["sse"][:, 0], s["npix"][:, 0]).cpu().numpy()
ss = s["ssim"].cpu().numpy()
fin = np.isfinite(pp)
log(f"(d) bf16 video scored against the fp16x2 video of the same {F} frames: PSNR mean {pp[fin].mean() if fin.any() else float('inf'):.2f} dB "
    f"over the {fin.sum()} frames that differ (min {pp.min():.2f} dB; {F - fin.sum()} identical), SSIM mean {ss.mean():.6f} (min {ss.min():.6f}); "
    f"bytes differing {float((vid_dev != ref).float().mean()) * 100:.3f} %, max |diff| {int((vid_dev.int() - ref.int()).abs().max())}")
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fp:
        fp.write("\n".join(lines) + "\n")
