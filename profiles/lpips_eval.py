"""Cost of LPIPS on the device and what it adds to held-out evaluation (results: profiles/r10_lpips.txt).

With seeded AlexNet / lpips-head weights in the released files' layouts (oracle/lpips_ref.seeded_state_dicts: the cost does not depend
on the values), in one process:
  (a) ops.lpips of one 450^2 frame pair: device time per call from CUDA events over a CUDA graph of 100 calls replayed 10 times (1 000
      calls), and per call issued back to back from Python (1 000 calls); the achieved rate from the 11.1 GFLOP of a pair (2 x 2.774
      GMAC) and its ratio to the fp32 FFMA floor (148 SMs x 128 FFMA / clock at the card's max SM clock; DESIGN quotes ~70 TFLOP/s);
  (b) the same call under torch.profiler (CUDA activity only): device time per kernel, to show which layer bounds it;
  (c) the kernel against the float64 oracle on the first 4 rendered frames of the split;
  (d) evaluate_split frames / s on the 200-frame synthetic val split of profiles/eval_split.py (450^2, bf16, perturb 0), without and with
      lpips=, alternated twice.
    python profiles/lpips_eval.py [--frames 200] [--out profiles/r10_lpips.txt]"""
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
from ideal_nerf_b200.evaluate import audio_codes, evaluate_split, load_lpips  # noqa: E402
from ideal_nerf_b200.frame import FrameRenderer  # noqa: E402
from oracle import lpips_ref as LR  # noqa: E402

GMAC_PER_IMAGE = {"conv1": 0.286, "conv2": 0.929, "conv3": 0.484, "conv4": 0.645, "conv5": 0.430}    # at 450^2

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


smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"], capture_output=True,
                     text=True)
log(f"# card: {torch.cuda.get_device_name(0)}; nvidia-smi name, power limit (W), max SM clock (MHz): {smi.stdout.strip() or 'n/a'}")
try:
    clk_mhz = float(smi.stdout.strip().split(",")[2])
except (IndexError, ValueError):
    clk_mhz = float("nan")
sms = torch.cuda.get_device_properties(0).multi_processor_count
floor_tflops = sms * 128 * 2 * clk_mhz * 1e6 / 1e12
flop_pair = 2 * 2 * sum(GMAC_PER_IMAGE.values()) * 1e9

# check the 450^2 MAC count against the layer shapes
sizes = LR.map_sizes(450, 450)
macs = [c * k * k * cin * h * w for (h, w), c, cin, k in zip(sizes, (64, 192, 384, 256, 256), (3, 64, 192, 384, 256), (11, 5, 3, 3, 3))]
assert np.allclose(np.array(macs) / 1e9, list(GMAC_PER_IMAGE.values()), atol=6e-4), macs

tmp = tempfile.mkdtemp()
t0 = time.perf_counter()
S.write_head_subject(tmp, 450, 450, n_frames=1, seed=0, torso_rows=40, val_frames=args.frames)
a = M.default_args(N_rand=0, mouth_rays=0, torso_rays=0, gt_dirs="head_imgs", near=S.NEAR, far=S.FAR, dim_aud=64, dim_expr=76, perturb=0.,
                   mlp_mode="bf16")
ds = DeviceHeadDataset(tmp, "aud.npy", "val", a)
F = len(ds)
log(f"# subject: {F} val frames of {ds.H} x {ds.W}, written and loaded in {time.perf_counter() - t0:.1f} s; bf16 mode, perturb 0, "
    "64 + 128 samples; seeded LPIPS weights")
alex, lin = LR.seeded_state_dicts(0)
w = load_lpips(alex, lin, device=dev)
torch.manual_seed(4321)
net = M.Network(ds.H, ds.W, ds.focal, S.NEAR, S.FAR, 8192, None, 64, 128, args=a)
net.apply(M.init_weights)
net = net.to(dev).eval()
latent = torch.ones(32, device=dev)
codes = audio_codes(net, ds)
rays = M.ops.get_rays_packed(ds.H, ds.W, ds.focal, ds.poses[0], S.NEAR, S.FAR)[::97].contiguous()
for fn in (net.face_nerf_coarse, net.face_nerf_fine):
    S.normalise_density_(fn, rays, codes[0], ds.exprs[0], latent)
r = FrameRenderer(net)


def wall(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


# (d) first, so that (a)-(c) use its rendered frames
with torch.no_grad():
    evaluate_split(r, ds, latent, codes, keep_video=False, lpips=w)                   # warm-up: modules, blobs, pinned buffers
    t_p, t_l = [], []
    for _ in range(2):
        t, plain = wall(lambda: evaluate_split(r, ds, latent, codes))
        t_p.append(t)
        t, res = wall(lambda: evaluate_split(r, ds, latent, codes, lpips=w))
        t_l.append(t)
assert np.array_equal(plain["video"], res["video"])

vid = torch.from_numpy(res["video"]).to(dev)
idx = torch.arange(F, dtype=torch.int64, device=dev)
one, i0 = vid[:1], idx[:1]
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

# (a) one 450^2 pair
for _ in range(20):
    M.ops.lpips(one, ds.frames, i0, w)
side = torch.cuda.Stream()
side.wait_stream(torch.cuda.current_stream())
with torch.cuda.stream(side):
    M.ops.lpips(one, ds.frames, i0, w)
torch.cuda.current_stream().wait_stream(side)
g = torch.cuda.CUDAGraph()
with torch.cuda.graph(g):
    for _ in range(100):
        M.ops.lpips(one, ds.frames, i0, w)
g.replay()
torch.cuda.synchronize()
per_graph = []
for _ in range(2):
    e0.record()
    for _ in range(10):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    per_graph.append(e0.elapsed_time(e1) / 1000)
n = 1000
e0.record()
for _ in range(n):
    M.ops.lpips(one, ds.frames, i0, w)
e1.record()
torch.cuda.synchronize()
per_py = e0.elapsed_time(e1) / n
best = min(per_graph)
rate = flop_pair / (best * 1e-3) / 1e12
log(f"(a) ops.lpips, one 450^2 frame pair (13 kernels): {best * 1e3:.1f} us per call replayed from a CUDA graph (100 calls x 10 replays, "
    f"two windows: {', '.join(f'{x * 1e3:.1f}' for x in per_graph)} us), {per_py * 1e3:.1f} us per call issued back to back from Python "
    f"({n} calls); {flop_pair / 1e9:.2f} GFLOP per pair -> {rate:.1f} TFLOP/s achieved, {rate / floor_tflops:.3f} of the fp32 FFMA floor "
    f"({floor_tflops:.1f} TFLOP/s = {sms} SMs x 128 FFMA x 2 x {clk_mhz:.0f} MHz; floor time {flop_pair / floor_tflops / 1e9:.3f} ms)")

# (b) per kernel
from torch.profiler import ProfilerActivity, profile  # noqa: E402
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(20):
        M.ops.lpips(one, ds.frames, i0, w)
    torch.cuda.synchronize()
per_kernel = {}
for ev in prof.key_averages():
    if ev.device_type.name == "CUDA" or getattr(ev, "device_time_total", 0) > 0:
        t_us = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)
        if t_us > 0 and ev.count > 0:
            per_kernel[ev.key] = (ev.count, t_us / 20)
tot = sum(t for _, t in per_kernel.values())
log(f"(b) torch.profiler, device time per call by kernel (20 calls; total {tot:.1f} us):")
for name, (cnt, t_us) in sorted(per_kernel.items(), key=lambda kv: -kv[1][1]):
    short = name.replace("void ", "").replace("(anonymous namespace)::", "").split("(")[0]
    log(f"      {t_us:8.1f} us  {t_us / tot * 100:5.1f} %  x{cnt // 20}  {short[:110]}")

# (c) against the oracle on rendered frames
k = min(4, F)
got = M.ops.lpips(vid[:k], ds.frames, idx[:k], w).double().cpu()
want = LR.lpips(res["video"][:k], ds.frames.cpu().numpy(), np.arange(k), alex, lin)
err = (got - want).abs()
log(f"(c) kernel vs float64 oracle on {k} rendered 450^2 frames: lpips {np.round(want.numpy(), 5).tolist()}, max |diff| {float(err.max()):.2e}, "
    f"max relative {float((err / want).max()):.2e}")

log(f"(d) evaluate_split without lpips: {F / min(t_p):7.2f} frames/s ({min(t_p) / F * 1e3:.2f} ms / frame; runs "
    f"{', '.join(f'{t:.2f}' for t in t_p)} s)")
log(f"    evaluate_split with lpips=:   {F / min(t_l):7.2f} frames/s ({min(t_l) / F * 1e3:.2f} ms / frame; runs "
    f"{', '.join(f'{t:.2f}' for t in t_l)} s)  -> LPIPS adds {(min(t_l) - min(t_p)) / F * 1e3:+.2f} ms / frame "
    f"({(min(t_l) / min(t_p) - 1) * 100:+.1f} %); mean LPIPS {res['mean_lpips']:.4f} (seeded weights, random-JPEG ground truth)")
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fp:
        fp.write("\n".join(lines) + "\n")
