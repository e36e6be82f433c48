"""Host cost of feeding the HeadNeRF training step from real data (results: profiles/r07_train_data_loop.txt).

Writes a synthetic subject in the reference's on-disk layout (450 x 450, 64 frames, torso rows in the parsing maps, a mouth box from the
landmarks), then in one process times 200 iterations (after warm-up) of
  (a) HeadDataset[i]              feeding TrainStep(mlp_mode="bf16", cuda_graph=True)   -- numpy sampling, JPEG / PNG decode per step;
  (b) DeviceHeadDataset.sample(i) feeding the same step                                 -- the batch drawn on the device;
  (c) the bare graph step on a fixed batch,
each iteration closed by a synchronise: the median wall time per iteration and the median host time until the step has been enqueued.
Then the sampler call alone (ops.sample_train_pixels, N_rand = 3072) with CUDA events over 1 000 launches.
    python profiles/train_data_loop.py [--iters 200] [--out profiles/r07_train_data_loop.txt]"""
import argparse
import os
import statistics
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
from ideal_nerf_b200.data import DeviceHeadDataset, HeadDataset  # noqa: E402
from ideal_nerf_b200.train import TrainStep  # noqa: E402

p = argparse.ArgumentParser()
p.add_argument("--iters", type=int, default=200)
p.add_argument("--warmup", type=int, default=10)
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
S.write_head_subject(tmp, 450, 450, n_frames=64, seed=0, torso_rows=40)
a = M.default_args(N_rand=3072, mouth_rays=512, torso_rays=0, sample_rate=0.95, gt_dirs="head_imgs", near=S.NEAR, far=S.FAR,
                   dim_aud=64, dim_expr=76, perturb=1.0, mlp_mode="bf16", lrate=3e-4, nosmo_iters=0)
t0 = time.perf_counter()
hd = HeadDataset(tmp, "aud.npy", "train", a)
ds = DeviceHeadDataset(tmp, "aud.npy", "train", a)
log(f"# subject: 64 frames of 450 x 450, N_rand 3072 = {ds.budgets} (rect, norect, mouth, torso); both datasets built in "
    f"{time.perf_counter() - t0:.1f} s")
torch.manual_seed(4321)
net = M.Network(450, 450, hd.focal, S.NEAR, S.FAR, 8192, None, 64, 128, args=a)
net.apply(M.init_weights)
net = net.to(dev).train()
ts = TrainStep(net, torch.ones(len(ds), 32, device=dev), a, cuda_graph=True)
rng = np.random.RandomState(0)
order = rng.randint(0, len(ds), args.iters + args.warmup)
idx_t = torch.zeros((), dtype=torch.int64, device=dev)


def loop_a(i):
    batch_rays, target_s, bc_rgb, auds, _, _, exp, index = hd[i]
    rays = M.ops.pack_rays(batch_rays[0], batch_rays[1], a.near, a.far)
    ts(rays, bc_rgb.float(), target_s, None, exp.to(dev), index, aud_window=net.audio_window(auds, index, len(hd)))


def loop_b(i):
    idx_t.fill_(int(i))
    b = ds.sample(idx_t)
    ts(b["rays"], b["bc_rgb"], b["target"], None, b["expr"], idx_t, aud_window=b["aud_window"])


fixed = ds.sample(0)


def loop_c(i):
    ts(fixed["rays"], fixed["bc_rgb"], fixed["target"], None, fixed["expr"], 0, aud_window=fixed["aud_window"])


def timed(fn):
    for i in order[:args.warmup]:
        fn(i)
    torch.cuda.synchronize()
    it_ms, host_ms = [], []
    for i in order[args.warmup:]:
        t0 = time.perf_counter()
        fn(i)
        t1 = time.perf_counter()
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        host_ms.append((t1 - t0) * 1e3)
        it_ms.append((t2 - t0) * 1e3)
    return statistics.median(it_ms), statistics.median(host_ms)


res = {}
for name, fn in (("c", loop_c), ("a", loop_a), ("b", loop_b), ("c", loop_c)):      # the bare step before and after, for drift
    res.setdefault(name, []).append(timed(fn))
log(f"(a) HeadDataset[i] -> TrainStep graph:        {res['a'][0][0]:8.3f} ms / iteration, host {res['a'][0][1]:8.3f} ms")
log(f"(b) DeviceHeadDataset.sample -> TrainStep:    {res['b'][0][0]:8.3f} ms / iteration, host {res['b'][0][1]:8.3f} ms")
log(f"(c) bare graph step (fixed batch), before/after: {res['c'][0][0]:.3f} / {res['c'][1][0]:.3f} ms / iteration, host "
    f"{res['c'][0][1]:.3f} / {res['c'][1][1]:.3f} ms")
log(f"    (b) / (c) = {res['b'][0][0] / statistics.mean([r[0] for r in res['c']]):.3f};  (a) / (b) = {res['a'][0][0] / res['b'][0][0]:.1f}")

for _ in range(20):
    ds.sample(idx_t)
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
n = 1000
e0.record()
for _ in range(n):
    M.ops.sample_train_pixels(idx_t, ds.budgets, ds.bounds, ds.torso_bits, ds.poses, ds.frames, ds.bc_img, ds.focal, ds.cx, ds.cy,
                              a.near, a.far, advance=False)
e1.record()
torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / n
log(f"sampler alone (ops.sample_train_pixels, 3072 rows of a 450^2 frame, memset + 4 kernels, back to back): {ms * 1e3:.1f} us per batch "
    f"(CUDA events over {n} launches)")
sums = {"loss_finite": bool(np.isfinite(float(ts(fixed['rays'], fixed['bc_rgb'], fixed['target'], None, fixed['expr'], 0,
                                                 aud_window=fixed['aud_window'])['loss'])))}
log(f"# {sums}")
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fp:
        fp.write("\n".join(lines) + "\n")
