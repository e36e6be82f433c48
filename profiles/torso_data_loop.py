"""Cost of feeding the torso stage's training step from data on disk (results: profiles/r09_torso_data_loop.txt).

Writes a synthetic subject in the reference's on-disk layout with com_imgs (450 x 450, 64 frames, 40 torso rows in the parsing maps, a
mouth box from the landmarks), builds DeviceTorsoDataset on it (targets from com_imgs, audio codes of a random-init head from
evaluate.audio_codes, the torso camera of train frame 0) and a random-init bf16 TorsoNetwork with the normalised-density preset, then in one
process times 200 iterations (after warm-up) of
  (a) DeviceTorsoDataset.sample(i) feeding TorsoTrainStep(cuda_graph=True)       -- the batch drawn on the device;
  (b) the bare graph step on a fixed batch, before and after (a), for drift,
each iteration closed by a synchronise: the median wall time per iteration and the median host time until the step has been enqueued.
Then DeviceTorsoDataset.sample alone and ops.masked_sse on one 450^2 frame, each with CUDA events over 1 000 calls, issued from Python and
replayed from a CUDA graph.
    python profiles/torso_data_loop.py [--iters 200] [--out profiles/r09_torso_data_loop.txt]"""
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
from ideal_nerf_b200.data import DeviceTorsoDataset, HeadDataset  # noqa: E402
from ideal_nerf_b200.evaluate import audio_codes  # noqa: E402
from ideal_nerf_b200.train import TorsoTrainStep  # noqa: E402

p = argparse.ArgumentParser()
p.add_argument("--iters", type=int, default=200)
p.add_argument("--warmup", type=int, default=10)
p.add_argument("--calls", type=int, default=1000)
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
S.write_head_subject(tmp, 450, 450, n_frames=64, seed=0, torso_rows=40, com_imgs=True)
a = M.default_args(N_rand=3072, mouth_rays=512, torso_rays=512, sample_rate=0.95, gt_dirs="com_imgs", near=S.NEAR, far=S.FAR,
                   dim_aud=64, dim_expr=76, perturb=1.0, mlp_mode="bf16", lrate=3e-4)
t0 = time.perf_counter()
torch.manual_seed(4321)
head = M.Network(450, 450, 1200., S.NEAR, S.FAR, 8192, None, 64, 128, args=a)
head.apply(M.init_weights)
codes = audio_codes(head.to(dev).eval(), HeadDataset(tmp, "aud.npy", "train", a))
ds = DeviceTorsoDataset(tmp, "aud.npy", "train", a, codes, torch.ones(64, 32, device=dev))
log(f"# subject: 64 frames of 450 x 450 (com_imgs), N_rand 3072 = {ds.budgets} (rect, norect, mouth, torso); bf16, perturb 1, 64 + 128 "
    f"samples per pair; audio codes + dataset built in {time.perf_counter() - t0:.1f} s")

torch.manual_seed(1234)
net = M.TorsoNetwork(450, 450, ds.focal, S.NEAR, S.FAR, 1 << 20, 64, 128, args=a, dim_expr=76)
net.apply(M.init_weights)
net = net.to(dev)
fixed = ds.sample(0)
for m in (net.face_nerf_coarse, net.face_nerf_fine):
    S.normalise_density_(m, fixed["rays_head"], fixed["aud_feature"], fixed["expr"], fixed["latent_code"])
sig = net.torso_signal(fixed["aud_feature"], fixed["pose"])
for m in (net.torso_coarse_nerf, net.torso_fine_nerf):
    S.normalise_density_(m, fixed["rays_torso"], sig, None, None)
step = TorsoTrainStep(net.train(), a, cuda_graph=True)
order = np.random.RandomState(0).randint(0, len(ds), args.iters + args.warmup)
idx_t = torch.zeros((), dtype=torch.int64, device=dev)


def loop_a(i):
    idx_t.fill_(int(i))
    step(**ds.sample(idx_t))


def loop_b(i):
    step(**fixed)


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
for name, fn in (("b", loop_b), ("a", loop_a), ("b", loop_b)):
    res.setdefault(name, []).append(timed(fn))
log(f"(a) DeviceTorsoDataset.sample -> TorsoTrainStep graph: {res['a'][0][0]:8.3f} ms / iteration, host {res['a'][0][1]:.3f} ms")
log(f"(b) bare graph step (fixed batch), before/after:      {res['b'][0][0]:.3f} / {res['b'][1][0]:.3f} ms / iteration, host "
    f"{res['b'][0][1]:.3f} / {res['b'][1][1]:.3f} ms")
log(f"    (a) / mean (b) = {res['a'][0][0] / statistics.mean([r[0] for r in res['b']]):.3f}")


def events(fn, n):
    """ms per call of fn() over n back-to-back calls (CUDA events), and the host ms per call of issuing them."""
    for _ in range(20):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    t0 = time.perf_counter()
    for _ in range(n):
        fn()
    t1 = time.perf_counter()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n, (t1 - t0) * 1e3 / n


def graphed(fn, n):
    """ms per call of fn() captured once in a CUDA graph and replayed n times (CUDA events)."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fn()
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    return events(g.replay, n)[0]


n = args.calls
idx_t.fill_(5)
ms, host = events(lambda: ds.sample(idx_t), n)
gms = graphed(lambda: ds.sample(idx_t), n)
log(f"DeviceTorsoDataset.sample alone (sampler memset + 4 kernels, inerf_get_rays_at, 4 row lookups; 3072 rows of a 450^2 frame): "
    f"{ms * 1e3:.1f} us per call issued from Python (host {host * 1e3:.1f} us per call), {gms * 1e3:.1f} us per call replayed from a CUDA "
    f"graph (CUDA events over {n} calls)")
pred = torch.randint(0, 256, (1, 450, 450, 3), dtype=torch.uint8, device=dev)
one = torch.full((1,), 5, dtype=torch.int64, device=dev)
ms, host = events(lambda: M.ops.masked_sse(pred, ds.frames, one, ds.torso_bits), n)
gms = graphed(lambda: M.ops.masked_sse(pred, ds.frames, one, ds.torso_bits), n)
sse, npix = M.ops.masked_sse(pred, ds.frames, one, ds.torso_bits)
log(f"ops.masked_sse, one 450^2 frame against its torso mask ({int(npix)} pixels; 2 memsets + 1 kernel): {ms * 1e3:.1f} us per call issued "
    f"from Python (host {host * 1e3:.1f} us per call), {gms * 1e3:.1f} us per call replayed from a CUDA graph (CUDA events over {n} calls)")
out = step(**fixed)
log(f"# loss finite: {bool(np.isfinite(float(out['loss'])))}")
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fp:
        fp.write("\n".join(lines) + "\n")
