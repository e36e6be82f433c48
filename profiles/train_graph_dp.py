"""Data-parallel training steps, eager and as one CUDA graph per rank (results: profiles/r11_train_graph_dp.txt).

    python profiles/train_graph_dp.py [--steps 200] [--out FILE]                                   # one GPU
    torchrun --nproc_per_node N profiles/train_graph_dp.py [--steps 200] [--out FILE]              # N GPUs, one process each

Weak scaling: every rank trains on its own N_rand = 3072 rays per step, bf16, 64 + 128 samples, perturb = 1, and the flat gradient is
averaged over the ranks with one NCCL all-reduce per step (inside the graph in graph mode).  At the launched world size it times
  * the head step (train.TrainStep): the workload of bench.py's train_step_bench, the audio window through AudioNet / AudioAttNet
    inside the step;
  * the torso step (train.TorsoTrainStep): frozen head pair + trained torso pair on 3072 rays each, as profiles/torso_train_step.py;
  * the head graph step fed from DeviceHeadDataset.sample(i, rank, world) on a synthetic 64-frame 450^2 subject: ONE batch of
    N_rand = 3072 per step split into complementary bands (the same Philox seed on every rank; the sampler draws at most 4 096 rows per
    region, so this batch does not grow with the world size), the frame index a device tensor: the whole loop with no host synchronise
    per step;
  * the NCCL all-reduce of the head step's flat gradient alone.
Each is timed with CUDA events over --steps back-to-back iterations after warm-up (the graph is captured in the warm-up); host ms is
the median time for one call to return when it starts on an idle device (the enqueue); both are maxima over ranks; rays/s counts all
ranks.  A graphed step also prints the capture_error_mode its capture succeeded in.  --out appends."""
import argparse
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import ideal_nerf_b200 as M  # noqa: E402
from ideal_nerf_b200 import ops, synthetic as S  # noqa: E402
from ideal_nerf_b200.data import DeviceHeadDataset  # noqa: E402
from ideal_nerf_b200.train import TorsoTrainStep, TrainStep  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--steps", type=int, default=200)
ap.add_argument("--warmup", type=int, default=5)
ap.add_argument("--out", default=None, help="append the report to this file")
args = ap.parse_args()
assert torch.cuda.is_available(), "this measurement needs a GPU"
rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
local = int(os.environ.get("LOCAL_RANK", "0"))
dev = torch.device("cuda", local)
torch.cuda.set_device(dev)
if world > 1:
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    dist.init_process_group("nccl", device_id=dev)
H = W = 450
N = 3072
lines = []


def log(s):
    if rank == 0:
        print(s, flush=True)
        lines.append(s)


def barrier():
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()


def timed(step):
    """(ms per step, host ms per step), each the maximum over ranks, of `step` after --warmup steps: CUDA events around --steps
    back-to-back steps, then the median time for one step call to return over --steps more calls, each started on an idle device (a
    long back-to-back loop fills the launch queue, and the host then waits for the GPU inside the call)."""
    for _ in range(args.warmup):
        step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    barrier()
    host = []
    for _ in range(args.steps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        step()
        host.append((time.perf_counter() - t0) * 1e3)
    barrier()
    t = torch.tensor([e0.elapsed_time(e1) / args.steps, statistics.median(host)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t[0]), float(t[1])


def row(what, ms, host, rays, extra=""):
    log(f"{what:44s} {ms:7.3f} ms/step  host {host:6.3f} ms/step  {rays / (ms * 1e-3) / 1e6:6.3f} M rays/s{extra}")


smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True)
log(f"# world {world}; card: {torch.cuda.get_device_name(dev)}; nvidia-smi:")
for s in (smi.stdout.strip() or "n/a").splitlines()[:1 + max(world, 1)]:
    log(f"#   {s}")
log(f"# bf16, N_rand {N} per rank, 64 + 128 samples, perturb 1; CUDA events over {args.steps} steps after {args.warmup} warm-up steps, "
    f"max over ranks")

# ---- head step: the workload of bench.py's train_step_bench --------------------------------------------------------------------
cam, fr = S.camera(), S.frame_inputs(0)


def head_step(graph):
    """train_step_bench's step (its seeds, arguments and inputs), returned as a closure so that it can be timed here."""
    a = M.default_args(dim_aud=64, dim_expr=76, perturb=1.0, mlp_mode="bf16", N_samples=64, N_importance=128, lrate=3e-4, nosmo_iters=0)
    net = M.Network(H, W, cam["focal"], S.NEAR, S.FAR, 8192, None, 64, 128, args=a)
    torch.manual_seed(4321)
    net.apply(M.init_weights)
    net = net.to(dev).train()
    g = torch.Generator().manual_seed(5 + rank)
    idx = torch.randperm(H * W, generator=g)[:N].to(dev)
    rays = ops.get_rays_packed(H, W, cam["focal"], cam["c2w"].to(dev), S.NEAR, S.FAR)[idx].contiguous()
    bc, tgt = fr["bc_rgb"].to(dev)[idx].contiguous(), torch.rand(N, 3, generator=g).to(dev)
    expr = fr["expr"].to(dev)
    auds = torch.randn(40, 16, 29, generator=torch.Generator().manual_seed(6)).to(dev)
    ts = TrainStep(net, torch.ones(40, 32, device=dev), a, world=world, cuda_graph=graph)
    win = net.audio_window(auds, 17, 40)
    return ts, lambda: ts(rays, bc, tgt, None, expr, 17, aud_window=win)


def mode_of(step):
    return f"  (captured in {step._static['capture_mode']!r} mode)" if step.cuda_graph else ""


for graph in (False, True):
    ts, fn = head_step(graph)
    ms, host = timed(fn)
    row(f"head TrainStep {'graph' if graph else 'eager'}", ms, host, N * world, mode_of(ts))
    del ts, fn
    torch.cuda.empty_cache()

# ---- torso step --------------------------------------------------------------------------------------------------------------------
g = torch.Generator().manual_seed(5 + rank)
idx = torch.randperm(H * W, generator=g)[:N].to(dev)
pose = cam["c2w"].clone()
pose[0, 3] += 0.01
rays_h = ops.get_rays_packed(H, W, cam["focal"], pose.to(dev), S.NEAR, S.FAR)[idx].contiguous()
rays_t = ops.get_rays_packed(H, W, cam["focal"], cam["c2w"].to(dev), S.NEAR, S.FAR)[idx].contiguous()
bc, tgt = fr["bc_rgb"].to(dev)[idx].contiguous(), torch.rand(N, 3, generator=g).to(dev)
aud, lat, pose = fr["aud"].to(dev), fr["latent"].to(dev), pose.to(dev)
expr79 = torch.randn(79, generator=torch.Generator().manual_seed(7)).to(dev)


def torso_network():
    torch.manual_seed(1234)
    net = M.TorsoNetwork(H, W, cam["focal"], S.NEAR, S.FAR, 1 << 20, 64, 128,
                         args=M.default_args(dim_aud=64, dim_expr=79, perturb=1., mlp_mode="bf16", lrate=3e-4))
    net.apply(M.init_weights)
    net = net.to(dev)
    for m in (net.face_nerf_coarse, net.face_nerf_fine):
        S.normalise_density_(m, rays_h, aud, expr79, lat)
    sig = net.torso_signal(aud, pose)
    for m in (net.torso_coarse_nerf, net.torso_fine_nerf):
        S.normalise_density_(m, rays_t, sig, None, None)
    return net.train()


for graph in (False, True):
    net = torso_network()
    st = TorsoTrainStep(net, net.args, world=world, cuda_graph=graph)
    ms, host = timed(lambda: st(rays_h, rays_t, bc, tgt, aud, pose, expr79, lat, perturb=1.))
    row(f"torso TorsoTrainStep {'graph' if graph else 'eager'}", ms, host, N * world, mode_of(st))
    del st, net
    torch.cuda.empty_cache()

# ---- head graph step fed from DeviceHeadDataset.sample(i, rank, world) -------------------------------------------------------------
paths = [tempfile.mkdtemp() if rank == 0 else None]
if world > 1:
    dist.broadcast_object_list(paths, 0)
tmp = paths[0]
if rank == 0:
    S.write_head_subject(tmp, H, W, n_frames=64, seed=0, torso_rows=40)
barrier()
a = M.default_args(N_rand=N, mouth_rays=512, torso_rays=0, sample_rate=0.95, gt_dirs="head_imgs", near=S.NEAR, far=S.FAR,
                   dim_aud=64, dim_expr=76, perturb=1.0, mlp_mode="bf16", lrate=3e-4, nosmo_iters=0)
ds = DeviceHeadDataset(tmp, "aud.npy", "train", a, device=dev)
torch.manual_seed(4321)
net = M.Network(H, W, ds.focal, S.NEAR, S.FAR, 8192, None, 64, 128, args=a)
net.apply(M.init_weights)
net = net.to(dev).train()
ts = TrainStep(net, torch.ones(len(ds), 32, device=dev), a, world=world, cuda_graph=True)
order = torch.from_numpy(np.random.RandomState(0).randint(0, len(ds), 256)).to(dev)
idx_t = torch.zeros((), dtype=torch.int64, device=dev)
calls = [0]
ops.seed_rng(11, dev, 0)                                               # the same stream on every rank: complementary bands


def data_step():
    idx_t.copy_(order[calls[0] % len(order)])
    calls[0] += 1
    b = ds.sample(idx_t, rank, world)
    ts(b["rays"], b["bc_rgb"], b["target"], None, b["expr"], idx_t, aud_window=b["aud_window"])


ms, host = timed(data_step)
row("head TrainStep graph fed by DeviceHeadDataset", ms, host, N,
    f"  (one {N}-ray batch {ds.budgets} per step, {N // world} rays per rank){mode_of(ts)}")
barrier()
if rank == 0:
    shutil.rmtree(tmp, ignore_errors=True)

# ---- the all-reduce alone ----------------------------------------------------------------------------------------------------------
if world > 1:
    grad = ts.flat.grad
    ms, host = timed(lambda: dist.all_reduce(grad, op=dist.ReduceOp.AVG))
    log(f"{'flat-gradient all-reduce alone (eager NCCL)':44s} {ms:7.3f} ms/call  host {host:6.3f} ms/call  "
        f"({grad.numel() * 4 / 1e6:.1f} MB, AVG)")

if rank == 0 and args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "a") as fp:
        fp.write("\n".join(lines) + "\n\n")
if world > 1:
    dist.destroy_process_group()
