"""The training driver's loop against a bare graph-step loop on the same dataset (results: profiles/r13_fit_loop.txt).

    python profiles/fit_loop.py [--steps 2000] [--out FILE]                                  # one GPU
    torchrun --nproc_per_node N profiles/fit_loop.py [--steps 2000] [--out FILE]             # N GPUs, one process each

A synthetic 64-frame 450^2 subject (write_head_subject), bf16, N_rand = 3072 per step split into bands over the ranks, 64 + 128
samples, perturb = 1, nosmo_iters = 0 (one audio phase).  Two loops of the same TrainStep(cuda_graph=True) fed from
DeviceHeadDataset.sample(idx, rank, world) with a device frame index:
  * bare: idx copied from a device table, sample, step -- nothing else;
  * fit:  fit.HeadFit(args).run(): the epoch permutation, the log ring, a log flush (one device-to-host copy) every i_print = 100 steps,
          and the Philox re-seed after each flush; no checkpoint, validation or image inside the timed window.
Each loop is warmed up (capture included), then timed with CUDA events over --steps steps; the two are alternated --reps times and
the medians reported, maxima over ranks."""
import argparse
import os
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from ideal_nerf_b200 import fit, ops, synthetic as S  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--steps", type=int, default=2000)
ap.add_argument("--warmup", type=int, default=50)
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--out", default=None, help="append the report to this file")
cli = ap.parse_args()
assert torch.cuda.is_available(), "this measurement needs a GPU"
rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
torch.cuda.set_device(dev)
if world > 1:
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    dist.init_process_group("nccl", device_id=dev)
lines = []


def log(s):
    if rank == 0:
        print(s, flush=True)
        lines.append(s)


def barrier():
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()


def timed(fn):
    """ms per step of fn(), which runs --steps steps: CUDA events around it, the maximum over ranks."""
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1) / cli.steps], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t)


smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True)
log(f"# world {world}; card: {torch.cuda.get_device_name(dev)}; nvidia-smi:")
for s in (smi.stdout.strip() or "n/a").splitlines()[:1 + max(world, 1)]:
    log(f"#   {s}")

tmp = [tempfile.mkdtemp() if rank == 0 else None]
if world > 1:
    dist.broadcast_object_list(tmp, 0)
tmp = tmp[0]
if rank == 0:
    S.write_head_subject(os.path.join(tmp, "subject"), 450, 450, n_frames=64, seed=0, torso_rows=40)
barrier()
args = fit.fit_parser().parse_args([])
for k, v in dict(datadir=os.path.join(tmp, "subject"), basedir=tmp, expname="run", N_rand=3072, mouth_rays=512, torso_rays=0,
                 sample_rate=0.95, near=S.NEAR, far=S.FAR, dim_aud=64, dim_expr=76, perturb=1.0, mlp_mode="bf16", lrate=3e-4,
                 nosmo_iters=0, i_print=100, i_weights=0, i_testset=0, i_img=0, N_iters=1000, no_reload=True).items():
    setattr(args, k, v)
log(f"# bf16, N_rand {args.N_rand} per step ({args.N_rand // world} rays per rank), 64 + 128 samples, perturb 1, 64 frames of 450^2, "
    f"i_print {args.i_print}; CUDA events over {cli.steps} steps after {cli.warmup} warm-up steps, median of {cli.reps}, max over ranks")

f = fit.HeadFit(args, rank, world)
step, ds = f.step, f.ds
f.run(cli.warmup)                                                          # eager step + capture
order = torch.from_numpy(np.random.RandomState(0).randint(0, len(ds), 4096)).to(dev)
idx_t = torch.zeros((), dtype=torch.int64, device=dev)


def bare():
    for i in range(cli.steps):
        idx_t.copy_(order[i % len(order)])
        b = ds.sample(idx_t, rank, world)
        step(b["rays"], b["bc_rgb"], b["target"], None, b["expr"], idx_t, aud_window=b["aud_window"])


def driver():
    f.run(step.global_step + cli.steps)


for _ in range(2):
    bare()
res = {"bare": [], "fit": []}
for _ in range(cli.reps):
    res["bare"].append(timed(bare))
    res["fit"].append(timed(driver))
b, d = statistics.median(res["bare"]), statistics.median(res["fit"])
log(f"{'bare graph-step loop':28s} {b:7.3f} ms/step   runs {', '.join(f'{v:.3f}' for v in res['bare'])}")
log(f"{'fit.HeadFit.run':28s} {d:7.3f} ms/step   runs {', '.join(f'{v:.3f}' for v in res['fit'])}   "
    f"({(d / b - 1) * 100:+.2f} % against bare, log flushes included)")
barrier()
if rank == 0:
    import shutil
    shutil.rmtree(tmp, ignore_errors=True)
    if cli.out:
        os.makedirs(os.path.dirname(os.path.abspath(cli.out)), exist_ok=True)
        with open(cli.out, "a") as fp:
            fp.write("\n".join(lines) + "\n\n")
if world > 1:
    dist.destroy_process_group()
