"""The torso stage's training step (train.TorsoTrainStep, NeRFs/TorsoNeRF/train_torso.py) on one GPU, with the head stage's
train.TrainStep in the same process as the yardstick.

    python profiles/torso_train_step.py [--steps 200] [--warmup 10] [--out FILE]

N_rand = 3072 rays (BASELINE config 3's batch) for both pairs, 64 + 128 samples per pair, perturb = 1; the four FaceNeRFs are random-init
with the normalised-density preset (the torso neither empty nor opaque).  For bf16 and fp32 mode, eager and as one CUDA graph:
  * ms per step: median of --steps timed steps after --warmup, each ended by a synchronise (host clock);
  * host ms per step: median time for the step call to return (the enqueue);
  * eager only, in a separate pass with CUDA events: the head render (no_grad, fused entry), the torso forward + backward (render,
    loss kernel, backward), and the rest (gradient gather, Adam, packed-cache drops), medians over --steps steps.  The pass runs the
    pieces of TorsoTrainStep._body with event pairs between them.
The head TrainStep runs the same way on the same 3072 head rays (audio code from an 8-frame DeepSpeech window inside the step).
"""
import argparse
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402
import ideal_nerf_b200 as M  # noqa: E402
from ideal_nerf_b200 import ops, synthetic as S  # noqa: E402
from ideal_nerf_b200.train import TorsoTrainStep, TrainStep  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--steps", type=int, default=200)
ap.add_argument("--warmup", type=int, default=10)
ap.add_argument("--out", default=None, help="also write the report to this file")
args = ap.parse_args()
assert torch.cuda.is_available(), "needs a GPU"
dev = torch.device("cuda", 0)
lines = []


def say(s):
    print(s, flush=True)
    lines.append(s)


try:
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                         timeout=60).stdout.strip().splitlines()[0]
except Exception as e:              # the measurement stands without it, but says so
    smi = f"nvidia-smi unavailable ({e})"
say(f"card: {torch.cuda.get_device_name(dev)}; nvidia-smi name, power limit: {smi}")
say(f"N_rand 3072, 64 + 128 samples per pair, perturb 1; {args.steps} timed steps after {args.warmup} warm-up steps")

H = W = 450
cam, fr = S.camera(), S.frame_inputs(0)
g = torch.Generator().manual_seed(5)
idx = torch.randperm(H * W, generator=g)[:3072].to(dev)
pose = cam["c2w"].clone()
pose[0, 3] += 0.01
rays_h = ops.get_rays_packed(H, W, cam["focal"], pose.to(dev), S.NEAR, S.FAR)[idx].contiguous()
rays_t = ops.get_rays_packed(H, W, cam["focal"], cam["c2w"].to(dev), S.NEAR, S.FAR)[idx].contiguous()    # frame-0 camera
bc, tgt = fr["bc_rgb"].to(dev)[idx].contiguous(), torch.rand(3072, 3, generator=g).to(dev)
aud, lat = fr["aud"].to(dev), fr["latent"].to(dev)
expr79 = torch.randn(79, generator=g).to(dev)
pose = pose.to(dev)


def torso_network(mode):
    torch.manual_seed(1234)
    net = M.TorsoNetwork(H, W, cam["focal"], S.NEAR, S.FAR, 1 << 20, 64, 128,
                         args=M.default_args(dim_aud=64, dim_expr=79, perturb=1., mlp_mode=mode, lrate=3e-4))
    net.apply(M.init_weights)
    net = net.to(dev)
    for m in (net.face_nerf_coarse, net.face_nerf_fine):
        S.normalise_density_(m, rays_h, aud, expr79, lat)
    sig = net.torso_signal(aud, pose)
    for m in (net.torso_coarse_nerf, net.torso_fine_nerf):
        S.normalise_density_(m, rays_t, sig, None, None)
    return net.train()


def head_step(mode, graph):
    a = M.default_args(dim_aud=64, dim_expr=76, perturb=1., mlp_mode=mode, lrate=3e-4, nosmo_iters=0)
    torch.manual_seed(4321)
    net = M.Network(H, W, cam["focal"], S.NEAR, S.FAR, 8192, None, 64, 128, args=a)
    net.apply(M.init_weights)
    net = net.to(dev).train()
    auds = torch.randn(40, 16, 29, generator=torch.Generator().manual_seed(6)).to(dev)
    ts = TrainStep(net, torch.ones(40, 32, device=dev), a, cuda_graph=graph)
    win = net.audio_window(auds, 17, 40)
    expr = fr["expr"].to(dev)
    return lambda: ts(rays_h, bc, tgt, None, expr, 17, aud_window=win)


def timed(fn):
    for _ in range(args.warmup):
        fn()
    torch.cuda.synchronize()
    step_ms, host_ms = [], []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        fn()
        t1 = time.perf_counter()
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        host_ms.append((t1 - t0) * 1e3)
        step_ms.append((t2 - t0) * 1e3)
    return statistics.median(step_ms), statistics.median(host_ms)


def split(mode):
    """Event-timed pieces of the eager step: head render | torso forward + backward | gather + Adam + the rest.  The loop restates
    train.TorsoTrainStep._body (plus the eager learning-rate update) to put event pairs between its pieces: keep it in step with _body."""
    net = torso_network(mode)
    st = TorsoTrainStep(net, net.args)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    parts = [[], [], []]
    for i in range(args.warmup + args.steps):
        for p in st.flat.params:
            p.grad = None
        ev[0].record()
        with torch.no_grad():
            head = net.render_pair("head", rays_h, bc, aud, expr79, lat, 1.)
        ev[1].record()
        torso = net.render_pair("torso", rays_t, bc, net.torso_signal(aud, pose), None, None, 1.)
        l2 = ops.head_torso_mse_pair(head["rgb_map"], head["rgb0"], torso["last_weight"], torso["last_weight0"], torso["rgb_map_fg"],
                                     torso["rgb_map_fg0"], tgt)
        (l2[0] + l2[1]).backward()
        ev[2].record()
        st.flat.gather_grads()
        st.optimizer.step()
        for m in st.trained:
            m.invalidate_packed()
        st._advance_lr()
        ev[3].record()
        torch.cuda.synchronize()
        if i >= args.warmup:
            for k in range(3):
                parts[k].append(ev[k].elapsed_time(ev[k + 1]))
    return [statistics.median(p) for p in parts]


results = {}
for mode in ("bf16", "fp32"):
    for graph in (False, True):
        net = torso_network(mode)
        st = TorsoTrainStep(net, net.args, cuda_graph=graph)
        ms, host = timed(lambda: st(rays_h, rays_t, bc, tgt, aud, pose, expr79, lat, perturb=1.))
        hms, hhost = timed(head_step(mode, graph))
        results[(mode, graph)] = (ms, hms)
        kind = "graph" if graph else "eager"
        say(f"{mode:5s} {kind}: TorsoTrainStep {ms:8.3f} ms/step (host {host:.3f} ms) | head TrainStep {hms:8.3f} ms/step "
            f"(host {hhost:.3f} ms) | ratio {ms / hms:.2f}")
        del st, net
        torch.cuda.empty_cache()
    h, t, r = split(mode)
    say(f"{mode:5s} eager split (CUDA events, medians): head render {h:.3f} ms | torso forward + backward {t:.3f} ms | "
        f"gather + Adam + rest {r:.3f} ms | sum {h + t + r:.3f} ms")

if args.out:
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")
