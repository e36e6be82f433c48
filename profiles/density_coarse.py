"""Coarse pass with and without its colour branch, on bench.py's frame (450 x 450, 64 + 128 samples, bf16).

In one process, alternating call by call, the fused entry (ops.render_rays_fused, gen = the whole frame) runs with rgb0 (the full coarse
FaceNeRF and compositor, what render_band does) and without it (the density-only coarse build and the sigma-only compositor, what
render_frame / render_video do).  Per arm: the five stage times of inerf_debug_render_stage_ms (CUDA events between the launches of one
call) as median, min and max over --frames calls, for perturb = 1 (bench.py `value`) and perturb = 0 (render_video, evaluate_split).
The card name, its power limit and the SM clock are read before and after and printed beside the numbers.

    python profiles/density_coarse.py [--frames 20] [--out profiles/r12_density_coarse.txt]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

STAGES = ("setup", "mlp_coarse", "composite_sample", "mlp_fine", "composite_final")


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm,power.draw"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                       capture_output=True, text=True)
    return dict(zip(q.split(","), (v.strip() for v in r.stdout.strip().split(",")))) if r.returncode == 0 else {"nvidia-smi": r.stderr.strip()}


def summary(rows):
    out = {}
    for k, name in enumerate(STAGES + ("total",)):
        v = [sum(r) for r in rows] if name == "total" else [r[k] for r in rows]
        out[name] = {"median": statistics.median(v), "min": min(v), "max": max(v)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=20, help="timed calls per arm and perturb setting")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the report here")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "profiles/density_coarse.py measures on the GPU"
    import bench
    from ideal_nerf_b200 import ops
    dev = torch.device("cuda", 0)
    _, net, fr, _ = bench.build_network("bf16", dev)
    H, W = net.H, net.W
    pose, bc = fr["pose"].to(dev), fr["bc_rgb"].to(dev).reshape(-1, 3)
    cond = (fr["aud"].to(dev), fr["expr"].to(dev), fr["latent"].to(dev))
    gen = dict(H=H, W=W, focal=net.focal, cx=W * .5, cy=H * .5, near=net.near, far=net.far, c2w=pose[:3, :4], first=0, count=H * W)
    a = net.args
    before = card()
    report = {"card_before": before, "frame": f"{H} x {W}, {a.N_samples} + {a.N_importance} samples, bf16", "frames_per_arm": args.frames}
    with torch.no_grad():
        for perturb in (1.0, 0.0):
            rows = {True: [], False: []}
            for i in range(2 * (args.frames + args.warmup)):
                coarse_rgb = i % 2 == 0
                ms = []
                ops.render_rays_fused(net.face_nerf_coarse, net.face_nerf_fine, cond, cond, bc, a.N_samples, a.N_importance, perturb, gen=gen,
                                      stage_ms=ms, coarse_rgb=coarse_rgb)
                if i >= 2 * args.warmup:
                    rows[coarse_rgb].append(ms[0])
            full, dens = summary(rows[True]), summary(rows[False])
            report[f"perturb={perturb:g}"] = {
                "with_rgb0": full, "without_rgb0": dens,
                "mlp_coarse_drop": 1 - dens["mlp_coarse"]["median"] / full["mlp_coarse"]["median"],
                "total_drop": 1 - dens["total"]["median"] / full["total"]["median"]}
    report["card_after"] = card()
    lines = [f"card: {before.get('name')}  power limit {before.get('power.limit')}  SM clock {before.get('clocks.sm')} "
             f"(max {before.get('clocks.max.sm')}) before, {report['card_after'].get('clocks.sm')} after",
             f"frame: {report['frame']}; {args.frames} calls per arm, arms alternating call by call; ms = CUDA events between the launches "
             "of one fused call (inerf_debug_render_stage_ms)"]
    for p in ("perturb=1", "perturb=0"):
        r = report[p]
        lines.append(f"{p}:  stage ms, median [min, max]")
        for name in STAGES + ("total",):
            f, d = r["with_rgb0"][name], r["without_rgb0"][name]
            lines.append(f"  {name:17s} with rgb0 {f['median']:8.3f} [{f['min']:.3f}, {f['max']:.3f}]   "
                         f"without {d['median']:8.3f} [{d['min']:.3f}, {d['max']:.3f}]")
        lines.append(f"  coarse FaceNeRF {100 * r['mlp_coarse_drop']:.1f} % faster, whole call {100 * r['total_drop']:.1f} % faster")
    text = "\n".join(lines)
    print(text)
    print(json.dumps(report))
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n" + json.dumps(report) + "\n")


if __name__ == "__main__":
    main()
