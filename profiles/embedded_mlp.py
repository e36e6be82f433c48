"""FaceNeRF.forward on embedded rows (x (P, 63+27), the reference module's own signature) against the fused (rays, z) entry.

    python profiles/embedded_mlp.py                      # card, power limit, points/s of the paths below, query hashes
    python profiles/embedded_mlp.py --hash-only --root T # only the sha256 of the bf16 and fp16x2 outputs below, with the package of tree T

On P = 202 500 x 64 rows (one 450 x 450 frame, 64 samples per ray; x is 4.7 GB, far larger than L2, and read once per call):
  * FaceNeRF.forward(x), mlp_mode="fp32" (FFMA kernel), "bf16" and "fp16x2" (tcgen05 embedded-row kernels);
  * FaceNeRF.query(rays, z) in bf16 and in fp16x2 on the same points (fused gamma, per-ray view bias);
  * Network.run_network at the reference's netchunk = 65 536 (embedding + FaceNeRF.forward per 65 536-row piece), and the forward calls
    alone on the pre-embedded pieces.
Times are CUDA-event times of whole calls after a warm-up.  TFLOP/s are algorithmic: 560 640 MAC per point for the fused form (view
columns folded into a per-ray bias), 560 640 + 3 456 for the embedded form, against the sustained cuBLAS bf16 figure of DESIGN.md §3;
for fp16x2 the issued rate of its three MMA passes (hi.hi + lo.hi + hi.lo) is printed as well.
The hashes are of raw from a seeded FaceNeRF.query (137 rays x {64, 192} samples) and of FaceNeRF.forward on the embedded rows of the
same points, each in bf16 and in fp16x2: equal hashes from two trees = the fused and embedded-row paths are unchanged bit for bit.
"""
import argparse
import hashlib
import os
import subprocess
import sys

ap = argparse.ArgumentParser()
ap.add_argument("--root", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))), help="tree whose package is imported")
ap.add_argument("--hash-only", action="store_true")
ap.add_argument("--out", default=None, help="also write the report to this file")
args = ap.parse_args()
sys.path.insert(0, os.path.abspath(args.root))

import torch  # noqa: E402
import ideal_nerf_b200 as M  # noqa: E402
from ideal_nerf_b200 import ops, synthetic as S  # noqa: E402

FLOP_FUSED = 2 * 560_640
FLOP_EMB = 2 * (560_640 + 3_456)
SUSTAINED_BF16_TFLOPS = 1376.0
lines = []


def say(s):
    print(s, flush=True)
    lines.append(s)


dev = torch.device("cuda", 0)
assert torch.cuda.is_available(), "needs a GPU"
cam, fr = S.camera(), S.frame_inputs(0)
aud, expr, lat = fr["aud"].to(dev), fr["expr"].to(dev), fr["latent"].to(dev)


def raw_hashes(mode):
    """sha256 of FaceNeRF.query(rays, z) and of FaceNeRF.forward(x) on the embedded rows of the same points."""
    torch.manual_seed(3)
    net = M.FaceNeRF(dim_aud=64, dim_latent=32, dim_expr=76, mlp_mode=mode).apply(M.init_weights).to(dev)
    rays = ops.get_rays_range(450, 450, cam["focal"], cam["c2w"].to(dev), S.NEAR, S.FAR, 90000, 137)
    e10, _ = M.get_embedder(10, 0)
    e4, _ = M.get_embedder(4, 0)
    hq, he = hashlib.sha256(), hashlib.sha256()
    with torch.no_grad():
        for s in (64, 192):
            z = torch.sort(S.NEAR + (S.FAR - S.NEAR) * torch.rand(137, s, device=dev, generator=torch.Generator(dev).manual_seed(s)), -1)[0]
            hq.update(net.query(rays, z.contiguous(), aud, expr, lat).cpu().numpy().tobytes())
            pts = (rays[:, None, 0:3] + rays[:, None, 3:6] * z[..., None]).reshape(-1, 3)
            x = torch.cat([e10(pts), e4(rays[:, None, 8:11].expand(137, s, 3).reshape(-1, 3))], -1).contiguous()
            he.update(net(x, aud, expr, lat).cpu().numpy().tobytes())
    return hq.hexdigest(), he.hexdigest()


for mode, tag in (("bf16", ""), ("fp16x2", "_fp16x2")):
    hq, he = raw_hashes(mode)
    say(f"query_raw_sha256{tag} {hq}  (package of {os.path.abspath(args.root)})")
    say(f"embedded_raw_sha256{tag} {he}  (package of {os.path.abspath(args.root)})")
if args.hash_only:
    sys.exit(0)

try:
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True, timeout=60).stdout.strip().splitlines()[0]
except Exception as e:          # the measurement stands without it, but says so
    smi = f"nvidia-smi unavailable ({e})"
say(f"card: {torch.cuda.get_device_name(0)}; nvidia-smi name, power limit, max SM clock: {smi}")


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def report(name, ms, n_pts, flop_per_pt, passes=1):
    tf = n_pts * flop_per_pt / (ms * 1e-3) / 1e12
    issued = f";  {passes * tf:7.1f} TFLOP/s issued ({passes} passes) = {passes * tf / SUSTAINED_BF16_TFLOPS:.3f}" if passes > 1 else ""
    say(f"{name:52s} {ms:9.3f} ms  {n_pts / (ms * 1e-3) / 1e6:9.1f} M points/s  {tf:7.1f} TFLOP/s algorithmic "
        f"= {tf / SUSTAINED_BF16_TFLOPS:.3f} of sustained bf16{issued}")
    return n_pts / (ms * 1e-3)


torch.manual_seed(1)
net = M.FaceNeRF(dim_aud=64, dim_latent=32, dim_expr=76, mlp_mode="bf16").apply(M.init_weights).to(dev)
n_rays, s = 202_500, 64
rays = ops.get_rays_packed(450, 450, cam["focal"], cam["c2w"].to(dev), S.NEAR, S.FAR)
z = torch.sort(S.NEAR + (S.FAR - S.NEAR) * torch.rand(n_rays, s, device=dev, generator=torch.Generator(dev).manual_seed(7)), -1)[0]
z = z.contiguous()
P = n_rays * s
with torch.no_grad():
    pts = rays[:, None, 0:3] + rays[:, None, 3:6] * z[..., None]
    e10, _ = M.get_embedder(10, 0)
    e4, _ = M.get_embedder(4, 0)
    x = torch.cat([e10(pts.reshape(-1, 3)), e4(rays[:, None, 8:11].expand(pts.shape).reshape(-1, 3))], -1).contiguous()
say(f"P = {n_rays} x {s} = {P} rows; x {tuple(x.shape)} fp32 = {x.numel() * 4 / 1e9:.2f} GB")

host = M.Network(450, 450, 1200., S.NEAR, S.FAR, 8192, None, 64, 128, args=M.default_args(dim_aud=64, dim_expr=76)).to(dev)
with torch.no_grad():
    net.mlp_mode = "fp32"
    r32 = report("FaceNeRF.forward(x)  fp32", timed(lambda: net(x, aud, expr, lat), 2), P, FLOP_EMB)
    out32 = net(x, aud, expr, lat)
    net.mlp_mode = "fp16x2"
    rx = report("FaceNeRF.forward(x)  fp16x2", timed(lambda: net(x, aud, expr, lat), 5), P, FLOP_EMB, passes=3)
    rxq = report("FaceNeRF.query(rays, z)  fp16x2 (same points)", timed(lambda: net.query(rays, z, aud, expr, lat), 5), P, FLOP_FUSED,
                 passes=3)
    outx = net(x, aud, expr, lat)
    scale = out32.abs().amax(0)
    dx32 = ((outx - out32).abs().amax(0) / scale).tolist()
    dxq = ((outx - net.query(rays, z, aud, expr, lat).reshape(-1, 4)).abs().amax(0) / scale).tolist()
    del outx
    net.mlp_mode = "bf16"
    r16 = report("FaceNeRF.forward(x)  bf16", timed(lambda: net(x, aud, expr, lat), 10), P, FLOP_EMB)
    rq = report("FaceNeRF.query(rays, z)  bf16 (same points)", timed(lambda: net.query(rays, z, aud, expr, lat), 10), P, FLOP_FUSED)
    rn = report("Network.run_network netchunk 65536  bf16", timed(lambda: host.run_network(pts, expr, rays[:, 8:11], aud, net, lat, 65536), 5),
                P, FLOP_EMB)
    pieces = lambda: [net(x[i:i + 65536], aud, expr, lat) for i in range(0, P, 65536)]
    rp = report("  of which FaceNeRF.forward on 65536-row pieces", timed(pieces, 5), P, FLOP_EMB)
    d = (net(x, aud, expr, lat) - net.query(rays, z, aud, expr, lat).reshape(-1, 4)).abs().amax(0)
say(f"bf16 embedded / bf16 fused: {r16 / rq:.3f};  bf16 embedded / fp32 embedded: {r16 / r32:.1f}x;  "
    f"run_network(netchunk 65536) / bf16 embedded: {rn / r16:.3f} (forward pieces alone {rp / r16:.3f})")
say(f"max |embedded - fused| per channel (r, g, b, sigma): {[f'{v:.2e}' for v in d.tolist()]}")
say(f"fp16x2 embedded / fp16x2 fused: {rx / rxq:.3f};  fp16x2 embedded / fp32 embedded: {rx / r32:.1f}x")
say(f"fp16x2 embedded, max-abs / scale of the fp32 kernel's raw per channel (r, g, b, sigma): vs fp32 embedded "
    f"{[f'{v:.2e}' for v in dx32]}, vs fp16x2 fused {[f'{v:.2e}' for v in dxq]}")
if args.out:
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")
