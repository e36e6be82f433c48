"""FaceNeRF.forward on embedded rows x (P, 63+27) in fp16x2 mode: the fp32-gate tensor-core embedded-row kernel (csrc/mlp_f16x2.cu, EMB
build, mode INERF_MLP_F16X2_EMB) against the fp32 kernel, the fused (rays, z) entry, the reference's goldens and the reference pipeline
with only FaceNeRF swapped; training in this mode still runs the fp32 kernels."""
import os
import subprocess
import sys

import pytest
import torch

from oracle import render_oracle as O
import test_gpu_parity as G
import test_embedded_bf16 as EB

pytestmark = pytest.mark.gpu

DEV = G.DEV
M = G.M            # module fixture: the built package on a B200
ROOT = EB.ROOT
P_RAGGED = EB.P_RAGGED
DIMS = EB.DIMS


def _fp32_bars(got, ref, what, bar=2e-5):
    """The bar of test_fp16x2_raw_matches_fp32_kernel: per channel, max-abs over the rows of `got` relative to the channel's scale over the
    whole batch `ref`."""
    scale = ref.abs().amax(0).clamp_min(1e-3)
    err = (got - ref[:got.shape[0]]).abs().amax(0) / scale
    print(f"{what}: max-abs / scale per channel {[f'{e:.2e}' for e in err.tolist()]}")
    assert bool((err < bar).all()), f"{what}: {err.tolist()}"


@pytest.mark.parametrize("preset", ["init", "dense"])
@pytest.mark.parametrize("net_kind", ["head", "torso"])
def test_embedded_f16x2_raw_vs_fp32_ragged(M, net_kind, preset):
    """raw of the fp16x2 embedded kernel against the fp32 embedded kernel for ragged row counts (P = 1 and P < 128 included); the first P
    rows of a call are bit-identical to the same rows of the largest call (rows never mix)."""
    dims = DIMS[net_kind]
    pts, dirs, b = EB._sample_points(max(P_RAGGED), 11)
    sd = EB._state(preset, dims, 5, b)
    nx, n32 = EB._net(M, sd, "fp16x2", dims), EB._net(M, sd, "fp32", dims)
    cond = [None if t is None else t.to(DEV) for t in EB._cond(dims, 5)]
    x = EB._embed(pts, dirs).to(DEV)
    with torch.no_grad():
        r32 = n32(x, *cond)
        rx_all = nx(x, *cond)
        for P in P_RAGGED:
            rx = nx(x[:P], *cond)
            assert rx.shape == (P, 4) and bool(torch.isfinite(rx).all())
            assert torch.equal(rx, rx_all[:P]), f"P={P}: rows depend on the call size"
            _fp32_bars(rx, r32, f"{net_kind}/{preset} P={P}")


def test_embedded_f16x2_matches_fused_query(M):
    """The same points through FaceNeRF.query (fused gamma, per-ray fp32 view bias) and FaceNeRF.forward (embedded rows, split-operand view
    K-block), x built by get_embedder as test_face_nerf_fused_query_matches_embedded builds it: fp32-level agreement."""
    b = O.synthetic_train_batch(0)
    n, s = 211, 64
    rays = b["rays"][:n].to(DEV)
    net = G.head_net(M, O.init_face_nerf(5), "fp16x2")
    aud, expr, lat = b["aud"].to(DEV), b["expr"].to(DEV), b["latent"].to(DEV)
    z = M.ops.sample_coarse(rays, s, torch.rand(n, s, device=DEV, generator=torch.Generator(device=DEV).manual_seed(4)))
    with torch.no_grad():
        raw = net.query(rays, z, aud, expr, lat).reshape(-1, 4)
        pts = rays[:, None, 0:3] + rays[:, None, 3:6] * z[..., None]
        e10, _ = M.get_embedder(10, 0); e4, _ = M.get_embedder(4, 0)
        x = torch.cat([e10(pts.reshape(-1, 3)), e4(rays[:, None, 8:11].expand(pts.shape).reshape(-1, 3))], -1)
        raw2 = net(x, aud, expr, lat)
    _fp32_bars(raw2, raw, "embedded vs fused query (fp16x2)")


def test_embedded_f16x2_golden(M, golden):
    """The reference's face_nerf goldens within 2e-5, the fp32 kernel's bar in test_face_nerf_forward_golden."""
    g = golden("face_nerf")
    net = G.head_net(M, O.init_face_nerf(int(g["seed_head"])), "fp16x2")
    net_t = G.head_net(M, O.init_face_nerf(int(g["seed_torso"]), 106, 0, 0), "fp16x2", dim_aud=106, dim_latent=0, dim_expr=0)
    with torch.no_grad():
        out = net(G.C(g["x"]), G.C(g["aud"]), G.C(g["expr"]), G.C(g["latent"]))
        out_t = net_t(G.C(g["x"]), G.C(g["aud_torso"]))
    print(f"golden max-abs: head {G.maxabs(out, g['out_head']):.3e}, torso {G.maxabs(out_t, g['out_torso']):.3e}")
    G.close(out, g["out_head"], 2e-5, "FaceNeRF head (fp16x2 embedded)")
    G.close(out_t, g["out_torso"], 2e-5, "FaceNeRF torso (fp16x2 embedded)")


@pytest.mark.parametrize("tag", ["init", "dense"])
def test_reference_render_with_f16x2_face_nerf_swapped_in(M, golden, tag):
    """The reference pipeline (oracle render_rays, the reference's run_network embedding and netchunk loop) with only FaceNeRF replaced by
    this package's module in fp16x2 mode, fed in netchunk pieces on the device, against the reference's own outputs: the fp32-gate bars
    of test_render_rays_fp16x2_meets_fp32_gate (init: every output within 1e-5; dense: at most 3 of 3072 rays over 1e-3, 99 % within
    3e-4, max-abs 1.5e-3 -- 10 rays, 6e-4 and 4e-3 for last_weight and the depth derived from disp)."""
    g = golden("render_3072")
    c, f = O.init_face_nerf(1), O.init_face_nerf(2)
    c["alpha_linear.weight"], c["alpha_linear.bias"] = torch.from_numpy(g[f"{tag}_alpha_w_c"]), torch.from_numpy(g[f"{tag}_alpha_b_c"])
    f["alpha_linear.weight"], f["alpha_linear.bias"] = torch.from_numpy(g[f"{tag}_alpha_w_f"]), torch.from_numpy(g[f"{tag}_alpha_b_f"])
    nets = {}
    orig = O.run_network

    def run_network_f16x2(sd, pts, viewdirs, a, e, l, netchunk=65536):
        key = id(sd)
        if key not in nets:
            nets[key] = G.head_net(M, sd, "fp16x2")
        flat = pts.reshape(-1, 3)
        enc = torch.cat([O.positional_encoding(flat, 10), O.positional_encoding(viewdirs[:, None].expand(pts.shape).reshape(-1, 3), 4)], -1)
        enc = enc.to(DEV)
        cond = [t.to(DEV) for t in (a, e, l)]
        outs = [nets[key](enc[i:i + netchunk], *cond) for i in range(0, enc.shape[0], netchunk)]
        return torch.cat(outs, 0).cpu().reshape(list(pts.shape[:-1]) + [4])

    rays, bc = torch.from_numpy(g["rays"]), torch.from_numpy(g["bc_rgb"])
    aud, expr, lat = (torch.from_numpy(g[k]) for k in ("aud", "expr", "latent"))
    O.run_network = run_network_f16x2
    try:
        with torch.no_grad():
            r = O.render_rays(rays, bc, c, f, aud, expr, lat)
    finally:
        O.run_network = orig
    assert len(nets) == 2
    outs = {k: (r[k], torch.from_numpy(g[f"{tag}_{k}"])) for k in ("rgb_map", "acc_map", "rgb0", "acc0", "last_weight", "z_std")}
    outs["depth (1/disp)"] = (1.0 / r["disp_map"], 1.0 / torch.from_numpy(g[f"{tag}_disp_map"]))
    for k, (a, b) in outs.items():
        err = (a.double() - b.double()).abs().reshape(a.shape[0], -1).amax(1)          # per ray
        e, n_over, q = float(err.max()), int((err > 1e-3).sum()), float(torch.quantile(err, 0.99))
        print(f"[{tag}] fp16x2 embedded FaceNeRF in the reference pipeline, {k}: max-abs {e:.3e}; rays over 1e-3: {n_over} of "
              f"{err.numel()}; 99th percentile {q:.2e}; 99.9th {float(torch.quantile(err, 0.999)):.2e}")
        if tag == "init":
            assert e <= 1e-5, f"{k}: {e:.3e}"
        else:
            loose = k in ("last_weight", "depth (1/disp)")
            assert e <= (4e-3 if loose else 1.5e-3), f"{k}: {e:.3e}"
            assert n_over <= (10 if loose else 3) and q <= (6e-4 if loose else 3e-4), f"{k}: {n_over} rays over 1e-3, 99th percentile {q:.2e}"


@pytest.mark.parametrize("P", [203, 12345])
def test_embedded_f16x2_training_runs_fp32_kernels(M, P):
    """Training through FaceNeRF.forward(x) in fp16x2 mode runs the fp32 kernels: raw equals the fp32 net's bit for bit and the gradients
    equal the fp32 net's to 1e-5 relative (atomic reductions: not bitwise); the new inference route does not leak into training."""
    pts, dirs, b = EB._sample_points(P, 13)
    sd = O.init_face_nerf(7)
    nx, n32 = G.head_net(M, sd, "fp16x2"), G.head_net(M, sd, "fp32")
    gen = torch.Generator(device=DEV).manual_seed(P)
    Gr = torch.randn(P, 4, device=DEV, generator=gen)
    x = EB._embed(pts, dirs).to(DEV)
    res = {}
    for tag, net in (("fp16x2", nx), ("fp32", n32)):
        net.train()
        aud, expr, lat = (b[k].to(DEV).clone().requires_grad_(True) for k in ("aud", "expr", "latent"))
        raw = net(x, aud, expr, lat)
        (raw * Gr).sum().backward()
        res[tag] = ({k: p.grad.clone() for k, p in net.named_parameters() if p.grad is not None}, raw.detach(), aud.grad, expr.grad,
                    lat.grad)
    assert torch.equal(res["fp16x2"][1], res["fp32"][1]), "training forward in fp16x2 mode must be the fp32 kernel"
    assert set(res["fp16x2"][0]) == set(res["fp32"][0])
    for k, g32 in res["fp32"][0].items():
        G.close(res["fp16x2"][0][k], g32, 1e-5 * max(float(g32.abs().max()), 1e-30), f"grad {k}")
    for i, nm in ((2, "d_aud"), (3, "d_expr"), (4, "d_latent")):
        G.close(res["fp16x2"][i], res["fp32"][i], 1e-5 * float(res["fp32"][i].abs().max()), nm)


_EMB_PAIR_VS_SINGLE = r"""
import hashlib, sys, torch
sys.path.insert(0, %r)
import ideal_nerf_b200 as M
dev = "cuda:0"
torch.manual_seed(3)
net = M.FaceNeRF(dim_aud=64, dim_latent=32, dim_expr=76, mlp_mode="fp16x2").apply(M.init_weights).to(dev)
g = torch.Generator(dev).manual_seed(5)
aud, expr, lat = (torch.randn(d, device=dev, generator=g) for d in (64, 76, 32))
h = hashlib.sha256()
for P in (1, 8769, 36 * 128 + 77):          # 1, 69 and 37 128-row slots: odd slot counts leave the peer CTA's last slot past the end
    x = torch.randn(P, 90, device=dev, generator=g)
    with torch.no_grad():
        h.update(net(x, aud, expr, lat).contiguous().cpu().numpy().tobytes())
torch.cuda.synchronize()
print("HASH", h.hexdigest())
"""


def test_embedded_f16x2_deterministic_and_pair_matches_single_cta(M):
    """A repeated call is bit-identical, and the CTA-pair build of the embedded-row kernel gives the same raw bit for bit as the single-CTA
    build (INERF_MLP_PAIR=0, read once per process)."""
    x = torch.randn(20000, 90, device=DEV, generator=torch.Generator(DEV).manual_seed(1))
    net = G.head_net(M, O.init_face_nerf(3), "fp16x2")
    b = O.synthetic_train_batch(0)
    cond = (b["aud"].to(DEV), b["expr"].to(DEV), b["latent"].to(DEV))
    with torch.no_grad():
        assert torch.equal(net(x, *cond), net(x, *cond))
    out = []
    for pair in ("1", "0"):
        r = subprocess.run([sys.executable, "-c", _EMB_PAIR_VS_SINGLE % ROOT], env={**os.environ, "INERF_MLP_PAIR": pair},
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        out.append([l for l in r.stdout.splitlines() if l.startswith("HASH")][-1])
    assert out[0] == out[1], out


def test_embedded_f16x2_packed_cache(M):
    """The embedded-row blob is cached per mode: a net switched bf16 -> fp16x2 -> bf16 gets the right blob each time and the outputs of a
    fresh net of that mode; an in-place weight update re-packs; invalidate_packed() drops the blob."""
    sd = O.init_face_nerf(3)
    b = O.synthetic_train_batch(0)
    cond = (b["aud"].to(DEV), b["expr"].to(DEV), b["latent"].to(DEV))
    x = torch.randn(300, 90, device=DEV, generator=torch.Generator(DEV).manual_seed(2))
    net = G.head_net(M, sd, "bf16")
    sizes = {}
    with torch.no_grad():
        for mode in ("bf16", "fp16x2", "bf16"):
            net.mlp_mode = mode
            out = net(x, *cond)
            assert torch.equal(out, G.head_net(M, sd, mode)(x, *cond)), f"switched to {mode}"
            sizes.setdefault(mode, net._packed_e.numel())
            assert net._packed_e.numel() == sizes[mode]
    assert sizes == {"bf16": 1130496, "fp16x2": 2260992}
    net.mlp_mode = "fp16x2"
    ps = net.kernel_params()
    e = net.packed_weights_emb(ps)
    assert e is net.packed_weights_emb(ps)
    with torch.no_grad():
        before = net(x, *cond)
        net.rgb_linear.bias.add_(1.0)
        net.pts_linears[3].weight.mul_(1.5)
        after = net(x, *cond)
    assert net.packed_weights_emb(net.kernel_params()) is not e
    assert not torch.equal(before, after)
    net.invalidate_packed()
    assert net._packed_e is None
