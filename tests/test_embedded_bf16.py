"""FaceNeRF.forward on embedded rows x (P, 63+27) in bf16 mode: the tcgen05 embedded-row kernel (csrc/mlp_bf16.cu, EMB build) for
inference and training, against the fp32 kernel, an emulation that rounds where the kernel rounds, the fused (rays, z) entry, the
reference's goldens and the reference pipeline with only FaceNeRF swapped."""
import os
import subprocess
import sys

import pytest
import torch

from oracle import render_oracle as O
import test_gpu_parity as G

pytestmark = pytest.mark.gpu

DEV = G.DEV
M = G.M            # module fixture: the built package on a B200
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P_RAGGED = [1, 127, 128, 129, 203, 255, 257, 12345, 65573]
DIMS = {"head": (64, 76, 32), "torso": (106, 0, 0)}


def _net(M, sd, mode, dims):
    da, de, dl = dims
    return G.head_net(M, sd, mode, dim_aud=da, dim_expr=de, dim_latent=dl)


def _cond(dims, seed):
    g = torch.Generator().manual_seed(seed)
    return tuple(torch.randn(d, generator=g) if d else None for d in dims)


def _sample_points(n_pts, seed):
    """Points on the synthetic batch's rays at depths in [near, far], with their view directions, as CPU tensors."""
    b = O.synthetic_train_batch(0)
    g = torch.Generator().manual_seed(seed)
    rays = b["rays"][torch.randint(0, b["rays"].shape[0], (n_pts,), generator=g)]
    z = O.NEAR + (O.FAR - O.NEAR) * torch.rand(n_pts, 1, generator=g)
    return rays[:, 0:3] + rays[:, 3:6] * z, rays[:, 8:11], b


def _embed(pts, dirs):
    return torch.cat([O.positional_encoding(pts, 10), O.positional_encoding(dirs, 4)], -1)


def _state(preset, dims, seed, b):
    sd = O.init_face_nerf(seed, *dims)
    if preset == "dense":
        aud, expr, lat = _cond(dims, seed)
        sd = O.normalise_density(sd, b["rays"][::7], aud, expr, lat)
    return sd


def _bf16_bars(got, ref, what, max_rel=6e-2, rms_rel=3e-2):
    """The bars of test_bf16_mlp_layers_and_raw, per channel, relative to the channel's scale over the whole batch `ref`."""
    got, ref = got.double(), ref.double()
    scale, rms_ref = ref.abs().amax(0), (ref ** 2).mean(0).sqrt()
    d = got - ref[:got.shape[0]]
    err, rms = d.abs().amax(0) / scale, (d ** 2).mean(0).sqrt() / rms_ref
    assert bool((err < max_rel).all()) and bool((rms < rms_rel).all()), f"{what}: max-rel {err.tolist()}, rms-rel {rms.tolist()}"


def _emulated_embedded(sd, pe, de, aud, expr, lat):
    """test_gpu_parity's emulation with gamma(v) and the view columns of views_linears.0 rounded to bf16 and fed through the matmul, as
    the embedded-row kernel does (the fused entry adds them as an fp32 per-ray bias instead)."""
    w = sd["views_linears.0.weight"]
    wv = w[:, 256:283]
    sd = dict(sd, **{"views_linears.0.weight": torch.cat([w[:, :256], wv + (G._bf(wv) - wv).detach(), w[:, 283:]], 1)})
    return G._emulated_bf16_forward(sd, pe, G._bf(de), aud, expr, lat)


@pytest.mark.parametrize("preset", ["init", "dense"])
@pytest.mark.parametrize("net_kind", ["head", "torso"])
def test_embedded_bf16_raw_vs_fp32_ragged(M, net_kind, preset):
    """raw of the bf16 embedded kernel against the fp32 embedded kernel for ragged row counts (P = 1 and P < 128 included); the first P
    rows of a call are bit-identical to the same rows of the largest call (rows never mix)."""
    dims = DIMS[net_kind]
    pts, dirs, b = _sample_points(max(P_RAGGED), 11)
    sd = _state(preset, dims, 5, b)
    n16, n32 = _net(M, sd, "bf16", dims), _net(M, sd, "fp32", dims)
    cond = [None if t is None else t.to(DEV) for t in _cond(dims, 5)]
    x = _embed(pts, dirs).to(DEV)
    with torch.no_grad():
        r32 = n32(x, *cond)
        r16_all = n16(x, *cond)
        for P in P_RAGGED:
            r16 = n16(x[:P], *cond)
            assert r16.shape == (P, 4) and bool(torch.isfinite(r16).all())
            assert torch.equal(r16, r16_all[:P]), f"P={P}: rows depend on the call size"
            _bf16_bars(r16, r32, f"{net_kind}/{preset} P={P}")


def test_embedded_bf16_vs_emulation(M):
    """Random-init weights, as test_bf16_training_grads compares its emulation: with the normalised-density preset (alpha_linear scaled
    ~100x) a pre-activation that lands on a bf16 rounding boundary in one computation and not in the other moves sigma by more than the
    bar; that preset is held to the fp32-kernel bars and the PSNR gate above."""
    dims = DIMS["head"]
    pts, dirs, b = _sample_points(4099, 12)
    sd = _state("init", dims, 6, b)
    aud, expr, lat = _cond(dims, 6)
    net = _net(M, sd, "bf16", dims)
    pe, de = O.positional_encoding(pts, 10), O.positional_encoding(dirs, 4)
    with torch.no_grad():
        got = net(torch.cat([pe, de], -1).to(DEV), aud.to(DEV), expr.to(DEV), lat.to(DEV))
        sdd = {k: v.to(DEV) for k, v in sd.items()}
        ref = _emulated_embedded(sdd, pe.to(DEV), de.to(DEV), aud.to(DEV), expr.to(DEV), lat.to(DEV))
    G.close(got, ref, 6e-3 * max(1.0, float(ref.abs().max())), "bf16 embedded vs emulation")


def test_embedded_bf16_matches_fused_query(M):
    """The same points through FaceNeRF.query (fused gamma, per-ray fp32 view bias) and FaceNeRF.forward (embedded rows, bf16 view
    K-block), x built as test_face_nerf_fused_query_matches_embedded builds it: agreement at bf16 level."""
    b = O.synthetic_train_batch(0)
    n, s = 211, 64
    rays = b["rays"][:n].to(DEV)
    net = G.head_net(M, O.init_face_nerf(5), "bf16")
    aud, expr, lat = b["aud"].to(DEV), b["expr"].to(DEV), b["latent"].to(DEV)
    z = M.ops.sample_coarse(rays, s, torch.rand(n, s, device=DEV, generator=torch.Generator(device=DEV).manual_seed(4)))
    with torch.no_grad():
        raw = net.query(rays, z, aud, expr, lat).reshape(-1, 4)
        pts = rays[:, None, 0:3] + rays[:, None, 3:6] * z[..., None]
        e10, _ = M.get_embedder(10, 0); e4, _ = M.get_embedder(4, 0)
        x = torch.cat([e10(pts.reshape(-1, 3)), e4(rays[:, None, 8:11].expand(pts.shape).reshape(-1, 3))], -1)
        raw2 = net(x, aud, expr, lat)
    _bf16_bars(raw2, raw, "embedded vs fused query (bf16)")


def test_embedded_bf16_golden(M, golden):
    g = golden("face_nerf")
    net = G.head_net(M, O.init_face_nerf(int(g["seed_head"])), "bf16")
    net_t = G.head_net(M, O.init_face_nerf(int(g["seed_torso"]), 106, 0, 0), "bf16", dim_aud=106, dim_latent=0, dim_expr=0)
    with torch.no_grad():
        out = net(G.C(g["x"]), G.C(g["aud"]), G.C(g["expr"]), G.C(g["latent"]))
        out_t = net_t(G.C(g["x"]), G.C(g["aud_torso"]))
    _bf16_bars(out, torch.as_tensor(g["out_head"]).to(DEV), "golden out_head")
    _bf16_bars(out_t, torch.as_tensor(g["out_torso"]).to(DEV), "golden out_torso")


@pytest.mark.parametrize("tag", ["init", "dense"])
def test_reference_render_with_bf16_face_nerf_swapped_in(M, golden, tag):
    """The reference pipeline (oracle render_rays, the reference's run_network embedding and netchunk loop) with only FaceNeRF replaced by
    this package's module in bf16 mode, fed in netchunk pieces on the device: the north-star gate of test_render_rays_bf16_psnr_gate."""
    g = golden("render_3072")
    c, f = O.init_face_nerf(1), O.init_face_nerf(2)
    c["alpha_linear.weight"], c["alpha_linear.bias"] = torch.from_numpy(g[f"{tag}_alpha_w_c"]), torch.from_numpy(g[f"{tag}_alpha_b_c"])
    f["alpha_linear.weight"], f["alpha_linear.bias"] = torch.from_numpy(g[f"{tag}_alpha_w_f"]), torch.from_numpy(g[f"{tag}_alpha_b_f"])
    nets = {}
    orig = O.run_network

    def run_network_bf16(sd, pts, viewdirs, a, e, l, netchunk=65536):
        key = id(sd)
        if key not in nets:
            nets[key] = G.head_net(M, sd, "bf16")
        flat = pts.reshape(-1, 3)
        enc = torch.cat([O.positional_encoding(flat, 10), O.positional_encoding(viewdirs[:, None].expand(pts.shape).reshape(-1, 3), 4)], -1)
        enc = enc.to(DEV)
        cond = [t.to(DEV) for t in (a, e, l)]
        outs = [nets[key](enc[i:i + netchunk], *cond) for i in range(0, enc.shape[0], netchunk)]
        return torch.cat(outs, 0).cpu().reshape(list(pts.shape[:-1]) + [4])

    rays, bc = torch.from_numpy(g["rays"]), torch.from_numpy(g["bc_rgb"])
    aud, expr, lat = (torch.from_numpy(g[k]) for k in ("aud", "expr", "latent"))
    O.run_network = run_network_bf16
    try:
        with torch.no_grad():
            r = O.render_rays(rays, bc, c, f, aud, expr, lat)
    finally:
        O.run_network = orig
    assert len(nets) == 2
    gen = torch.Generator(device=DEV).manual_seed(30)
    for key in ("rgb_map", "rgb0"):
        ref = torch.from_numpy(g[f"{tag}_{key}"]).to(DEV)
        tgt = ref + 0.0316 * torch.randn(ref.shape, device=DEV, generator=gen)
        ours = r[key].to(DEV)
        psnr_ref, psnr_ours = G._psnr(ref, tgt), G._psnr(ours, tgt)
        print(f"[{tag}] {key}: PSNR vs target: reference {psnr_ref:.4f} dB, bf16 embedded FaceNeRF {psnr_ours:.4f} dB "
              f"(delta {abs(psnr_ours - psnr_ref):.4f}); PSNR(ours, reference render) {G._psnr(ours, ref):.2f} dB")
        assert 29.5 < psnr_ref < 30.5
        assert abs(psnr_ours - psnr_ref) <= 0.05, "north_star gate: PSNR delta <= 0.05 dB in bf16-MLP mode"


@pytest.mark.parametrize("P", [203, 12345])
def test_embedded_bf16_training_grads(M, P):
    """bf16 training through FaceNeRF.forward(x) (saving forward + the bf16 backward chain, dW and conditioning kernels): against
    autograd of the emulation and against the fp32 kernels, with the bars of test_bf16_training_grads."""
    pts, dirs, b = _sample_points(P, 13)
    sd = O.init_face_nerf(7)
    n16, n32 = G.head_net(M, sd, "bf16"), G.head_net(M, sd, "fp32")
    gen = torch.Generator(device=DEV).manual_seed(P)
    Gr = torch.randn(P, 4, device=DEV, generator=gen) * torch.tensor([1., 1., 1., 0.3], device=DEV)
    pe, de = O.positional_encoding(pts, 10).to(DEV), O.positional_encoding(dirs, 4).to(DEV)
    x = torch.cat([pe, de], -1)
    grads = {}
    for tag, net in (("bf16", n16), ("fp32", n32)):
        aud, expr, lat = b["aud"].to(DEV).clone().requires_grad_(True), b["expr"].to(DEV)[None].clone().requires_grad_(True), \
            b["latent"].to(DEV).clone().requires_grad_(True)
        raw = net(x, aud, expr, lat)
        (raw * Gr).sum().backward()
        assert aud.grad.shape == aud.shape and expr.grad.shape == expr.shape and lat.grad.shape == lat.shape
        grads[tag] = ({k: p.grad.clone() for k, p in net.named_parameters() if p.grad is not None}, aud.grad, expr.grad.reshape(-1),
                      lat.grad, raw.detach())
    with torch.no_grad():
        assert torch.equal(grads["bf16"][4], n16(x, b["aud"].to(DEV), b["expr"].to(DEV), b["latent"].to(DEV))), \
            "the saving build must not change raw"
    sdg = {k: v.to(DEV).clone().requires_grad_(True) for k, v in sd.items()}
    aud, expr, lat = (b[k].to(DEV).clone().requires_grad_(True) for k in ("aud", "expr", "latent"))
    raw_e = _emulated_embedded(sdg, pe, de, aud, expr, lat)
    (raw_e * Gr).sum().backward()
    G.close(grads["bf16"][4], raw_e, 6e-3 * max(1.0, float(raw_e.abs().max())), "bf16 training forward vs emulation")
    for k, gk in grads["bf16"][0].items():
        ref, r32 = sdg[k].grad, grads["fp32"][0][k]
        if float(r32.abs().max()) == 0.0:
            continue
        rel = float((gk - ref).norm() / ref.norm())
        cos = float(torch.nn.functional.cosine_similarity(gk.flatten().double(), r32.flatten().double(), dim=0))
        print(f"[P={P}] {k:26s} rel-L2 vs emulation {rel:.3e}   cos vs fp32 kernels {cos:.5f}")
        assert rel <= 0.1, (k, rel)
        assert cos >= 0.97, (k, cos)
    for i, nm in ((1, "d_aud"), (2, "d_expr"), (3, "d_latent")):
        ref = (aud, expr, lat)[i - 1].grad
        rel = float((grads["bf16"][i] - ref).norm() / ref.norm())
        print(f"[P={P}] {nm}: rel-L2 vs emulation {rel:.3e}")
        assert rel <= 0.1, (nm, rel)


def test_embedded_bf16_vs_fp32_training_500_steps(M):
    """test_bf16_vs_fp32_training_500_steps through embedded rows: a FaceNeRF trained with FaceNeRF.forward(x) for 500 Adam steps (lr 1e-3
    decaying one decade per 300 steps, so the run ends at a converged point) to reproduce the raw output of a teacher network on 65 536
    embedded points of the synthetic batch's rays, same initial weights in both modes.  Final PSNR of raw (mean of the last 50 steps) of
    bf16 mode within 0.1 dB of fp32 mode; both improve by more than 1 dB."""
    pts, dirs, b = _sample_points(65536, 14)
    x = _embed(pts, dirs).to(DEV)
    aud, expr, lat = b["aud"].to(DEV), b["expr"].to(DEV), b["latent"].to(DEV)
    with torch.no_grad():
        target = G.head_net(M, O.init_face_nerf(41), "fp32")(x, aud, expr, lat)
    curves = {}
    for mode in ("fp32", "bf16"):
        net = G.head_net(M, O.init_face_nerf(43), mode).train()
        opt = torch.optim.Adam(net.parameters(), lr=1e-3, betas=(0.9, 0.999))
        psnr = []
        for i in range(500):
            for gr in opt.param_groups:
                gr["lr"] = 1e-3 * 0.1 ** (i / 300)
            opt.zero_grad(set_to_none=True)
            loss = torch.mean((net(x, aud, expr, lat) - target) ** 2)
            loss.backward()
            opt.step()
            psnr.append(-10. * torch.log10(loss.detach()))
        curves[mode] = torch.stack(psnr).cpu()
    p32, p16 = curves["fp32"], curves["bf16"]
    print(f"PSNR step 0: fp32 {float(p32[0]):.3f} bf16 {float(p16[0]):.3f}; last-50 mean: fp32 {float(p32[-50:].mean()):.3f} "
          f"bf16 {float(p16[-50:].mean()):.3f}; max |delta| over the run {float((p32 - p16).abs().max()):.3f} dB")
    assert float(p32[-50:].mean()) > float(p32[0]) + 1.0 and float(p16[-50:].mean()) > float(p16[0]) + 1.0
    assert abs(float(p32[-50:].mean()) - float(p16[-50:].mean())) <= 0.1


_EMB_PAIR_VS_SINGLE = r"""
import hashlib, sys, torch
sys.path.insert(0, %r)
import ideal_nerf_b200 as M
from ideal_nerf_b200 import ops
dev = "cuda:0"
torch.manual_seed(3)
net = M.FaceNeRF(dim_aud=64, dim_latent=32, dim_expr=76, mlp_mode="bf16").apply(M.init_weights).to(dev)
g = torch.Generator(dev).manual_seed(5)
aud, expr, lat = (torch.randn(d, device=dev, generator=g) for d in (64, 76, 32))
h = hashlib.sha256()
upd = lambda t: h.update(t.detach().contiguous().cpu().numpy().tobytes())
params = [p.detach() for p in net.kernel_params()]
for P in (1, 8769, 35 * 256 + 77):          # 1, 35 and 36 256-row chunks: odd chunk counts leave the peer CTA's last chunk past the end
    x = torch.randn(P, 90, device=dev, generator=g)
    with torch.no_grad():
        upd(net(x, aud, expr, lat))
        cond = ops.fold_cond(net._dims, params, aud, expr, lat)
        raw, acts, mask, n_points = ops.mlp_fwd_train_bf16(net._dims, params, net.packed_weights_emb(net.kernel_params()), cond, x=x)
        upd(raw); upd(acts); upd(mask)
torch.cuda.synchronize()
print("HASH", h.hexdigest())
"""


def test_embedded_bf16_deterministic_and_pair_matches_single_cta(M):
    """A repeated call is bit-identical, and the CTA-pair builds of the embedded-row kernel (inference and activation saving) give the
    same raw, saved images and ReLU masks bit for bit as the single-CTA builds (INERF_MLP_PAIR=0, read once per process)."""
    x = torch.randn(20000, 90, device=DEV, generator=torch.Generator(DEV).manual_seed(1))
    net = G.head_net(M, O.init_face_nerf(3), "bf16")
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


def test_embedded_bf16_packed_cache(M):
    """FaceNeRF keeps the embedded-row blob beside the fused entry's: the same key rules (re-packed after an in-place update) and dropped
    by invalidate_packed()."""
    net = G.head_net(M, O.init_face_nerf(3), "bf16")
    ps = net.kernel_params()
    e = net.packed_weights_emb(ps)
    assert e is net.packed_weights_emb(ps) and e.numel() > net.packed_weights(ps).numel()
    x = torch.randn(300, 90, device=DEV, generator=torch.Generator(DEV).manual_seed(2))
    b = O.synthetic_train_batch(0)
    cond = (b["aud"].to(DEV), b["expr"].to(DEV), b["latent"].to(DEV))
    with torch.no_grad():
        before = net(x, *cond)
        net.rgb_linear.bias.add_(1.0)
        net.pts_linears[3].weight.mul_(1.5)
        after = net(x, *cond)
    assert net.packed_weights_emb(net.kernel_params()) is not e
    assert not torch.equal(before, after)
    net.invalidate_packed()
    assert net._packed_e is None
