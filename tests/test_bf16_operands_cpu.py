"""CPU twin of test_bf16_operands.py: the ray generator's spread, the float64 reference helpers against the torch emulation of the bf16
kernels (test_gpu_parity._emulated_bf16_forward), and every checker with its negative control on images built on the CPU in the
kernels' own layout."""
import pytest
import torch

from oracle import bf16_operands_ref as R
from oracle import render_oracle as O
import test_gpu_parity as G

DIMS = {"head": (64, 76, 32), "head79": (64, 79, 32), "torso": (106, 0, 0)}


def test_hetero_rays_spread():
    rays = R.hetero_rays(3072, 1)
    assert rays.shape == (3072, 11) and rays.dtype == torch.float32
    ang = R.adjacent_view_angles(rays)
    assert float(ang.min()) >= 0.6, float(ang.min())                           # adjacent view directions differ by > 34 degrees
    assert float(rays[:, 10].max()) <= 0.0                                     # one hemisphere
    norm = rays[:, 3:6].norm(dim=-1)
    assert 0.5 - 1e-6 <= float(norm.min()) and float(norm.max()) <= 2.0 + 1e-6
    assert bool((rays[:, 7] > rays[:, 6]).all()) and rays[:, 6].unique().numel() == 3072 and rays[:, 0].unique().numel() == 3072
    assert torch.equal(rays[:, 8:11], O.pack_rays(rays[:, 0:3], rays[:, 3:6], 0., 1.)[:, 8:11])
    assert torch.equal(rays, R.hetero_rays(3072, 1))
    for s in (43, 45, 64, 192):
        n = R.odd_chunk_rays(s, 12000 // s)
        assert ((n * s + 255) // 256) % 2 == 1 and (n * s) % 256 != 0


def _emulate(sd, dims, cv, pe, view_enc, d_raw):
    """The bf16 kernels' arithmetic in fp32 torch on the CPU, keeping what they save: activation images (bf16 values), masks (pre >= 0),
    the gamma images, delta images, as {image: (P, 64) columns} and {layer: (P, width) bool}."""
    da, de, dl = dims
    C = da + de + dl
    c = R.cond_vector(*cv)
    W = lambda k: sd[k]
    bf = G._bf
    imgs, masks, pres = {R.IMG_PE: torch.cat([bf(pe), torch.zeros(pe.shape[0], 1)], 1)}, {}, {}
    x = bf(pe)
    h = None
    for l in range(11):
        if l < 8:
            w, b = W(f"pts_linears.{l}.weight"), W(f"pts_linears.{l}.bias")
            if l == 0:
                pre = x @ bf(w[:, :63]).T + (w[:, 63:] @ c + b)
            elif l == 5:
                pre = x @ bf(w[:, :63]).T + h @ bf(w[:, 63 + C:]).T + (w[:, 63:63 + C] @ c + b)
            else:
                pre = h @ bf(w).T + b
        else:
            w, b = W(f"views_linears.{l - 8}.weight"), W(f"views_linears.{l - 8}.bias")
            if l == 8:
                pre = h @ bf(w[:, :256]).T + view_enc.float() @ w[:, 256:283].T + (w[:, 283:] @ c[da:da + de] + b)
            else:
                pre = h @ bf(w).T + b
        pres[l] = pre
        masks[l] = pre >= 0
        h = bf(torch.relu(pre))
        first, n = R.lay_img(l)
        for k in range(n):
            imgs[first + k] = h[:, 64 * k:64 * k + 64]
    imgs[R.IMG_DIR] = torch.cat([bf(view_enc.float()), torch.zeros(pe.shape[0], 37)], 1)
    deltas = {R.IMG_DOUT: torch.cat([bf(d_raw), torch.zeros(d_raw.shape[0], 60)], 1)}
    d = bf(torch.where(masks[10], d_raw[:, :3] @ W("rgb_linear.weight"), torch.zeros(())))
    dl_ = {10: d}
    for l in range(10, 0, -1):
        w = W(f"pts_linears.{l}.weight") if l < 8 else W(f"views_linears.{l - 8}.weight")
        wa = w[:, :256] if l == 8 else (w[:, 63 + C:] if l == 5 else w)
        dh = d @ bf(wa)
        if l == 8:
            dh = dh + d_raw[:, 3:4] * W("alpha_linear.weight")
        d = bf(torch.where(masks[l - 1], dh, torch.zeros(())))
        dl_[l - 1] = d
    for l, v in dl_.items():
        first, n = R.lay_img(l)
        for k in range(n):
            deltas[first + k] = v[:, 64 * k:64 * k + 64]
    return imgs, masks, deltas, pres


def _pad(cols, T):
    return {i: torch.cat([v, torch.zeros(T * 128 - v.shape[0], 64)], 0) for i, v in cols.items()}


def _setup(dims, P=300, seed=3, dense=True):
    rays = R.hetero_rays(P, seed)
    g = torch.Generator().manual_seed(seed)
    cv = tuple(torch.randn(d, generator=g) if d else None for d in dims)
    sd = O.init_face_nerf(seed, *dims)
    if dense:
        sd = O.normalise_density(sd, rays, *cv)
    z = rays[:, 6:7] + (rays[:, 7:8] - rays[:, 6:7]) * torch.rand(P, 1, generator=g)
    pts = rays[:, 0:3] + rays[:, 3:6] * z
    pe = R.pe_doubling(pts)                                    # the fused kernel's gamma(p) arithmetic
    view_enc = O.positional_encoding(rays[:, 8:11].double(), 4)
    d_raw = (torch.randn(P, 4, generator=g) + 0.5) * torch.tensor([1., 1., 1., 0.3])
    T = ((P + 255) // 256) * 2
    imgs, masks, deltas, pres = _emulate(sd, dims, cv, pe, view_enc, d_raw)
    from ideal_nerf_b200 import ops
    A = ops.decode_images(R.encode_images(_pad(imgs, T), T), T)
    D = ops.decode_images(R.encode_images(_pad(deltas, T), T), T)
    mask = R.encode_mask({l: torch.cat([m, torch.zeros(T * 128 - P, m.shape[1], dtype=torch.bool)]) for l, m in masks.items()}, T)
    return dict(rays=rays, sd=sd, cv=cv, pe=pe, pts=pts, view_enc=view_enc, d_raw=d_raw, T=T, A=A, D=D, mask=mask, masks=masks,
                pres=pres, P=P)


def test_image_and_mask_encoding_round_trip():
    T, P = 4, 512
    v = torch.randn(T * 128, 64)
    A = __import__("ideal_nerf_b200").ops.decode_images(R.encode_images({5: v}, T), T)
    assert torch.equal(R.img_cols(A, 5, 1), G._bf(v)) and float(A[:, 4].abs().max()) == 0
    bits = torch.rand(T * 128, 256) < 0.5
    assert torch.equal(R.mask_bits(R.encode_mask({3: bits}, T), T, 3), bits)


@pytest.mark.parametrize("net_kind", list(DIMS))
def test_reference_agrees_with_emulation_and_checkers_pass(net_kind):
    """The float64 reference of each layer, fed the emulation's images, reproduces the emulation's pre-activations to the bound, every
    checker passes the emulated images, and the emulation's raw equals test_gpu_parity._emulated_bf16_forward."""
    dims = DIMS[net_kind]
    e = _setup(dims)
    P, A, D = e["P"], e["A"], e["D"]
    net = R.Net64(e["sd"], dims, *e["cv"])
    for l in range(11):
        pre, bound = R.forward_ref(net, l, R.layer_input(net, l, A, P, dir_img=False), e["view_enc"])
        assert bool(((pre - e["pres"][l].double()).abs() <= bound).all()), l
    mfn = lambda l: R.mask_bits(e["mask"], e["T"], l)
    f, st = R.check_forward(net, A, mfn, None, P, view_enc=e["view_enc"], max_mism_frac=1e-2)
    assert not f, f
    assert not R.check_pe_fused(A, e["pts"], P)[0]
    assert not R.check_dir_fused(A, e["view_enc"], P)[0]
    f, _ = R.check_chain(net, D, mfn, e["d_raw"], P, max_mism_frac=1e-2)
    assert not f, f
    if dims[1]:
        # random-init weights and the bar of test_embedded_bf16_vs_emulation: the two emulations fold the conditioning in a different fp32
        # order, so a pre-activation on a bf16 rounding boundary can round differently (with the density preset that moves sigma ~100x more)
        e = _setup(dims, dense=False)
        ref = G._emulated_bf16_forward(e["sd"], e["pe"], e["view_enc"].float(), *e["cv"])
        W = e["sd"]
        sig = torch.relu(e["pres"][7]) @ W["alpha_linear.weight"].T + W["alpha_linear.bias"]
        rgb = torch.relu(e["pres"][10]) @ W["rgb_linear.weight"].T + W["rgb_linear.bias"]
        G.close(torch.cat([rgb, sig], -1), ref, 6e-3 * max(1.0, float(ref.abs().max())), "emulation vs _emulated_bf16_forward")


def test_negative_controls_are_rejected():
    """Each corruption of the issue's list makes its checker fail on the CPU-built images, which pass uncorrupted."""
    dims = DIMS["head"]
    e = _setup(dims, P=2000)
    P, A, D = e["P"], e["A"], e["D"]
    net = R.Net64(e["sd"], dims, *e["cv"])
    mfn = lambda l: R.mask_bits(e["mask"], e["T"], l)
    kw = dict(view_enc=e["view_enc"], max_mism_frac=1e-2)
    assert not R.check_forward(net, A, mfn, None, P, **kw)[0]
    assert R.check_forward(R.Net64(e["sd"], dims, *e["cv"], bias_round=R.bf16), A, mfn, None, P, **kw)[0]
    assert R.check_forward(net, A, mfn, None, P, corrupt=("kblock", 3, 32), layers=[3], **kw)[0]
    assert R.check_dir_fused(A, e["view_enc"].roll(-1, 0), P)[0]
    acc = R.DwAccum()
    acc.add(net, A, D, P)
    g = [None] * 26
    for key, ref in acc.ref.items():                                # gradients as the kernel would give them: fp32 of the exact sums
        kind, l = key
        idx = {"alpha": 22, "rgb": 24}.get(l, 2 * l if isinstance(l, int) and l < 8 else (16 + 2 * (l - 8) if isinstance(l, int) else 0))
        if kind == "b":
            g[idx + 1] = ref.float()
    C = sum(dims)
    g[0] = torch.cat([acc.ref[("w", 0)].float(), torch.zeros(256, C)], 1)
    g[10] = torch.cat([acc.ref[("w", 5)][:, :63].float(), torch.zeros(256, C), acc.ref[("w", 5)][:, 63:].float()], 1)
    g[16] = torch.cat([acc.ref[("w", 8)].float(), torch.zeros(128, dims[1])], 1)
    for l in (1, 2, 3, 4, 6, 7, 9, 10):
        g[2 * l if l < 8 else 16 + 2 * (l - 8)] = acc.ref[("w", l)].float()
    g[22], g[24] = acc.ref[("w", "alpha")].float(), acc.ref[("w", "rgb")].float()
    c, _ = R.dw_constant(e["T"])
    assert not R.check_dw(net, g, acc, c)[0]
    row = int(g[2].norm(dim=1).argmax())
    assert R.check_dw(net, g, acc, c, scale_row=(("w", 1), row))[0]
