"""Every operand of the bf16 FaceNeRF training kernels, element by element, against float64 (oracle/bf16_operands_ref.py), on ray
batches where every ray has its own origin, near / far and a view direction far from its neighbours' (R.hetero_rays), beside the
synthetic camera's rays.

Bars (each checker is also run on a corrupted copy below and must reject it), with what one B200 measured (all shapes, both ray kinds):
  * saved activations, chain deltas: bit-equal to bf16_rn of the float64 value wherever that value lies farther than the bound
    R.acc_eps(K) * sum|terms| from a bf16 rounding boundary (one truncating fp32 MMA step per 16 of K) -- measured: no decided
    mismatch, at most 1 ulp anywhere except chain deltas with cancelling terms (still within the bound); within bound + 1 ulp everywhere; 1-ulp mismatches at most MAX_MISM of a layer plus two elements -- measured at most 6.0e-4 at
    >= 12 000 points (one element of 256 at P = 1), the bar 2e-3 is ~3x that;
  * ReLU mask bits: the sign of the float64 pre-activation wherever |pre| exceeds the bound;
  * sigma / rgb of raw: within 2^-8 * sum|w h| of the heads applied to the saved h7 / v2 images -- measured at most 0.24 / 0.32 of it;
  * gamma(p) image (fused path): bit-equal to bf16 of the kernel's arithmetic (sincosf once, then angle doubling), whose fp32 value lies
    within 3.1^f * 2^-22 of float64 gamma at octave f (measured 7.5e-8 at octave 0 growing ~3x per octave to 9.7e-4 at octave 9; the
    1-ulp mismatch fraction against float64 gamma grows from 1e-5 to 1.2e-2); gamma(v) image within 1 ulp of float64 (measured:
    bit-equal); both bit-equal to bf16(x) on embedded rows;
  * dW / db: |got - delta^T X| <= c * |delta|^T |X|, c = (8 * tiles per work item + ranges + 8) * 2^-23 -- measured at most 0.14 of
    the bound at 4 tiles per work item and 0.32 at the 3072 x 192 size (185 tiles per work item, c = 1.8e-4);
  * folded biases within 2^-20 of sum |terms| (measured 0.08 of it); conditioning columns of the gradients == db (x) c bit for bit
    (c = [aud | RN(expr / 3) | latent]); d_cond within 2^-18 of sum |W db| (measured 0.014 of it).
The 3072 x 192 run (4 608 tiles, 1 331 of them past 2 GiB) takes ~1 s of float64 checks after 0.01 s of kernels.
"""
import time

import pytest
import torch

from oracle import bf16_operands_ref as R
from oracle import render_oracle as O
import test_gpu_parity as G

pytestmark = pytest.mark.gpu

DEV = G.DEV
M = G.M            # module fixture: the built package on a B200
NETS = {"head": (64, 76, 32), "head79": (64, 79, 32), "torso": (106, 0, 0)}
MAX_MISM = 2e-3
G_SCALE = torch.tensor([1., 1., 1., 0.3])


def _cond(dims, seed):
    g = torch.Generator().manual_seed(seed)
    return tuple(torch.randn(d, generator=g) if d else None for d in dims)


def _model(M, dims, seed, rays):
    """A FaceNeRF of `dims` with the normalised-density preset on `rays`, its conditioning vectors (CPU) and the bf16 module."""
    sd = O.init_face_nerf(seed, *dims)
    cv = _cond(dims, seed)
    sd = O.normalise_density(sd, rays, *cv)
    da, de, dl = dims
    return sd, cv, G.head_net(M, sd, "bf16", dim_aud=da, dim_expr=de, dim_latent=dl)


def _dev(t):
    return None if t is None else t.to(DEV)


def _train_bf16(M, net, cv, d_raw, rays=None, z=None, x=None):
    ops = M.ops
    ps = net.kernel_params()
    params = [p.detach() for p in ps]
    cvd = [_dev(t) for t in cv]
    cond = ops.fold_cond(net._dims, params, *cvd)
    packed = net.packed_weights(ps) if x is None else net.packed_weights_emb(ps)
    raw, acts, mask, P = ops.mlp_fwd_train_bf16(net._dims, params, packed, cond, rays, z, x)
    g, d_cond = ops.mlp_bwd_bf16(net._dims, params, net.packed_weights_bwd(ps), *cvd, acts, mask, d_raw, P, keep_deltas=True)
    return dict(raw=raw, acts=acts, mask=mask, P=P, g=g, d_cond=d_cond, deltas=ops.mlp_bwd_bf16.deltas, cond=cond)


def _d_raw(P, seed):
    gen = torch.Generator(device=DEV).manual_seed(seed)
    return (torch.randn(P, 4, device=DEV, generator=gen) + 0.5) * G_SCALE.to(DEV)      # a mean: deltas of one sign dominate, as in training


def _check_all(M, tag, dims, sd, cv, out, *, rays=None, z=None, s=None, x=None, controls=False):
    """Items 2-4 of the operand checks on one run; prints the measured numbers; with controls, runs each checker on a corrupted copy."""
    ops = M.ops
    P = out["P"]
    T = ((P + 255) // 256) * 2
    A, D = ops.decode_images(out["acts"], T), ops.decode_images(out["deltas"], T)
    mfn = lambda l: R.mask_bits(out["mask"], T, l)
    sdd = {k: v.to(DEV) for k, v in sd.items()}
    net = R.Net64(sdd, dims, *cv)
    emb = x is not None
    fails = []
    view_enc = None if emb else R.dir_ref(rays, s, P)
    f, st = R.check_forward(net, A, mfn, out["raw"], P, view_enc=view_enc, emb=emb, max_mism_frac=MAX_MISM)
    fails += f
    for l in range(11):
        print(f"[{tag}] fwd layer {l:2d}: max {st[l]['max_ulp']} ulp, 1-ulp mismatches {st[l]['mism_frac']:.2e}, undecided "
              f"{st[l]['undecided'] / st[l]['n']:.2e}, decided mismatches {st[l]['dec_mism']}, mask errors {st[l]['mask_bad']}")
    print(f"[{tag}] heads: max error / bound sigma {st['heads']['sigma']:.3f} rgb {st['heads']['rgb']:.3f}")
    if emb:
        fails += R.check_embedded_inputs(A, x, P)
    else:
        pts = (rays[:, None, 0:3] + rays[:, None, 3:6] * z[..., None]).reshape(-1, 3)
        f, pst = R.check_pe_fused(A, pts, P)
        fails += f
        print(f"[{tag}] PE vs float64 gamma per octave: 1-ulp mismatch fraction " + " ".join(f"{v:.1e}" for v in pst["mism"])
              + "; max |fp32 gamma - float64| " + " ".join(f"{v:.1e}" for v in pst["err"]))
        f, dst = R.check_dir_fused(A, view_enc, P)
        fails += f
        print(f"[{tag}] DIR: max {dst['max_ulp']} ulp, 1-ulp mismatches {dst['mism'] / dst['n']:.2e}")
    f, cst = R.check_chain(net, D, mfn, out["d_raw"], P, max_mism_frac=MAX_MISM)
    fails += f
    for l in range(11):
        print(f"[{tag}] chain delta {l:2d}: max {cst[l]['max_ulp']} ulp, 1-ulp mismatches {cst[l]['mism_frac']:.2e}, "
              f"decided mismatches {cst[l]['dec_mism']}")
    acc = R.DwAccum()
    acc.add(net, A, D, P)
    c, per = R.dw_constant(T, torch.cuda.get_device_properties(DEV).multi_processor_count)
    f, wst = R.check_dw(net, out["g"], acc, c)
    fails += f
    print(f"[{tag}] dW / db: c = {c:.2e} ({per} tiles per work item); max error / bound {max(wst.values()):.3e}")
    f, fr = R.check_fold(net, out["cond"])
    fails += f
    f2, cr = R.check_cond_grads(sdd, dims, out["g"], out["d_cond"], *[_dev(t) for t in cv])
    fails += f2
    print(f"[{tag}] fold max error / bound {fr:.3f}; d_cond max error / bound {cr:.3f}")
    assert not fails, "\n".join(fails)
    if controls:
        bad = R.Net64(sdd, dims, *cv, bias_round=R.bf16)
        assert R.check_forward(bad, A, mfn, None, P, view_enc=view_enc, emb=emb, max_mism_frac=MAX_MISM)[0], "bias lo half dropped"
        assert R.check_forward(net, A, mfn, None, P, view_enc=view_enc, emb=emb, max_mism_frac=MAX_MISM, corrupt=("kblock", 3, 32),
                               layers=[3])[0], "one K-block zeroed"
        if not emb:
            assert R.check_dir_fused(A, R.dir_ref(rays.roll(-1, 0), s, P), P)[0], "DIR image of the neighbouring ray"
        row = int(out["g"][2].norm(dim=1).argmax())
        assert R.check_dw(net, out["g"], acc, c, scale_row=(("w", 1), row))[0], "dW row scaled by 1.001"


FUSED = [(s, k) for s in (43, 45, 64, 192) for k in NETS]


@pytest.mark.parametrize("s,net_kind", FUSED)
@pytest.mark.parametrize("rays_kind", ["hetero", "camera"])
def test_bf16_operands_fused(M, s, net_kind, rays_kind):
    """The (rays, z) saving build, chain and dW at s in {43 (a slot touches exactly four rays), 45, 64, 192}, odd chunk counts."""
    n = R.odd_chunk_rays(s, 12000 // s)
    rays = R.hetero_rays(n, s) if rays_kind == "hetero" else O.synthetic_train_batch(0)["rays"][:n]
    dims = NETS[net_kind]
    sd, cv, net = _model(M, dims, 3 + s, rays)
    rays = rays.to(DEV)
    gen = torch.Generator(device=DEV).manual_seed(s)
    z = M.ops.sample_coarse(rays, s, torch.rand(n, s, device=DEV, generator=gen))
    d_raw = _d_raw(n * s, s)
    out = _train_bf16(M, net, cv, d_raw, rays=rays, z=z)
    out["d_raw"] = d_raw
    assert ((n * s + 255) // 256) % 2 == 1
    _check_all(M, f"{rays_kind} {net_kind} s={s} n={n}", dims, sd, cv, out, rays=rays, z=z, s=s,
               controls=(s == 43 and net_kind == "head" and rays_kind == "hetero"))


@pytest.mark.parametrize("P", [1, 127, 128, 129, 257, 12345])
@pytest.mark.parametrize("net_kind", list(NETS))
def test_bf16_operands_embedded(M, P, net_kind):
    """The embedded-row saving build (producer warps write gamma(p) / gamma(v) from x; the extra view K-block), chain and dW."""
    rays = R.hetero_rays(P, 100 + P)
    g = torch.Generator().manual_seed(P)
    zz = rays[:, 6:7] + (rays[:, 7:8] - rays[:, 6:7]) * torch.rand(P, 1, generator=g)
    pts = rays[:, 0:3] + rays[:, 3:6] * zz
    x = torch.cat([O.positional_encoding(pts, 10), O.positional_encoding(rays[:, 8:11], 4)], -1).to(DEV)
    dims = NETS[net_kind]
    sd, cv, net = _model(M, dims, 5, R.hetero_rays(256, 7))
    d_raw = _d_raw(P, P)
    out = _train_bf16(M, net, cv, d_raw, x=x)
    out["d_raw"] = d_raw
    _check_all(M, f"embedded {net_kind} P={P}", dims, sd, cv, out, x=x, controls=(P == 12345 and net_kind == "head"))


@pytest.mark.parametrize("net_kind", list(NETS))
def test_fp32_conditioning_gradients(M, net_kind):
    """The fp32 training path's conditioning columns (same conditioning kernel): bit-equal db (x) c, d_cond against float64."""
    ops = M.ops
    dims = NETS[net_kind]
    rays = R.hetero_rays(61, 9).to(DEV)
    sd, cv, _ = _model(M, dims, 11, rays.cpu())
    da, de, dl = dims
    net = G.head_net(M, sd, "fp32", dim_aud=da, dim_expr=de, dim_latent=dl)
    params = [p.detach() for p in net.kernel_params()]
    cvd = [_dev(t) for t in cv]
    cond = ops.fold_cond(net._dims, params, *cvd)
    z = ops.sample_coarse(rays, 43)
    raw, acts, P = ops.mlp_fwd_train(net._dims, params, cond, rays, z)
    g, d_cond = ops.mlp_bwd(net._dims, params, *cvd, acts, _d_raw(P, 3), P)
    sdd = {k: v.to(DEV) for k, v in sd.items()}
    f, fr = R.check_fold(R.Net64(sdd, dims, *cvd), cond)
    f2, cr = R.check_cond_grads(sdd, dims, g, d_cond, *cvd)
    print(f"[fp32 {net_kind}] fold max error / bound {fr:.3f}; d_cond max error / bound {cr:.3f}")
    assert not f + f2, f + f2


def test_bf16_operands_production_size(M):
    """One training fine pass: 3072 rays x 192 samples (4608 tiles, ~3 GB of saved images, so offsets past 2 GiB), saving forward,
    chain and dW, every element checked; the float64 reference streams over batches of 256 tiles."""
    ops = M.ops
    n, s = 3072, 192
    rays_c = R.hetero_rays(n, 2024)
    dims = NETS["head"]
    sd, cv, net = _model(M, dims, 21, rays_c)
    rays = rays_c.to(DEV)
    t0 = time.time()
    z = ops.sample_coarse(rays, s, torch.rand(n, s, device=DEV, generator=torch.Generator(device=DEV).manual_seed(1)))
    P = n * s
    d_raw = _d_raw(P, 5)
    out = _train_bf16(M, net, cv, d_raw, rays=rays, z=z)
    torch.cuda.synchronize()
    t1 = time.time()
    T = P // 128
    assert out["acts"].numel() >= T * 40 * 16384 > 2 ** 31          # the last 1 331 tiles lie past 2 GiB
    sdd = {k: v.to(DEV) for k, v in sd.items()}
    net64 = R.Net64(sdd, dims, *cv)
    view_enc = R.dir_ref(rays, s, P)
    pts = (rays[:, None, 0:3] + rays[:, None, 3:6] * z[..., None]).reshape(-1, 3)
    raw = out["raw"].reshape(-1, 4)
    acc, fails, worst = R.DwAccum(), [], {}
    B = 256
    for t0_ in range(0, T, B):
        nt = min(B, T - t0_)
        r0, rows = t0_ * 128, nt * 128
        A = ops.decode_images(out["acts"][t0_ * 40 * 16384:], nt)
        D = ops.decode_images(out["deltas"][t0_ * 40 * 16384:], nt)
        msk = out["mask"][t0_ * 76 * 512:(t0_ + nt) * 76 * 512]
        mfn = lambda l: R.mask_bits(msk, nt, l)
        f, st = R.check_forward(net64, A, mfn, raw[r0:r0 + rows], rows, view_enc=view_enc[r0:r0 + rows], max_mism_frac=MAX_MISM)
        fails += [f"tiles {t0_}+: {m}" for m in f]
        f, _ = R.check_pe_fused(A, pts[r0:r0 + rows], rows)
        fails += f
        fails += R.check_dir_fused(A, view_enc[r0:r0 + rows], rows)[0]
        f, cst = R.check_chain(net64, D, mfn, d_raw[r0:r0 + rows], rows, max_mism_frac=MAX_MISM)
        fails += [f"tiles {t0_}+: {m}" for m in f]
        for l in range(11):
            worst[l] = max(worst.get(l, 0.0), st[l]["mism_frac"], cst[l]["mism_frac"])
        acc.add(net64, A, D, rows)
        del A, D
    c, per = R.dw_constant(T, torch.cuda.get_device_properties(DEV).multi_processor_count)
    f, wst = R.check_dw(net64, out["g"], acc, c)
    fails += f
    torch.cuda.synchronize()
    t2 = time.time()
    print(f"[production {n}x{s}] kernels {t1 - t0:.2f} s, float64 checks {t2 - t1:.2f} s; worst 1-ulp mismatch fraction per layer "
          + " ".join(f"{worst[l]:.1e}" for l in range(11)) + f"; dW c = {c:.2e} ({per} tiles per work item), max error / bound "
          f"{max(wst.values()):.3e}")
    assert not fails, "\n".join(fails[:20])


# ------------------------------------------------------------------------------------------------
# the same rays through the rest of the path
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("lindisp", [False, True])
def test_sample_coarse_hetero_bit_exact(M, lindisp):
    from oracle import philox_ref as PH
    n = 777
    rays_c = R.hetero_rays(n, 31)
    rays = rays_c.to(DEV)
    near, far = rays_c[:, 6:7], rays_c[:, 7:8]
    for s in (64, 45, 7):
        assert G.bits_equal(M.ops.sample_coarse(rays, s, None, lindisp), O.stratified_z(near, far, s, n, None, lindisp))
        t = torch.rand(n, s, generator=torch.Generator().manual_seed(s))
        assert G.bits_equal(M.ops.sample_coarse(rays, s, t.to(DEV), lindisp), O.stratified_z(near, far, s, n, t, lindisp))
    st = torch.tensor([77, 3], dtype=torch.int64, device=DEV)
    z = M.ops.sample_coarse_rng(rays, 64, st, lindisp, advance=False)
    u = torch.from_numpy(PH.draws_u01(77, 3, 1, n * 64)).reshape(n, 64)
    assert G.bits_equal(z, O.stratified_z(near, far, 64, n, u, lindisp))


def _dense_fp32(M, rays_c, seed=7):
    b = O.synthetic_train_batch(0)
    sd = O.normalise_density(O.init_face_nerf(seed), rays_c, b["aud"], b["expr"], b["latent"])
    return sd, b


def test_fp32_and_fp16x2_query_hetero(M):
    """The FFMA query against float64 run_network per point (on the fp32 points the kernel forms), and the fp16x2 query against the FFMA
    kernel at the bar of test_fp16x2_raw_matches_fp32_kernel."""
    n, s = 211, 43
    rays_c = R.hetero_rays(n, 41)
    sd, b = _dense_fp32(M, rays_c)
    rays = rays_c.to(DEV)
    aud, expr, lat = b["aud"].to(DEV), b["expr"].to(DEV), b["latent"].to(DEV)
    z = M.ops.sample_coarse(rays, s, torch.rand(n, s, device=DEV, generator=torch.Generator(device=DEV).manual_seed(2)))
    with torch.no_grad():
        r32 = G.head_net(M, sd, "fp32").query(rays, z, aud, expr, lat)
        rx = G.head_net(M, sd, "fp16x2").query(rays, z, aud, expr, lat)
    pts = (rays[:, None, 0:3] + rays[:, None, 3:6] * z[..., None]).cpu()
    ref = O.run_network({k: v.double() for k, v in sd.items()}, pts.double(), rays_c[:, 8:11].double(), b["aud"].double(),
                        b["expr"].double(), b["latent"].double())
    scale = ref.abs().amax((0, 1)).clamp_min(1.0)
    err = ((r32.cpu().double() - ref).abs().amax((0, 1)) / scale)
    print(f"FFMA query vs float64: max-abs / max(1, scale) per channel {err.tolist()}")
    assert bool((err < 5e-5).all()), err.tolist()
    sc = r32.abs().amax((0, 1)).clamp_min(1e-3)
    ex = (rx - r32).abs().amax((0, 1)) / sc
    print(f"fp16x2 vs FFMA: {ex.tolist()}")
    assert bool((ex < 2e-5).all()), ex.tolist()


@pytest.mark.parametrize("n", [47, 203])
def _masked_forward64(sd, x, aud, expr, lat, masks):
    """O.face_nerf_forward in float64 with each ReLU replaced by the fp32 kernel's own decision (masks[l] = its saved activation > 0):
    float64 autograd then differs from the kernel by rounding only, not by the ReLU flips two correct forwards make where a
    pre-activation is within rounding of zero."""
    P = x.shape[0]
    e3 = expr / 3
    first = torch.cat([x[:, :63], aud[None].expand(P, -1), e3[None].expand(P, -1), lat[None].expand(P, -1)], -1)
    h = first
    for i in range(8):
        h = torch.nn.functional.linear(h, sd[f"pts_linears.{i}.weight"], sd[f"pts_linears.{i}.bias"]) * masks[i]
        if i == 4:
            h = torch.cat([first, h], -1)
    sigma = torch.nn.functional.linear(h, sd["alpha_linear.weight"], sd["alpha_linear.bias"])
    h = torch.cat([h, x[:, 63:], e3[None].expand(P, -1)], -1)
    for i in range(3):
        h = torch.nn.functional.linear(h, sd[f"views_linears.{i}.weight"], sd[f"views_linears.{i}.bias"]) * masks[8 + i]
    return torch.cat([torch.nn.functional.linear(h, sd["rgb_linear.weight"], sd["rgb_linear.bias"]), sigma], -1)


@pytest.mark.parametrize("n", [5, 47])
def test_fp32_training_grads_hetero(M, n):
    """fp32 training through (rays, z) at s = 43 (n = 5: 215 points, not a multiple of the 64-row tile) against float64 autograd of the
    reference forward taken through the kernel's own ReLU decisions."""
    s = 43
    rays_c = R.hetero_rays(n, 50 + n)
    sd, b = _dense_fp32(M, rays_c, 9)
    rays = rays_c.to(DEV)
    net = G.head_net(M, sd, "fp32")
    z = M.ops.sample_coarse(rays, s, torch.rand(n, s, device=DEV, generator=torch.Generator(device=DEV).manual_seed(n)))
    gout = torch.randn(n, s, 4, device=DEV, generator=torch.Generator(device=DEV).manual_seed(1))
    aud, expr, lat = (b[k].to(DEV).clone().requires_grad_(True) for k in ("aud", "expr", "latent"))
    (net.query(rays, z, aud, expr, lat) * gout).sum().backward()
    with torch.no_grad():
        params = [p.detach() for p in net.kernel_params()]
        cond = M.ops.fold_cond(net._dims, params, aud.detach(), expr.detach(), lat.detach())
        _, acts, P = M.ops.mlp_fwd_train(net._dims, params, cond, rays, z)
    acts = acts.reshape(-1, 2528)[:P].cpu()          # rows padded to the 64-row tile; 2528 floats a row (csrc/mlp_common.cuh SAVE_W)
    masks = [acts[:, 256 * l:256 * l + 256] > 0 for l in range(8)] + [acts[:, 2048 + 128 * l:2048 + 128 * l + 128] > 0 for l in range(3)]
    pts = (rays[:, None, 0:3] + rays[:, None, 3:6] * z[..., None]).reshape(-1, 3).cpu().double()
    x = torch.cat([O.positional_encoding(pts, 10), O.positional_encoding(rays_c[:, 8:11].double().repeat_interleave(s, 0), 4)], -1)
    sdr = {k: v.double().requires_grad_(True) for k, v in sd.items()}
    cr = [b[k].double().requires_grad_(True) for k in ("aud", "expr", "latent")]
    (_masked_forward64(sdr, x, *cr, masks) * gout.cpu().double().reshape(-1, 4)).sum().backward()
    worst = 0.0
    for name, p in net.named_parameters():
        ref = sdr[name].grad
        if ref is None:
            continue
        e = G.maxabs(p.grad, ref) / max(1.0, float(ref.abs().max()))
        worst = max(worst, e)
        assert e <= 2e-5, (name, e)
    for t, r in zip((aud, expr, lat), cr):
        e = G.maxabs(t.grad, r.grad) / max(1.0, float(r.grad.abs().max()))
        worst = max(worst, e)
        assert e <= 2e-5, e
    print(f"[n={n}] fp32 gradients vs float64 autograd: worst max-abs / max(1, scale) {worst:.2e}")


def test_render_rays_fp32_and_fused_entry_hetero(M):
    """render_rays (fp32 kernels) against the oracle's render_rays at the 1e-3 gate, and the fused render entry bit-equal to the stage
    calls, on rays with their own origins, near / far and directions."""
    from ideal_nerf_b200 import ops
    from ideal_nerf_b200.render import _render_rays_impl
    n = 1003
    rays_c = R.hetero_rays(n, 61)
    b = O.synthetic_train_batch(0)
    c = O.normalise_density(O.init_face_nerf(1), rays_c, b["aud"], b["expr"], b["latent"])
    f = O.normalise_density(O.init_face_nerf(2), rays_c, b["aud"], b["expr"], b["latent"])
    bc = torch.rand(n, 3, generator=torch.Generator().manual_seed(3))
    out = {}
    for mode in ("fp32", "bf16"):
        args = M.default_args(dim_aud=64, dim_expr=76, perturb=0., mlp_mode=mode)
        net = M.Network(450, 450, 1200., O.NEAR, O.FAR, 8192, None, 64, 128, args=args)
        net.face_nerf_coarse.load_state_dict(c)
        net.face_nerf_fine.load_state_dict(f)
        net = net.to(DEV)
        cond = (b["aud"].to(DEV), b["expr"].to(DEV), b["latent"].to(DEV))
        for perturb in (0., 1.):
            res = []
            for fused in (True, False):
                ops.FUSED_RENDER = fused
                ops.seed_rng(5, DEV)
                try:
                    with torch.no_grad():
                        res.append(_render_rays_impl(rays_c.to(DEV), bc.to(DEV), net.face_nerf_coarse, net.face_nerf_fine, *cond, 64, 128,
                                                     perturb=perturb))
                finally:
                    ops.FUSED_RENDER = True
            for k in ("rgb_map", "disp_map", "acc_map", "rgb0", "z_std", "last_weight"):
                assert G.bits_equal(res[0][k], res[1][k]), (mode, perturb, k)
            out[(mode, perturb)] = res[0]
    with torch.no_grad():
        ref = O.render_rays(rays_c, bc, c, f, b["aud"], b["expr"], b["latent"])
    for k in ("rgb_map", "acc_map", "rgb0", "z_std"):
        e = G.maxabs(out[("fp32", 0.)][k], ref[k])
        print(f"render_rays fp32 vs oracle, {k}: max-abs {e:.2e}")
        assert e <= 1e-3, (k, e)
