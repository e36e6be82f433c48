"""The coarse pass without its colour (ops.render_rays_fused(coarse_rgb=False), what FrameRenderer.render_frame and render_video run): the
density-only build of the bf16 coarse FaceNeRF and the sigma-only coarse compositor must leave every output but rgb0 bit-identical to the
full coarse pass -- maps, depth, last_weight, disp0, acc0, z_std and the merged depths, on both coarse paths of the fused entry, for rays
and generated frames, ragged sizes, the single-CTA build, fp16x2 mode and the non-finite flags."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = ("rgb_map", "disp_map", "acc_map", "_depth_map", "last_weight", "disp0", "acc0", "z_std", "_z_vals")


@pytest.fixture(scope="module")
def M():
    import ideal_nerf_b200 as m
    assert torch.cuda.is_available(), "-m gpu tests need a GPU"
    from ideal_nerf_b200 import _lib
    _lib.check(m.lib().inerf_device_check(), "inerf_device_check")
    return m


def make_net(M, mode, s1=64, s2=128, seed=1234):
    """bench.py's network (xavier init, normalised-density preset) at 450 x 450 in `mode`"""
    from ideal_nerf_b200 import ops, synthetic as S
    cam, fr = S.camera(), S.frame_inputs(0)
    a = M.default_args(dim_aud=64, dim_expr=76, perturb=1.0, mlp_mode=mode, N_samples=s1, N_importance=s2, near=S.NEAR, far=S.FAR)
    net = M.Network(450, 450, cam["focal"], S.NEAR, S.FAR, 1 << 20, None, s1, s2, args=a)
    torch.manual_seed(seed)
    net.apply(M.init_weights)
    net = net.to(DEV).eval()
    rays = ops.get_rays_packed(450, 450, cam["focal"], cam["c2w"].to(DEV), S.NEAR, S.FAR)[::197].contiguous()
    for fn in (net.face_nerf_coarse, net.face_nerf_fine):
        S.normalise_density_(fn, rays, fr["aud"].to(DEV), fr["expr"].to(DEV), fr["latent"].to(DEV))
    return net, fr, cam


@pytest.fixture(scope="module")
def bf16(M):
    return make_net(M, "bf16")


def both_arms(net, fr, cam, perturb, first=0, count=450 * 450, rays=False, aud=None, check_numerics=False):
    """(with rgb0, without rgb0) of one fused call on the same RNG state; rays=True: the packed rays instead of gen"""
    from ideal_nerf_b200 import ops, synthetic as S
    c2w = fr["pose"][:3, :4].to(DEV)
    gen = dict(H=450, W=450, focal=cam["focal"], cx=225., cy=225., near=S.NEAR, far=S.FAR, c2w=c2w, first=first, count=count)
    r = ops.get_rays_range(450, 450, cam["focal"], c2w, S.NEAR, S.FAR, first, count) if rays else None
    bc = fr["bc_rgb"].to(DEV).reshape(-1, 3)[first:first + count].contiguous()
    cond = (fr["aud"].to(DEV) if aud is None else aud, fr["expr"].to(DEV), fr["latent"].to(DEV))
    a = net.args
    out = []
    for coarse_rgb in (True, False):
        ops.seed_rng(7, DEV)
        with torch.no_grad():
            out.append(ops.render_rays_fused(net.face_nerf_coarse, net.face_nerf_fine, cond, cond, bc, a.N_samples, a.N_importance, perturb,
                                             rays=r, gen=None if rays else gen, want_z=True, check_numerics=check_numerics,
                                             coarse_rgb=coarse_rgb))
    torch.cuda.synchronize()
    return out


def assert_bits(full, dens, what):
    assert "rgb0" in full and "rgb0" not in dens, what
    for k in KEYS:
        a, b = full[k].cpu().numpy(), dens[k].cpu().numpy()
        assert a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32)), (what, k)


@pytest.mark.parametrize("perturb", [1.0, 0.0])
@pytest.mark.parametrize("rays", [False, True])
def test_arms_bit_equal(M, bf16, perturb, rays):
    """n = 1, 3 071 and the full 202 500-ray frame, plus the three ragged bands of a 3-way split (the pair build's trailing chunk lies
    past the end); perturb 1 = the fused 64 + 128 compositor + sampler, perturb 0 = composite + inerf_importance_sample"""
    net, fr, cam = bf16
    spans = [(225 * 450 + 3, 1), (1000, 3071), (0, 450 * 450)] + [(k * 67500, 67500) for k in range(3)]
    for first, count in spans:
        full, dens = both_arms(net, fr, cam, perturb, first, count, rays=rays)
        assert_bits(full, dens, (perturb, rays, first, count))
        if count == 450 * 450:
            assert 0.05 < float(full["last_weight"].mean()) < 0.95      # the preset renders a non-trivial image


@pytest.mark.parametrize("perturb", [1.0, 0.0])
def test_second_sample_config(M, perturb):
    """44 + 84 samples: the general coarse path (stand-alone sampler) also when perturb > 0, a coarse compositor with one 64-sample chunk
    not full, and the bf16 kernels at s = 44 / 128"""
    net, fr, cam = make_net(M, "bf16", 44, 84, seed=77)
    for first, count in ((0, 4097), (450 * 450 - 333, 333)):
        full, dens = both_arms(net, fr, cam, perturb, first, count)
        assert_bits(full, dens, (perturb, first, count))


def test_fp16x2_strided_sigma(M):
    """fp16x2 mode has no density-only build: the coarse net runs in full and the compositor reads the sigma lane (stride 4)"""
    net, fr, cam = make_net(M, "fp16x2", seed=5)
    for perturb in (1.0, 0.0):
        full, dens = both_arms(net, fr, cam, perturb, 3000, 5003)
        assert_bits(full, dens, ("fp16x2", perturb))


def test_nonfinite_flags(M, bf16):
    """a NaN audio code: both arms flag the fine maps and the coarse disp0 / acc0 / z_std alike; only the full arm flags rgb0"""
    net, fr, cam = bf16
    bad = fr["aud"].to(DEV).clone()
    bad[3] = float("nan")
    for perturb in (1.0, 0.0):
        full, dens = both_arms(net, fr, cam, perturb, 0, 640, aud=bad, check_numerics=True)
        assert "rgb0" in full["_nonfinite"] and "rgb_map" in full["_nonfinite"], full["_nonfinite"]
        assert set(dens["_nonfinite"]) == set(full["_nonfinite"]) - {"rgb0"}, (perturb, full["_nonfinite"], dens["_nonfinite"])
    full, dens = both_arms(net, fr, cam, 1.0, 0, 640, check_numerics=True)
    assert full["_nonfinite"] == [] and dens["_nonfinite"] == []


def test_render_frame_and_video(M, bf16):
    """render_frame (no rgb0) == render_band(...)['rgb_map'] (with rgb0) bit for bit at perturb 0 and 1; render_video's bytes == to8b of
    the full path's frames"""
    from ideal_nerf_b200 import ops
    from ideal_nerf_b200.frame import FrameRenderer, render_video
    from ideal_nerf_b200 import synthetic as S
    net, fr, cam = bf16
    frs = [S.frame_inputs(i) for i in range(3)]
    lat, bc = frs[0]["latent"].to(DEV), frs[0]["bc_rgb"].to(DEV)
    frames = [(f["pose"].to(DEV), f["aud"].to(DEV), f["expr"].to(DEV)) for f in frs]
    r = FrameRenderer(net)
    with torch.no_grad():
        for perturb in (0.0, 1.0):
            pose, aud, expr = frames[1]
            ops.seed_rng(3, DEV)
            a = r.render_frame(pose, aud, expr, lat, bc, perturb).clone()
            ops.seed_rng(3, DEV)
            ret, _ = r.render_band(pose, aud, expr, lat, bc, perturb)
            assert "rgb0" in ret
            assert np.array_equal(a.cpu().numpy().view(np.uint32), ret["rgb_map"].cpu().numpy().view(np.uint32)), perturb
        vid = render_video(r, frames, lat, bc)
        for i, (pose, aud, expr) in enumerate(frames):
            ret, _ = r.render_band(pose, aud, expr, lat, bc, 0.)
            assert np.array_equal(vid[i].numpy().reshape(-1, 3), ops.to8b(ret["rgb_map"]).cpu().numpy()), i


_SINGLE_CTA = r"""
import sys
sys.path.insert(0, %r)
sys.path.insert(0, %r)
import torch
import ideal_nerf_b200 as M
from test_density_coarse import make_net, both_arms, assert_bits
net, fr, cam = make_net(M, "bf16")
for perturb in (1.0, 0.0):
    for first, count in ((0, 450 * 450), (1000, 3071), (67500, 67500), (7, 1)):
        full, dens = both_arms(net, fr, cam, perturb, first, count)
        assert_bits(full, dens, (perturb, first, count))
print("SINGLE_CTA_OK")
"""


def test_single_cta_build(M):
    """INERF_MLP_PAIR=0 (read once per process, hence a subprocess): the single-CTA density-only build, same bits"""
    env = dict(os.environ, INERF_MLP_PAIR="0")
    r = subprocess.run([sys.executable, "-c", _SINGLE_CTA % (ROOT, os.path.join(ROOT, "tests"))], env=env, capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0 and "SINGLE_CTA_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
