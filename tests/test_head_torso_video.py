"""GPU tests of the head + torso video path (test_torso.py:516-531): the fused blend-to-uint8 kernel inerf_head_torso_to8b,
frame.HeadTorsoFrameRenderer against TorsoNetwork.forward, the band partition at several GPU counts, render_head_torso_video, and the
config-4 oracle bar through the new renderer.

The networks are built as in test_gpu_parity.test_head_torso_frame_band_config4: four init_face_nerf presets with normalised density,
the torso rays from the frame-0 camera.  Most checks use a reduced 95 x 121 frame: 11 495 rays, which no world size of 2, 3 or 8
divides, so the tail band is ragged."""
import numpy as np
import pytest
import torch

from oracle import render_oracle as O

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
H, W = 95, 121


@pytest.fixture(scope="module")
def M():
    import ideal_nerf_b200 as m
    assert torch.cuda.is_available(), "-m gpu tests need a GPU"
    m.lib()                                       # raises if the extension is missing: no fallback
    m._lib.check(m.lib().inerf_device_check(), "inerf_device_check")
    return m


def bits_equal(a, b):
    a, b = a.detach().cpu().numpy(), b.detach().cpu().numpy()
    return a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a.view(np.uint32) if a.dtype == np.float32 else a,
                                                                        b.view(np.uint32) if b.dtype == np.float32 else b)


def to8b_np(x):
    return (255 * np.clip(x.detach().cpu().numpy(), 0, 1)).astype(np.uint8)


def _pose(i):
    """Head pose of frame i: the synthetic camera turned by 0.02 i rad about y and shifted (frame 0 shifted like the config-4 test)."""
    c2w = O.synthetic_camera()["c2w"].clone()
    c, s = float(np.cos(0.02 * i)), float(np.sin(0.02 * i))
    c2w[:3, :3] = torch.tensor([[c, 0., s], [0., 1., 0.], [-s, 0., c]])
    c2w[:3, 3] += torch.tensor([0.01 + 0.003 * i, -0.02, 0.0])
    return c2w


def _oracle_rays(h, w, focal, pose):
    ro, rd = O.get_rays(h, w, focal, pose, w * .5, h * .5)
    return O.pack_rays(ro.reshape(-1, 3), rd.reshape(-1, 3), O.NEAR, O.FAR)


def _torso_signal(aud, pose):
    et = O.pose_to_euler_trans(pose[None])
    return torch.cat([aud[:64], O.positional_encoding(et[:, :3], 3).squeeze(0), O.positional_encoding(et[:, 3:], 3).squeeze(0)])


def _setup(h, w):
    """State dicts of the four nets (normalised density on this frame's rays) and the frame's host inputs."""
    cam = O.synthetic_camera()
    focal = cam["focal"] * w / 450
    pose, pose0 = _pose(0), cam["c2w"]
    g = torch.Generator().manual_seed(4)
    aud, expr, lat = torch.randn(64, generator=g), torch.randn(79, generator=g), torch.ones(32)
    bc = torch.rand(h * w, 3, generator=g)
    sig = _torso_signal(aud, pose)
    rays_h, rays_t = _oracle_rays(h, w, focal, pose), _oracle_rays(h, w, focal, pose0)
    sds = {"face_nerf_coarse": O.init_face_nerf(21, 64, 79, 32), "face_nerf_fine": O.init_face_nerf(22, 64, 79, 32),
           "torso_coarse_nerf": O.init_face_nerf(23, 106, 0, 0), "torso_fine_nerf": O.init_face_nerf(24, 106, 0, 0)}
    for k in sds:
        head = "face" in k
        sds[k] = O.normalise_density(sds[k], rays_h[::7] if head else rays_t[::7], aud if head else sig, expr if head else None,
                                     lat if head else None)
    return dict(sds=sds, focal=focal, pose=pose, pose0=pose0, aud=aud, expr=expr, lat=lat, bc=bc, sig=sig, rays_h=rays_h, rays_t=rays_t)


@pytest.fixture(scope="module")
def small():
    return _setup(H, W)


def _net(M, s, mode, h=H, w=W):
    args = M.default_args(dim_aud=64, dim_expr=79, perturb=0., mlp_mode=mode)
    net = M.TorsoNetwork(h, w, s["focal"], O.NEAR, O.FAR, 1 << 20, 64, 128, args=args)
    for k, sd in s["sds"].items():
        getattr(net, k).load_state_dict(sd)
    return net.to(DEV).eval()


def _dev(s):
    return {k: s[k].to(DEV) for k in ("pose", "pose0", "aud", "expr", "lat", "bc")}


# ------------------------------------------------------------------------------------------------
# the kernel
# ------------------------------------------------------------------------------------------------
def _kernel_inputs(n, gen):
    head = torch.rand(n, 3, generator=gen) * 1.6 - 0.3                  # below 0 and above 1
    lw = torch.rand(n, generator=gen)
    fg = torch.rand(n, 3, generator=gen) * 1.6 - 0.3
    k = min(n, 6)
    lw[:k] = torch.tensor([1., 0., 1., 0.5, 1., 0.25])[:k]
    head[:k, 0] = torch.tensor([0.5, 0.7, 1., 0.5, 0., 2.])[:k]        # ray 0: 0.5 * 1 + 0.5 = exactly 1; ray 2: 1 * 1 + 0 = 1
    fg[:k, 0] = torch.tensor([0.5, 1., 0., 0.75, 1., -0.5])[:k]         # ray 1: exactly 1 from fg alone; ray 5: 2 * 0.25 - 0.5 = 0
    return head, lw, fg


def _view(flat_len, off, dtype):
    """A contiguous tensor of flat_len elements starting `off` elements into a fresh allocation (off > 0: not 16-byte aligned)."""
    return torch.empty(flat_len + off, dtype=dtype, device=DEV)[off:]


@pytest.mark.parametrize("n", [1001, 7, 1, 4096])
def test_head_torso_to8b_kernel_exact(M, n):
    """out_u8 == to8b(head_torso_blend(...)) and out_rgb == head_torso_blend(...) bit for bit, for aligned and offset pointers (the
    vector path and the scalar path), against both the two-kernel path and numpy."""
    ops = M.ops
    gen = torch.Generator().manual_seed(n)
    head, lw, fg = _kernel_inputs(n, gen)
    want_rgb = ops.head_torso_blend(head.to(DEV), lw.to(DEV), fg.to(DEV))
    want_u8 = ops.to8b(want_rgb)
    rgb_np = head.numpy() * lw.numpy()[:, None] + fg.numpy()           # float32: product rounded, then the sum: no FMA
    assert bits_equal(want_rgb.cpu(), torch.from_numpy(rgb_np))
    assert np.array_equal(want_u8.cpu().numpy(), to8b_np(torch.from_numpy(rgb_np)))
    if n >= 6:
        assert {0, 255} <= set(np.unique(want_u8.cpu().numpy()).tolist())
    for off_in, off_lw, off_u8, off_rgb in ((0, 0, 0, 0), (1, 0, 0, 0), (0, 0, 1, 0), (0, 0, 0, 3), (2, 1, 3, 1), (3, 3, 2, 2)):
        a, b, c = _view(3 * n, off_in, torch.float32), _view(n, off_lw, torch.float32), _view(3 * n, off_in, torch.float32)
        a.copy_(head.reshape(-1)); b.copy_(lw); c.copy_(fg.reshape(-1))
        out, rgb = _view(3 * n, off_u8, torch.uint8), _view(3 * n, off_rgb, torch.float32)
        r = ops.head_torso_to8b(a.view(n, 3), b, c.view(n, 3), out=out.view(n, 3), out_rgb=rgb)
        assert r.data_ptr() == out.data_ptr()
        assert bits_equal(out.view(n, 3), want_u8), (off_in, off_lw, off_u8, off_rgb)
        assert bits_equal(rgb.view(n, 3), want_rgb), (off_in, off_lw, off_u8, off_rgb)
        assert bits_equal(ops.head_torso_to8b(a.view(n, 3), b, c.view(n, 3)), want_u8)          # out_rgb = NULL
    assert ops.head_torso_to8b(torch.zeros(0, 3, device=DEV), torch.zeros(0, device=DEV), torch.zeros(0, 3, device=DEV)).shape == (0, 3)


# ------------------------------------------------------------------------------------------------
# the frame renderer
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_render_frame_equals_torso_network_forward(M, small, mode):
    """world = 1, perturb = 0: HeadTorsoFrameRenderer.render_frame == TorsoNetwork.forward(rays_head(pose), rays_torso(torso_pose))[0]
    bit for bit, and render_band's rgb0 == forward's rgb_com0."""
    from ideal_nerf_b200.frame import HeadTorsoFrameRenderer
    net, d = _net(M, small, mode), _dev(small)
    with torch.no_grad():
        r = HeadTorsoFrameRenderer(net, d["pose0"])
        rgb = r.render_frame(d["pose"], d["aud"], d["expr"], d["lat"], d["bc"])
        ret, span = r.render_band(d["pose"], d["aud"], d["expr"], d["lat"], d["bc"])
        rays_h = M.ops.get_rays_packed(H, W, small["focal"], d["pose"], O.NEAR, O.FAR)
        rays_t = M.ops.get_rays_packed(H, W, small["focal"], d["pose0"], O.NEAR, O.FAR)
        want, want0 = net(rays_h, rays_t, d["bc"], d["aud"], d["pose"], d["expr"], d["lat"], perturb=0.)
    assert span == (0, H * W) and rgb.shape == (H * W, 3) and bool(torch.isfinite(rgb).all())
    lw = float(ret["torso"]["last_weight"].mean())
    assert 0.02 < lw < 0.98, f"torso preset must be neither empty nor opaque (mean last_weight {lw})"
    assert bits_equal(rgb, want)
    assert bits_equal(ret["rgb_map"], want)
    assert bits_equal(ret["rgb0"], want0)


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_bands_concatenate_to_the_world1_frame(M, small, mode):
    """Every rank's render_band (and render_band_u8), rendered on the one GPU and concatenated, == the world = 1 frame bit for bit, for
    world 2, 3 and 8 (ragged tail bands): the single-GPU stand-in for the multi-GPU video checksum."""
    from ideal_nerf_b200.frame import HeadTorsoFrameRenderer, band
    net, d = _net(M, small, mode), _dev(small)
    args = (d["pose"], d["aud"], d["expr"], d["lat"], d["bc"])
    with torch.no_grad():
        full = HeadTorsoFrameRenderer(net, d["pose0"]).render_frame(*args)
        full8 = to8b_np(full)
        for world in (2, 3, 8):
            parts, parts8 = [], []
            for rank in range(world):
                r = HeadTorsoFrameRenderer(net, d["pose0"], rank=rank, world=world)
                ret, span = r.render_band(*args)
                assert span == band(H * W, rank, world)
                parts.append(ret["rgb_map"])
                u8, span8 = r.render_band_u8(*args)
                assert span8 == span and u8.dtype == torch.uint8
                parts8.append(u8.cpu().numpy())
            assert bits_equal(torch.cat(parts), full), world
            assert np.array_equal(np.concatenate(parts8), full8), world


def test_render_head_torso_video(M, small):
    """render_head_torso_video on 4 frames, each with its own pose, aud and expr, == to8b of the per-frame render_frame output exactly;
    the fp32 driver render_video on the same renderer gives the same bytes."""
    from ideal_nerf_b200.frame import HeadTorsoFrameRenderer, render_head_torso_video, render_video
    net, d = _net(M, small, "bf16"), _dev(small)
    gen = torch.Generator().manual_seed(11)
    frames = [(_pose(i).to(DEV), (small["aud"] + 0.3 * torch.randn(64, generator=gen)).to(DEV), torch.randn(79, generator=gen).to(DEV))
              for i in range(4)]
    with torch.no_grad():
        r = HeadTorsoFrameRenderer(net, d["pose0"])
        vid = render_head_torso_video(r, frames, d["lat"], d["bc"])
        assert vid.shape == (4, H, W, 3) and vid.dtype == torch.uint8 and vid.is_pinned()
        per_frame = [to8b_np(r.render_frame(pose, aud, expr, d["lat"], d["bc"])) for pose, aud, expr in frames]
        vid32 = render_video(r, frames, d["lat"], d["bc"])
    for i in range(4):
        assert np.array_equal(vid[i].numpy().reshape(-1, 3), per_frame[i]), i
    assert np.array_equal(vid.numpy(), vid32.numpy())
    assert not np.array_equal(per_frame[0], per_frame[3]), "frames with different inputs must differ"


def test_frame_450_matches_oracle_config4(M):
    """The config-4 bar through the new renderer: a 450 x 450 composited frame in fp32 mode, three image rows against the CPU oracle's
    head + torso composite, <= 1e-3 max-abs."""
    from ideal_nerf_b200.frame import HeadTorsoFrameRenderer
    s = _setup(450, 450)
    net, d = _net(M, s, "fp32", 450, 450), _dev(s)
    rows = slice(210 * 450, 213 * 450)
    with torch.no_grad():
        rgb = HeadTorsoFrameRenderer(net, d["pose0"]).render_frame(d["pose"], d["aud"], d["expr"], d["lat"], d["bc"])
    assert rgb.shape == (202500, 3) and bool(torch.isfinite(rgb).all())
    sd = s["sds"]
    h = O.render_rays(s["rays_h"][rows], s["bc"][rows], sd["face_nerf_coarse"], sd["face_nerf_fine"], s["aud"], s["expr"], s["lat"],
                      with_fg=True)
    t = O.render_rays(s["rays_t"][rows], s["bc"][rows], sd["torso_coarse_nerf"], sd["torso_fine_nerf"], s["sig"], None, None, with_fg=True)
    assert 0.02 < float(t["last_weight"].mean()) < 0.98, "torso preset must be neither empty nor opaque"
    want = O.head_torso_blend(h["rgb_map"], t["last_weight"], t["rgb_map_fg"])
    err = float((rgb[rows].cpu().double() - want.double()).abs().max())
    assert err <= 1e-3, f"config 4 frame rows through HeadTorsoFrameRenderer: max-abs {err:.3e}"
