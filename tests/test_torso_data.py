"""GPU tests of the torso stage's data path: DeviceTorsoDataset.sample against its parts (DeviceHeadDataset.sample, ops.get_rays_at and
the sampler with the torso camera in every pose slot, the row lookups), its targets from com_imgs, the multi-GPU bands, a device index
inside a captured CUDA graph, and TorsoTrainStep fed from it, eager against graphed; then the kernel inerf_masked_sse (ops.masked_sse)
against the numpy oracle and evaluate_split on a torso val split."""
import inspect

import numpy as np
import pytest
import torch

from oracle import masked_sse_ref as MS

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def M():
    import ideal_nerf_b200 as m
    assert torch.cuda.is_available(), "-m gpu tests need a GPU"
    m.lib()                                       # raises if the extension is missing: no fallback
    m._lib.check(m.lib().inerf_device_check(), "inerf_device_check")
    return m


def state_now(M):
    s = M.ops.rng_state(DEV).cpu().tolist()
    return s[0], s[1]


@pytest.fixture(scope="module")
def subject(M, tmp_path_factory):
    """A 128 x 96 subject of 12 frames with com_imgs; the torso and head datasets of its train split, and the codes the torso one holds."""
    from ideal_nerf_b200 import synthetic as S
    from ideal_nerf_b200.data import DeviceHeadDataset, DeviceTorsoDataset
    d = str(tmp_path_factory.mktemp("torso_subject"))
    S.write_head_subject(d, 128, 96, n_frames=12, seed=1, torso_rows=10, com_imgs=True)
    args = M.default_args(N_rand=1024, mouth_rays=128, torso_rays=64, sample_rate=0.9, gt_dirs="com_imgs", near=0.3, far=1.4, dim_aud=64)
    g = torch.Generator().manual_seed(3)
    aud, lat = torch.randn(12, 64, generator=g).to(DEV), torch.randn(12, 32, generator=g).to(DEV)
    return d, DeviceTorsoDataset(d, "aud.npy", "train", args, aud, lat), DeviceHeadDataset(d, "aud.npy", "train", args), aud, lat


def sampler(M, ds, f, poses, seed, off):
    """ops.sample_train_pixels on the dataset's tables with the given poses, from Philox state (seed, off)."""
    M.ops.seed_rng(seed, DEV, off)
    idx = torch.tensor(f, dtype=torch.int64, device=DEV)
    return M.ops.sample_train_pixels(idx, ds.budgets, ds.bounds, ds.torso_bits, poses, ds.frames, ds.bc_img, ds.focal, ds.cx, ds.cy,
                                     ds.args.near, ds.args.far, want_coords=True)


def test_sample_against_its_parts(M, subject):
    from ideal_nerf_b200.train import TorsoTrainStep
    _, ds, hd, aud, lat = subject
    keys = [k for k in inspect.signature(TorsoTrainStep.__call__).parameters if k not in ("self", "perturb")]
    torso_poses = ds.torso_pose.expand(len(ds), 3, 4).contiguous()
    assert not torch.equal(ds.poses[5], ds.torso_pose)
    for f, seed, off in ((0, 3, 0), (5, 4, 7), (11, 2 ** 40 + 5, 123)):
        M.ops.seed_rng(seed, DEV, off)
        b = ds.sample(f)
        assert state_now(M) == (seed, off + 1)                                                  # one draw
        assert sorted(b) == sorted(keys)
        M.ops.seed_rng(seed, DEV, off)
        h = hd.sample(f)
        assert torch.equal(b["rays_head"], h["rays"]) and torch.equal(b["target"], h["target"]) and torch.equal(b["bc_rgb"], h["bc_rgb"])
        rays, _, _, coords = sampler(M, ds, f, ds.poses, seed, off)
        assert torch.equal(rays, b["rays_head"])
        assert torch.equal(b["rays_torso"], M.ops.get_rays_at(coords, ds.focal, ds.torso_pose, ds.args.near, ds.args.far, ds.cx, ds.cy))
        rays_t, target_t, _, coords_t = sampler(M, ds, f, torso_poses, seed, off)
        assert torch.equal(b["rays_torso"], rays_t) and torch.equal(coords_t, coords) and torch.equal(target_t, b["target"])
        assert torch.equal(b["rays_torso"], b["rays_head"]) == (f == 0)                          # the torso camera is frame 0's
        assert torch.equal(b["aud_feature"], aud[f]) and torch.equal(b["latent_code"], lat[f])
        assert torch.equal(b["pose"], ds.poses[f]) and b["pose"].shape == (3, 4) and torch.equal(b["expr"], ds.exprs[f])
    batch_rays, target_s, bc_rgb, auds, raw_img, pose, exp, index = ds[3]                        # DeviceHeadDataset's tuple
    assert batch_rays.shape == (2, 1024, 3) and target_s.shape == (1024, 3) and index == 3 and torch.equal(raw_img, ds.frames[3])


def test_targets_come_from_com_imgs(M, subject):
    import os
    from ideal_nerf_b200.data import _imread_rgb
    d, ds, _, _, _ = subject
    for f in (0, 7):
        com = torch.from_numpy(_imread_rgb(os.path.join(d, "com_imgs", f"{f}.jpg"))[:, :, ::-1].copy()).to(DEV)   # BGR, as stored
        head = torch.from_numpy(_imread_rgb(os.path.join(d, "head_imgs", f"{f}.jpg"))[:, :, ::-1].copy()).to(DEV)
        assert torch.equal(ds.frames[f], com) and not torch.equal(ds.frames[f], head)
        M.ops.seed_rng(6, DEV, f)
        b = ds.sample(f)
        _, _, _, coords = sampler(M, ds, f, ds.poses, 6, f)
        assert torch.equal(b["target"], com[coords[:, 0], coords[:, 1]].float() / 255.0)
        torso = b["target"][-ds.budgets[3]:]                                                   # the torso rows are the painted colour
        assert float((torso * 255 - torch.tensor([90., 150., 40.], device=DEV)).abs().median()) <= 10    # BGR; JPEG blurs the edge


def test_bands_concatenate_to_the_batch(M, subject):
    _, ds, _, _, _ = subject
    M.ops.seed_rng(9, DEV, 2)
    whole = ds.sample(4)
    for world in (2, 3):
        parts = []
        for rank in range(world):
            M.ops.seed_rng(9, DEV, 2)
            parts.append(ds.sample(4, rank, world))
        for k in ("rays_head", "rays_torso", "target", "bc_rgb"):
            assert torch.equal(torch.cat([p[k] for p in parts]), whole[k]), (world, k)
        for k in ("aud_feature", "pose", "expr", "latent_code"):
            assert all(torch.equal(p[k], whole[k]) for p in parts), (world, k)


def test_device_index_in_a_captured_graph(M, subject):
    _, ds, _, _, _ = subject
    idx = torch.zeros((), dtype=torch.int64, device=DEV)
    M.ops.seed_rng(77, DEV, 0)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        ds.sample(idx)                                                                          # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = ds.sample(idx)
    prev = None
    for f in (2, 7, 7, 0):
        idx.fill_(f)
        seed, off = state_now(M)
        g.replay()
        torch.cuda.synchronize()
        assert state_now(M) == (seed, off + 1)
        got = {k: v.clone() for k, v in out.items()}
        M.ops.seed_rng(seed, DEV, off)
        want = ds.sample(f)                                                                     # eager, host index, same state
        for k in want:
            assert torch.equal(got[k], want[k]), (f, k)
        if prev is not None:
            assert not torch.equal(prev, got["rays_head"])                                      # consecutive replays draw fresh pixels
        prev = got["rays_head"]


def torso_network(M, ds, a):
    """A TorsoNetwork of the subject's camera, random-init with the normalised-density preset on the subject's rays."""
    from ideal_nerf_b200 import synthetic as S
    torch.manual_seed(1234)
    net = M.TorsoNetwork(ds.H, ds.W, ds.focal, a.near, a.far, 1 << 20, 64, 128, args=a, dim_expr=76)
    net.apply(M.init_weights)
    net = net.to(DEV)
    M.ops.seed_rng(5, DEV, 0)
    b = ds.sample(0)
    for m in (net.face_nerf_coarse, net.face_nerf_fine):
        S.normalise_density_(m, b["rays_head"], b["aud_feature"], b["expr"], b["latent_code"])
    sig = net.torso_signal(b["aud_feature"], b["pose"])
    for m in (net.torso_coarse_nerf, net.torso_fine_nerf):
        S.normalise_density_(m, b["rays_torso"], sig, None, None)
    return net.train()


def test_torso_step_fed_from_sample_graph_matches_eager(M, subject):
    """20 bf16 TorsoTrainStep iterations fed from sample(), eager and as one CUDA graph, each from the same seed (so the same batches):
    the tolerance of test_torso_step_cuda_graph_matches_eager -- losses within 2e-4 relative, parameters within 0.75 of the 20 x lr they
    can have moved."""
    from ideal_nerf_b200.data import DeviceTorsoDataset
    from ideal_nerf_b200.train import TorsoTrainStep
    d, _, _, aud, lat = subject
    a = M.default_args(N_rand=1024, mouth_rays=128, torso_rays=64, sample_rate=0.9, gt_dirs="com_imgs", near=0.5772005200386048,
                       far=1.1772005200386046, dim_aud=64, dim_expr=76, perturb=0., mlp_mode="bf16", lrate=1e-4, lrate_decay=1)
    ds = DeviceTorsoDataset(d, "aud.npy", "train", a, aud, lat)
    sd = {k: v.clone() for k, v in torso_network(M, ds, a).state_dict().items()}
    nets, curves, firsts = [], [], []
    order = np.random.RandomState(0).randint(0, len(ds), 20)
    idx = torch.zeros((), dtype=torch.int64, device=DEV)
    for graph in (False, True):
        net = torso_network(M, ds, a)
        net.load_state_dict(sd)
        step = TorsoTrainStep(net, a, cuda_graph=graph)
        M.ops.seed_rng(11, DEV, 0)
        curve = []
        for k, f in enumerate(order):
            idx.fill_(int(f))
            b = ds.sample(idx)
            if k == 0:
                firsts.append(b["rays_head"].clone())
            out = step(**b)
            curve.append((float(out["img_loss"]), float(out["img_loss0"]), float(out["loss"])))
        assert step.global_step == 20
        if graph:
            assert step._static["graph"] is not None
        nets.append(net)
        curves.append(curve)
    print("eager :", curves[0]); print("graph :", curves[1])
    assert torch.equal(firsts[0], firsts[1])
    assert all(np.isfinite(curves[0]).ravel())
    for x, y in zip(np.ravel(curves[0]), np.ravel(curves[1])):
        assert abs(x - y) <= 2e-4 * max(1.0, abs(x)), (curves[0], curves[1])
    for (k, p), q in zip(nets[0].state_dict().items(), nets[1].state_dict().values()):
        e = float((p.double() - q.double()).abs().max())
        assert e <= 0.75 * 20 * 1e-4, f"parameter {k} after 20 steps: max-abs {e:.3e}"


# ------------------------------------------------------------------------------------------------
# inerf_masked_sse
# ------------------------------------------------------------------------------------------------
def masks_of(H, W, seed):
    """(5, ceil(H*W/32)) uint32 mask words: empty, full, ragged random, torso rows, a single pixel at the end; every padding bit set."""
    from ideal_nerf_b200.data import torso_bits
    rng = np.random.RandomState(seed)
    parses = np.zeros((5, H, W, 3), np.uint8)
    parses[1, ..., 0] = 255
    parses[2][rng.rand(H, W) < 0.3] = (255, 0, 0)
    parses[3, H - max(1, H // 5):, :, 0] = 255
    parses[4, H - 1, W - 1, 0] = 255
    bits = np.stack([torso_bits(p) for p in parses])
    pad = -(H * W) % 32
    bits[:, -1] |= np.uint32(((1 << pad) - 1) << (32 - pad))
    return bits


INDEX = [0, 1, 2, 2, 3, 4, 1, 5, -1, 3]


@pytest.mark.parametrize("H,W", [(11, 11), (37, 101), (450, 450)])
def test_masked_sse_against_oracle(M, H, W):
    rng = np.random.RandomState(H + W)
    gt = rng.randint(0, 256, (5, H, W, 3)).astype(np.uint8)
    pred = rng.randint(0, 256, (len(INDEX), H, W, 3)).astype(np.uint8)
    pred[3] = gt[2]                                                                             # an exact copy
    bits = masks_of(H, W, H * W)
    t = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(DEV)
    sse, npix = M.ops.masked_sse(t(pred), t(gt), t(np.asarray(INDEX, np.int64)), t(bits.view(np.int32)))
    want_sse, want_npix = MS.masked_sse(pred, gt, INDEX, bits)
    assert np.array_equal(sse.cpu().numpy(), want_sse) and np.array_equal(npix.cpu().numpy(), want_npix)
    n = npix.cpu().numpy()
    assert n[0] == 0 and n[1] == H * W and n[5] == 1 and n[7] == 0 and n[8] == 0                # empty, full, one pixel, out of range
    assert sse[3] == 0 and n[3] > 0 and sse[0] == 0 and sse[7] == 0 and sse[8] == 0


def test_masked_sse_graph_replay(M):
    H, W = 37, 101
    rng = np.random.RandomState(1)
    gt = torch.from_numpy(rng.randint(0, 256, (5, H, W, 3)).astype(np.uint8)).to(DEV)
    pred = torch.from_numpy(rng.randint(0, 256, (len(INDEX), H, W, 3)).astype(np.uint8)).to(DEV)
    bits = masks_of(H, W, 2)
    bits_t = torch.from_numpy(bits.view(np.int32)).to(DEV)
    idx = torch.tensor(INDEX, dtype=torch.int64, device=DEV)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        M.ops.masked_sse(pred, gt, idx, bits_t)                                                 # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = M.ops.masked_sse(pred, gt, idx, bits_t)
    for index in (INDEX, [4] * 9 + [5], [2, 3, 4, 0, 1, 2, 3, 4, 0, 1]):
        idx.copy_(torch.tensor(index, dtype=torch.int64))
        g.replay()
        torch.cuda.synchronize()
        want = MS.masked_sse(pred.cpu().numpy(), gt.cpu().numpy(), index, bits)
        assert np.array_equal(out[0].cpu().numpy(), want[0]) and np.array_equal(out[1].cpu().numpy(), want[1]), index


def test_ops_masked_sse_rejects_bad_tensors(M):
    u8 = lambda *s: torch.zeros(s, dtype=torch.uint8, device=DEV)
    idx = torch.zeros(2, dtype=torch.int64, device=DEV)
    bits = torch.zeros(1, 8, dtype=torch.int32, device=DEV)
    with pytest.raises(ValueError, match="bits"):
        M.ops.masked_sse(u8(2, 16, 16, 3), u8(1, 16, 16, 3), idx, bits[:, :7])
    with pytest.raises(ValueError, match="bits"):
        M.ops.masked_sse(u8(2, 16, 16, 3), u8(1, 16, 16, 3), idx, bits.long())
    with pytest.raises(ValueError, match="frame_index"):
        M.ops.masked_sse(u8(2, 16, 16, 3), u8(1, 16, 16, 3), idx[:1], bits)
    with pytest.raises(RuntimeError, match="argument error"):
        M.ops.masked_sse(u8(2, 10, 16, 3), u8(1, 10, 16, 3), idx, bits[:, :5])


# ------------------------------------------------------------------------------------------------
# evaluate_split on a torso val split
# ------------------------------------------------------------------------------------------------
def test_evaluate_split_torso(M, tmp_path):
    from ideal_nerf_b200 import synthetic as S
    from ideal_nerf_b200.data import DeviceHeadDataset, DeviceTorsoDataset
    from ideal_nerf_b200.evaluate import audio_codes, evaluate_split, psnr
    from ideal_nerf_b200.frame import HeadTorsoFrameRenderer
    d = str(tmp_path)
    S.write_head_subject(d, 72, 56, n_frames=2, seed=3, torso_rows=12, val_frames=4, com_imgs=True)
    args = M.default_args(N_rand=0, mouth_rays=0, torso_rays=0, gt_dirs="com_imgs", near=S.NEAR, far=S.FAR, dim_aud=64, dim_expr=76,
                          perturb=0., mlp_mode="bf16")
    hd = DeviceHeadDataset(d, "aud.npy", "val", args)
    torch.manual_seed(12)
    head = M.Network(hd.H, hd.W, hd.focal, S.NEAR, S.FAR, 8192, None, 64, 128, args=args)
    head.apply(M.init_weights)
    codes = audio_codes(head.to(DEV).eval(), hd)
    ds = DeviceTorsoDataset(d, "aud.npy", "val", args, codes)
    torch.manual_seed(13)
    net = M.TorsoNetwork(ds.H, ds.W, ds.focal, S.NEAR, S.FAR, 8192, 64, 128, args=args, dim_expr=76)
    net.apply(M.init_weights)
    net = net.to(DEV).eval()
    latent = torch.ones(32, device=DEV)
    res = evaluate_split(HeadTorsoFrameRenderer(net, ds.torso_pose), ds, latent, codes)
    video, n = res["video"], len(ds)
    gt = ds.frames.cpu().numpy()
    # the torso keys: the oracle on the returned bytes against com_imgs
    sse, npix = MS.masked_sse(video, gt, np.arange(n), ds.torso_bits.cpu().numpy())
    assert np.array_equal(res["sse_torso"], sse) and np.array_equal(res["npix_torso"], npix)
    assert np.array_equal(npix, [12 * 56] * n) and (sse > 0).all()
    assert np.array_equal(res["psnr_torso"], psnr(sse, npix).numpy()) and res["psnr_torso"].shape == (n,)
    assert abs(res["mean_psnr_torso"] - res["psnr_torso"].mean()) < 1e-12
    # the existing keys: inerf_image_metrics on the same bytes
    im = M.ops.image_metrics(torch.from_numpy(video).to(DEV), ds.frames, torch.arange(n, dtype=torch.int64, device=DEV), ds.bounds)
    assert np.array_equal(res["sse"], im["sse"].cpu().numpy()) and np.array_equal(res["npix"], im["npix"].cpu().numpy())
    assert np.abs(res["ssim"] - im["ssim"].cpu().numpy()).max() <= 1e-12
    assert np.array_equal(res["psnr"], psnr(res["sse"], res["npix"]).numpy())
    # a DeviceHeadDataset of the same split: the same scores and video, no torso keys
    plain = evaluate_split(HeadTorsoFrameRenderer(net, ds.torso_pose), hd, latent, codes)
    assert sorted(plain) == sorted(k for k in res if not k.endswith("_torso"))
    assert np.array_equal(plain["video"], video) and np.array_equal(plain["sse"], res["sse"])
