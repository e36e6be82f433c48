"""GPU checks of the training-batch pixel sampler (inerf_sample_train_pixels, ops.sample_train_pixels, data.DeviceHeadDataset): the drawn
coordinates bit for bit against the numpy oracle of the contract, the batch contents against HeadDataset's, the multi-GPU bands, replay
inside a CUDA graph, and a short training run fed from it."""
import numpy as np
import pytest
import torch

from oracle import pixel_sampler_ref as PS

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def M():
    import ideal_nerf_b200 as m
    m.build()
    return m


def state_now(M):
    s = M.ops.rng_state(DEV).cpu().tolist()
    return s[0], s[1]


def tables(M, H, W, n_frames, seed, mouth_boxes, rect, torso_rows):
    """Device tables of n_frames random frames (bounds from data.region_bounds of the given landmark boxes)."""
    from ideal_nerf_b200.data import region_bounds, torso_bits
    rng = np.random.RandomState(seed)
    bounds, bits, masks = [], [], []
    for f in range(n_frames):
        lo, hi = mouth_boxes[f % len(mouth_boxes)]
        lm = rng.rand(68, 2) * 5 + 10
        lm[48:] = lo + rng.rand(20, 2) * (np.array(hi) - lo)
        bounds.append(region_bounds(np.array(rect, np.int32), lm, H, W))
        parse = np.zeros((H, W, 3), np.uint8)
        parse[H - torso_rows:, :, 0] = 255
        bits.append(torso_bits(parse))
        masks.append(parse[:, :, 0] == 255)
    t = dict(bounds=torch.from_numpy(np.stack(bounds)).to(DEV), torso_bits=torch.from_numpy(np.stack(bits).view(np.int32)).to(DEV),
             poses=torch.from_numpy(rng.randn(n_frames, 3, 4).astype(np.float32)).to(DEV),
             frames=torch.from_numpy(rng.randint(0, 256, (n_frames, H, W, 3)).astype(np.uint8)).to(DEV),
             bc_img=torch.from_numpy(rng.rand(H, W, 3).astype(np.float32)).to(DEV))
    return t, np.stack(bounds), masks


def draw(M, t, f, budgets, H, W, **kw):
    idx = torch.tensor(f, dtype=torch.int64, device=DEV)
    return M.ops.sample_train_pixels(idx, budgets, t["bounds"], t["torso_bits"], t["poses"], t["frames"], t["bc_img"], 1200. * W / 450,
                                     W / 2, H / 2, 0.5, 1.2, want_coords=True, **kw)


CASES = {
    # 450^2, the reference's budgets, with and without torso rays; several frames and offsets
    "450_torso0": (450, 450, (2432, 128, 512, 0), [((230., 185.), (270., 215.))], [56, 56, 281, 337], 40),
    "450_torso": (450, 450, (2000, 300, 512, 260), [((230., 185.), (270., 215.)), ((100.5, 300.5), (140., 330.))], [56, 56, 281, 337], 40),
    # ragged frame (H*W = 1665, not a multiple of 32); the mouth box sticks out of the rect and out of the frame
    # (torso = one row of 37 pixels: a budget equal to the region's size)
    "ragged_mouth_outside": (45, 37, (300, 200, 150, 37), [((30., 40.), (38., 45.))], [5, 4, 20, 20], 1),
    # rect and torso budgets equal to their regions' sizes, no mouth
    "rect_full": (45, 37, (0, 0, 0, 0), [((-30., -30.), (-25., -25.))], [0, 0, 9, 9], 2),
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_coordinates_bit_exact_against_oracle(M, case):
    H, W, budgets, boxes, rect, torso_rows = CASES[case]
    t, bounds, masks = tables(M, H, W, 3, 11, boxes, rect, torso_rows)
    if case == "rect_full":
        sizes = PS.region_masks(bounds[0], masks[0], H, W).sum(1)
        budgets = (int(sizes[0]), 100, 0, int(sizes[3]))
    for f, (seed, off) in ((0, (5, 0)), (1, (5, 3)), (2, (2 ** 40 + 7, 123456))):
        M.ops.seed_rng(seed, DEV, off)
        rays, target, bc, coords = draw(M, t, f, budgets, H, W)
        assert state_now(M) == (seed, off + 1)                                      # advanced by one
        want = PS.select(seed, off, budgets, bounds[f], masks[f], H, W)
        got = coords.cpu().numpy()
        assert np.array_equal(got[:, 0] * W + got[:, 1], want), (case, f)
        sel = coords
        ref = M.ops.get_rays_at(sel, 1200. * W / 450, t["poses"][f], 0.5, 1.2, W / 2, H / 2)
        assert torch.equal(rays, ref)
        assert torch.equal(target, t["frames"][f][sel[:, 0], sel[:, 1]].float() / 255.0)
        assert torch.equal(bc, t["bc_img"][sel[:, 0], sel[:, 1]])


@pytest.fixture(scope="module")
def subject(M, tmp_path_factory):
    from ideal_nerf_b200 import synthetic as S
    from ideal_nerf_b200.data import DeviceHeadDataset, HeadDataset
    d = str(tmp_path_factory.mktemp("subject"))
    S.write_head_subject(d, 128, 96, n_frames=12, seed=1, torso_rows=10)
    args = M.default_args(N_rand=1024, mouth_rays=128, torso_rays=64, sample_rate=0.9, gt_dirs="head_imgs", near=0.3, far=1.4)
    return HeadDataset(d, "aud.npy", "train", args), DeviceHeadDataset(d, "aud.npy", "train", args)


def test_batch_contents_match_head_dataset(M, subject):
    from ideal_nerf_b200.data import _imread_rgb, torso_bits
    hd, ds = subject
    a = ds.args
    H, W = ds.H, ds.W
    for f, seed in ((0, 3), (5, 4), (11, 5)):
        M.ops.seed_rng(seed, DEV, 0)
        b = ds.sample(f)
        bits = torso_bits(_imread_rgb(hd.all_parse_imgs[f]))
        torso = ((bits[np.arange(H * W) >> 5] >> (np.arange(H * W) & 31).astype(np.uint32)) & 1).astype(bool)
        p = PS.select(seed, 0, ds.budgets, ds.bounds[f].cpu().numpy(), torso, H, W)
        sel = torch.from_numpy(np.stack([p // W, p % W], 1)).to(DEV)
        # HeadDataset.__getitem__'s tensors at the same pixels
        raw_img = torch.tensor(_imread_rgb(hd.all_imgs[f])[:, :, ::-1].copy())
        target_s = (raw_img.to(DEV).float() / 255.0)[sel[:, 0], sel[:, 1]]
        pose = torch.tensor(hd.all_poses[f][:3, :4], dtype=torch.float32, device=DEV)
        r01 = M.ops.get_rays_at(sel, hd.focal, pose, 0.0, 1.0, hd.cx, hd.cy)
        assert torch.equal(b["rays"], M.ops.pack_rays(r01[:, 0:3], r01[:, 3:6], a.near, a.far))
        assert torch.equal(b["rays"], M.ops.get_rays_at(sel, hd.focal, pose, a.near, a.far, hd.cx, hd.cy))
        assert torch.equal(b["target"], target_s)
        assert torch.equal(b["bc_rgb"], hd.background_img[sel[:, 0], sel[:, 1]].float())
        assert torch.equal(b["pose"], pose)
        assert torch.equal(b["expr"].cpu(), torch.tensor(hd.all_exprs[f], dtype=torch.float32))
    net = M.Network(H, W, hd.focal, a.near, a.far, 8192, None, 64, 128, args=M.default_args(dim_aud=64, dim_expr=76))
    for f in (0, 1, 6, 10, 11):                                                            # both padded ends and the interior
        want = net.audio_window(hd.auds, f, len(hd))
        got = ds.sample(torch.tensor(f, device=DEV))["aud_window"]
        assert got.shape == want.shape and torch.equal(got, want), f
    batch_rays, target_s, bc_rgb, auds, raw_img, pose, exp, index = ds[3]
    assert batch_rays.shape == (2, 1024, 3) and target_s.shape == (1024, 3) and bc_rgb.shape == (1024, 3) and index == 3
    assert torch.equal(raw_img.cpu(), torch.tensor(_imread_rgb(hd.all_imgs[3])[:, :, ::-1].copy())) and exp.shape == (76,)


def test_bands_concatenate_to_the_batch(M, subject):
    _, ds = subject
    M.ops.seed_rng(9, DEV, 2)
    whole = ds.sample(4)
    for world in (2, 3):
        parts = []
        for rank in range(world):
            M.ops.seed_rng(9, DEV, 2)
            parts.append(ds.sample(4, rank, world))
        for k in ("rays", "target", "bc_rgb"):
            assert torch.equal(torch.cat([p[k] for p in parts]), whole[k]), (world, k)


def test_cuda_graph_replay_draws_fresh_batches(M, subject):
    hd, ds = subject
    a = ds.args
    idx = torch.zeros((), dtype=torch.int64, device=DEV)
    M.ops.seed_rng(77, DEV, 0)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        ds.sample(idx)                                                                    # warm-up outside the capture
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
        bits = ds.torso_bits[f].cpu().numpy().view(np.uint32)
        pix = np.arange(ds.H * ds.W)
        torso = ((bits[pix >> 5] >> (pix & 31).astype(np.uint32)) & 1).astype(bool)
        p = PS.select(seed, off, ds.budgets, ds.bounds[f].cpu().numpy(), torso, ds.H, ds.W)
        sel = torch.from_numpy(np.stack([p // ds.W, p % ds.W], 1)).to(DEV)
        assert torch.equal(out["rays"], M.ops.get_rays_at(sel, hd.focal, ds.poses[f], a.near, a.far, hd.cx, hd.cy)), f
        assert torch.equal(out["expr"], ds.exprs[f]) and torch.equal(out["pose"], ds.poses[f])
        if prev is not None:
            assert not np.array_equal(prev, p)                                            # consecutive replays draw different pixels
        prev = p


def test_train_step_fed_from_device_dataset(M, tmp_path):
    from ideal_nerf_b200 import synthetic as S
    from ideal_nerf_b200 import train as T
    from ideal_nerf_b200.data import DeviceHeadDataset
    S.write_head_subject(str(tmp_path), 96, 96, n_frames=1, seed=2, torso_rows=8, constant_rgb=(200, 60, 30), n_aud=1)
    a = M.default_args(N_rand=1024, mouth_rays=128, torso_rays=64, sample_rate=0.9, gt_dirs="head_imgs", near=S.NEAR, far=S.FAR,
                       dim_aud=64, dim_expr=76, perturb=1.0, mlp_mode="bf16", lrate=5e-4, nosmo_iters=0)
    ds = DeviceHeadDataset(str(tmp_path), "aud.npy", "train", a)
    torch.manual_seed(4321)
    net = M.Network(ds.H, ds.W, ds.focal, S.NEAR, S.FAR, 8192, None, 64, 128, args=a)
    net.apply(M.init_weights)
    net = net.to(DEV).train()
    ts = T.TrainStep(net, torch.ones(1, 32, device=DEV), a, cuda_graph=True)
    idx = torch.zeros((), dtype=torch.int64, device=DEV)
    M.ops.seed_rng(1, DEV, 0)
    losses = []
    for _ in range(30):
        b = ds.sample(idx)
        out = ts(b["rays"], b["bc_rgb"], b["target"], None, b["expr"], idx, aud_window=b["aud_window"])
        losses.append(float(out["img_loss"]))
    assert all(np.isfinite(losses))
    assert np.mean(losses[-5:]) < np.mean(losses[:5]), losses
