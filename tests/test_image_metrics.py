"""GPU tests of the image metrics: the kernel inerf_image_metrics (ops.image_metrics) against the numpy oracle on random, smooth, identical
and constant frames at 11 x 11, 37 x 101 (ragged tiles) and 450 x 450, with empty, clipped and overlapping boxes, a device frame index
with repeats and an out-of-range row, and replay in a CUDA graph; then evaluate.evaluate_split on a synthetic subject, head and head +
torso, against the video drivers and the oracle."""
import numpy as np
import pytest
import torch

from oracle import image_metrics_ref as IM

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def M():
    import ideal_nerf_b200 as m
    assert torch.cuda.is_available(), "-m gpu tests need a GPU"
    m.lib()                                       # raises if the extension is missing: no fallback
    m._lib.check(m.lib().inerf_device_check(), "inerf_device_check")
    return m


def frames_of(H, W, seed):
    """Ground truth (5, H, W, 3): random bytes, a smooth gradient, a constant, another random, another gradient."""
    rng = np.random.RandomState(seed)
    yy, xx = np.meshgrid(np.arange(H), np.arange(W), indexing="ij")
    grad = np.stack([yy * 255 // (H - 1), xx * 255 // (W - 1), (yy + xx) * 255 // (H + W - 2)], -1).astype(np.uint8)
    return np.stack([rng.randint(0, 256, (H, W, 3)), grad, np.full((H, W, 3), 201), rng.randint(0, 256, (H, W, 3)), 255 - grad]
                    ).astype(np.uint8)


def bounds_of(H, W):
    """(5, 8) boxes: overlapping rect and mouth; an empty rect (r0 > r1) and a mouth clipped at the border; both beyond the frame; the
    whole frame; a one-pixel rect inside a clipped mouth."""
    return np.array([[2, H // 2, 3, W // 2, H // 4, H - 3, W // 4, W - 2],
                     [5, 4, 0, W - 1, -7, 3, W - 4, W + 20],
                     [H + 2, H + 9, 0, 3, 0, 4, W, W + 3],
                     [0, H - 1, 0, W - 1, 0, H - 1, 0, W - 1],
                     [H // 2, H // 2, W // 2, W // 2, -100, H + 100, 1, 2]], np.int32)


def preds_of(gt, seed):
    """Rendered stand-ins (8, H, W, 3) for the frame index [0, 1, 1, 2, 3, 4, 0, 9] (repeats; row 7 out of range): noisy copies, an
    exact copy of frame 1 (row 2), a constant against the constant (row 3), and random bytes."""
    rng = np.random.RandomState(seed)
    noisy = lambda f, s: np.clip(gt[f].astype(int) + rng.randint(-s, s + 1, gt[f].shape), 0, 255).astype(np.uint8)
    H, W = gt.shape[1:3]
    return np.stack([noisy(0, 30), noisy(1, 4), gt[1], np.full((H, W, 3), 37, np.uint8), rng.randint(0, 256, (H, W, 3)).astype(np.uint8),
                     noisy(4, 60), gt[2], noisy(3, 5)])


INDEX = [0, 1, 1, 2, 3, 4, 0, 9]


def run(M, pred, gt, index, bounds):
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    r = M.ops.image_metrics(t(pred), t(gt), t(np.asarray(index, np.int64)), None if bounds is None else t(bounds))
    return {k: v.cpu().numpy() for k, v in r.items()}


@pytest.mark.parametrize("H,W", [(11, 11), (37, 101), (450, 450)])
def test_kernel_against_oracle(M, H, W):
    gt = frames_of(H, W, H + W)
    pred = preds_of(gt, H * W)
    bounds = bounds_of(H, W)
    got = run(M, pred, gt, INDEX, bounds)
    sse, npix, ssim_sum = IM.image_metrics(pred, gt, INDEX, bounds)
    assert np.array_equal(got["sse"], sse) and np.array_equal(got["npix"], npix)
    want = ssim_sum / (3 * (H - 10) * (W - 10))
    assert np.abs(got["ssim"] - want).max() <= 1e-5, (got["ssim"], want)
    assert got["sse"][2].sum() == 0 and abs(got["ssim"][2] - 1) <= 1e-6                  # identical frames
    assert not got["sse"][7].any() and not got["npix"][7].any() and got["ssim"][7] == 0    # out-of-range index
    assert np.array_equal(got["npix"][:, 0], [H * W] * 7 + [0])
    assert got["npix"][1, 1] == 0 and got["npix"][4, 1] == H * W                          # empty rect; a box holding the frame
    nob = run(M, pred, gt, INDEX, None)                                                   # no boxes: full frame only
    assert np.array_equal(nob["sse"][:, 0], sse[:, 0]) and not nob["sse"][:, 1:].any() and not nob["npix"][:, 1:].any()
    assert np.array_equal(nob["ssim"], got["ssim"])


def test_device_index_and_graph_replay(M):
    """The frame index is read on the device: a captured call scores whatever the index tensor holds at replay, equal to the eager call."""
    H, W = 45, 70
    gt = torch.from_numpy(frames_of(H, W, 1)).to(DEV)
    pred = torch.from_numpy(preds_of(frames_of(H, W, 1), 2)).to(DEV)
    bounds = torch.from_numpy(bounds_of(H, W)).to(DEV)
    idx = torch.tensor(INDEX, dtype=torch.int64, device=DEV)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        M.ops.image_metrics(pred, gt, idx, bounds)                                        # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = M.ops.image_metrics(pred, gt, idx, bounds)
    for index in (INDEX, [4, 4, 4, 4, 3, 2, 1, -1], [0, 1, 2, 3, 4, 0, 1, 2]):
        idx.copy_(torch.tensor(index, dtype=torch.int64))
        g.replay()
        eager = M.ops.image_metrics(pred, gt, idx, bounds)
        torch.cuda.synchronize()
        for k in ("sse", "npix", "ssim"):
            assert torch.equal(out[k], eager[k]), (index, k)
        sse, npix, _ = IM.image_metrics(pred.cpu().numpy(), gt.cpu().numpy(), index, bounds.cpu().numpy())
        assert np.array_equal(out["sse"].cpu().numpy(), sse) and np.array_equal(out["npix"].cpu().numpy(), npix)


def test_ops_rejects_bad_tensors(M):
    u8 = lambda *s: torch.zeros(s, dtype=torch.uint8, device=DEV)
    idx = torch.zeros(2, dtype=torch.int64, device=DEV)
    with pytest.raises(ValueError, match="pred_u8"):
        M.ops.image_metrics(u8(2, 16, 16, 3).float(), u8(1, 16, 16, 3), idx)
    with pytest.raises(ValueError, match="must be"):
        M.ops.image_metrics(u8(2, 16, 17, 3), u8(1, 16, 16, 3), idx)
    with pytest.raises(ValueError, match="frame_index"):
        M.ops.image_metrics(u8(2, 16, 16, 3), u8(1, 16, 16, 3), idx[:1])
    with pytest.raises(ValueError, match="bounds"):
        M.ops.image_metrics(u8(2, 16, 16, 3), u8(1, 16, 16, 3), idx, torch.zeros(2, 8, dtype=torch.int32, device=DEV))
    with pytest.raises(RuntimeError, match="argument error"):
        M.ops.image_metrics(u8(2, 10, 16, 3), u8(1, 10, 16, 3), idx)


# ------------------------------------------------------------------------------------------------
# evaluate_split
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def subject(M, tmp_path_factory):
    from ideal_nerf_b200 import synthetic as S
    from ideal_nerf_b200.data import DeviceHeadDataset
    d = str(tmp_path_factory.mktemp("subject"))
    S.write_head_subject(d, 72, 56, n_frames=2, seed=3, torso_rows=12, val_frames=4)
    args = M.default_args(N_rand=0, mouth_rays=0, torso_rays=0, gt_dirs="head_imgs", near=S.NEAR, far=S.FAR, dim_aud=64, dim_expr=76,
                          perturb=0., mlp_mode="bf16")
    return DeviceHeadDataset(d, "aud.npy", "val", args)


def head_net(M, ds):
    from ideal_nerf_b200 import synthetic as S
    torch.manual_seed(12)
    net = M.Network(ds.H, ds.W, ds.focal, S.NEAR, S.FAR, 8192, None, 64, 128, args=ds.args)
    net.apply(M.init_weights)
    return net.to(DEV).eval()


def check_scores(res, ds, video):
    from ideal_nerf_b200.evaluate import psnr
    n = len(ds)
    sse, npix, ssim_sum = IM.image_metrics(video, ds.frames.cpu().numpy(), np.arange(n), ds.bounds.cpu().numpy())
    assert np.array_equal(res["sse"], sse) and np.array_equal(res["npix"], npix)
    assert np.abs(res["ssim"] - ssim_sum / (3 * (ds.H - 10) * (ds.W - 10))).max() <= 1e-5
    assert np.array_equal(res["psnr"], psnr(sse, npix).numpy()) and res["psnr"].shape == (n, 3)
    assert np.allclose(res["mean_psnr"], res["psnr"].mean(0)) and abs(res["mean_ssim"] - res["ssim"].mean()) < 1e-12
    assert np.isfinite(res["psnr"]).all() and (npix[:, 1:] > 0).all()


def test_audio_codes_bit_exact(M, subject):
    from ideal_nerf_b200.evaluate import audio_codes
    net = head_net(M, subject)
    codes = audio_codes(net, subject)
    assert codes.shape == (len(subject), 64)
    with torch.no_grad():
        for i in range(len(subject)):
            assert torch.equal(codes[i], net.audio_feature(subject.auds, i, len(subject))), i


def test_evaluate_split_head(M, subject):
    from ideal_nerf_b200.evaluate import audio_codes, evaluate_split
    from ideal_nerf_b200.frame import FrameRenderer, render_video
    ds = subject
    net = head_net(M, ds)
    codes = audio_codes(net, ds)
    latent = torch.ones(32, device=DEV)
    res = evaluate_split(FrameRenderer(net), ds, latent, codes)
    with torch.no_grad():
        want = render_video(FrameRenderer(net), [(ds.poses[i], codes[i], ds.exprs[i]) for i in range(len(ds))], latent, ds.bc_img)
    assert res["video"].shape == (len(ds), ds.H, ds.W, 3) and np.array_equal(res["video"], want.numpy())
    check_scores(res, ds, res["video"])
    assert evaluate_split(FrameRenderer(net), ds, latent, codes, keep_video=False)["video"] is None


def test_evaluate_split_head_torso(M, subject):
    from ideal_nerf_b200 import synthetic as S
    from ideal_nerf_b200.evaluate import audio_codes, evaluate_split
    from ideal_nerf_b200.frame import HeadTorsoFrameRenderer, render_head_torso_video
    ds = subject
    codes = audio_codes(head_net(M, ds), ds)
    torch.manual_seed(13)
    net = M.TorsoNetwork(ds.H, ds.W, ds.focal, S.NEAR, S.FAR, 8192, 64, 128, args=ds.args, dim_expr=76)
    net.apply(M.init_weights)
    net = net.to(DEV).eval()
    latent = torch.ones(32, device=DEV)
    r = HeadTorsoFrameRenderer(net, ds.poses[0])
    res = evaluate_split(r, ds, latent, codes)
    with torch.no_grad():
        want = render_head_torso_video(r, [(ds.poses[i], codes[i], ds.exprs[i]) for i in range(len(ds))], latent, ds.bc_img)
    assert np.array_equal(res["video"], want.numpy())
    check_scores(res, ds, res["video"])
