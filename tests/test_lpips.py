"""GPU tests of LPIPS: the kernels behind inerf_lpips (ops.lpips) against the float64 oracle on seeded weights in the released files' key
layouts, on random, smooth-gradient, constant and noisy-copy frames with R != B at 31 x 31, 37 x 101 (ragged tiles) and 450 x 450, with a
device frame index holding repeats and an out-of-range row; exact zeros; bit-identical eager calls and CUDA-graph replay; and
evaluate_split(lpips=...) on a synthetic subject, head and head + torso.  test_against_lpips_package runs only where the lpips package and
the two released weight files are available (INERF_LPIPS_ALEXNET, INERF_LPIPS_LIN)."""
import os

import numpy as np
import pytest
import torch

from oracle import lpips_ref as LR

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
INDEX = [0, 1, 1, 2, 3, 4, 0, 9]                     # repeats; row 7 out of range


@pytest.fixture(scope="module")
def M():
    import ideal_nerf_b200 as m
    assert torch.cuda.is_available(), "-m gpu tests need a GPU"
    m.lib()                                       # raises if the extension is missing: no fallback
    m._lib.check(m.lib().inerf_device_check(), "inerf_device_check")
    return m


@pytest.fixture(scope="module")
def state():
    """Seeded (alexnet, lin) state dicts in the key layouts of alexnet-owt-7be5be79.pth and lpips' v0.1 alex.pth."""
    return LR.seeded_state_dicts(2024)


@pytest.fixture(scope="module")
def weights(M, state):
    from ideal_nerf_b200.evaluate import load_lpips
    return load_lpips(*state, device=DEV)


def frames_of(H, W, seed):
    """Ground truth (5, H, W, 3) BGR: random bytes, a smooth gradient, a constant, another random, another gradient; R != B throughout."""
    rng = np.random.RandomState(seed)
    yy, xx = np.meshgrid(np.arange(H), np.arange(W), indexing="ij")
    grad = np.stack([yy * 255 // (H - 1), xx * 255 // (W - 1), 255 - (yy + xx) * 255 // (H + W - 2)], -1).astype(np.uint8)
    return np.stack([rng.randint(0, 256, (H, W, 3)), grad, np.broadcast_to(np.array([30, 140, 220]), (H, W, 3)),
                     rng.randint(0, 256, (H, W, 3)), grad[::-1, ::-1]]).astype(np.uint8)


def preds_of(gt, seed):
    """Rendered stand-ins (8, H, W, 3) for INDEX: noisy copies, an exact copy of frame 1 (row 2), a constant against the constant
    (row 3), random bytes, and the channel-swapped frame 0 (row 6)."""
    rng = np.random.RandomState(seed)
    noisy = lambda f, s: np.clip(gt[f].astype(int) + rng.randint(-s, s + 1, gt[f].shape), 0, 255).astype(np.uint8)
    H, W = gt.shape[1:3]
    return np.stack([noisy(0, 30), noisy(1, 4), gt[1], np.full((H, W, 3), 37, np.uint8), rng.randint(0, 256, (H, W, 3)).astype(np.uint8),
                     noisy(4, 60), gt[0, ..., ::-1], noisy(3, 5)])


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


@pytest.mark.parametrize("H,W", [(31, 31), (37, 101), (450, 450)])
def test_kernel_against_oracle(M, state, weights, H, W):
    gt = frames_of(H, W, H + W)
    pred = preds_of(gt, H * W)
    got = M.ops.lpips(dev(pred), dev(gt), dev(np.asarray(INDEX, np.int64)), weights)
    assert got.dtype == torch.float32 and got.shape == (8,) and got.device == torch.device(DEV)
    got = got.double().cpu()
    want = LR.lpips(pred, gt, INDEX, *state)
    err = (got - want).abs()
    print(f"\nlpips {H} x {W}: oracle {np.round(want.numpy(), 6).tolist()}\n  max |kernel - oracle| {float(err.max()):.3e}, "
          f"max relative {float((err / want.clamp_min(1e-12))[want > 0].max()):.3e}")
    assert (err <= 1e-6 + 1e-3 * want).all(), (got, want)
    assert got[2] == 0 and got[7] == 0                                                    # identical frames; out-of-range index
    assert (want[[0, 1, 3, 4, 5, 6]] > 1e-4).all()                                        # every other row scores, the swap included


def test_deterministic_and_graph_replay(M, weights):
    """Two eager calls are bit-identical, and a captured call replays the eager bits for whatever the device index holds."""
    H, W = 67, 90
    gt = dev(frames_of(H, W, 1))
    pred = dev(preds_of(frames_of(H, W, 1), 2))
    idx = torch.tensor(INDEX, dtype=torch.int64, device=DEV)
    a, b = M.ops.lpips(pred, gt, idx, weights), M.ops.lpips(pred, gt, idx, weights)
    assert torch.equal(a, b)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        M.ops.lpips(pred, gt, idx, weights)                                              # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = M.ops.lpips(pred, gt, idx, weights)
    for index in (INDEX, [4, 4, 4, 4, 3, 2, 1, -1], [0, 1, 2, 3, 4, 0, 1, 2]):
        idx.copy_(torch.tensor(index, dtype=torch.int64))
        g.replay()
        eager = M.ops.lpips(pred, gt, idx, weights)
        torch.cuda.synchronize()
        assert torch.equal(out, eager), index
    assert torch.equal(M.ops.lpips(pred[:3], gt, idx[:3], weights), eager[:3])            # a row's bits do not depend on the batch


def test_ops_lpips_rejects_bad_tensors(M, weights):
    u8 = lambda *s: torch.zeros(s, dtype=torch.uint8, device=DEV)
    idx = torch.zeros(2, dtype=torch.int64, device=DEV)
    with pytest.raises(ValueError, match="pred_u8"):
        M.ops.lpips(u8(2, 32, 32, 3).float(), u8(1, 32, 32, 3), idx, weights)
    with pytest.raises(ValueError, match="must be"):
        M.ops.lpips(u8(2, 32, 33, 3), u8(1, 32, 32, 3), idx, weights)
    with pytest.raises(ValueError, match="frame_index"):
        M.ops.lpips(u8(2, 32, 32, 3), u8(1, 32, 32, 3), idx[:1], weights)
    with pytest.raises(ValueError, match="15"):
        M.ops.lpips(u8(2, 32, 32, 3), u8(1, 32, 32, 3), idx, weights[:14])
    with pytest.raises(ValueError, match=r"weights\[3\]"):
        M.ops.lpips(u8(2, 32, 32, 3), u8(1, 32, 32, 3), idx, weights[:3] + [weights[3].double()] + weights[4:])
    with pytest.raises(RuntimeError, match="argument error"):
        M.ops.lpips(u8(2, 30, 32, 3), u8(1, 30, 32, 3), idx, weights)
    assert M.ops.lpips(u8(0, 32, 32, 3), u8(1, 32, 32, 3), idx[:0], weights).shape == (0,)


# ------------------------------------------------------------------------------------------------
# evaluate_split(lpips=...)
# ------------------------------------------------------------------------------------------------
HEAD_KEYS = ["mean_psnr", "mean_ssim", "npix", "psnr", "sse", "ssim", "video"]
TORSO_KEYS = HEAD_KEYS + ["mean_psnr_torso", "npix_torso", "psnr_torso", "sse_torso"]


def same_values(a, b):
    assert sorted(a) == sorted(b)
    for k in a:
        if isinstance(a[k], np.ndarray):
            assert np.array_equal(a[k], b[k]), k
        else:
            assert a[k] == b[k], k


def check_lpips(M, res, ds, weights):
    n = len(ds)
    want = M.ops.lpips(torch.from_numpy(res["video"]).to(DEV), ds.frames, torch.arange(n, dtype=torch.int64, device=DEV), weights)
    assert res["lpips"].dtype == np.float64 and res["lpips"].shape == (n,)
    assert np.array_equal(res["lpips"], want.double().cpu().numpy())
    assert abs(res["mean_lpips"] - res["lpips"].mean()) < 1e-12 and (res["lpips"] > 0).all()


def test_evaluate_split_head(M, weights, tmp_path):
    from ideal_nerf_b200 import synthetic as S
    from ideal_nerf_b200.data import DeviceHeadDataset
    from ideal_nerf_b200.evaluate import audio_codes, evaluate_split
    from ideal_nerf_b200.frame import FrameRenderer
    d = str(tmp_path)
    S.write_head_subject(d, 72, 56, n_frames=2, seed=3, torso_rows=12, val_frames=4)
    args = M.default_args(N_rand=0, mouth_rays=0, torso_rays=0, gt_dirs="head_imgs", near=S.NEAR, far=S.FAR, dim_aud=64, dim_expr=76,
                          perturb=0., mlp_mode="bf16")
    ds = DeviceHeadDataset(d, "aud.npy", "val", args)
    torch.manual_seed(12)
    net = M.Network(ds.H, ds.W, ds.focal, S.NEAR, S.FAR, 8192, None, 64, 128, args=args)
    net.apply(M.init_weights)
    net = net.to(DEV).eval()
    codes = audio_codes(net, ds)
    latent = torch.ones(32, device=DEV)
    plain = evaluate_split(FrameRenderer(net), ds, latent, codes)
    res = evaluate_split(FrameRenderer(net), ds, latent, codes, lpips=weights)
    assert sorted(plain) == HEAD_KEYS                                                    # without lpips=: the keys it always had
    same_values(plain, {k: v for k, v in res.items() if k not in ("lpips", "mean_lpips")})
    check_lpips(M, res, ds, weights)


def test_evaluate_split_head_torso(M, weights, tmp_path):
    from ideal_nerf_b200 import synthetic as S
    from ideal_nerf_b200.data import DeviceHeadDataset, DeviceTorsoDataset
    from ideal_nerf_b200.evaluate import audio_codes, evaluate_split
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
    r = HeadTorsoFrameRenderer(net, ds.torso_pose)
    plain = evaluate_split(r, ds, latent, codes)
    res = evaluate_split(r, ds, latent, codes, lpips=weights)
    assert sorted(plain) == sorted(TORSO_KEYS)
    same_values(plain, {k: v for k, v in res.items() if k not in ("lpips", "mean_lpips")})
    assert "psnr_torso" in res and "lpips" in res                                        # LPIPS beside the torso region's PSNR
    check_lpips(M, res, ds, weights)
    head_only = evaluate_split(r, hd, latent, codes, lpips=weights)                      # the same split as a head dataset
    assert sorted(head_only) == sorted(HEAD_KEYS + ["lpips", "mean_lpips"])
    assert np.array_equal(head_only["lpips"], res["lpips"])


def test_against_lpips_package(M):
    """The kernel against lpips.LPIPS(net='alex') on the released weights, on a few frame pairs.  Needs the lpips package and the two
    files: INERF_LPIPS_ALEXNET=<alexnet-owt-7be5be79.pth>, INERF_LPIPS_LIN=<lpips/weights/v0.1/alex.pth>."""
    lp = pytest.importorskip("lpips")
    pa, pl = os.environ.get("INERF_LPIPS_ALEXNET"), os.environ.get("INERF_LPIPS_LIN")
    if not (pa and pl and os.path.exists(pa) and os.path.exists(pl)):
        pytest.skip("INERF_LPIPS_ALEXNET / INERF_LPIPS_LIN do not name the released weight files")
    from ideal_nerf_b200.evaluate import load_lpips
    w = load_lpips(pa, pl, device=DEV)
    gt = frames_of(96, 128, 5)
    pred = preds_of(gt, 6)[:6]
    idx = [0, 1, 1, 2, 3, 4]
    got = M.ops.lpips(dev(pred), dev(gt), dev(np.asarray(idx, np.int64)), w).double().cpu()
    net = lp.LPIPS(net="alex", version="0.1", verbose=False).eval()
    to_t = lambda a: torch.from_numpy(np.ascontiguousarray(a[..., ::-1])).permute(0, 3, 1, 2).double() / 127.5 - 1.
    with torch.no_grad():
        want = net.double()(to_t(pred), to_t(gt[idx])).reshape(-1)
    err = (got - want).abs()
    print(f"\nlpips package: max |kernel - package| {float(err.max()):.3e}")
    assert (err <= 1e-6 + 1e-3 * want).all(), (got, want)
