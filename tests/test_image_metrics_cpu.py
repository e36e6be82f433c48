"""CPU-side checks of the image metrics: the numpy oracle of inerf_image_metrics against a brute-force per-window SSIM and against the
reflect-filter-then-crop form skimage computes, evaluate.psnr's edge cases, the argument checks of the C entry point (all returned before
any device work), and the held-out split of synthetic.write_head_subject."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import image_metrics_ref as IM

A16 = 0x10000          # fake device address (never dereferenced: every call below returns before a launch)


@pytest.fixture(scope="module")
def M():
    import ideal_nerf_b200 as m
    m.build()
    return m


def brute_ssim_map(x, y):
    """SSIM of every position whose 11 x 11 window lies inside the frame, one window at a time with the 2-D weights outer(g, g)."""
    g = IM.gaussian_taps()
    w2 = np.outer(g, g)
    H, W = x.shape
    out = np.empty((H - 10, W - 10))
    for i in range(H - 10):
        for j in range(W - 10):
            a, b = x[i:i + 11, j:j + 11].astype(np.float64), y[i:i + 11, j:j + 11].astype(np.float64)
            ua, ub = (w2 * a).sum(), (w2 * b).sum()
            va, vb, cov = (w2 * a * a).sum() - ua * ua, (w2 * b * b).sum() - ub * ub, (w2 * a * b).sum() - ua * ub
            out[i, j] = ((2 * ua * ub + IM.C1) * (2 * cov + IM.C2)) / ((ua * ua + ub * ub + IM.C1) * (va + vb + IM.C2))
    return out


def test_gaussian_taps():
    g = IM.gaussian_taps()
    assert g.shape == (11,) and abs(g.sum() - 1) < 1e-15 and np.allclose(g, g[::-1])
    assert np.allclose(g[6] / g[5], np.exp(-0.5 / 1.5 ** 2))


@pytest.mark.parametrize("H,W", [(11, 11), (13, 17), (20, 12)])
def test_oracle_against_brute_force_windows(H, W):
    rng = np.random.RandomState(H * W)
    x = rng.randint(0, 256, (H, W)).astype(np.uint8)
    for y in (rng.randint(0, 256, (H, W)).astype(np.uint8), np.clip(x.astype(int) + rng.randint(-9, 10, (H, W)), 0, 255).astype(np.uint8),
              np.full((H, W), 200, np.uint8), x):
        got = IM.ssim_map(x, y)
        assert got.shape == (H - 10, W - 10)
        np.testing.assert_allclose(got, brute_ssim_map(x, y), rtol=0, atol=1e-12)
    assert np.allclose(IM.ssim_map(x, x), 1.0, atol=1e-12)


def test_oracle_is_skimage_reflect_then_crop():
    """skimage filters the whole image with reflection and averages the SSIM map cropped by 5 pixels: the same numbers as 'valid'."""
    nd = pytest.importorskip("scipy.ndimage")
    rng = np.random.RandomState(3)
    x = rng.randint(0, 256, (23, 31, 3)).astype(np.uint8)
    y = np.clip(x.astype(int) + rng.randint(-40, 41, x.shape), 0, 255).astype(np.uint8)
    per = []
    for c in range(3):
        a, b = x[..., c].astype(np.float64), y[..., c].astype(np.float64)
        f = lambda t: nd.gaussian_filter(t, sigma=1.5, truncate=3.5, mode="reflect")
        ua, ub = f(a), f(b)
        va, vb, cov = f(a * a) - ua * ua, f(b * b) - ub * ub, f(a * b) - ua * ub
        s = ((2 * ua * ub + IM.C1) * (2 * cov + IM.C2)) / ((ua * ua + ub * ub + IM.C1) * (va + vb + IM.C2))
        per.append(s[5:-5, 5:-5].mean())
    assert abs(IM.ssim(x, y) - np.mean(per)) < 1e-12


def test_oracle_regions_and_index():
    rng = np.random.RandomState(4)
    H, W = 12, 14
    gt = rng.randint(0, 256, (2, H, W, 3)).astype(np.uint8)
    pred = rng.randint(0, 256, (3, H, W, 3)).astype(np.uint8)
    bounds = np.array([[2, 5, 3, 7, 4, 20, -3, 4], [6, 5, 0, 13, 0, 11, 0, 13]], np.int32)      # clipped mouth; empty rect, full mouth
    sse, npix, ssim_sum = IM.image_metrics(pred, gt, [1, 0, 2], bounds)
    assert np.array_equal(npix, [[H * W, 0, H * W], [H * W, 4 * 5, 8 * 5], [0, 0, 0]])
    assert sse[0, 0] == sse[0, 2] == ((pred[0].astype(int) - gt[1]) ** 2).sum() and sse[0, 1] == 0
    assert sse[1, 1] == ((pred[1, 2:6, 3:8].astype(int) - gt[0, 2:6, 3:8]) ** 2).sum()
    assert not sse[2].any() and ssim_sum[2] == 0
    sse0, npix0, _ = IM.image_metrics(pred, gt, [1, 0, 2])
    assert np.array_equal(sse0[:, 0], sse[:, 0]) and not sse0[:, 1:].any() and not npix0[:, 1:].any()


def test_psnr_edge_cases():
    from ideal_nerf_b200.evaluate import psnr
    npix = torch.tensor([[100, 7, 0]], dtype=torch.int64)
    p = psnr(torch.tensor([[0, 3 * 7 * 255 ** 2, 0]]), npix)
    assert p.dtype == torch.float64 and p.shape == (1, 3)
    assert p[0, 0] == float("inf") and p[0, 1] == 0. and p[0, 2] == float("inf")         # identical, maximal error, empty region
    assert abs(float(psnr(np.array([300]), np.array([100]))[0]) - 20 * np.log10(255.)) < 1e-12     # mean squared error 1
    big = psnr(torch.tensor([1]), torch.tensor([1 << 40]))                                  # int64 counts beyond 2^32
    assert abs(float(big) - 10 * np.log10(255. ** 2 * 3 * 2 ** 40)) < 1e-9


def test_abi_argument_checks_before_any_launch(M):
    L = M.lib()
    assert M._lib.INERF_IMAGE_METRICS_MAX_PIXELS == 1 << 24

    def run(**over):
        a = dict(pred=A16, gt=A16, idx=A16, bounds=A16, B=2, H=45, W=37, F=3, sse=A16, npix=A16, ssim=A16)
        a.update(over)
        return L.inerf_image_metrics(a["pred"], a["gt"], a["idx"], a["bounds"], a["B"], a["H"], a["W"], a["F"], a["sse"], a["npix"],
                                     a["ssim"], None)

    for name in ("pred", "gt", "idx", "sse", "npix", "ssim"):
        assert run(**{name: None}) == -1, name
        assert b"NULL" in L.inerf_last_error()
    assert run(B=-1) == -1 and run(F=-1) == -1
    for over in ({"H": 10}, {"W": 10}, {"H": 0}, {"H": 4097, "W": 4097}):
        assert run(**over) == -2, over
        assert b"inerf_image_metrics" in L.inerf_last_error()
    assert run(B=0) == 0                                                                   # nothing to score, nothing enqueued
    assert run(B=0, bounds=None, H=11, W=11) == 0
    assert run(B=0, H=4096, W=4096) == 0                                                   # exactly the pixel limit


def test_ops_image_metrics_checks_arguments(M):
    u8 = lambda *s: torch.zeros(s, dtype=torch.uint8)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        M.ops.image_metrics(u8(1, 16, 16, 3), u8(2, 16, 16, 3), torch.zeros(1, dtype=torch.int64))


def test_subject_val_split(tmp_path):
    """val_frames writes transforms_exp_val.json with held-out frames and appends their audio; the train split is unchanged; a val split
    too small for the training budgets still loads as an evaluation dataset with zero budgets."""
    from ideal_nerf_b200 import default_args
    from ideal_nerf_b200 import synthetic as S
    from ideal_nerf_b200.data import DeviceHeadDataset, HeadDataset
    a, b = str(tmp_path / "a"), str(tmp_path / "b")
    S.write_head_subject(a, 30, 24, n_frames=3, seed=2, torso_rows=1)
    S.write_head_subject(b, 30, 24, n_frames=3, seed=2, torso_rows=1, val_frames=2)
    assert not os.path.exists(os.path.join(a, "transforms_exp_val.json"))
    assert open(os.path.join(a, "transforms_exp_train.json")).read() == open(os.path.join(b, "transforms_exp_train.json")).read()
    for i in range(3):
        assert open(os.path.join(a, "head_imgs", f"{i}.jpg"), "rb").read() == open(os.path.join(b, "head_imgs", f"{i}.jpg"), "rb").read()
    val = json.load(open(os.path.join(b, "transforms_exp_val.json")))["frames"]
    assert [f["img_id"] for f in val] == [3, 4] and [f["aud_id"] for f in val] == [3, 4]
    aud_a, aud_b = np.load(os.path.join(a, "aud.npy")), np.load(os.path.join(b, "aud.npy"))
    assert aud_b.shape == (5, 16, 29) and np.array_equal(aud_b[:3], aud_a)
    train_args = default_args(N_rand=64, mouth_rays=8, torso_rays=32, sample_rate=0.9, gt_dirs="head_imgs")
    hd = HeadDataset(b, "aud.npy", "val", train_args, device="cpu")
    assert len(hd) == 2 and torch.equal(hd.auds, torch.from_numpy(aud_b[3:]))
    with pytest.raises(ValueError, match="fewer than its budget"):                         # e.g. 24 torso pixels, 32 torso rays
        DeviceHeadDataset(b, "aud.npy", "val", train_args, device="cpu")
    ds = DeviceHeadDataset(b, "aud.npy", "val", default_args(N_rand=0, mouth_rays=0, torso_rays=0, gt_dirs="head_imgs"), device="cpu")
    assert ds.frames.shape == (2, 30, 24, 3) and ds.budgets == (0, 0, 0, 0)
