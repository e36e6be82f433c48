"""CPU-side checks of the torso stage's data path: DeviceTorsoDataset's construction (the default and explicit torso camera, the shape
checks of its tables), the com_imgs of synthetic.write_head_subject, the argument checks of inerf_masked_sse (all returned before any
device work) and its numpy oracle against a brute-force loop."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import masked_sse_ref as MS

A16 = 0x10000          # fake device address (never dereferenced: every call below returns before a launch)


@pytest.fixture(scope="module")
def M():
    import ideal_nerf_b200 as m
    m.build()
    return m


def eval_args(**over):
    from ideal_nerf_b200 import default_args
    kw = dict(N_rand=0, mouth_rays=0, torso_rays=0, gt_dirs="com_imgs", dim_aud=64)
    kw.update(over)
    return default_args(**kw)


@pytest.fixture(scope="module")
def subject(tmp_path_factory):
    from ideal_nerf_b200 import synthetic as S
    d = str(tmp_path_factory.mktemp("torso_subject"))
    S.write_head_subject(d, 48, 40, n_frames=3, seed=5, torso_rows=16, val_frames=2, com_imgs=True)
    return d


def train_pose(d, i=0):
    return np.array(json.load(open(os.path.join(d, "transforms_exp_train.json")))["frames"][i]["transform_matrix"], np.float32)


def test_default_torso_pose_is_train_frame_0(subject):
    from ideal_nerf_b200.data import DeviceTorsoDataset
    want = torch.from_numpy(train_pose(subject)[:3])
    assert not np.array_equal(train_pose(subject, 1), train_pose(subject, 0))                  # the poses differ per frame
    tr = DeviceTorsoDataset(subject, "aud.npy", "train", eval_args(), torch.zeros(3, 64), torch.zeros(3, 32), device="cpu")
    va = DeviceTorsoDataset(subject, "aud.npy", "val", eval_args(), torch.zeros(2, 64), device="cpu")
    for ds in (tr, va):
        assert ds.torso_pose.shape == (3, 4) and ds.torso_pose.dtype == torch.float32
        assert torch.equal(ds.torso_pose, want)
    assert not torch.equal(va.poses[0], want)                                                   # a val frame's own pose is not it
    assert va.latent_codes is None
    with pytest.raises(ValueError, match="latent_codes"):
        va.sample(0)


def test_explicit_torso_pose(subject):
    from ideal_nerf_b200.data import DeviceTorsoDataset
    p4 = np.eye(4)
    p4[:3, 3] = [0.1, 0.2, 0.3]
    for pose in (p4, p4[:3], torch.tensor(p4[:3], dtype=torch.float64)):
        ds = DeviceTorsoDataset(subject, "aud.npy", "val", eval_args(), torch.zeros(2, 64), torso_pose=pose, device="cpu")
        assert torch.equal(ds.torso_pose, torch.tensor(p4[:3], dtype=torch.float32))
    for bad in (np.eye(3), np.zeros((4, 3)), np.zeros(12), np.zeros((2, 3, 4))):
        with pytest.raises(ValueError, match="torso_pose"):
            DeviceTorsoDataset(subject, "aud.npy", "val", eval_args(), torch.zeros(2, 64), torso_pose=bad, device="cpu")


def test_table_shapes_checked(subject):
    from ideal_nerf_b200.data import DeviceTorsoDataset

    def make(aud, lat, mode="train", **over):
        return DeviceTorsoDataset(subject, "aud.npy", mode, eval_args(**over), aud, lat, device="cpu")

    ds = make(torch.randn(3, 64, dtype=torch.float64), np.ones((3, 32)))
    assert ds.aud_codes.dtype == torch.float32 and ds.latent_codes.shape == (3, 32)
    for aud, lat, name in ((torch.zeros(2, 64), torch.zeros(3, 32), "aud_codes"), (torch.zeros(3, 63), torch.zeros(3, 32), "aud_codes"),
                           (torch.zeros(3, 64, 1), torch.zeros(3, 32), "aud_codes"), (torch.zeros(3, 64), torch.zeros(4, 32), "latent_codes"),
                           (torch.zeros(3, 64), torch.zeros(3, 31), "latent_codes"), (torch.zeros(3, 64), None, "latent_codes")):
        with pytest.raises(ValueError, match=name):
            make(aud, lat)
    make(torch.zeros(3, 76), torch.zeros(3, 32), dim_aud=76)                                     # the width follows args.dim_aud
    with pytest.raises(ValueError, match="aud_codes"):
        make(torch.zeros(3, 64), torch.zeros(3, 32), dim_aud=76)
    with pytest.raises(ValueError, match="aud_codes"):                                          # the val split has 2 frames
        make(torch.zeros(3, 64), None, mode="val")


def test_device_torso_dataset_keeps_head_tables(subject):
    """The head part is DeviceHeadDataset's: same frames (from com_imgs), bounds, torso bits, poses and expressions."""
    from ideal_nerf_b200.data import DeviceHeadDataset, DeviceTorsoDataset
    hd = DeviceHeadDataset(subject, "aud.npy", "train", eval_args(), device="cpu")
    ds = DeviceTorsoDataset(subject, "aud.npy", "train", eval_args(), torch.zeros(3, 64), torch.zeros(3, 32), device="cpu")
    for k in ("frames", "bounds", "torso_bits", "poses", "exprs", "bc_img", "auds_padded"):
        assert torch.equal(getattr(ds, k), getattr(hd, k)), k
    head = DeviceHeadDataset(subject, "aud.npy", "train", eval_args(gt_dirs="head_imgs"), device="cpu")
    assert not torch.equal(head.frames, ds.frames)


def test_com_imgs_default_writes_the_same_bytes(tmp_path):
    from ideal_nerf_b200 import synthetic as S
    a, b = str(tmp_path / "a"), str(tmp_path / "b")
    S.write_head_subject(a, 32, 24, n_frames=2, seed=7, torso_rows=8, val_frames=1)
    S.write_head_subject(b, 32, 24, n_frames=2, seed=7, torso_rows=8, val_frames=1, com_imgs=True)
    files = lambda d: sorted(os.path.relpath(os.path.join(r, f), d) for r, _, fs in os.walk(d) for f in fs)
    fa, fb = files(a), files(b)
    assert not os.path.exists(os.path.join(a, "com_imgs"))
    assert sorted(set(fb) - set(fa)) == [os.path.join("com_imgs", f"{i}.jpg") for i in range(3)] and set(fa) <= set(fb)
    for f in fa:
        assert open(os.path.join(a, f), "rb").read() == open(os.path.join(b, f), "rb").read(), f


def test_com_imgs_differ_from_head_imgs_in_the_torso_rows_only(tmp_path):
    """The boundary row H - torso_rows is a multiple of 16 (the JPEG's MCU height at 4:2:0), so the blocks above it are encoded from the
    same pixels; the decoder's chroma upsampling reads one chroma row across the boundary, so the last pixel row above it may differ."""
    from ideal_nerf_b200 import synthetic as S
    from ideal_nerf_b200.data import _imread_rgb
    H, W, rows = 64, 48, 16
    S.write_head_subject(str(tmp_path), H, W, n_frames=3, seed=1, torso_rows=rows, com_imgs=True)
    for i in range(3):
        head = _imread_rgb(str(tmp_path / "head_imgs" / f"{i}.jpg")).astype(int)
        com = _imread_rgb(str(tmp_path / "com_imgs" / f"{i}.jpg")).astype(int)
        assert np.array_equal(head[:H - rows - 1], com[:H - rows - 1]), i
        torso = com[H - rows + 8:]                                                              # away from the boundary's blocks
        assert np.abs(torso - np.array(S.TORSO_RGB)).max() <= 8, i
        assert np.abs(head[H - rows:] - com[H - rows:]).mean() > 30, i


def brute_masked_sse(pred, gt, index, bits):
    B, H, W = pred.shape[:3]
    sse, npix = [0] * B, [0] * B
    for b, f in enumerate(index):
        if not 0 <= f < gt.shape[0]:
            continue
        for r in range(H):
            for c in range(W):
                p = r * W + c
                if (int(bits[f][p // 32]) >> (p % 32)) & 1:
                    npix[b] += 1
                    sse[b] += sum((int(pred[b, r, c, k]) - int(gt[f, r, c, k])) ** 2 for k in range(3))
    return np.array(sse, np.int64), np.array(npix, np.int64)


@pytest.mark.parametrize("H,W", [(11, 11), (7, 9), (5, 13)])
def test_oracle_against_brute_force(H, W):
    from ideal_nerf_b200.data import torso_bits
    rng = np.random.RandomState(H * W)
    gt = rng.randint(0, 256, (3, H, W, 3)).astype(np.uint8)
    pred = rng.randint(0, 256, (5, H, W, 3)).astype(np.uint8)
    parses = [np.zeros((H, W, 3), np.uint8), np.zeros((H, W, 3), np.uint8), np.zeros((H, W, 3), np.uint8)]
    parses[1][..., 0] = 255                                                                     # full mask
    parses[2][rng.rand(H, W) < 0.4] = (255, 0, 0)                                               # ragged random mask
    parses[2][0, 0] = (255, 0, 1)                                                               # not pure red: not torso
    bits = np.stack([torso_bits(p) for p in parses])
    pad = -(H * W) % 32
    bits[:, -1] |= np.uint32(((1 << pad) - 1) << (32 - pad))                                    # padding bits past H * W are ignored
    index = [2, 1, 0, 2, 3]
    sse, npix = MS.masked_sse(pred, gt, index, bits)
    want_sse, want_npix = brute_masked_sse(pred, gt, index, bits)
    assert np.array_equal(sse, want_sse) and np.array_equal(npix, want_npix)
    assert npix[1] == H * W and npix[2] == 0 and sse[2] == 0 and npix[4] == 0 and sse[4] == 0
    assert np.array_equal(MS.masked_sse(pred, gt, index, bits.view(np.int32))[0], sse)         # int32 words hold the same bits


def test_abi_argument_checks_before_any_launch(M):
    L = M.lib()

    def run(**over):
        a = dict(pred=A16, gt=A16, idx=A16, bits=A16, B=2, H=45, W=37, F=3, sse=A16, npix=A16)
        a.update(over)
        return L.inerf_masked_sse(a["pred"], a["gt"], a["idx"], a["bits"], a["B"], a["H"], a["W"], a["F"], a["sse"], a["npix"], None)

    for name in ("pred", "gt", "idx", "bits", "sse", "npix"):
        assert run(**{name: None}) == -1, name
        assert b"NULL" in L.inerf_last_error()
    assert run(B=-1) == -1 and run(F=-1) == -1
    for over in ({"H": 10}, {"W": 10}, {"H": 0}, {"H": 4097, "W": 4097}):
        assert run(**over) == -2, over
        assert b"inerf_masked_sse" in L.inerf_last_error()
    assert run(B=0) == 0                                                                        # nothing to score, nothing enqueued
    assert run(B=0, H=11, W=11) == 0
    assert run(B=0, H=4096, W=4096) == 0                                                        # exactly the pixel limit


def test_ops_masked_sse_checks_arguments(M):
    u8 = lambda *s: torch.zeros(s, dtype=torch.uint8)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        M.ops.masked_sse(u8(1, 16, 16, 3), u8(2, 16, 16, 3), torch.zeros(1, dtype=torch.int64), torch.zeros(2, 8, dtype=torch.int32))
