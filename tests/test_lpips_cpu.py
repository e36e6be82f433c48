"""CPU-side checks of LPIPS: the float64 oracle of inerf_lpips against an independent construction from torchvision's AlexNet and the
lpips package's structure, the layer map sizes and the 31-pixel bound, the workspace size and argument checks of the C entry points (all
returned before any device work), evaluate.load_lpips' key mapping and checks, and evaluate_split's unchanged default."""
import inspect

import numpy as np
import pytest
import torch
import torch.nn as nn

from oracle import lpips_ref as LR

A16 = 0x10000          # fake device address (never dereferenced: every call below returns before a launch)


@pytest.fixture(scope="module")
def M():
    import ideal_nerf_b200 as m
    m.build()
    return m


def frames_of(n, H, W, seed):
    rng = np.random.RandomState(seed)
    yy, xx = np.meshgrid(np.arange(H), np.arange(W), indexing="ij")
    grad = np.stack([yy * 255 // (H - 1), xx * 255 // (W - 1), 255 - (yy + xx) * 255 // (H + W - 2)], -1)
    out = [rng.randint(0, 256, (H, W, 3)), grad, np.clip(grad + rng.randint(-20, 21, (H, W, 3)), 0, 255)]
    return np.stack([out[i % 3] for i in range(n)]).astype(np.uint8)


class PackageStyleLPIPS(nn.Module):
    """LPIPS v0.1 (AlexNet) as the lpips package structures it: ScalingLayer, torchvision's alexnet().features cut into slice1..slice5
    at relu1..relu5, normalize_tensor, NetLinLayer (Dropout, then a bias-free 1 x 1 Conv2d) and spatial_average, summed over the layers.
    Its input is im2tensor's: an RGB image / 127.5 - 1."""

    def __init__(self, alexnet_sd, lin_sd):
        super().__init__()
        tv = pytest.importorskip("torchvision")
        f = tv.models.alexnet(weights=None).features
        f.load_state_dict({k[len("features."):]: v for k, v in alexnet_sd.items() if k.startswith("features.")})
        self.slices = nn.ModuleList([f[0:2], f[2:5], f[5:8], f[8:10], f[10:12]])
        self.register_buffer("shift", torch.tensor([-.030, -.088, -.188])[None, :, None, None])
        self.register_buffer("scale", torch.tensor([.458, .448, .450])[None, :, None, None])
        self.lins = nn.ModuleList()
        for k, c in enumerate((64, 192, 384, 256, 256)):
            lin = nn.Sequential(nn.Dropout(), nn.Conv2d(c, 1, 1, 1, 0, bias=False))
            lin[1].weight.data.copy_(lin_sd[f"lin{k}.model.1.weight"])
            self.lins.append(lin)

    def forward(self, in0, in1):
        x0, x1 = (in0 - self.shift) / self.scale, (in1 - self.shift) / self.scale
        val = 0
        for sl, lin in zip(self.slices, self.lins):
            x0, x1 = sl(x0), sl(x1)
            n0 = x0 / (torch.sqrt(torch.sum(x0 ** 2, dim=1, keepdim=True)) + 1e-10)
            n1 = x1 / (torch.sqrt(torch.sum(x1 ** 2, dim=1, keepdim=True)) + 1e-10)
            val = val + lin((n0 - n1) ** 2).mean([2, 3], keepdim=True)
        return val


def im2tensor_bgr(frames_u8):
    """lpips.im2tensor of the RGB image behind each stored BGR frame."""
    rgb = np.ascontiguousarray(frames_u8[..., ::-1]).astype(np.float64)
    return torch.from_numpy(rgb / (255. / 2.) - 1.).permute(0, 3, 1, 2).contiguous()


@pytest.mark.parametrize("H,W", [(31, 31), (37, 101), (64, 48)])
def test_oracle_against_package_structure(H, W):
    """The oracle against an independent construction of lpips.LPIPS(net='alex', version='0.1') on the same seeded weights, in float64."""
    alex, lin = LR.seeded_state_dicts(7)
    ref = PackageStyleLPIPS(alex, lin).double().eval()
    gt = frames_of(3, H, W, H * W)
    rng = np.random.RandomState(1)
    pred = np.clip(gt.astype(int) + rng.randint(-40, 41, gt.shape), 0, 255).astype(np.uint8)
    pred[2] = gt[1]                                                                        # row 2 identical to its ground truth
    index = [0, 2, 1]
    got = LR.lpips(pred, gt, index, alex, lin)
    with torch.no_grad():
        want = ref(im2tensor_bgr(pred), im2tensor_bgr(gt[index])).reshape(-1)
    assert got.dtype == torch.float64 and got.shape == (3,)
    torch.testing.assert_close(got, want, rtol=1e-7, atol=1e-12)           # the package holds shift / scale as float32 values
    assert got[2] == 0 and (got[:2] > 1e-3).all()
    # BGR as stored: the swapped channel order gives another score
    swapped = LR.lpips(pred[..., ::-1].copy(), gt[..., ::-1].copy(), index, alex, lin)
    assert (swapped[:2] - got[:2]).abs().min() > 1e-6


def test_oracle_out_of_range_rows():
    alex, lin = LR.seeded_state_dicts(3)
    gt = frames_of(2, 33, 35, 0)
    pred = frames_of(4, 33, 35, 1)
    got = LR.lpips(pred, gt, [1, -1, 2, 0], alex, lin)
    assert got[1] == 0 and got[2] == 0 and got[0] > 0 and got[3] > 0
    assert torch.equal(got[[0, 3]], LR.lpips(pred[[0, 3]], gt, [1, 0], alex, lin))
    assert not LR.lpips(pred[:1], gt, [5], alex, lin).any()


def test_layer_map_sizes():
    assert LR.map_sizes(450, 450) == [(111, 111), (55, 55), (27, 27), (27, 27), (27, 27)]
    assert LR.map_sizes(31, 31) == [(7, 7), (3, 3), (1, 1), (1, 1), (1, 1)]
    assert LR.map_sizes(37, 101) == [(8, 24), (3, 11), (1, 5), (1, 5), (1, 5)]
    for H, W in ((30, 40), (40, 30), (30, 30)):
        with pytest.raises(RuntimeError):
            LR.map_sizes(H, W)


def test_workspace_bytes_follow_the_maps(M):
    """inerf_lpips_workspace_bytes holds the seven fp32 maps of both images of every row and the head partials, each region rounded up
    to 256 bytes, with the map sizes torch.nn.functional gives."""
    import ctypes
    L = M.lib()
    for B, H, W in ((1, 450, 450), (3, 31, 31), (2, 37, 101), (5, 64, 48)):
        s = LR.map_sizes(H, W)
        hw = [h * w for h, w in s]
        pooled = [s[1][0] * s[1][1], s[2][0] * s[2][1]]
        up = lambda n: (n + 63) // 64 * 64
        maps = [64 * hw[0], 64 * pooled[0], 192 * hw[1], 192 * pooled[1], 384 * hw[2], 256 * hw[3], 256 * hw[4]]
        floats = sum(up(2 * B * m) for m in maps) + sum(up(B * ((n + 31) // 32)) for n in hw)
        got = ctypes.c_size_t(0)
        assert L.inerf_lpips_workspace_bytes(B, H, W, ctypes.byref(got)) == 0
        assert got.value == 4 * floats, (B, H, W)


def test_abi_argument_checks_before_any_launch(M):
    import ctypes
    L = M.lib()
    assert M._lib.INERF_LPIPS_N_PARAMS == 15 and M._lib.INERF_LPIPS_MAX_ROWS == 65535
    need = ctypes.c_size_t(0)
    assert L.inerf_lpips_workspace_bytes(2, 45, 37, ctypes.byref(need)) == 0
    params = (ctypes.c_void_p * 15)(*([A16] * 15))

    def run(**over):
        a = dict(params=params, pred=A16, gt=A16, idx=A16, B=2, H=45, W=37, F=3, ws=A16, nbytes=need.value, out=A16)
        a.update(over)
        return L.inerf_lpips(a["params"], a["pred"], a["gt"], a["idx"], a["B"], a["H"], a["W"], a["F"], a["ws"], a["nbytes"], a["out"], None)

    for name in ("params", "pred", "gt", "idx", "ws", "out"):
        assert run(**{name: None}) == -1, name
        assert b"NULL" in L.inerf_last_error()
    for i in range(15):
        p = (ctypes.c_void_p * 15)(*([A16] * 15))
        p[i] = None
        assert run(params=p) == -1, i
    assert run(B=-1) == -1 and run(F=-1) == -1
    for over in ({"H": 30}, {"W": 30}, {"H": 0}, {"H": 4097, "W": 4097}, {"B": 65536}, {"nbytes": need.value - 1}):
        assert run(**over) == -2, over
        assert b"inerf_lpips" in L.inerf_last_error()
    assert run(B=0, nbytes=0) == 0                                                         # nothing to score, nothing enqueued
    assert run(B=0, H=31, W=31, nbytes=0) == 0
    assert L.inerf_lpips_workspace_bytes(1, 45, 37, None) == -1
    assert L.inerf_lpips_workspace_bytes(-1, 45, 37, ctypes.byref(need)) == -1
    assert L.inerf_lpips_workspace_bytes(1, 30, 37, ctypes.byref(need)) == -2
    assert L.inerf_lpips_workspace_bytes(0, 31, 31, ctypes.byref(need)) == 0 and need.value == 0


def test_load_lpips_key_mapping(tmp_path):
    from ideal_nerf_b200 import ops
    from ideal_nerf_b200.evaluate import load_lpips
    alex, lin = LR.seeded_state_dicts(5)
    w = load_lpips(alex, lin, device="cpu")
    assert len(w) == 15 and [tuple(t.shape) for t in w] == ops.LPIPS_SHAPES
    assert all(t.dtype == torch.float32 and t.is_contiguous() for t in w)
    for k, i in enumerate((0, 3, 6, 8, 10)):
        assert torch.equal(w[2 * k], alex[f"features.{i}.weight"]) and torch.equal(w[2 * k + 1], alex[f"features.{i}.bias"])
        assert torch.equal(w[10 + k], lin[f"lin{k}.model.1.weight"].reshape(-1))
    pa, pl = str(tmp_path / "alexnet.pth"), str(tmp_path / "alex.pth")                    # paths, as the released files come
    torch.save({k: v.double() for k, v in alex.items()}, pa)
    torch.save(lin, pl)
    for a, b in zip(load_lpips(pa, pl, device="cpu"), w):
        assert a.dtype == torch.float32 and torch.equal(a, b)


def test_load_lpips_rejects_bad_files():
    from ideal_nerf_b200.evaluate import load_lpips
    alex, lin = LR.seeded_state_dicts(5)
    no_cls = {k: v for k, v in alex.items() if not k.startswith("classifier")}            # classifier.* is not needed
    assert all(torch.equal(a, b) for a, b in zip(load_lpips(no_cls, lin, device="cpu"), load_lpips(alex, lin, device="cpu")))
    for sd, other, key in ((alex, lin, "features.8.bias"), (lin, alex, "lin3.model.1.weight")):
        broken = {k: v for k, v in sd.items() if k != key}
        args = (broken, other) if sd is alex else (other, broken)
        with pytest.raises(ValueError, match=f"missing key {key}"):
            load_lpips(*args, device="cpu")
    bad = dict(alex, **{"features.3.weight": torch.zeros(192, 64, 3, 3)})
    with pytest.raises(ValueError, match=r"features\.3\.weight has shape"):
        load_lpips(bad, lin, device="cpu")
    bad = dict(lin, **{"lin0.model.1.weight": torch.zeros(64)})
    with pytest.raises(ValueError, match=r"lin0\.model\.1\.weight has shape"):
        load_lpips(alex, bad, device="cpu")
    with pytest.raises(ValueError, match="path or a state dict"):
        load_lpips(alex, [1, 2], device="cpu")


def test_ops_lpips_needs_cuda_tensors():
    from ideal_nerf_b200 import ops
    u8 = lambda *s: torch.zeros(s, dtype=torch.uint8)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        ops.lpips(u8(1, 32, 32, 3), u8(2, 32, 32, 3), torch.zeros(1, dtype=torch.int64), [])


def test_evaluate_split_default_is_unchanged():
    from ideal_nerf_b200.evaluate import evaluate_split
    p = inspect.signature(evaluate_split).parameters
    assert list(p) == ["renderer", "dataset", "latent", "codes", "perturb", "keep_video", "lpips"]
    assert p["lpips"].default is None and p["perturb"].default == 0. and p["keep_video"].default is True
