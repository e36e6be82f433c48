"""CPU-side checks of the training-batch pixel sampler: the argument validation of inerf_sample_train_pixels (returns before any device
work), the struct layout, the integer region bounds and torso bits DeviceHeadDataset builds against sample_pixels' float predicates, its
construction checks, and the numpy oracle of the draw."""
import ctypes
import types

import numpy as np
import pytest

from oracle import pixel_sampler_ref as PS

A16 = 0x10000          # fake device address (never dereferenced: every call below fails before a launch)


@pytest.fixture(scope="module")
def M():
    import ideal_nerf_b200 as m
    m.build()
    return m


def reference_masks(face_rect, landmark, parse_img, H, W):
    """The region predicates of HeadDataset.sample_pixels, verbatim: (rect & ~mouth, ~rect, mouth, torso) over p = row * W + col."""
    lm = landmark[48:]
    max_x, min_x = np.max(lm[:, 0]) + 20, np.min(lm[:, 0]) - 20
    max_y, min_y = np.max(lm[:, 1]) + 20, np.min(lm[:, 1]) - 20
    rr, cc = np.meshgrid(np.arange(H), np.arange(W), indexing="ij")
    coords = np.stack([rr, cc], -1).reshape(-1, 2)
    mouth = (coords[:, 0] >= min_x) & (coords[:, 0] <= max_x) & (coords[:, 1] >= min_y) & (coords[:, 1] <= max_y)
    rect = (coords[:, 0] >= face_rect[0]) & (coords[:, 0] <= face_rect[0] + face_rect[2]) & \
           (coords[:, 1] >= face_rect[1]) & (coords[:, 1] <= face_rect[1] + face_rect[3])
    torso = ((parse_img[:, :, 0] == 255) & (parse_img[:, :, 1] == 0) & (parse_img[:, :, 2] == 0)).reshape(-1)
    return np.stack([rect & ~mouth, ~rect, mouth, torso])


def valid_args(M, **over):
    a = M._lib.InerfPixelSampleArgs(H=45, W=37, n_frames=2, k=(ctypes.c_int32 * 4)(40, 10, 8, 2), first=0, count=60,
                                    focal=100., cx=18.5, cy=22.5, near_=0.5, far_=1.2)
    for name in ("frame_index", "bounds", "torso_bits", "poses", "frames", "bc_img", "rng_state", "rays", "target", "bc_rgb", "coords"):
        setattr(a, name, A16)
    for k, v in over.items():
        if k == "k":
            v = (ctypes.c_int32 * 4)(*v)
        setattr(a, k, v)
    return a


def test_struct_size_matches_library(M):
    assert M.lib().inerf_sizeof(4) == ctypes.sizeof(M._lib.InerfPixelSampleArgs)
    assert M.lib().inerf_sizeof(3) == 0


def test_argument_checks_before_any_launch(M):
    L = M.lib()
    need = ctypes.c_size_t(0)
    assert L.inerf_pixel_sampler_workspace_bytes(ctypes.byref(valid_args(M)), ctypes.byref(need)) == 0 and need.value > 0
    assert L.inerf_pixel_sampler_workspace_bytes(None, ctypes.byref(need)) == -1
    assert L.inerf_pixel_sampler_workspace_bytes(ctypes.byref(valid_args(M, H=0)), ctypes.byref(need)) == -2

    def run(args, ws=A16, nbytes=None):
        return L.inerf_sample_train_pixels(None if args is None else ctypes.byref(args), ws, need.value if nbytes is None else nbytes, None)

    assert run(None) == -1
    for name in ("frame_index", "bounds", "torso_bits", "poses", "frames", "bc_img", "rng_state", "rays", "target", "bc_rgb"):
        assert run(valid_args(M, **{name: None})) == -1, name
        assert b"NULL" in L.inerf_last_error()
    assert run(valid_args(M), ws=None) == -1
    for over in ({"H": 0}, {"W": -3}, {"n_frames": 0}, {"H": 2049, "W": 2049}, {"k": (40, -1, 8, 2)},
                 {"first": -1}, {"count": -1}, {"first": 1}, {"count": 61}):
        assert run(valid_args(M, **over)) == -2, over
        assert b"inerf_sample_train_pixels" in L.inerf_last_error()
    assert run(valid_args(M, H=0, frames=None)) == -2                                   # shapes are checked before the pointers
    assert run(valid_args(M, k=(4097, 10, 8, 2), count=10)) == -4                        # one CTA sorts at most 4096 rows of a region
    assert run(valid_args(M), nbytes=need.value - 1) == -2                              # workspace too small
    assert run(valid_args(M), ws=A16 + 8) == -2                                         # or not 256-byte aligned
    assert run(valid_args(M, coords=None, count=0)) == 0                                # nothing to write, nothing enqueued


def adversarial_landmarks(rng, H, W):
    """Mouth landmarks whose thresholds are integral, x.5, negative or beyond the frame."""
    out = []
    for lo, hi in ((np.array([30., 40.]), np.array([50., 61.])),                       # integral thresholds
                   (np.array([30.5, 40.5]), np.array([50.5, 61.5])),                   # x.5 thresholds
                   (np.array([-35.25, 5.]), np.array([10., 15.75])),                   # negative
                   (np.array([H - 5., W - 3.]), np.array([H + 40., W + 100.])),        # beyond the frame
                   (np.array([-100., -100.]), np.array([H + 100., W + 100.])),         # covers everything
                   (np.array([H + 30., 2.]), np.array([H + 50., 9.]))):                # entirely outside
        lm = rng.rand(68, 2) * 10 + 20
        lm[48:] = lo + rng.rand(20, 2) * (hi - lo)
        lm[48], lm[49] = lo, hi
        out.append(lm)
    lm = rng.rand(68, 2) * 10 + 20
    lm[48:] = np.round(rng.rand(20, 2) * 30 + 10) + 0.5                                 # every landmark on a half-integer
    out.append(lm)
    return out


@pytest.mark.parametrize("H,W", [(45, 37), (64, 64)])
def test_integer_bounds_select_the_reference_regions(H, W):
    from ideal_nerf_b200.data import region_bounds
    rng = np.random.RandomState(0)
    parse = np.zeros((H, W, 3), np.uint8)
    parse[H - 6:, :, 0] = 255
    parse[H - 3:, :4, 1] = 7                                                            # not pure red
    rects = ([5, 4, 30, 25], [0, 0, H - 1, W - 1], [-10, -5, 20, 300], [H + 3, 2, 5, 5], [10, 12, 0, 0])
    for lm in adversarial_landmarks(rng, H, W):
        for fr in rects:
            b = region_bounds(np.array(fr, np.int32), lm, H, W)
            assert b.dtype == np.int32
            want = reference_masks(np.array(fr, np.int32), lm, parse, H, W)
            got = PS.region_masks(b, want[3].reshape(H, W), H, W)
            assert np.array_equal(got, want), (fr, lm[48:].min(0), lm[48:].max(0))


@pytest.mark.parametrize("H,W", [(45, 37), (32, 32), (1, 5)])
def test_torso_bits(H, W):
    from ideal_nerf_b200.data import torso_bits
    rng = np.random.RandomState(1)
    parse = rng.randint(0, 2, (H, W, 3)).astype(np.uint8) * 255
    bits = torso_bits(parse)
    assert bits.dtype == np.uint32 and bits.shape == ((H * W + 31) // 32,)
    p = np.arange(H * W)
    unpacked = (bits[p >> 5] >> (p & 31).astype(np.uint32)) & 1
    want = ((parse[:, :, 0] == 255) & (parse[:, :, 1] == 0) & (parse[:, :, 2] == 0)).reshape(-1)
    assert np.array_equal(unpacked.astype(bool), want)
    tail = np.arange(H * W, bits.size * 32)
    assert not ((bits[tail >> 5] >> (tail & 31).astype(np.uint32)) & 1).any()             # padding bits are clear


def test_budgets_and_region_size_checks():
    from ideal_nerf_b200.data import check_region_sizes, region_bounds, region_budgets, region_sizes
    a = types.SimpleNamespace(N_rand=3072, mouth_rays=512, torso_rays=0, sample_rate=0.95)
    assert region_budgets(a) == (int(2560 * 0.95), 2560 - int(2560 * 0.95), 512, 0)
    for bad in (dict(mouth_rays=-1), dict(torso_rays=-5), dict(N_rand=100, mouth_rays=80, torso_rays=30), dict(sample_rate=1.5)):
        with pytest.raises(ValueError, match="negative region budget"):
            region_budgets(types.SimpleNamespace(**dict(vars(a), **bad)))
    H, W = 45, 37
    rng = np.random.RandomState(2)
    lms = adversarial_landmarks(rng, H, W)[:4]
    fr = np.array([5, 4, 30, 25], np.int32)
    torso = np.zeros((H, W), bool)
    torso[H - 4:] = True
    bounds = np.stack([region_bounds(fr, lm, H, W) for lm in lms])
    sizes = region_sizes(bounds, [torso.sum()] * len(lms), H, W)
    for f in range(len(lms)):
        assert np.array_equal(sizes[f], PS.region_masks(bounds[f], torso, H, W).sum(1))
    check_region_sizes(sizes, tuple(sizes.min(0)))                                      # a budget equal to the region's size is fine
    budgets = list(sizes.min(0))
    budgets[2] = int(sizes[1, 2]) + 1                                                   # frame 1's mouth is one pixel short
    short = np.argwhere(sizes[:, 2] < budgets[2])[0, 0]
    with pytest.raises(ValueError, match=rf"frame {short} \(f{short}.jpg\): region 'mouth' has"):
        check_region_sizes(sizes, tuple(budgets), [f"f{i}.jpg" for i in range(len(lms))])


@pytest.mark.parametrize("H,W,budgets", [(45, 37, (300, 120, 60, 40)), (64, 64, (500, 900, 100, 0))])
def test_oracle_selection(H, W, budgets):
    from ideal_nerf_b200.data import region_bounds
    rng = np.random.RandomState(3)
    lm = adversarial_landmarks(rng, H, W)[1]
    b = region_bounds(np.array([5, 4, 30, 25], np.int32), lm, H, W)
    torso = np.zeros((H, W), bool)
    torso[H - 5:] = True
    masks = PS.region_masks(b, torso, H, W)
    picks = []
    for seed, off in ((7, 0), (7, 1), (123456789012, 5)):
        sel = PS.select(seed, off, budgets, b, torso, H, W)
        assert sel.shape == (sum(budgets),) and sel.dtype == np.int64
        keys = PS.pixel_keys(seed, off, H * W)[[0, 0, 1, 2]]
        lo = 0
        for r, k in enumerate(budgets):
            part = sel[lo:lo + k]
            lo += k
            assert masks[r][part].all() and len(np.unique(part)) == k
            v = (keys[r][part].astype(np.uint64) << np.uint64(32)) | part.astype(np.uint64)
            assert (np.diff(v.astype(np.float64)) > 0).all() or k <= 1                   # ascending (key << 32 | p)
            rest = np.setdiff1d(np.nonzero(masks[r])[0], part)
            if len(rest) and k:                                                           # the k smallest of the region
                vr = (keys[r][rest].astype(np.uint64) << np.uint64(32)) | rest.astype(np.uint64)
                assert vr.min() > v.max()
        picks.append(sel)
    assert not np.array_equal(picks[0], picks[1])                                         # a new offset draws a new batch
    with pytest.raises(ValueError):
        PS.select(1, 0, (int(masks[0].sum()) + 1, 0, 0, 0), b, torso, H, W)
