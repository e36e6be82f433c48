"""The pixel draw of inerf_sample_train_pixels in numpy -- TEST INFRASTRUCTURE ONLY (checker of ideal-nerf_b200/csrc/pixel_sampler.cu).

The contract is the one written above InerfPixelSampleArgs in include/inerf_b200.h: pixel p = row * W + col is keyed by the words
(x, y, z, w) of Philox4x32-10 block p of stream INERF_RNG_STREAM_PIXELS; the regions rect = R & ~M, norect = ~R, mouth = M, torso = T use
the words x, x, y, z; each region keeps its k members with the smallest (key << 32 | p), in ascending order of that value; the regions
are concatenated rect, norect, mouth, torso."""
import numpy as np

from oracle.philox_ref import philox4x32_10

STREAM_PIXELS = 3


def pixel_keys(seed, offset, n):
    """(4, n) uint32: the Philox words of pixels 0..n-1."""
    p = np.arange(n, dtype=np.uint64)
    off = (int(offset) + (STREAM_PIXELS << 56)) & 0xFFFFFFFFFFFFFFFF
    w = philox4x32_10((p & np.uint64(0xFFFFFFFF)).astype(np.uint32), (p >> np.uint64(32)).astype(np.uint32),
                      np.uint32(off & 0xFFFFFFFF), np.uint32(off >> 32), seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    return np.stack(w)


def region_masks(bounds, torso, H, W):
    """Boolean (4, H*W) masks of rect, norect, mouth, torso from the int32 bounds of data.region_bounds and a (H, W) torso mask."""
    rr, cc = np.meshgrid(np.arange(H), np.arange(W), indexing="ij")
    rr, cc = rr.reshape(-1), cc.reshape(-1)
    b = bounds
    R = (rr >= b[0]) & (rr <= b[1]) & (cc >= b[2]) & (cc <= b[3])
    M = (rr >= b[4]) & (rr <= b[5]) & (cc >= b[6]) & (cc <= b[7])
    return np.stack([R & ~M, ~R, M, np.asarray(torso, bool).reshape(-1)])


def select(seed, offset, budgets, bounds, torso, H, W):
    """(N_rand,) int64 pixel indices in output order (rect, norect, mouth, torso)."""
    keys = pixel_keys(seed, offset, H * W)[[0, 0, 1, 2]]
    masks = region_masks(bounds, torso, H, W)
    out = []
    for r, k in enumerate(budgets):
        members = np.nonzero(masks[r])[0]
        if len(members) < k:
            raise ValueError(f"region {r} has {len(members)} members, fewer than {k}")
        order = np.lexsort((members, keys[r][members]))          # by key, then by pixel index
        out.append(members[order[:k]])
    return np.concatenate(out).astype(np.int64)
