"""numpy restatement of inerf_masked_sse (include/inerf_b200.h): the exact squared error of uint8 frames over a per-frame pixel mask given
as data.torso_bits words (bit p & 31 of word p >> 5 for pixel p = row * W + col)."""
import numpy as np


def unpack_bits(words, n_pixels):
    """(n_pixels,) bool of one frame's mask words; the bits past n_pixels are ignored."""
    w = np.asarray(words).astype(np.uint32)
    p = np.arange(n_pixels)
    return ((w[p >> 5] >> (p & 31).astype(np.uint32)) & 1).astype(bool)


def masked_sse(pred, gt_frames, frame_index, bits):
    """inerf_masked_sse on host arrays: pred (B, H, W, 3) uint8, gt_frames (F, H, W, 3) uint8, frame_index (B,), bits (F, ceil(H*W/32))
    uint32 (or int32 holding the same bits).  Returns (sse (B,) int64, npix (B,) int64); a row whose index is outside [0, F) is zero."""
    pred, gt_frames = np.asarray(pred), np.asarray(gt_frames)
    B, H, W = pred.shape[:3]
    F = gt_frames.shape[0]
    sse, npix = np.zeros(B, np.int64), np.zeros(B, np.int64)
    for b, f in enumerate(np.asarray(frame_index).reshape(-1)):
        if not 0 <= f < F:
            continue
        m = unpack_bits(bits[f], H * W)
        e = ((pred[b].astype(np.int64) - gt_frames[f].astype(np.int64)) ** 2).sum(-1).reshape(-1)
        sse[b], npix[b] = e[m].sum(), m.sum()
    return sse, npix
