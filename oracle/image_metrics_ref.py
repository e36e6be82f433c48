"""numpy float64 restatement of inerf_image_metrics (include/inerf_b200.h): exact SSE over the full frame, the face rect and the mouth box,
and SSIM as skimage.metrics.structural_similarity(x, y, channel_axis=-1, gaussian_weights=True, sigma=1.5, use_sample_covariance=False,
data_range=255) computes it.  skimage filters with reflection and then crops the 5 border pixels, so only windows inside the frame count:
here the separable filter runs in 'valid' mode instead, which gives the same numbers without the padding."""
import numpy as np

SIGMA, RADIUS = 1.5, 5                      # skimage: truncate 3.5 -> radius int(3.5 * 1.5 + 0.5) = 5, an 11-tap window
C1, C2 = (0.01 * 255) ** 2, (0.03 * 255) ** 2


def gaussian_taps():
    """scipy.ndimage's 1-D Gaussian of gaussian_filter(sigma=1.5, truncate=3.5): (11,) float64, sums to 1."""
    x = np.arange(-RADIUS, RADIUS + 1, dtype=np.float64)
    w = np.exp(-0.5 / SIGMA ** 2 * x ** 2)
    return w / w.sum()


def _filter_valid(img, w):
    """Separable correlation of (H, W) float64 with the taps w along both axes, valid positions only: (H - 10, W - 10)."""
    k = len(w)
    h = sum(w[i] * img[:, i:img.shape[1] - k + 1 + i] for i in range(k))
    return sum(w[i] * h[i:h.shape[0] - k + 1 + i, :] for i in range(k))


def ssim_map(x, y):
    """Per-position SSIM of one channel: x, y (H, W) -> (H - 10, W - 10) float64."""
    x, y = np.asarray(x, np.float64), np.asarray(y, np.float64)
    w = gaussian_taps()
    ux, uy = _filter_valid(x, w), _filter_valid(y, w)
    vx = _filter_valid(x * x, w) - ux * ux
    vy = _filter_valid(y * y, w) - uy * uy
    vxy = _filter_valid(x * y, w) - ux * uy
    return ((2 * ux * uy + C1) * (2 * vxy + C2)) / ((ux * ux + uy * uy + C1) * (vx + vy + C2))


def ssim(x, y):
    """Mean SSIM of two (H, W, 3) images over the channels and the valid positions (skimage's mssim with channel_axis=-1)."""
    return float(np.mean([ssim_map(x[..., c], y[..., c]).mean() for c in range(x.shape[-1])]))


def box_mask(box, H, W):
    """(H, W) bool of the inclusive box {r0, r1, c0, c1}."""
    rr, cc = np.meshgrid(np.arange(H), np.arange(W), indexing="ij")
    return (rr >= box[0]) & (rr <= box[1]) & (cc >= box[2]) & (cc <= box[3])


def image_metrics(pred, gt_frames, frame_index, bounds=None):
    """inerf_image_metrics on host arrays: pred (B, H, W, 3) uint8, gt_frames (F, H, W, 3) uint8, frame_index (B,), bounds (F, 8) or None.
    Returns (sse (B, 3) int64, npix (B, 3) int64, ssim_sum (B,) float64); a row whose index is outside [0, F) is all zeros, and without
    bounds columns 1 and 2 of sse and npix are 0."""
    pred, gt_frames = np.asarray(pred), np.asarray(gt_frames)
    B, H, W = pred.shape[:3]
    F = gt_frames.shape[0]
    sse, npix, ssim_sum = np.zeros((B, 3), np.int64), np.zeros((B, 3), np.int64), np.zeros(B, np.float64)
    for b, f in enumerate(np.asarray(frame_index).reshape(-1)):
        if not 0 <= f < F:
            continue
        x, y = pred[b], gt_frames[f]
        e = ((x.astype(np.int64) - y.astype(np.int64)) ** 2).sum(-1)
        masks = [np.ones((H, W), bool)] + ([box_mask(bounds[f][:4], H, W), box_mask(bounds[f][4:], H, W)] if bounds is not None else [])
        for j, m in enumerate(masks):
            sse[b, j], npix[b, j] = e[m].sum(), m.sum()
        ssim_sum[b] = sum(ssim_map(x[..., c], y[..., c]).sum() for c in range(3))
    return sse, npix, ssim_sum
