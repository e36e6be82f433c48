"""float64 torch-CPU restatement of inerf_lpips (include/inerf_b200.h): LPIPS v0.1 with the AlexNet trunk of Zhang et al., "The
Unreasonable Effectiveness of Deep Features as a Perceptual Metric" (CVPR 2018), eq. 1,

    d(x, x0) = sum_l 1 / (H_l W_l) sum_{h, w} || w_l * (y^l_hw - y0^l_hw) ||_2^2,

where y^l_hw is the layer-l AlexNet feature at (h, w) unit-normalised over the channels, as the lpips package's v0.1 computes it
(lpips.LPIPS(net='alex', version='0.1'), normalize=False): im2tensor's x = byte / 127.5 - 1, the ScalingLayer, features relu1..relu5,
normalize_tensor f / (sqrt(sum_c f^2) + 1e-10), NetLinLayer (a 1 x 1 convolution without bias) and spatial_average.  Frames are uint8
(H, W, 3) BGR as stored; AlexNet is fed R, G, B.  State dicts as the two released files hold them: torchvision's AlexNet
(features.{0,3,6,8,10}.{weight,bias}) and lpips' alex.pth (lin{0..4}.model.1.weight, (1, C, 1, 1))."""
import torch
import torch.nn.functional as F

SHIFT = (-.030, -.088, -.188)
SCALE = (.458, .448, .450)
CONV = (0, 3, 6, 8, 10)                                 # torchvision's features index of conv1..conv5
GEOMETRY = ((4, 2), (1, 2), (1, 1), (1, 1), (1, 1))    # (stride, padding) of conv1..conv5
POOL_AFTER = (True, True, False, False, False)


def scaled_input(frames_u8):
    """(N, H, W, 3) uint8 BGR -> (N, 3, H, W) float64 RGB after im2tensor and the ScalingLayer."""
    x = torch.as_tensor(frames_u8).to(torch.float64).flip(-1).permute(0, 3, 1, 2)
    x = x / 127.5 - 1.
    shift = torch.tensor(SHIFT, dtype=torch.float64).view(1, 3, 1, 1)
    scale = torch.tensor(SCALE, dtype=torch.float64).view(1, 3, 1, 1)
    return (x - shift) / scale


def features(x, alexnet):
    """relu1..relu5 of AlexNet on scaled input x (N, 3, H, W) float64."""
    out = []
    for k, (i, (stride, pad)) in enumerate(zip(CONV, GEOMETRY)):
        w = alexnet[f"features.{i}.weight"].to(torch.float64)
        b = alexnet[f"features.{i}.bias"].to(torch.float64)
        x = F.relu(F.conv2d(x, w, b, stride=stride, padding=pad))
        out.append(x)
        if POOL_AFTER[k]:
            x = F.max_pool2d(x, 3, 2)
    return out


def map_sizes(H, W):
    """(h, w) of relu1..relu5 for H x W frames, from the shapes torch.nn.functional gives."""
    x = torch.zeros(1, 3, H, W, dtype=torch.float64)
    sizes = []
    for k, (stride, pad) in enumerate(GEOMETRY):
        ks = (11, 5, 3, 3, 3)[k]
        x = F.conv2d(x, torch.zeros(1, x.shape[1], ks, ks, dtype=torch.float64), stride=stride, padding=pad)
        sizes.append(tuple(x.shape[2:]))
        if POOL_AFTER[k]:
            x = F.max_pool2d(x, 3, 2)
    return sizes


def seeded_state_dicts(seed):
    """(alexnet, lin) state dicts in the two released files' key layouts, scaled like trained weights so that no layer saturates or dies:
    Kaiming-uniform convolutions (bound sqrt(6 / fan_in)), biases 0.01 +- 0.005, non-negative lin weights as in the released heads, and
    classifier.* entries that LPIPS does not use."""
    g = torch.Generator().manual_seed(seed)
    u = lambda shape, lo, hi: lo + (hi - lo) * torch.rand(shape, generator=g, dtype=torch.float32)
    alexnet = {}
    for i, (cout, cin, k) in zip(CONV, ((64, 3, 11), (192, 64, 5), (384, 192, 3), (256, 384, 3), (256, 256, 3))):
        bound = (6. / (cin * k * k)) ** .5
        alexnet[f"features.{i}.weight"] = u((cout, cin, k, k), -bound, bound)
        alexnet[f"features.{i}.bias"] = u((cout,), .005, .015)
    alexnet["classifier.1.weight"] = u((16, 9216), -.01, .01)
    alexnet["classifier.1.bias"] = u((16,), -.01, .01)
    lin = {f"lin{k}.model.1.weight": u((1, c, 1, 1), 0., .2) for k, c in enumerate((64, 192, 384, 256, 256))}
    return alexnet, lin


def lpips(pred, gt_frames, frame_index, alexnet, lin):
    """inerf_lpips on host data: pred (B, H, W, 3) uint8, gt_frames (F, H, W, 3) uint8, frame_index (B,).  Returns (B,) float64; a row
    whose index is outside [0, F) is 0."""
    pred, gt_frames = torch.as_tensor(pred), torch.as_tensor(gt_frames)
    index = [int(f) for f in torch.as_tensor(frame_index).reshape(-1)]
    out = torch.zeros(len(index), dtype=torch.float64)
    live = [b for b, f in enumerate(index) if 0 <= f < gt_frames.shape[0]]
    if not live:
        return out
    fa = features(scaled_input(pred[live]), alexnet)
    fb = features(scaled_input(gt_frames[[index[b] for b in live]]), alexnet)
    total = torch.zeros(len(live), dtype=torch.float64)
    for k, (a, g) in enumerate(zip(fa, fb)):
        na = a / (a.pow(2).sum(1, keepdim=True).sqrt() + 1e-10)
        ng = g / (g.pow(2).sum(1, keepdim=True).sqrt() + 1e-10)
        w = lin[f"lin{k}.model.1.weight"].to(torch.float64).reshape(1, -1, 1, 1)
        total = total + ((na - ng) ** 2 * w).sum(1).mean((1, 2))
    out[live] = total
    return out
