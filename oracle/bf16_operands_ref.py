"""Float64 restatements of the operands of the bf16 FaceNeRF training kernels (csrc/mlp_bf16.cu saving builds, mlp_bf16_bwd.cu,
mlp_bf16_dw.cu, the conditioning kernel of mlp_fp32_bwd.cu), and element-wise checkers built on them.

Every saved operand is predicted from the kernel's OWN saved inputs, so no error compounds across layers:
  * a saved activation is bf16_rn(relu(pre)), pre = X . bf16(W)^T + b in float64 from the saved input image X, the bf16-rounded weights
    and the float64-folded bias.  The kernel's pre-activation differs from that by fp32 accumulation in tensor memory, the bias split
    into two bf16 halves (16 significant bits) and the fp32 fold, together at most acc_eps(K) of the sum of the magnitudes of the terms
    (`bound`).  Where the float64 value lies farther than `bound` from a bf16 rounding boundary the saved value is decided and must be
    bit-equal; everywhere it must lie within `bound` + 1 bf16 ulp.
  * the ReLU mask bit is the sign of pre wherever |pre| > bound;
  * a chain delta is bf16_rn(mask * (delta_l . bf16(W_l))) with the same rule;
  * dW / db are delta^T X / sum delta over the saved images, to c * (|delta|^T |X|) with c from the number of fp32 additions.
The checkers return a list of failure strings (empty = pass) and a dict of measured statistics, so a test can run them on corrupted
copies and assert that they reject.  Only tests import this module."""
import math

import torch

from oracle import render_oracle as O

EPS_FP32 = 2.0 ** -23       # one fp32 addition that truncates: at most one ulp of the running magnitude
HEAD_EPS = 2.0 ** -8        # sigma / rgb heads: fp32 dot products on the UN-rounded activations vs the same on the bf16 images


def acc_eps(k):
    """Bound of |kernel accumulator - float64| relative to the sum of |terms| for a K-wide product plus its bias: one tcgen05.mma per 16
    of K plus the bias MMA, each aligning its 16 products and the accumulator to the largest exponent with truncation (at most one fp32
    ulp per addend and one for the sum, 18 in all).  It also covers the bias split into two bf16 halves (2^-17 |b|) and the fp32 fold."""
    return ((k + 15) // 16 + 1) * 18 * EPS_FP32


N_SMS = 148                 # B200: the dW launcher's work split depends on it


# ------------------------------------------------------------------------------------------------
# rays
# ------------------------------------------------------------------------------------------------
def hetero_rays(n, seed, min_angle=0.6):
    """(n, 11) packed rays [o, d, near, far, d/|d|] where every ray has its own origin (in [-0.5, 0.5]^3), its own near / far
    (near in [0.2, 0.7], far - near in [0.3, 1.2]), a direction on the hemisphere z < 0 with |d| in [0.5, 2], and the view direction of
    each ray at least `min_angle` rad from the previous ray's (rejection sampling, seeded)."""
    g = torch.Generator().manual_seed(seed)
    o = torch.rand(n, 3, generator=g) - 0.5
    norm = 0.5 + 1.5 * torch.rand(n, 1, generator=g)
    near = 0.2 + 0.5 * torch.rand(n, 1, generator=g)
    far = near + 0.3 + 0.9 * torch.rand(n, 1, generator=g)
    u = torch.empty(n, 3)
    prev = None
    for i in range(n):
        while True:
            v = torch.randn(3, generator=g, dtype=torch.float64)
            v = v / v.norm()
            v[2] = -abs(float(v[2]))
            if prev is None or float(torch.dot(v, prev)) < math.cos(min_angle):
                break
        u[i] = v.float()
        prev = v
    d = (u * norm).float()
    viewdirs = d / torch.norm(d, dim=-1, keepdim=True)          # as pack_rays computes it
    return torch.cat([o, d, near, far, viewdirs], -1).contiguous()


def adjacent_view_angles(rays):
    v = rays[:, 8:11].double()
    return torch.arccos((v[1:] * v[:-1]).sum(-1).clamp(-1, 1))


def odd_chunk_rays(s, approx):
    """A ray count near `approx` for which n * s points fill an odd number of 256-point chunks, the last one partly."""
    n = approx
    while ((n * s + 255) // 256) % 2 == 0 or (n * s) % 256 == 0:
        n += 1
    return n


# ------------------------------------------------------------------------------------------------
# bf16 helpers
# ------------------------------------------------------------------------------------------------
def bf16(x):
    return x.to(torch.bfloat16).to(x.dtype)


def ulp_bf16(x):
    """ulp of bf16 at |x| (8 significant bits); 2^-133 at 0."""
    _, e = torch.frexp(x.abs())
    return torch.ldexp(torch.ones_like(x), (e - 8).clamp_min(-133))


def _ordered(x):
    b = x.to(torch.bfloat16).view(torch.int16).int()
    return torch.where(b < 0, -(b & 0x7FFF), b)


def bits_bf16(x):
    return x.to(torch.bfloat16).view(torch.int16)


def rounding_stats(got, ref, bound, relu):
    """got: the kernel's bf16 values (any float dtype); ref: the float64 value before rounding (pre-activation if relu);
    bound: per-element bound of |kernel value before rounding - ref|.  Returns the counts the checkers assert on."""
    got, ref = got.double(), ref.double()
    bound = torch.as_tensor(bound, dtype=torch.float64, device=ref.device).expand_as(ref)
    r = ref.clamp_min(0) if relu else ref
    want = bf16(r)
    m, e = torch.frexp(want)
    u = torch.ldexp(torch.ones_like(want), e - 8)
    u = torch.where(m.abs() == 0.5, u / 2, u)                   # below a power of two the boundary is half as far
    dist = u / 2 - (r - want).abs()                             # distance of r to the nearest rounding boundary
    dec = (want != 0) & (dist > bound)
    # an exact float64 zero is decided only when every term is zero (masked, or zero inputs): a sum of bf16 products cancels exactly in
    # float64 while the fp32 accumulator keeps a residual within the bound
    dec = dec | ((ref < -bound) if relu else ((ref == 0) & (bound == 0)))
    mism = got != want
    tol = bound + ulp_bf16(torch.maximum(got.abs(), r.abs()))
    over = (got - r).abs() > tol
    ul = (_ordered(got) - _ordered(want)).abs()
    big = r.abs() > bound
    out = dict(n=ref.numel(), mism=int(mism.sum()), dec_mism=int((mism & dec).sum()), undecided=int((~dec).sum()),
               over=int(over.sum()), max_ulp=int(ul[big].max()) if bool(big.any()) else 0)
    if out["dec_mism"]:                     # the worst decided mismatch: where it is, and how far past the bound the kernel must have been
        idx = (mism & dec).nonzero()
        k = int((dist[mism & dec] / bound[mism & dec]).argmax())
        i = tuple(idx[k].tolist())
        out["worst"] = dict(at=i, got=float(got[i]), want=float(want[i]), ref=float(ref[i]), bound=float(bound[i]), dist=float(dist[i]))
    return out


# ------------------------------------------------------------------------------------------------
# image / mask layout (include/inerf_b200.h, csrc/mlp_common.cuh)
# ------------------------------------------------------------------------------------------------
def img_cols(A, first, n_img):
    """(T, imgs, 128, 64) decoded images -> (T*128, 64*n_img) point-major columns."""
    return A[:, first:first + n_img].permute(0, 2, 1, 3).reshape(-1, 64 * n_img)


def lay_img(l):
    return (4 * l, 4) if l < 8 else (32 + 2 * (l - 8), 2)


IMG_PE, IMG_DIR, IMG_DOUT = 38, 39, 38


def mask_bits(mask, n_tiles, l):
    """(T*128, width) bool: bit (31 - j) of word w of a row = pre-activation 32 w + j of layer l is >= 0."""
    mw = mask.view(torch.int32).reshape(n_tiles, 76, 128)
    w0, nw = (8 * l, 8) if l < 8 else (64 + 4 * (l - 8), 4)
    words = mw[:, w0:w0 + nw].permute(0, 2, 1).reshape(-1, nw)
    sh = 31 - torch.arange(32, device=mask.device)
    return ((words[:, :, None] >> sh[None, None, :]) & 1).reshape(-1, nw * 32).bool()


def encode_images(cols_by_img, n_tiles):
    """Inverse of img_cols + ops.decode_images for CPU-built images: {image index: (T*128, 64) values} -> the swizzled byte buffer."""
    buf = torch.zeros(n_tiles, 40, 128, 8, 8, dtype=torch.bfloat16)
    r = torch.arange(128) & 7
    phys = torch.arange(8)[None, :] ^ r[:, None]                # logical chunk c lives at c ^ (row & 7)
    for i, v in cols_by_img.items():
        t = v.to(torch.bfloat16).reshape(n_tiles, 128, 8, 8)
        out = torch.zeros_like(t)
        out.scatter_(2, phys[None, :, :, None].expand(n_tiles, 128, 8, 8), t)
        buf[:, i] = out
    return buf.reshape(-1).view(torch.uint8)


def encode_mask(bits_by_layer, n_tiles):
    """Inverse of mask_bits: {layer: (T*128, width) bool} -> the mask buffer (uint8 view of [T][76][128] int32 words)."""
    words = torch.zeros(n_tiles, 76, 128, dtype=torch.int64)
    for l, b in bits_by_layer.items():
        w0, nw = (8 * l, 8) if l < 8 else (64 + 4 * (l - 8), 4)
        sh = 31 - torch.arange(32)
        w = (b.reshape(n_tiles, 128, nw, 32).long() << sh).sum(-1)
        words[:, w0:w0 + nw] = w.permute(0, 2, 1)
    words = torch.where(words >= 2 ** 31, words - 2 ** 32, words)
    return words.to(torch.int32).reshape(-1).view(torch.uint8)


# ------------------------------------------------------------------------------------------------
# the folded network in float64
# ------------------------------------------------------------------------------------------------
def cond_vector(aud, expr, lat):
    """[aud | expr / 3 | latent] as the kernels form it: expr / 3 in fp32 round-to-nearest."""
    parts = [t.float().reshape(-1) for t in (aud,) if t is not None]
    if expr is not None:
        parts.append((expr.double().reshape(-1) / 3.0).float())       # RN division (x / 3 never lies on a double-rounding tie)
    if lat is not None:
        parts.append(lat.float().reshape(-1))
    return torch.cat(parts) if parts else torch.zeros(0)


class Net64:
    """The folded network of one FaceNeRF state dict in float64: per layer the activation-column weights (bf16-rounded as the kernel
    streams them), the folded bias and |W_cond| . |c| for the bound."""

    def __init__(self, sd, dims, aud, expr, lat, bias_round=None):
        da, de, dl = dims
        self.C, self.E, self.da = da + de + dl, de, da
        dev = sd["pts_linears.0.weight"].device
        c = cond_vector(aud, expr, lat).to(dev).double()
        self.c32 = cond_vector(aud, expr, lat).to(dev)
        W = lambda k: sd[k].double()
        C, E = self.C, self.E
        self.w, self.b, self.babs = {}, {}, {}
        for l in range(11):
            if l < 8:
                w, b = W(f"pts_linears.{l}.weight"), W(f"pts_linears.{l}.bias")
                if l == 0:
                    wa, wc, cc = w[:, :63], w[:, 63:63 + C], c
                elif l == 5:
                    wa, wc, cc = torch.cat([w[:, :63], w[:, 63 + C:]], 1), w[:, 63:63 + C], c
                else:
                    wa, wc, cc = w, w[:, :0], c[:0]
            else:
                w, b = W(f"views_linears.{l - 8}.weight"), W(f"views_linears.{l - 8}.bias")
                if l == 8:
                    wa, wc, cc = w[:, :256], w[:, 283:283 + E], c[da:da + E]
                    self.wdir = w[:, 256:283]
                else:
                    wa, wc, cc = w, w[:, :0], c[:0]
            self.w[l] = bf16(wa)
            fb = b + wc @ cc
            self.b[l] = fb if bias_round is None else bias_round(fb)
            self.babs[l] = b.abs() + wc.abs() @ cc.abs()
        self.aw, self.ab = W("alpha_linear.weight")[0], W("alpha_linear.bias")[0]
        self.rw, self.rb = W("rgb_linear.weight"), W("rgb_linear.bias")
        self.chain_w = {l: (self.w[l][:, 63:] if l == 5 else self.w[l]) for l in range(1, 11)}


def layer_input(net, l, A, P, dir_img=True):
    """X of layer l from the saved images (float64, P rows): gamma(p) for L0, gamma(p) + h4 for L5, h7 (+ the bf16 gamma(v) image on
    the embedded path) for V0, the previous layer's image otherwise."""
    pe = img_cols(A, IMG_PE, 1)[:P, :63].double()
    if l == 0:
        return pe
    prev = img_cols(A, *lay_img(l - 1))[:P].double()
    if l == 5:
        return torch.cat([pe, prev], 1)
    if l == 8 and dir_img:
        return torch.cat([prev, img_cols(A, IMG_DIR, 1)[:P, :27].double()], 1)
    return prev


def forward_ref(net, l, X, view_enc=None, emb=False, zero_kblock=None):
    """float64 pre-activation of layer l and its bound.  view_enc: float64 gamma(v) per point (fused path: fp32 weights, added as a bias);
    emb: X carries the bf16 gamma(v) image in its last 27 columns, multiplied by bf16 weights.  zero_kblock: (first column) of a 16-wide
    K-block of the weight stage to drop (negative control)."""
    w = net.w[l]
    if l == 8 and emb:
        w = torch.cat([w, bf16(net.wdir)], 1)
    if zero_kblock is not None:
        w = w.clone()
        w[:, zero_kblock:zero_kblock + 16] = 0
    pre = X @ w.T + net.b[l]
    mag = X.abs() @ w.abs().T + net.babs[l]
    if l == 8 and not emb:
        pre = pre + view_enc @ net.wdir.T
        mag = mag + view_enc.abs() @ net.wdir.abs().T
    bound = acc_eps(256 + 64 if l == 8 and emb else w.shape[1]) * mag          # the view K-block is 64 wide
    if l == 8 and not emb:
        bound = bound + 2.0 ** -18 * (view_enc.abs() @ net.wdir.abs().T)        # 27 fp32 FMAs on sincosf values, 2^-24 each
    return pre, bound


# ------------------------------------------------------------------------------------------------
# checkers
# ------------------------------------------------------------------------------------------------
def check_forward(net, A, mask_fn, raw, P, *, view_enc=None, emb=False, max_mism_frac, corrupt=None, layers=range(11)):
    """Every layer's saved activation image and ReLU mask, and raw's sigma / rgb, at all P points.  mask_fn(l) -> (>= P, width) bool.
    corrupt: None, ('kblock', layer, col) to zero a K-block of that layer's reference weights.  Returns (failures, per-layer stats)."""
    fails, stats = [], {}
    for l in layers:
        X = layer_input(net, l, A, P, dir_img=emb)
        zk = corrupt[2] if corrupt is not None and corrupt[0] == "kblock" and corrupt[1] == l else None
        pre, bound = forward_ref(net, l, X, view_enc, emb, zk)
        got = img_cols(A, *lay_img(l))[:P]
        st = rounding_stats(got, pre, bound, relu=True)
        mb = mask_fn(l)[:P]
        sure = pre.abs() > bound
        st["mask_bad"] = int((mb[sure] != (pre[sure] > 0)).sum())
        st["mism_frac"] = st["mism"] / max(1, st["n"])
        stats[l] = st
        if st["dec_mism"] or st["over"] or st["mask_bad"] or st["mism"] > max_mism_frac * st["n"] + 2:
            fails.append(f"layer {l}: {st}")
    if raw is not None:
        h7, v2 = img_cols(A, *lay_img(7))[:P].double(), img_cols(A, *lay_img(10))[:P].double()
        sig = h7 @ net.aw + net.ab
        sb = HEAD_EPS * (h7.abs() @ net.aw.abs()) + EPS_FP32 * net.ab.abs()
        rgb = v2 @ net.rw.T + net.rb
        rbd = HEAD_EPS * (v2.abs() @ net.rw.abs().T) + EPS_FP32 * net.rb.abs()
        r = raw.reshape(-1, 4)[:P].double()
        e_s, e_r = (r[:, 3] - sig).abs() / sb.clamp_min(1e-30), (r[:, :3] - rgb).abs() / rbd.clamp_min(1e-30)
        stats["heads"] = dict(sigma=float(e_s.max()), rgb=float(e_r.max()))
        if float(e_s.max()) > 1 or float(e_r.max()) > 1:
            fails.append(f"heads: max error / bound sigma {float(e_s.max()):.3f} rgb {float(e_r.max()):.3f}")
    return fails, stats


def pe_ref(pts32):
    """gamma_10 in float64 of the fp32 points the kernel forms (fl(o + fl(d z)))."""
    return O.positional_encoding(pts32.double(), 10)


def pe_doubling(pts32):
    """gamma_10 as the fused kernel computes it, in fp32: sin / cos of p once (torch.sin / torch.cos, which on the GPU are the same CUDA
    sinf / cosf as the kernel's sincosf), then per octave sin 2a = fl(2 sin a * cos a) and cos 2a = fl(1 - 2 sin^2 a) (one FMA).  Each
    step is formed exactly in float64 and rounded once, as the kernel rounds."""
    s, c = torch.sin(pts32), torch.cos(pts32)
    parts = [pts32, s, c]
    for _ in range(1, 10):
        sd, cd = s.double(), c.double()
        s, c = (2.0 * sd * cd).float(), (1.0 - 2.0 * sd * sd).float()
        parts += [s, c]
    return torch.cat(parts, -1)


def check_pe_fused(A, pts32, P):
    """PE image == bf16_rn of the kernel's documented gamma(p) arithmetic (pe_doubling) bit for bit, image column 63 zero.  Also measures,
    per octave f, the 1-ulp mismatch fraction against bf16_rn(gamma(p)) in float64 and the largest |fp32 gamma - float64 gamma|: the
    doubling is not the 2^f-growth the angle alone would give -- an amplitude error is multiplied by 4 sin^2 a per step, so the error
    at octave f is bounded by ~3.1^f (two consecutive steps multiply it by at most 9.5) times 2^-23, not 2^f; returns those per octave.
    Returns (failures, {"mism": [...], "err": [...]})."""
    got = img_cols(A, IMG_PE, 1)[:P].double()
    emu = pe_doubling(pts32[:P])
    ref = pe_ref(pts32[:P])
    fails = []
    bad = got[:, :63] != bf16(emu.double())
    if bool(bad.any()):
        fails.append(f"PE image: {int(bad.sum())} entries differ from bf16 of the kernel's gamma(p) arithmetic, "
                     f"columns {sorted(set((bad.nonzero()[:, 1]).tolist()))[:12]}")
    if float(got[:, 63].abs().max()) != 0.0:
        fails.append("PE: column 63 not zero")
    mism, err = [], []
    for f in range(10):
        cols = slice(3 + 6 * f, 9 + 6 * f)
        mism.append(float((got[:, cols] != bf16(ref[:, cols])).double().mean()))
        e = float((emu[:, cols].double() - ref[:, cols]).abs().max())
        err.append(e)
        if e > 3.1 ** f * 2.0 ** -22:
            fails.append(f"PE octave {f}: fp32 gamma {e:.2e} from float64, over 3.1^f * 2^-22")
    return fails, dict(mism=mism, err=err)


def dir_ref(rays, s, P):
    """gamma_4 in float64 of the view direction of ray p // s, per point."""
    v = rays[:, 8:11].double()
    return O.positional_encoding(v, 4).repeat_interleave(s, 0)[:P]


def check_dir_fused(A, ref_enc, P):
    """DIR image vs bf16_rn(ref_enc), ref_enc = gamma_4 in float64 of the view direction of ray p // s per point (dir_ref): within 1 ulp,
    bit-equal where decided (sincosf of exact 2^f multiples); columns 27..63 zero."""
    got = img_cols(A, IMG_DIR, 1)[:P].double()
    st = rounding_stats(got[:, :27], ref_enc[:P], 2.0 ** -22, relu=False)
    fails = [f"DIR: {st}"] if st["over"] or st["dec_mism"] else []
    if float(got[:, 27:].abs().max()) != 0.0:
        fails.append("DIR: columns 27..63 not zero")
    return fails, st


def check_embedded_inputs(A, x, P):
    """Embedded rows: PE image == bf16(x[:, :63]) and DIR image == bf16(x[:, 63:90]) bit for bit, padding columns zero."""
    pe, di = img_cols(A, IMG_PE, 1)[:P], img_cols(A, IMG_DIR, 1)[:P]
    fails = []
    if not torch.equal(bits_bf16(pe[:, :63]), bits_bf16(x[:P, :63].float())) or float(pe[:, 63].abs().max()) != 0:
        fails.append("PE image != bf16(x[:, :63])")
    if not torch.equal(bits_bf16(di[:, :27]), bits_bf16(x[:P, 63:90].float())) or float(di[:, 27:].abs().max()) != 0:
        fails.append("DIR image != bf16(x[:, 63:90])")
    return fails


def check_chain(net, D, mask_fn, d_raw, P, *, max_mism_frac):
    """The chain's delta images against the float64 product of the NEXT layer's saved delta image with bf16(W), masked with the kernel's
    own mask, bf16 rounded; d_v2 from d_raw through rgb_linear (fp32 FMAs); the d_raw image == bf16(d_raw); rows past P zero."""
    fails, stats = [], {}
    dr = d_raw.reshape(-1, 4)[:P]
    dout = img_cols(D, IMG_DOUT, 1)
    if not torch.equal(bits_bf16(dout[:P, :4]), bits_bf16(dr.float())) or float(dout[:P, 4:].abs().max()) != 0:
        fails.append("d_raw image != bf16(d_raw)")
    dr64 = dr.double()
    for l in range(10, -1, -1):
        if l == 10:
            pre, mag = dr64[:, :3] @ net.rw, dr64[:, :3].abs() @ net.rw.abs()
        else:
            dn = img_cols(D, *lay_img(l + 1))[:P].double()
            w = net.chain_w[l + 1]
            pre, mag = dn @ w, dn.abs() @ w.abs()
            if l == 7:
                pre = pre + dr64[:, 3:4] * net.aw[None, :]
                mag = mag + dr64[:, 3:4].abs() * net.aw.abs()[None, :]
        m = mask_fn(l)[:P]
        ref = torch.where(m, pre, torch.zeros((), dtype=pre.dtype, device=pre.device))
        got = img_cols(D, *lay_img(l))
        st = rounding_stats(got[:P], ref, acc_eps(w.shape[0] + (1 if l == 7 else 0) if l < 10 else 3) * mag, relu=False)
        st["mism_frac"] = st["mism"] / max(1, st["n"])
        st["tail"] = float(got[P:].abs().max()) if got.shape[0] > P else 0.0
        stats[l] = st
        if st["dec_mism"] or st["over"] or st["tail"] != 0.0 or st["mism"] > max_mism_frac * st["n"] + 2:
            fails.append(f"delta of layer {l}: {st}")
    return fails, stats


def dw_constant(n_tiles, n_sms=N_SMS, n_tasks=24):
    """c of the dW bound: a work item accumulates 8 MMAs (K = 16) per 128-point tile of its range in fp32, then the ranges meet in
    fp32 atomic adds; each addition may lose up to 2^-23 of the running magnitude (truncating accumulation included)."""
    chunks = max(1, min((4 * n_sms + n_tasks - 1) // n_tasks, n_tiles))
    per = (n_tiles + chunks - 1) // chunks
    n_chunks = (n_tiles + per - 1) // per
    return (8 * per + n_chunks + 8) * 2.0 ** -23, per


class DwAccum:
    """delta^T X, |delta|^T |X|, sum delta, sum |delta| of every weight gradient in float64, accumulated over batches of tiles."""

    def __init__(self):
        self.ref, self.mag = {}, {}

    def _add(self, key, v, m):
        if key in self.ref:
            self.ref[key] += v
            self.mag[key] += m
        else:
            self.ref[key], self.mag[key] = v, m

    def add(self, net, A, D, rows):
        """rows: the valid rows of this batch of tiles (points < P)."""
        for l in range(11):
            d = img_cols(D, *lay_img(l))[:rows].double()
            X = layer_input(net, l, A, rows, dir_img=True)
            self._add(("w", l), d.T @ X, d.abs().T @ X.abs())
            self._add(("b", l), d.sum(0), d.abs().sum(0))
        do = img_cols(D, IMG_DOUT, 1)[:rows, :4].double()
        h7, v2 = img_cols(A, *lay_img(7))[:rows].double(), img_cols(A, *lay_img(10))[:rows].double()
        self._add(("w", "alpha"), do[:, 3:4].T @ h7, do[:, 3:4].abs().T @ h7)
        self._add(("w", "rgb"), do[:, :3].T @ v2, do[:, :3].abs().T @ v2)
        self._add(("b", "alpha"), do[:, 3].sum(0, keepdim=True), do[:, 3].abs().sum(0, keepdim=True))
        self._add(("b", "rgb"), do[:, :3].sum(0), do[:, :3].abs().sum(0))


def dw_got(g, net, key):
    """The kernel's gradient entries that key's reference covers (nn.Linear layout, activation columns)."""
    kind, l = key
    C, E = net.C, net.E
    if l == "alpha":
        return g[22] if kind == "w" else g[23]
    if l == "rgb":
        return g[24] if kind == "w" else g[25]
    wi = 2 * l if l < 8 else 16 + 2 * (l - 8)
    if kind == "b":
        return g[wi + 1]
    if l == 0:
        return g[0][:, :63]
    if l == 5:
        return torch.cat([g[10][:, :63], g[10][:, 63 + C:]], 1)
    if l == 8:
        return g[16][:, :283]
    return g[wi]


def check_dw(net, g, acc, c, scale_row=None):
    """Every dW / db entry: |got - delta^T X| <= c * (|delta|^T |X|).  scale_row: (key, row) of the kernel's gradient to multiply by
    1.001 first (negative control).  Returns (failures, max error / bound per key)."""
    fails, stats = [], {}
    for key in acc.ref:
        got = dw_got(g, net, key).double()
        if scale_row is not None and scale_row[0] == key:
            got = got.clone()
            got[scale_row[1]] *= 1.001
        ratio = (got - acc.ref[key]).abs() / (c * acc.mag[key]).clamp_min(1e-300)
        zero_ok = bool(((acc.mag[key] == 0) <= (got == 0)).all())
        stats[key] = float(ratio.max())
        if stats[key] > 1.0 or not zero_ok:
            fails.append(f"{key}: max error / bound {stats[key]:.3f}")
    return fails, stats


def check_fold(net, cond_buf):
    """The fp32 folded biases of inerf_mlp_fold_cond against float64: |got - b| <= 2^-20 (|b| + |W_cond| |c|)."""
    got = cond_buf[:8 * 256 + 3 * 128].double()
    ref = torch.cat([net.b[l] for l in range(11)])
    mag = torch.cat([net.babs[l] for l in range(11)])
    r = float(((got - ref).abs() / (2.0 ** -20 * mag)).max())
    return ([f"fold: max error / bound {r:.3f}"] if r > 1 else []), r


def check_cond_grads(sd, dims, g, d_cond, aud, expr, lat):
    """Folded conditioning columns of the weight gradients == db (x) c bit for bit (one fp32 product each, c = [aud | fp32(expr / 3) |
    latent]); d_cond == W_cond^T db in float64 (expr part / 3) to 2^-18 of sum |W db|."""
    da, de, dl = dims
    C = da + de + dl
    c = cond_vector(aud, expr, lat).to(g[0].device)
    fails = []
    jobs = [(0, 1, 63, 0, C), (10, 11, 63, 0, C)] + ([(16, 17, 283, da, de)] if de else [])
    ref = torch.zeros(C, dtype=torch.float64, device=c.device)
    mag = torch.zeros_like(ref)
    for wi, bi, col0, j0, nj in jobs:
        got = g[wi][:, col0:col0 + nj]
        want = g[bi][:, None] * c[None, j0:j0 + nj]
        if not torch.equal(got.view(torch.int32), want.view(torch.int32)):
            fails.append(f"cond columns of grad {wi}: {int((got != want).sum())} entries differ from db (x) c")
        w = sd[["pts_linears.0.weight", "pts_linears.5.weight", "views_linears.0.weight"][[0, 10, 16].index(wi)]].double()
        wc, db = w[:, col0:col0 + nj], g[bi].double()
        ref[j0:j0 + nj] += wc.T @ db
        mag[j0:j0 + nj] += wc.abs().T @ db.abs()
    ref[da:da + de] /= 3
    mag[da:da + de] /= 3
    r = float(((d_cond[:C].double() - ref).abs() / (2.0 ** -18 * mag).clamp_min(1e-300)).max()) if C else 0.0
    if r > 1:
        fails.append(f"d_cond: max error / bound {r:.3f}")
    return fails, r
