"""FaceNeRF: the audio/expression-conditioned NeRF MLP of models/face_nerf.py:8-80.

Same constructor, same ``forward(x, aud, expr, latent_code)`` signature and -- because the layers are
ordinary ``nn.Linear`` modules with the reference's attribute names -- the same ``state_dict`` keys
(``pts_linears.0-7``, ``views_linears.0-2``, ``feature_linear``, ``alpha_linear``, ``rgb_linear``),
so ``head.tar`` / ``*_torso.tar`` checkpoints load unchanged.  The arithmetic is one fused CUDA kernel
(csrc/mlp_fp32.cu or csrc/mlp_bf16.cu) fed with the conditioning folded into biases.
"""
import torch
import torch.nn as nn

from . import _lib, ops

# "bf16": tcgen05 kernels for inference and training, on both entries -- query(rays, z) and forward(x) on embedded rows (the latter with
# its own packed blob, INERF_MLP_BF16_EMB).  "fp16x2": tensor cores at fp32-gate accuracy (fp16 hi/lo operand pairs, three MMA passes)
# for inference on both entries (forward(x) with its own blob and mode, INERF_MLP_F16X2_EMB); training in this mode runs the fp32
# kernels, like "fp32"
MODES = {"fp32": _lib.INERF_MLP_FP32, "bf16": _lib.INERF_MLP_BF16, "fp16x2": _lib.INERF_MLP_F16X2}


class FaceNeRF(nn.Module):
    def __init__(self, D=8, W=256, input_ch=63, input_ch_views=27, dim_aud=64, dim_latent=0, dim_expr=0,
                 output_ch=4, skips=None, use_viewdirs=True, mlp_mode="fp32"):
        super(FaceNeRF, self).__init__()
        if skips is None:
            skips = [4]
        if not (D == 8 and W == 256 and input_ch == 63 and input_ch_views == 27 and list(skips) == [4]
                and use_viewdirs):
            raise NotImplementedError("ideal-nerf_b200 builds the configuration every reference script uses: "
                                      "D=8, W=256, input_ch=63, input_ch_views=27, skips=[4], use_viewdirs=True")
        self.D, self.W = D, W
        self.input_xyz_ch, self.input_views_ch = input_ch, input_ch_views
        self.dim_aud, self.dim_expr, self.dim_latent = dim_aud, dim_expr, dim_latent
        self.skips, self.use_viewdirs = skips, use_viewdirs
        self.mlp_mode = mlp_mode

        input_ch_all = input_ch + dim_aud + dim_expr + dim_latent
        self.pts_linears = nn.ModuleList(
            [nn.Linear(input_ch_all, W)] + [nn.Linear(W, W) if i not in skips else nn.Linear(W + input_ch_all, W)
                                            for i in range(D - 1)])
        self.views_linears = nn.ModuleList([nn.Linear(input_ch_views + W + dim_expr, W // 2)] +
                                           [nn.Linear(W // 2, W // 2) for _ in range(D // 4)])
        self.feature_linear = nn.Linear(W, W)     # constructed, never applied (face_nerf.py:34) -- kept for checkpoints
        self.alpha_linear = nn.Linear(W, 1)
        self.rgb_linear = nn.Linear(W // 2, 3)
        self._dims = ops.net_dims(dim_aud, dim_expr, dim_latent)
        self._packed = None
        self._packed_key = None
        self._packed_t = None
        self._packed_t_key = None
        self._packed_e = None
        self._packed_e_key = None

    # -- plumbing -------------------------------------------------------------------------------
    def kernel_params(self):
        """The 26 tensors in include/inerf_b200.h order."""
        ps = []
        for l in self.pts_linears:
            ps += [l.weight, l.bias]
        for l in self.views_linears:
            ps += [l.weight, l.bias]
        ps += [self.alpha_linear.weight, self.alpha_linear.bias, self.rgb_linear.weight, self.rgb_linear.bias]
        return ps

    def _mode(self):
        try:
            return MODES[self.mlp_mode]
        except KeyError:
            raise ValueError(f"mlp_mode must be one of {sorted(MODES)}, got {self.mlp_mode!r}")

    def invalidate_packed(self):
        """Drop the cached packed weights.  The cache key is (data_ptr, _version) of every parameter, which in-place updates that bypass
        autograd's version counters do not change -- torch.optim.Adam(fused=True) is one -- so the training path never trusts it (it
        re-packs on every call and invalidates afterwards) and train() / eval() switches drop it as well."""
        self._packed = self._packed_key = None
        self._packed_t = self._packed_t_key = None
        self._packed_e = self._packed_e_key = None

    def train(self, mode=True):
        self.invalidate_packed()
        return super().train(mode)

    def packed_weights(self, params, out=None):
        """Mode-specific packed weights, re-packed whenever a parameter was updated in place.  out: a blob of this mode's size that must
        hold them (a captured CUDA graph reads it): the weights are packed into it unless it already is the current cached blob."""
        mode = self._mode()
        if mode == _lib.INERF_MLP_FP32:
            return None
        key = (mode, tuple((p.data_ptr(), p._version) for p in params))
        if key != self._packed_key or (out is not None and self._packed is not out):
            self._packed = ops.pack_weights(mode, self._dims, [p.detach() for p in params], out=out)
            self._packed_key = key
        return self._packed

    def packed_weights_bwd(self, params):
        """Transposed stage images for the bf16 backward chain (re-packed when a parameter changed)."""
        key = tuple((p.data_ptr(), p._version) for p in params)
        if key != getattr(self, "_packed_t_key", None):
            self._packed_t = ops.pack_weights(_lib.INERF_MLP_BF16_BWD, self._dims, [p.detach() for p in params])
            self._packed_t_key = key
        return self._packed_t

    def packed_weights_emb(self, params):
        """Stage images of the embedded-row kernel (FaceNeRF.forward) of the current tensor-core mode -- INERF_MLP_BF16_EMB or
        INERF_MLP_F16X2_EMB -- re-packed when a parameter or the mode changed."""
        mode = _lib.INERF_MLP_F16X2_EMB if self._mode() == _lib.INERF_MLP_F16X2 else _lib.INERF_MLP_BF16_EMB
        key = (mode, tuple((p.data_ptr(), p._version) for p in params))
        if key != self._packed_e_key:
            self._packed_e = ops.pack_weights(mode, self._dims, [p.detach() for p in params])
            self._packed_e_key = key
        return self._packed_e

    def _prep(self, aud, expr, latent_code):
        params = self.kernel_params()
        for p in params:
            if not p.is_cuda:
                raise RuntimeError("FaceNeRF parameters must live on a CUDA device (no CPU path)")
        if (aud is None) != (self.dim_aud == 0) or (expr is None) != (self.dim_expr == 0) \
                or (latent_code is None) != (self.dim_latent == 0):
            raise ValueError("aud/expr/latent_code must be given exactly for the non-zero dim_aud/dim_expr/dim_latent")
        return params

    # -- reference signature --------------------------------------------------------------------
    def forward(self, x, aud, expr=None, latent_code=None):
        """x (P, 63+27) already embedded, as in face_nerf.py:40.  Returns (P, 4) = [rgb, sigma] pre-activation."""
        params = self._prep(aud, expr, latent_code)
        return _MlpFn.apply(self, (True, self._wants_grad(params, aud, expr, latent_code)), x, None, aud, expr, latent_code, *params)

    # -- fused entry used by render_rays ----------------------------------------------------------
    def query(self, rays, z_vals, aud, expr=None, latent_code=None):
        """run_network on the points o + d*z of packed rays (n,11) / depths (n,s): returns raw (n,s,4)."""
        params = self._prep(aud, expr, latent_code)
        return _MlpFn.apply(self, (False, self._wants_grad(params, aud, expr, latent_code)), rays, z_vals, aud, expr, latent_code, *params)

    @staticmethod
    def _wants_grad(params, *cond):
        """Training path only when autograd is recording (grad mode is always off INSIDE Function.forward, and
        needs_input_grad ignores torch.no_grad(), so this is decided here)."""
        return torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in list(params) + list(cond))


class _MlpFn(torch.autograd.Function):
    """run_network + FaceNeRF as one op.  Inference: one fused kernel in the module's mlp_mode.  Training (any
    parameter or conditioning vector requires grad): the forward keeps its activations and backward() runs the analytic
    gradient kernels -- fp32 FFMA (csrc/mlp_fp32_bwd.cu) or bf16 tcgen05 (csrc/mlp_bf16_bwd.cu + mlp_bf16_dw.cu) by mlp_mode."""

    @staticmethod
    def forward(ctx, net, flags, a, b, aud, expr, latent, *params):
        embedded, train = flags
        mode = net._mode()
        pd = [p.detach() for p in params]
        f = lambda t: None if t is None else ops.f32c(t.detach(), "conditioning").reshape(-1)
        aud_d, expr_d, lat_d = f(aud), f(expr), f(latent)
        cond = ops.fold_cond(net._dims, pd, aud_d, expr_d, lat_d)
        if train:
            ctx.net, ctx.has = net, (aud is not None, expr is not None, latent is not None)
            ctx.cond_shapes = tuple(None if t is None else t.shape for t in (aud, expr, latent))
            if mode == _lib.INERF_MLP_BF16:
                net.invalidate_packed()                       # optimiser steps may not bump parameter versions (fused Adam)
                if embedded:
                    out, acts, mask, n_points = ops.mlp_fwd_train_bf16(net._dims, pd, net.packed_weights_emb(params), cond, x=a)
                else:
                    out, acts, mask, n_points = ops.mlp_fwd_train_bf16(net._dims, pd, net.packed_weights(params), cond, a, b)
                ctx.n_points, ctx.bf16 = n_points, True
                ctx.save_for_backward(acts, mask, *[t for t in (aud_d, expr_d, lat_d) if t is not None], *pd)
                ctx.packed_t = net.packed_weights_bwd(params)
                net.invalidate_packed()                       # ... and the next inference call must not reuse this step's pack
                return out
            net.invalidate_packed()                           # a later bf16 inference call must re-pack: in-place optimiser updates
            out, acts, n_points = ops.mlp_fwd_train(net._dims, pd, cond, x=a) if embedded else \
                ops.mlp_fwd_train(net._dims, pd, cond, rays=a, z=b)                                 # do not bump parameter versions
            ctx.n_points, ctx.bf16 = n_points, False
            ctx.save_for_backward(acts, *[t for t in (aud_d, expr_d, lat_d) if t is not None], *pd)
            return out
        if embedded and mode == _lib.INERF_MLP_BF16:
            return ops.mlp_fwd_embedded(mode, net._dims, pd, net.packed_weights_emb(params), cond, a)
        if embedded and mode == _lib.INERF_MLP_F16X2:       # the embedded-row kernel has its own mode value: the blobs differ
            return ops.mlp_fwd_embedded(_lib.INERF_MLP_F16X2_EMB, net._dims, pd, net.packed_weights_emb(params), cond, a)
        packed = net.packed_weights(params)
        if embedded:
            return ops.mlp_fwd_embedded(mode, net._dims, pd, packed, cond, a)
        return ops.mlp_fwd(mode, net._dims, pd, packed, cond, a, b)

    @staticmethod
    def backward(ctx, g):
        saved = list(ctx.saved_tensors)
        acts = saved.pop(0)
        mask = saved.pop(0) if ctx.bf16 else None
        aud = saved.pop(0) if ctx.has[0] else None
        expr = saved.pop(0) if ctx.has[1] else None
        latent = saved.pop(0) if ctx.has[2] else None
        params = saved
        d = ctx.net._dims
        if ctx.bf16:
            grads, d_cond = ops.mlp_bwd_bf16(d, params, ctx.packed_t, aud, expr, latent, acts, mask, g, ctx.n_points)
        else:
            grads, d_cond = ops.mlp_bwd(d, params, aud, expr, latent, acts, g, ctx.n_points)
        da, de = d.dim_aud, d.dim_expr
        sh = ctx.cond_shapes                                  # the conditioning vectors may arrive as (C,), (1, C), ...: same shape back
        g_aud = d_cond[:da].view(sh[0]) if aud is not None else None
        g_expr = d_cond[da:da + de].view(sh[1]) if expr is not None else None
        g_lat = d_cond[da + de:da + de + d.dim_latent].view(sh[2]) if latent is not None else None
        return (None, None, None, None, g_aud, g_expr, g_lat, *grads)
