"""The render_rays pipeline: host-side mirror of the reference's renderer classes/functions.

  Network (class form)      NeRFs/HeadNeRF/train/audio_exp_nerf.py:198-439 (== test/eval_aud_exp_nerf.py:191-432)
  TorsoNetwork              NeRFs/TorsoNeRF/train_torso.py:186-431 (head + torso, composite at :269-270)
  raw2outputs               NeRFs/HeadNeRF/train/baseline.py:325-375; torso variant NeRFs/TorsoNeRF/test_torso.py:352-402
  render_rays (functional)  NeRFs/HeadNeRF/train/baseline.py:378-448

Each stage is one CUDA kernel behind include/inerf_b200.h:
  stratified depths -> inerf_sample_coarse, points+PE+FaceNeRF -> inerf_mlp_fwd,
  raw2outputs -> inerf_composite_fwd/bwd, sample_pdf+sort+std -> inerf_importance_sample.
No (P,90) embedding, no (N,S,3) point tensor and no torch.cat of netchunks is ever materialised.
"""
import logging
from types import SimpleNamespace

import numpy as np
import torch
import torch.nn as nn

from . import _lib, ops
from .audio_net import AudioNet, AudioAttNet
from .face_nerf import FaceNeRF
from .helper import config_parser, get_embedder

logger = logging.getLogger('adnerf')


def default_args(**over):
    args = config_parser().parse_args([])
    for k, v in over.items():
        setattr(args, k, v)
    return args


# ------------------------------------------------------------------------------------------------
# raw2outputs
# ------------------------------------------------------------------------------------------------
def _noise(raw, raw_noise_std, pytest):
    if not raw_noise_std > 0.:
        return None
    shape = raw[..., 3].shape
    if pytest:                                               # baseline.py:356-359 (note: rand, not randn)
        np.random.seed(0)
        return torch.Tensor(np.random.rand(*list(shape)) * raw_noise_std).to(raw.device)
    return torch.randn(shape, device=raw.device) * raw_noise_std


def raw2outputs(raw, z_vals, rays_d, bc_rgb, raw_noise_std=0., white_bkgd=False, pytest=False):
    """baseline.py:325 -> (rgb_map, disp_map, acc_map, weights, depth_map)."""
    return ops.composite(raw, z_vals, rays_d, bc_rgb, _noise(raw, raw_noise_std, pytest), white_bkgd, False)


def raw2outputs_torso(raw, z_vals, rays_d, bc_rgb, raw_noise_std=0, white_bkgd=False, pytest=False):
    """test_torso.py:352 -> (rgb_map, disp_map, acc_map, weights, depth_map, rgb_map_fg)."""
    return ops.composite(raw, z_vals, rays_d, bc_rgb, _noise(raw, raw_noise_std, pytest), white_bkgd, True)


# ------------------------------------------------------------------------------------------------
# the path
# ------------------------------------------------------------------------------------------------
def _fusable(net_coarse, net_fine, aud, expr, latent, N_samples, N_importance, retraw=False, raw_noise_std=0., pytest=False,
             pdf_policy=_lib.INERF_PDF_EXACT_TORCH_CPU):
    """True when the call can run as inerf_render_rays_fused: an inference call (autograd not recording anything the nets could need)
    of a two-pass shape the fused entry takes, without the extras that materialise per-sample tensors (retraw, noise, pytest tables).
    Per-kernel event timing (ops.kernel_timing) keeps the stage-by-stage path so that every kernel gets its own event pair."""
    if ops._timing is not None or retraw or raw_noise_std > 0. or pytest or not ops.FUSED_RENDER or pdf_policy != _lib.INERF_PDF_EXACT_TORCH_CPU:
        return False
    if not (N_importance > 0 and N_samples >= 4 and N_samples % 2 == 0 and (N_samples + N_importance) % 2 == 0 and N_samples + N_importance <= 256):
        return False
    if net_coarse.mlp_mode != net_fine.mlp_mode:
        return False
    cond = (aud, expr, latent)
    return not any(FaceNeRF._wants_grad(n.kernel_params(), *cond) for n in (net_coarse, net_fine))


def _render_rays_impl(rays, bc_rgb, net_coarse, net_fine, aud, expr, latent, N_samples, N_importance, retraw=False,
                      lindisp=False, perturb=0., white_bkgd=False, raw_noise_std=0., pytest=False, with_fg=False,
                      pdf_policy=_lib.INERF_PDF_EXACT_TORCH_CPU, check_numerics=False, gen=None, coarse_rgb=True):
    """audio_exp_nerf.py:297-371 (torso extras: train_torso.py:290-363).  gen: instead of `rays`, the frame / camera / pixel range whose
    rays the fused entry generates itself (frame.FrameRenderer).  coarse_rgb=False: the caller does not read 'rgb0', so the fused entry
    leaves it out and skips the coarse colour (ops.render_rays_fused); the stage-by-stage path still returns it."""
    net_f = net_coarse if net_fine is None else net_fine
    if gen is not None or _fusable(net_coarse, net_f, aud, expr, latent, N_samples, N_importance, retraw, raw_noise_std, pytest, pdf_policy):
        # inference: the whole call is ONE C entry point (inerf_render_rays_fused), five launches in the reference's configuration
        ret = ops.render_rays_fused(net_coarse, net_f, (aud, expr, latent), (aud, expr, latent), bc_rgb, N_samples, N_importance, perturb,
                                    rays=rays, gen=gen, lindisp=lindisp, white_bkgd=white_bkgd, with_fg=with_fg,
                                    check_numerics=check_numerics, coarse_rgb=coarse_rgb)
        for k in ret.get('_nonfinite', ()):
            logger.info(f"! [Numerical Error] {k} contains nan or inf.")
        return ret
    rays = ops.f32c(rays, "rays")
    bc_rgb = ops.f32c(bc_rgb, "bc_rgb")
    if rays.shape[-1] <= 8:
        raise NotImplementedError("use_viewdirs=False rays (8 columns) are not built; pass the (N,11) packed rays")
    N_rays = rays.shape[0]
    rays_d = rays[:, 3:6]                                    # strided view; the kernels take the row stride

    # perturb > 0: the reference draws torch.rand(N, S) / torch.rand(N, N_importance) from the global generator (:321-328, helper.py:282);
    # here the draws are made inside the sampling kernels (Philox, ops.rng_state) unless pytest=True asks for the numpy-seeded tables
    in_kernel_rng = perturb > 0. and not pytest
    if in_kernel_rng:
        rng = ops.rng_state(rays.device)
        z_vals = ops.sample_coarse_rng(rays, N_samples, rng, lindisp, advance=False)
    else:
        t_rand = None
        if perturb > 0.:                                     # :323-325
            np.random.seed(0)
            t_rand = torch.Tensor(np.random.rand(N_rays, N_samples)).to(rays.device)
        z_vals = ops.sample_coarse(rays, N_samples, t_rand, lindisp)

    raw = net_coarse.query(rays, z_vals, aud, expr, latent)
    outs = ops.composite(raw, z_vals, rays_d, bc_rgb, _noise(raw, raw_noise_std, pytest), white_bkgd, with_fg)
    rgb_map, disp_map, acc_map, weights, depth_map = outs[:5]

    ret = {}
    if N_importance > 0:
        rgb_map_0, disp_map_0, acc_map_0 = rgb_map, disp_map, acc_map
        outs0 = outs
        det = (perturb == 0.)
        if in_kernel_rng:
            _, z_vals, z_std = ops.importance_sample_rng(z_vals, weights, N_importance, rng, advance=False)
            ops.rng_advance(rng)                             # one bump per render_rays call; the two kernels use different streams
        else:
            if pytest:                                       # helper.py:285-293
                np.random.seed(0)
                u = (torch.Tensor(np.linspace(0., 1., N_importance)) if det
                     else torch.Tensor(np.random.rand(N_rays, N_importance))).to(rays.device)
            else:
                u = ops.linspace_table(N_importance, rays.device)
            z_samples, z_vals, z_std, _ = ops.importance_sample(z_vals, weights, u, pdf_policy)

        run_fn = net_coarse if net_fine is None else net_fine
        raw = run_fn.query(rays, z_vals, aud, expr, latent)
        outs = ops.composite(raw, z_vals, rays_d, bc_rgb, _noise(raw, raw_noise_std, pytest), white_bkgd, with_fg)
        rgb_map, disp_map, acc_map, weights, depth_map = outs[:5]

    ret.update({'rgb_map': rgb_map, 'disp_map': disp_map, 'acc_map': acc_map})
    if with_fg:
        ret['rgb_map_fg'] = outs[5]
    if retraw:
        ret['raw'] = raw
    if N_importance > 0:
        ret['rgb0'] = rgb_map_0
        ret['disp0'] = disp_map_0
        ret['acc0'] = acc_map_0
        ret['z_std'] = z_std
        ret['last_weight'] = weights[..., -1]
        if with_fg:
            ret['last_weight0'] = outs0[3][..., -1]
            ret['rgb_map_fg0'] = outs0[5]
    if in_kernel_rng and not N_importance > 0:
        ops.rng_advance(rng)
    if check_numerics:
        # the reference scans every output with .any() -- nine host synchronisations per call (:367-369); here ONE kernel ORs a bit per
        # tensor into a device flag and the host reads that flag once
        keys = list(ret)
        flag = torch.zeros((1,), dtype=torch.int32, device=rays.device)
        ops.flag_nonfinite([ret[k] for k in keys], flag)
        bits = int(flag.item())
        for i, k in enumerate(keys):
            if bits >> i & 1:
                logger.info(f"! [Numerical Error] {k} contains nan or inf.")
        ret['_nonfinite'] = [k for i, k in enumerate(keys) if bits >> i & 1]
    ret['_z_vals'] = z_vals
    ret['_weights'] = weights
    ret['_depth_map'] = depth_map
    return ret


_PRIVATE = ('_z_vals', '_weights', '_depth_map', '_nonfinite')


def render_rays(ray_batch, bc_rgb, aud_para, network_fn, network_query_fn=None, N_samples=64, retraw=False,
                lindisp=False, perturb=0., N_importance=0, network_fine=None, white_bkgd=False, raw_noise_std=0.,
                verbose=False, pytest=False, expr=None, latent_code=None):
    """Functional form, baseline.py:378.  ``network_fn``/``network_fine`` are FaceNeRF modules; the fused
    kernel replaces ``network_query_fn`` (accepted and ignored so call sites need no edit)."""
    ret = _render_rays_impl(ray_batch, bc_rgb, network_fn, network_fine, aud_para, expr, latent_code, N_samples,
                            N_importance, retraw, lindisp, perturb, white_bkgd, raw_noise_std, pytest)
    return {k: v for k, v in ret.items() if k not in _PRIVATE}


class _DeepSpeechAudNetKeys(nn.Module):
    """models/audio_net.py:72-87, parameters only (state_dict compatibility): the reference uses it when dim_aud <= 29, which none of
    its configurations does."""

    def __init__(self):
        super().__init__()
        self.encoder_fc = nn.Sequential(nn.Linear(16, 1), nn.LeakyReLU(0.02, True))


class Network(nn.Module):
    """Class-form HeadNeRF renderer, audio_exp_nerf.py:198.  ``args`` carries the reference's flags
    (helper.config_parser); the reference reads them from a module-level global."""

    def __init__(self, H, W, focal, near, far, chunk, intrinsic, N_samlpes, N_importance, args=None):
        super(Network, self).__init__()
        self.args = args if args is not None else default_args(dim_aud=64, dim_expr=76)
        a = self.args
        self.H, self.W, self.focal = H, W, focal
        self.near, self.far = near, far
        self.chunk = chunk
        self.intrinsic = intrinsic
        self.N_samples = N_samlpes
        self.N_importance = N_importance
        self.output_ch = 4
        self.skips = [4]
        self.embed_fn, input_ch = get_embedder(a.multires, a.i_embed)
        self.embed_dirs_fn, input_ch_views = get_embedder(a.multires_views, a.i_embed)
        mode = getattr(a, "mlp_mode", "fp32")
        self.face_nerf_coarse = FaceNeRF(D=a.netdepth, W=a.netwidth, input_ch=input_ch, dim_aud=a.dim_aud,
                                         output_ch=self.output_ch, skips=self.skips, dim_latent=32,
                                         dim_expr=a.dim_expr, input_ch_views=input_ch_views,
                                         use_viewdirs=a.use_viewdirs, mlp_mode=mode)
        self.face_nerf_fine = FaceNeRF(D=a.netdepth, W=a.netwidth, input_ch=input_ch, dim_aud=a.dim_aud,
                                       dim_latent=32, dim_expr=a.dim_expr, output_ch=self.output_ch,
                                       skips=self.skips, input_ch_views=input_ch_views,
                                       use_viewdirs=a.use_viewdirs, mlp_mode=mode)
        # the conditioning nets of audio_exp_nerf.py:224-226, same attribute names so that head.tar's model_state_dict loads
        self.aud_net = AudioNet(a.dim_aud, getattr(a, "win_size", 16))
        self.aud_att_net = AudioAttNet()
        self.ds_aud_net = _DeepSpeechAudNetKeys()

    def audio_feature(self, auds, index, dataset_size, global_step=None):
        """The per-frame audio code of audio_exp_nerf.py:241-266: the smo_size-frame window around `index` (zero padded at the ends of
        the sequence) through AudioNet, then AudioAttNet; a single AudioNet call before `nosmo_iters`.  auds: (T, 16, 29) DeepSpeech
        windows on the device.  Runs in the CUDA kernels of csrc/audio_net.cu; differentiable in both nets' parameters when autograd is recording."""
        a = self.args
        if a.dim_aud <= 29:
            raise NotImplementedError("dim_aud <= 29 (DeepSpeechAudNet) is not a configuration the reference's configs use")
        if global_step is None or global_step >= getattr(a, "nosmo_iters", 0):
            return self.aud_att_net(self.aud_net(self.audio_window(auds, index, dataset_size)))
        return self.aud_net(auds[index:index + 1].contiguous())

    def audio_window(self, auds, index, dataset_size):
        """The smo_size-frame window of DeepSpeech features around frame `index`, zero padded past either end (:243-262): (smo_size, 16, 29)."""
        half = int(getattr(self.args, "smo_size", 8) / 2)
        left, right = index - half, index + half
        pad_l, pad_r = max(0, -left), max(0, right - dataset_size)
        win = auds[max(left, 0):min(right, dataset_size)]
        if pad_l:
            win = torch.cat((torch.zeros_like(win)[:pad_l], win), 0)
        if pad_r:
            win = torch.cat((win, torch.zeros_like(win)[:pad_r]), 0)
        return win.contiguous()

    def set_mlp_mode(self, mode):
        for m in self.modules():
            if isinstance(m, FaceNeRF):
                m.mlp_mode = mode

    def forward(self, inputs):
        """audio_exp_nerf.py:228 with the conditioning features already computed (AudioNet is not on the hot path):
        inputs = [(batch_rays(2,N,3), bg_img, aud_feature(dim_aud), pose, expr, latent_code), global_step, dataset_size]."""
        x, global_step, dataset_size = inputs
        batch_rays, bg_img, aud_feature, pose, expr, latent_code = x
        expr_feature = expr if self.args.dim_expr > 0 else None
        render_poses = None if self.training is True else pose[:3, :4]
        return self.render_dynamic_face(H=self.H, W=self.W, focal=self.focal, expr=expr_feature, poses=pose,
                                        latent_code=latent_code, render_poses=render_poses, chunk=self.args.chunk,
                                        near=self.near, far=self.far, rays=batch_rays, bc_rgb=bg_img,
                                        aud_para=aud_feature, ndc=False)

    def batchify_rays(self, rays, bc_rgb, aud_para, poses, latent_code, expr, chunk=1024 * 32, **kw):
        all_ret = {}
        for i in range(0, rays.shape[0], chunk):
            ret = self.render_rays(rays[i:i + chunk], bc_rgb[i:i + chunk], aud_para, poses, latent_code, expr, **kw)
            for k in ret:
                all_ret.setdefault(k, []).append(ret[k])
        return {k: (v[0] if len(v) == 1 else torch.cat(v, 0)) for k, v in all_ret.items()}

    def render_rays(self, rays, bc_rgb, aud_para, poses, latent_code, expr, retraw=False, lindisp=False,
                    perturb=None, white_bkgd=False, raw_noise_std=0., attention_embed_ln=0, pytest=False):
        perturb = self.args.perturb if perturb is None else perturb
        ret = _render_rays_impl(rays, bc_rgb, self.face_nerf_coarse, self.face_nerf_fine, aud_para, expr, latent_code,
                                self.args.N_samples, self.args.N_importance, retraw, lindisp, perturb, white_bkgd,
                                raw_noise_std, pytest, check_numerics=getattr(self.args, "check_numerics", False))
        return {k: v for k, v in ret.items() if k not in _PRIVATE}

    def raw2outputs(self, raw, z_vals, rays_d, bc_rgb, raw_noise_std=0, white_bkgd=False, pytest=False):
        return raw2outputs(raw, z_vals, rays_d, bc_rgb, raw_noise_std, white_bkgd, pytest)

    def run_network(self, inputs, expr, viewdirs, aud, nerf_model, latent_code, netchunk=1024 * 64):
        """audio_exp_nerf.py:376 on explicit points (N,S,3): embed + FaceNeRF.forward in netchunk pieces."""
        inputs_flat = torch.reshape(inputs, [-1, inputs.shape[-1]])
        embeded = self.embed_fn(inputs_flat)
        input_dirs = viewdirs[:, None].expand(inputs.shape)
        embeded = torch.cat([embeded, self.embed_dirs_fn(torch.reshape(input_dirs, [-1, 3]))], -1)
        outs = [nerf_model(embeded[i:i + netchunk], aud, expr, latent_code) for i in range(0, embeded.shape[0], netchunk)]
        outputs_flat = outs[0] if len(outs) == 1 else torch.cat(outs, 0)
        return torch.reshape(outputs_flat, list(inputs.shape[:-1]) + [outputs_flat.shape[-1]])

    def render_dynamic_face(self, H, W, focal, expr, poses, latent_code, render_poses=None, chunk=1024 * 32, near=0.,
                            far=1., rays=None, bc_rgb=None, aud_para=None, ndc=False, use_viewdirs=True, **kw):
        if ndc:
            raise NotImplementedError("ndc rays are never used by the reference's talking-head scripts")
        if render_poses is not None:
            packed = ops.get_rays_packed(H, W, focal, render_poses, near, far)    # cx, cy default to W/2, H/2 (:401)
            bc_rgb = bc_rgb.reshape(-1, 3)
            sh = (H, W, 3)
        else:
            rays_o, rays_d = rays
            sh = rays_d.shape
            packed = ops.pack_rays(rays_o, rays_d, near, far)
        all_ret = self.batchify_rays(packed, bc_rgb, aud_para, poses=poses, latent_code=latent_code, expr=expr,
                                     chunk=chunk, **kw)
        for k in all_ret:
            all_ret[k] = torch.reshape(all_ret[k], list(sh[:-1]) + list(all_ret[k].shape[1:]))
        k_extract = ['rgb_map', 'disp_map', 'acc_map', 'last_weight']
        ret_list = [all_ret[k] for k in k_extract]
        ret_dict = {k: all_ret[k] for k in all_ret if k not in k_extract}
        return ret_list + [ret_dict]


class TorsoNetwork(nn.Module):
    """Head + torso renderer, train_torso.py:186.  Two FaceNeRF pairs; the torso pair is conditioned on
    [aud_feature[:dim_aud_body] | gamma_3(euler) | gamma_3(trans)] and has no expr/latent inputs."""

    def __init__(self, H, W, focal, near, far, chunk, N_samlpes, N_importance, args=None, dim_expr=79):
        super(TorsoNetwork, self).__init__()
        self.args = args if args is not None else default_args(dim_aud=64, dim_expr=dim_expr)
        a = self.args
        self.H, self.W, self.focal, self.near, self.far, self.chunk = H, W, focal, near, far, chunk
        self.N_samples, self.N_importance = N_samlpes, N_importance
        self.embed_torso_aud_fn, input_ch_torso_aud = get_embedder(3, 0)          # train_torso.py:41
        mode = getattr(a, "mlp_mode", "fp32")
        mk = lambda **kw: FaceNeRF(D=a.netdepth, W=a.netwidth, input_ch=63, output_ch=4, skips=[4],
                                   input_ch_views=27, use_viewdirs=a.use_viewdirs, mlp_mode=mode, **kw)
        self.face_nerf_coarse = mk(dim_aud=a.dim_aud, dim_latent=32, dim_expr=dim_expr)
        self.face_nerf_fine = mk(dim_aud=a.dim_aud, dim_latent=32, dim_expr=dim_expr)
        dim_torso = a.dim_aud_body + 2 * input_ch_torso_aud
        self.torso_coarse_nerf = mk(dim_aud=dim_torso)
        self.torso_fine_nerf = mk(dim_aud=dim_torso)

    def torso_signal(self, aud_feature, pose):
        """train_torso.py:237-240."""
        et = pose_to_euler_trans(pose.unsqueeze(0))
        embed_et = torch.cat((self.embed_torso_aud_fn(et[:, :3]), self.embed_torso_aud_fn(et[:, 3:])), dim=1)
        return torch.cat((aud_feature[..., :self.args.dim_aud_body], torch.squeeze(embed_et)), dim=-1)

    def render_pair(self, which, rays, bc_rgb, aud, expr, latent, perturb=None, **kw):
        a = self.args
        nets = (self.face_nerf_coarse, self.face_nerf_fine) if which == "head" else \
            (self.torso_coarse_nerf, self.torso_fine_nerf)
        perturb = a.perturb if perturb is None else perturb
        return _render_rays_impl(rays, bc_rgb, nets[0], nets[1], aud, expr, latent, a.N_samples, a.N_importance,
                                 perturb=perturb, with_fg=True, **kw)

    def forward(self, rays_head, rays_torso, bc_rgb, aud_feature, pose, expr, latent_code, perturb=None, **kw):
        """Returns (rgb_com, rgb_com0), train_torso.py:247-271.  rays_*: packed (N,11)."""
        head = self.render_pair("head", rays_head, bc_rgb, aud_feature, expr, latent_code, perturb, **kw)
        torso = self.render_pair("torso", rays_torso, bc_rgb, self.torso_signal(aud_feature, pose), None, None,
                                 perturb, **kw)
        rgb_com = ops.head_torso_blend(head['rgb_map'], torso['last_weight'], torso['rgb_map_fg'])
        rgb_com0 = ops.head_torso_blend(head['rgb0'], torso['last_weight0'], torso['rgb_map_fg0'])
        return rgb_com, rgb_com0


def pose_to_euler_trans(poses):
    """run_nerf_helpers.py:26-47: (B,3|4,4) -> (B,6).  Once per frame on 9 numbers; plain tensor ops."""
    R = poses[:, :3, :3]
    e = torch.stack([torch.atan2(R[:, 2, 2], R[:, 1, 2]), torch.asin(-R[:, 0, 2]),
                     torch.atan2(R[:, 0, 0], -R[:, 0, 1])], 1)
    return torch.cat((e, poses[:, :3, 3]), dim=1)


def init_weights(m):
    """audio_exp_nerf.py:442-448."""
    if isinstance(m, nn.Linear):
        torch.nn.init.xavier_uniform_(m.weight)
        m.bias.data.fill_(0.01)
    if isinstance(m, nn.Conv1d):
        torch.nn.init.xavier_uniform_(m.weight)
        m.bias.data.fill_(0.01)
