"""Argument rules of the coarse pass without its colour (InerfRenderArgs.rgb0 == NULL, ops.render_rays_fused(coarse_rgb=False)), checked
on the host: the workspace plan, the torso-extras rule and the Python keyword."""
import ctypes

import pytest


@pytest.fixture(scope="module")
def M():
    import ideal_nerf_b200 as m
    m.lib()
    return m


def _args(M, mode, rgb0):
    from ideal_nerf_b200._lib import InerfNetDims, InerfRenderArgs
    a = InerfRenderArgs()
    a.mode, a.n, a.n_samples, a.n_importance, a.perturb = mode, 100, 64, 128, 1
    for net in (a.coarse, a.fine):
        net.dims = InerfNetDims(64, 76, 32, 256, 8, 63, 27)
    a.rgb0 = rgb0
    return a


def test_workspace_coarse_buffer(M):
    """rgb0 == NULL shrinks the coarse raw buffer to one float per sample in bf16 mode only (the other modes run the full coarse net)"""
    from ideal_nerf_b200 import _lib
    L = M.lib()
    up = lambda b: (b + 255) // 256 * 256
    size = {}
    for mode in (_lib.INERF_MLP_FP32, _lib.INERF_MLP_BF16, _lib.INERF_MLP_F16X2):
        for rgb0 in (256, None):
            nb = ctypes.c_size_t()
            assert L.inerf_render_workspace_bytes(ctypes.byref(_args(M, mode, rgb0)), ctypes.byref(nb)) == 0
            size[mode, rgb0] = nb.value
    assert size[_lib.INERF_MLP_BF16, 256] - size[_lib.INERF_MLP_BF16, None] == up(100 * 64 * 16) - up(100 * 64 * 4)
    for mode in (_lib.INERF_MLP_FP32, _lib.INERF_MLP_F16X2):
        assert size[mode, None] == size[mode, 256] == size[_lib.INERF_MLP_BF16, 256]


def test_torso_extras_need_rgb0(M):
    """rgb_map_fg0 is a coarse colour: the torso extras without rgb0 are refused before any device work"""
    from ideal_nerf_b200 import _lib
    L = M.lib()
    a = _args(M, _lib.INERF_MLP_BF16, None)
    nb = ctypes.c_size_t()
    assert L.inerf_render_workspace_bytes(ctypes.byref(a), ctypes.byref(nb)) == 0
    a.workspace, a.workspace_bytes = 1 << 20, nb.value          # never dereferenced: the call fails in its host checks
    for k in ("bc_rgb", "t_vals", "rgb_map", "disp_map", "acc_map", "depth_map", "last_weight", "disp0", "acc0", "z_std", "rng_state",
              "rgb_map_fg", "rgb_map_fg0", "last_weight0"):
        setattr(a, k, 1 << 20)
    a.gen_rays = 0
    a.rays, a.ray_stride = 1 << 20, 11
    assert L.inerf_render_rays_fused(ctypes.byref(a), None) == -1
    assert b"torso extras need rgb0" in L.inerf_last_error()


def test_python_keyword(M):
    with pytest.raises(ValueError, match="coarse_rgb=True"):
        M.ops.render_rays_fused(None, None, None, None, None, 64, 128, 1.0, with_fg=True, coarse_rgb=False)
