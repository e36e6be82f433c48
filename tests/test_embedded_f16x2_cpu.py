"""CPU-side checks of the fp16x2 embedded-row entry (FaceNeRF.forward on x (P, 63+27) at fp32-gate accuracy, mode INERF_MLP_F16X2_EMB):
the packed-blob sizes and the argument validation, which returns before any device work."""
import ctypes

import pytest

from ideal_nerf_b200 import _lib
from ideal_nerf_b200._lib import InerfNetDims

A16, A8 = 0x10000, 0x10008          # fake device addresses: 16-byte aligned / 8-byte aligned (never dereferenced)


@pytest.fixture(scope="module")
def L():
    import ideal_nerf_b200 as m
    m.build()
    return m.lib()


def _params():
    arr = _lib.ParamArray()
    for i in range(_lib.N_PARAMS):
        arr[i] = A16 + 256 * i
    return arr


@pytest.mark.parametrize("dims", [(64, 76, 32), (106, 0, 0)])
def test_packed_sizes(L, dims):
    d = InerfNetDims(*dims, 256, 8, 63, 27)
    n, e = ctypes.c_size_t(), ctypes.c_size_t()
    assert L.inerf_mlp_packed_bytes(_lib.INERF_MLP_F16X2, ctypes.byref(d), ctypes.byref(n)) == 0
    assert n.value == 2228224                       # the fused entry's blob is unchanged: 152 stages
    assert L.inerf_mlp_packed_bytes(_lib.INERF_MLP_F16X2_EMB, ctypes.byref(d), ctypes.byref(e)) == 0
    assert e.value == n.value + 32768               # + (hi, lo) 64-row x 64-column fp16 view K-blocks, one per half of views_linears.0
    assert L.inerf_mlp_pack(_lib.INERF_MLP_F16X2_EMB, ctypes.byref(d), None, None, None) == -1


def test_embedded_entry_argument_checks(L):
    d = InerfNetDims(64, 76, 32, 256, 8, 63, 27)
    f = L.inerf_mlp_fwd_embedded
    P = _params()
    m = _lib.INERF_MLP_F16X2_EMB
    assert f(m, ctypes.byref(d), P, None, A16, A16, 5, A16, None) == -1        # the INERF_MLP_F16X2_EMB blob is required
    assert b"INERF_MLP_F16X2_EMB" in L.inerf_last_error()
    assert f(m, ctypes.byref(d), P, A16, A16, A8, 5, A16, None) == -3          # x 16-byte aligned
    assert f(m, ctypes.byref(d), P, A8, A16, A16, 5, A16, None) == -3          # ... and the blob
    assert f(m, ctypes.byref(d), P, A16, A16, A16, -1, A16, None) == -2
    assert f(m, ctypes.byref(d), P, A16, A16, A16, 0, A16, None) == 0          # nothing to do
    bad = InerfNetDims(64, 76, 32, 128, 8, 63, 27)
    assert f(m, ctypes.byref(bad), P, A16, A16, A16, 5, A16, None) == -4
    assert f(_lib.INERF_MLP_F16X2, ctypes.byref(d), P, A16, A16, A16, 5, A16, None) == -4      # the fused entry's mode and blob
    assert b"INERF_MLP_F16X2_EMB" in L.inerf_last_error()


def test_other_entries_reject_the_embedded_mode(L):
    d = InerfNetDims(64, 76, 32, 256, 8, 63, 27)
    P = _params()
    assert L.inerf_mlp_fwd(_lib.INERF_MLP_F16X2_EMB, ctypes.byref(d), P, A16, A16, A16, 11, A16, 4, 64, A16, None) == -4
    assert L.inerf_mlp_fwd_trace(_lib.INERF_MLP_F16X2_EMB, ctypes.byref(d), P, A16, A16, A16, 11, A16, 4, 64, A16, A16, None) == -4
    a = _lib.InerfRenderArgs(mode=_lib.INERF_MLP_F16X2_EMB, n=0, n_samples=64, n_importance=128)
    a.coarse.dims = a.fine.dims = d
    assert L.inerf_render_rays_fused(ctypes.byref(a), None) == -4
    assert b"INERF_MLP_F16X2_EMB" in L.inerf_last_error()
