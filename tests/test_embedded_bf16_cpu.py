"""CPU-side checks of the bf16 embedded-row entry points (FaceNeRF.forward on x (P, 63+27)): the packed-blob sizes and the argument
validation, which returns before any device work."""
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
    assert L.inerf_mlp_packed_bytes(_lib.INERF_MLP_BF16, ctypes.byref(d), ctypes.byref(n)) == 0
    assert n.value == 1114112                       # the fused entry's blob is unchanged: 76 stages
    assert L.inerf_mlp_packed_bytes(_lib.INERF_MLP_BF16_EMB, ctypes.byref(d), ctypes.byref(e)) == 0
    assert e.value == n.value + 2 * 64 * 64 * 2     # + one 64-row x 64-column bf16 view K-block per half of views_linears.0
    assert L.inerf_mlp_packed_bytes(_lib.INERF_MLP_BF16_BWD, ctypes.byref(d), ctypes.byref(n)) == 0
    assert n.value == 1048576 + 2 * 4096            # the backward chain's transposed weight stages, then its two alpha tiles
    assert L.inerf_mlp_pack(_lib.INERF_MLP_BF16_EMB, ctypes.byref(d), None, None, None) == -1


def test_train_entry_argument_checks(L):
    d = InerfNetDims(64, 76, 32, 256, 8, 63, 27)
    f = L.inerf_mlp_fwd_train_bf16_embedded
    P = _params()
    ok = dict(packed=A16, cond=A16, x=A16, p=5, raw=A16, acts=A16, mask=A16)

    def call(**kw):
        a = dict(ok, **kw)
        return f(ctypes.byref(d), P, a["packed"], a["cond"], a["x"], a["p"], a["raw"], a["acts"], a["mask"], None)

    for k in ("packed", "cond", "x", "raw", "acts", "mask"):
        assert call(**{k: None}) == -1, k
        assert b"NULL" in L.inerf_last_error()
    assert f(ctypes.byref(d), None, A16, A16, A16, 5, A16, A16, A16, None) == -1
    assert call(p=-1) == -2
    assert call(p=0) == 0 and call(p=0, x=None, raw=None) == 0          # nothing to do: no pointer is needed
    for k in ("x", "raw", "acts", "mask"):
        assert call(**{k: A8}) == -3, k
    bad = InerfNetDims(64, 76, 32, 128, 8, 63, 27)
    assert f(ctypes.byref(bad), P, A16, A16, A16, 5, A16, A16, A16, None) == -4


def test_embedded_inference_entry_modes(L):
    d = InerfNetDims(64, 76, 32, 256, 8, 63, 27)
    f = L.inerf_mlp_fwd_embedded
    P = _params()
    assert f(_lib.INERF_MLP_F16X2, ctypes.byref(d), P, A16, A16, A16, 5, A16, None) == -4       # fp16x2: fused entry only
    assert f(_lib.INERF_MLP_BF16, ctypes.byref(d), P, None, A16, A16, 5, A16, None) == -1       # bf16 needs the EMB blob
    assert f(_lib.INERF_MLP_BF16, ctypes.byref(d), P, A16, A16, A8, 5, A16, None) == -3        # x 16-byte aligned
    assert f(_lib.INERF_MLP_BF16, ctypes.byref(d), P, A16, A16, A16, -1, A16, None) == -2
    assert f(_lib.INERF_MLP_BF16, ctypes.byref(d), P, A16, A16, A16, 0, A16, None) == 0
