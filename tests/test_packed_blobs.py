"""The packed weight blobs of every tensor-core mode and the folded `cond` buffer, byte for byte: SHA-256 digests of what inerf_mlp_pack
and inerf_mlp_fold_cond write for seeded weights and conditioning, recorded when each tensor-core kernel still had its own schedule, pack
kernel and bias-tile offsets.  A change to a stage order, a pack conversion or the bias-tile layout of `cond` changes a digest."""
import hashlib

import pytest
import torch

from oracle import render_oracle as O
import test_gpu_parity as G

pytestmark = pytest.mark.gpu

DEV = G.DEV
M = G.M            # module fixture: the built package on a B200

MODES = ("INERF_MLP_BF16", "INERF_MLP_BF16_EMB", "INERF_MLP_BF16_BWD", "INERF_MLP_F16X2", "INERF_MLP_F16X2_EMB")

DIGESTS = {
    (64, 76, 32): {
        "INERF_MLP_BF16": "215ee636843352b01a41c1d8474c22cfc06c890a0ef1552f946a4291fbce6428",
        "INERF_MLP_BF16_EMB": "e306be4cfb9accac119726851a90a0c5e968cc286e2b5503fffcca944b001474",
        "INERF_MLP_BF16_BWD": "08d771cc78750a98cfd0f698e29c32bc04944ae86d8b84e088335eac8a281103",
        "INERF_MLP_F16X2": "81afe46ee83e57c5e91b23547bc5ed3fd91703f0bb4074cf30bfb3bbf51c3cf6",
        "INERF_MLP_F16X2_EMB": "b30a34b93e16c0b66edf954e6619033a1a68fbc751d63ad2dc5428686a1aecd0",
        "cond": "341cb338c6a8dfe2359dfe591717671aebc15ac27d9a5216ffa48134cd4320ee",
    },
    (106, 0, 0): {
        "INERF_MLP_BF16": "87ea98d0783b1db505a3ef978f49fda21c33fb16d4455ae3e92b15a0d9f830c8",
        "INERF_MLP_BF16_EMB": "6b905a49e9d69b925ff777e87302027d779e983bbee48734a11845cc89e88703",
        "INERF_MLP_BF16_BWD": "bacb30ba8f878dcfc59b51915bfe3c0ebf8e8264a20851bac1bdfd8e43cbb880",
        "INERF_MLP_F16X2": "9f75f283c380e4dde8ce5dfe62dd4bf3d3c76a29955904b5c6445a8623de5f81",
        "INERF_MLP_F16X2_EMB": "34fa974fa839edc30685b66c46f01c823a20c5da6c7569dc77a8f287ca23bad7",
        "cond": "9a3cd3776b5295e38aca514fb24ce7e01d603c27eeebdb5a36728b117ce5fe7e",
    },
}


def _digests(M, dims):
    net = M.FaceNeRF(dim_aud=dims[0], dim_expr=dims[1], dim_latent=dims[2])
    net.load_state_dict(O.init_face_nerf(3, *dims))
    net = net.to(DEV)
    params = [p.detach() for p in net.kernel_params()]
    g = torch.Generator().manual_seed(4)
    aud, expr, lat = (torch.randn(d, generator=g).to(DEV) if d else None for d in dims)
    out = {}
    for mode in MODES:
        blob = M.ops.pack_weights(getattr(M._lib, mode), net._dims, params)
        out[mode] = hashlib.sha256(blob.cpu().numpy().tobytes()).hexdigest()
    cond = M.ops.fold_cond(net._dims, params, aud, expr, lat)
    out["cond"] = hashlib.sha256(cond.cpu().numpy().tobytes()).hexdigest()
    torch.cuda.synchronize()
    return out


@pytest.mark.parametrize("dims", [(64, 76, 32), (106, 0, 0)])
def test_packed_blobs_and_cond_are_unchanged(M, dims):
    got = _digests(M, dims)
    for k, v in got.items():
        print(f"{dims} {k}: {v}")
    assert got == DIGESTS[dims]
