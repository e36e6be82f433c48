"""CPU-side checks: the C-ABI library builds/loads and exports every symbol of include/inerf_b200.h,
argument validation works without a GPU, and the host mirror keeps the reference's surface."""
import ctypes
import inspect
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def M():
    import ideal_nerf_b200 as m
    m.build()
    return m


def header_symbols():
    txt = open(os.path.join(ROOT, "include", "inerf_b200.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(inerf_[a-z0-9_]+)\s*\(", txt)))


def test_library_exports_every_declared_symbol(M):
    L = M.lib()
    syms = header_symbols()
    assert len(syms) >= 18
    for s in syms:
        assert hasattr(L, s), f"{s} declared in include/inerf_b200.h but not exported"
    from ideal_nerf_b200 import _lib
    assert sorted(_lib.SIGNATURES) == syms, "ctypes signature table and header disagree"
    assert L.inerf_version() == 100


def test_argument_validation_without_gpu(M):
    """Entry points validate shapes/pointers before touching the device: safe to call on a CPU box."""
    L = M.lib()
    from ideal_nerf_b200._lib import InerfNetDims
    assert L.inerf_composite_fwd(None, None, None, 3, None, None, 4, 64, 0, None, None, None, None, None, None, None) == -1
    assert b"NULL" in L.inerf_last_error()
    assert L.inerf_composite_fwd(None, None, None, 3, None, None, 4, 5000, 0, None, None, None, None, None, None, None) == -2
    assert L.inerf_composite_fwd(None, None, None, 3, None, None, 0, 64, 0, None, None, None, None, None, None, None) == 0
    assert L.inerf_sample_pdf(None, 63, None, 62, 8, 1, 128, None, 0, 0, None, None, None, 0, None, None, None) == -2
    bad = InerfNetDims(64, 76, 32, 128, 8, 63, 27)
    n = ctypes.c_size_t()
    assert L.inerf_mlp_cond_floats(ctypes.byref(bad), ctypes.byref(n)) == -4
    ok = InerfNetDims(64, 76, 32, 256, 8, 63, 27)
    assert L.inerf_mlp_cond_floats(ctypes.byref(ok), ctypes.byref(n)) == 0 and n.value == 8 * 256 + 3 * 128 + 4 + 2 * (16 * 4096 + 6 * 2048) // 4
    assert L.inerf_mlp_fwd(7, ctypes.byref(ok), None, None, None, None, 11, None, 1, 1, None, None) == -1


def test_fused_render_entry_validates_without_gpu(M):
    """inerf_render_rays_fused / inerf_render_workspace_bytes: struct layout agrees with the header, shapes are checked before any
    device work, and the workspace plan is the sum of the buffers DESIGN.md lists."""
    L = M.lib()
    from ideal_nerf_b200._lib import InerfNetDims, InerfRenderArgs, InerfRenderNet
    assert [L.inerf_sizeof(i) for i in range(4)] == [ctypes.sizeof(InerfNetDims), ctypes.sizeof(InerfRenderNet), ctypes.sizeof(InerfRenderArgs), 0]
    a = InerfRenderArgs()
    nb = ctypes.c_size_t()
    assert L.inerf_render_workspace_bytes(None, ctypes.byref(nb)) == -1
    a.n, a.n_samples, a.n_importance = 100, 64, 0
    assert L.inerf_render_workspace_bytes(ctypes.byref(a), ctypes.byref(nb)) == -2            # coarse-only renders use the stage entry points
    a.n_importance = 128
    assert L.inerf_render_workspace_bytes(ctypes.byref(a), ctypes.byref(nb)) == -4            # dims not set: unsupported geometry
    for net in (a.coarse, a.fine):
        net.dims = InerfNetDims(64, 76, 32, 256, 8, 63, 27)
    a.perturb = 1
    assert L.inerf_render_workspace_bytes(ctypes.byref(a), ctypes.byref(nb)) == 0
    up = lambda b: (b + 255) // 256 * 256
    cond = (8 * 256 + 3 * 128 + 4) * 4 + 2 * (16 * 4096 + 6 * 2048)
    want = 2 * up(cond) + up(100 * 64 * 4) + up(100 * 64 * 16) + up(100 * 192 * 4) + up(100 * 192 * 16) + up(100 * 4)
    assert nb.value == want, (nb.value, want)
    a.gen_rays, a.perturb = 1, 0                                                               # + rays, coarse weights, z_samples
    assert L.inerf_render_workspace_bytes(ctypes.byref(a), ctypes.byref(nb)) == 0
    assert nb.value == want + up(100 * 11 * 4) + up(100 * 64 * 4) + up(100 * 128 * 4)
    assert L.inerf_render_rays_fused(ctypes.byref(a), None) == -1 and b"workspace" in L.inerf_last_error()
    a.n = 0
    assert L.inerf_render_rays_fused(ctypes.byref(a), None) == 0                               # empty batch: nothing to enqueue


def test_no_cpu_fallback(M):
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        M.raw2outputs(torch.zeros(2, 4, 4), torch.zeros(2, 4), torch.zeros(2, 3), torch.zeros(2, 3))
    with pytest.raises(RuntimeError, match="CUDA"):
        M.sample_pdf(torch.zeros(2, 5), torch.zeros(2, 4), 8, det=True)
    net = M.FaceNeRF(dim_aud=64, dim_latent=32, dim_expr=76)
    with pytest.raises(RuntimeError, match="CUDA"):
        net(torch.zeros(4, 90), torch.zeros(64), torch.zeros(76), torch.zeros(32))


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "ideal-nerf_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dp, f)).read()
                assert not re.search(r"^\s*(import|from)\s+oracle", src, flags=re.M), f"{f} imports oracle/"
                assert "render_oracle" not in src or f == "sample_pdf.cu", f


def test_reference_surface(M):
    """Names and signatures of the reference's Python surface (SURVEY.md 8b)."""
    sig = inspect.signature
    assert list(sig(M.raw2outputs).parameters) == ["raw", "z_vals", "rays_d", "bc_rgb", "raw_noise_std", "white_bkgd", "pytest"]
    assert list(sig(M.sample_pdf).parameters)[:5] == ["bins", "weights", "N_samples", "det", "pytest"]
    assert list(sig(M.get_embedder).parameters) == ["multires", "i", "input_dims"]
    assert list(sig(M.get_rays).parameters) == ["H", "W", "focal", "c2w", "cx", "cy"]
    assert list(sig(M.FaceNeRF.forward).parameters) == ["self", "x", "aud", "expr", "latent_code"]
    assert list(sig(M.FaceNeRF.__init__).parameters)[1:11] == ["D", "W", "input_ch", "input_ch_views", "dim_aud", "dim_latent",
                                                             "dim_expr", "output_ch", "skips", "use_viewdirs"]
    rr = list(sig(M.Network.render_rays).parameters)
    assert rr[:7] == ["self", "rays", "bc_rgb", "aud_para", "poses", "latent_code", "expr"]
    assert rr[7:] == ["retraw", "lindisp", "perturb", "white_bkgd", "raw_noise_std", "attention_embed_ln", "pytest"]
    fr = list(sig(M.render_rays).parameters)
    assert fr[:15] == ["ray_batch", "bc_rgb", "aud_para", "network_fn", "network_query_fn", "N_samples", "retraw", "lindisp",
                       "perturb", "N_importance", "network_fine", "white_bkgd", "raw_noise_std", "verbose", "pytest"]
    net = M.Network(450, 450, 1200., 0.57, 1.17, 8192, None, 64, 128)
    keys = set(net.state_dict())
    for pre in ("face_nerf_coarse.", "face_nerf_fine."):
        for l in [f"pts_linears.{i}" for i in range(8)] + [f"views_linears.{i}" for i in range(3)] + \
                ["feature_linear", "alpha_linear", "rgb_linear"]:
            assert pre + l + ".weight" in keys and pre + l + ".bias" in keys
    assert net.face_nerf_coarse.pts_linears[0].weight.shape == (256, 63 + 64 + 76 + 32)
    assert net.face_nerf_coarse.pts_linears[5].weight.shape == (256, 256 + 235)
    assert net.face_nerf_coarse.views_linears[0].weight.shape == (128, 27 + 256 + 76)


def test_config_flags(M, tmp_path):
    p = M.config_parser()
    a = p.parse_args([])
    assert (a.N_samples, a.N_importance, a.chunk, a.netchunk, a.perturb) == (64, 128, 8192, 65536, 1.0)
    assert a.use_viewdirs is True and a.white_bkgd is True                 # store_false flags default to True
    a = p.parse_args(["--N_sample", "32", "--dim_aud", "64", "--dim_expr", "76", "--near", "0.5772", "--far", "1.1772"])
    assert a.N_samples == 32 and a.dim_aud == 64 and a.dim_expr == 76    # README's N_sample spelling still works
    cfg = tmp_path / "paper_model.txt"
    cfg.write_text("expname=torso_bg\nN_sample=64\nN_importance=128\nlrate=3e-4\nN_rand=3072\nmouth_rays=512\ndim_expr=79\ndim_aud=64\n"
                   "near=0.5674083709716797\nfar=1.1674083709716796\n")
    a = p.parse_args(["--config", str(cfg), "--N_rand", "1024"])
    assert a.N_samples == 64 and a.lrate == 3e-4 and a.mouth_rays == 512 and a.dim_expr == 79
    assert a.N_rand == 1024 and abs(a.near - 0.5674083709716797) < 1e-15


def test_network_state_dict_matches_reference_keys_and_checkpoint_round_trip(M, tmp_path):
    """head.tar layout (audio_exp_nerf.py:584-591): the Network exposes the reference's parameter names -- FaceNeRF x2, AudioNet,
    AudioAttNet, DeepSpeechAudNet -- and a checkpoint written with the reference's keys round-trips; --ft_path files load with the three
    width-dependent weights dropped (:498-514)."""
    import torch
    from ideal_nerf_b200 import checkpoint as ck
    net = M.Network(450, 450, 1200., 0.57, 1.17, 8192, None, 64, 128)
    keys = set(net.state_dict())
    for k in ("aud_net.encoder_conv.0.weight", "aud_net.encoder_conv.6.bias", "aud_net.encoder_fc1.2.weight",
              "aud_att_net.attentionConvNet.8.weight", "aud_att_net.attentionNet.0.bias", "ds_aud_net.encoder_fc.0.weight"):
        assert k in keys, k
    assert net.aud_net.encoder_fc1[2].weight.shape == (64, 64) and net.aud_att_net.attentionConvNet[0].weight.shape == (16, 32, 3)
    lat = torch.ones(5, 32)
    opt = torch.optim.Adam(list(net.parameters()) + [lat], lr=3e-4)
    p = str(tmp_path / "head.tar")
    ck.save_head_checkpoint(p, net, opt, lat * 2, 1234)
    raw = torch.load(p, weights_only=False)
    assert set(raw) == {"global_step", "model_state_dict", "optimizer", "latent_codes"}
    net2 = M.Network(450, 450, 1200., 0.57, 1.17, 8192, None, 64, 128)
    lat2 = torch.zeros(5, 32)
    assert ck.load_head_checkpoint(p, net2, None, lat2) == 1234
    assert all(torch.equal(a, b) for a, b in zip(net.state_dict().values(), net2.state_dict().values()))
    assert torch.equal(lat2, lat * 2)
    # fine-tune source with a different conditioning width: first-layer weights are dropped, everything else loads
    src = M.Network(450, 450, 1200., 0.57, 1.17, 8192, None, 64, 128, args=M.default_args(dim_aud=64, dim_expr=0))
    ft = str(tmp_path / "ft.tar")
    torch.save({"network_fn_state_dict": src.face_nerf_coarse.state_dict(), "network_fine_state_dict": src.face_nerf_fine.state_dict(),
                "network_audnet_state_dict": src.aud_net.state_dict(), "network_audattnet_state_dict": src.aud_att_net.state_dict()}, ft)
    before = net2.face_nerf_coarse.pts_linears[0].weight.clone()
    ck.load_finetune_checkpoint(ft, net2)
    assert torch.equal(net2.face_nerf_coarse.pts_linears[0].weight, before)                      # dropped key: untouched
    assert torch.equal(net2.face_nerf_coarse.pts_linears[1].weight, src.face_nerf_coarse.pts_linears[1].weight)
    assert torch.equal(net2.aud_net.encoder_conv[0].weight, src.aud_net.encoder_conv[0].weight)


def test_flat_params_adam_equals_per_parameter_adam():
    """train.FlatParams: one-tensor Adam over the re-homed parameters == torch.optim.Adam over the separate parameters (audio_exp_nerf.py:529,
    the reference's optimiser), including a parameter that never receives a gradient; views stay 256-byte aligned and live."""
    import torch
    from ideal_nerf_b200.train import FlatParams
    torch.manual_seed(3)
    mk = lambda: torch.nn.ModuleList([torch.nn.Linear(7, 5), torch.nn.Linear(5, 3), torch.nn.Linear(3, 3)])     # the last one is never used
    a, b = mk(), mk()
    b.load_state_dict(a.state_dict())
    opt_a = torch.optim.Adam(a.parameters(), lr=1e-2)
    fp = FlatParams(list(b.parameters()))
    opt_b = torch.optim.Adam([fp.flat], lr=1e-2)
    for p in b.parameters():
        assert p.data_ptr() % 256 == fp.flat.data_ptr() % 256 and p.is_contiguous()
    x = torch.randn(11, 7)
    for _ in range(4):
        opt_a.zero_grad(set_to_none=True)
        a[1](torch.relu(a[0](x))).square().mean().backward()
        opt_a.step()
        for p in b.parameters():
            p.grad = None
        b[1](torch.relu(b[0](x))).square().mean().backward()
        fp.gather_grads()
        opt_b.step()
    for pa, pb in zip(a.parameters(), b.parameters()):
        assert torch.allclose(pa, pb, rtol=0, atol=1e-7), float((pa - pb).abs().max())


def test_bench_reference_arm_prints_one_json_line():
    """bench.py --impl reference (the reference's own renderer from oracle/_ref on the host cores; the oracle port when absent) honours the driver's contract without a GPU: exactly one stdout
    line, the metric / unit / config of the product arm, impl = reference, a cpu_baseline and an e2e object of its own."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-400:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout[:400]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "rays/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["metric"].startswith("rays/sec render") and "workload" in d["config"]
    from oracle import ref_import
    assert d["cpu_baseline"]["kind"] == ("reference" if ref_import.available() else "port")     # oracle/_ref (or /root/reference) present?
    assert d["cpu_baseline"]["cores"] >= 1 and "sample" in d["cpu_baseline"]
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0


def test_network_layout_matches_reference_network(M):
    """The 'optimizer' entry of head.tar indexes the reference's per-parameter Adam state by position in list(Network.parameters()), so
    the parameter order is part of the file format.  Name and shape of every parameter, in order (feature_linear and ds_aud_net
    included), against the reference's Network(450, 450, 1200., 0.57, 1.17, 8192, None, 64, 128): from tests/golden/head_tar_layout.npz
    (tests/golden/make_golden_head_tar.py) when it is committed, else from the reference tree when oracle/ref_import.py finds one."""
    import numpy as np
    from oracle import ref_import
    path = os.path.join(ROOT, "tests", "golden", "head_tar_layout.npz")
    if os.path.exists(path):
        with np.load(path) as z:
            ref = [(str(n), tuple(int(d) for d in s[1:1 + s[0]])) for n, s in zip(z["names"], z["shapes"])]
    elif ref_import.available():
        head = ref_import.import_head(force_cpu=True)
        ref = [(n, tuple(p.shape)) for n, p in head.Network(450, 450, 1200., 0.57, 1.17, 8192, None, 64, 128).named_parameters()]
    else:
        pytest.skip("neither tests/golden/head_tar_layout.npz nor the reference tree is present")
    net = M.Network(450, 450, 1200., 0.57, 1.17, 8192, None, 64, 128)
    assert [(n, tuple(p.shape)) for n, p in net.named_parameters()] == ref


def test_network_parameter_order_matches_reference(M, golden):
    """Parameter order (see test_network_layout_matches_reference_network) against what the committed fixtures made from the reference's
    own modules record: the order of the FaceNeRF parameters that receive a gradient (train_step.npz; feature_linear receives none and is
    not in it) and of AudioNet(64) / AudioAttNet (audio_nets.npz).  The positions of feature_linear and of ds_aud_net are not in these
    fixtures; test_network_layout_matches_reference_network pins them."""
    net = M.Network(450, 450, 1200., 0.57, 1.17, 8192, None, 64, 128)
    names = [n for n, _ in net.named_parameters()]
    assert list(net.state_dict()) == names                                     # no buffers: state_dict order == parameter order
    modules = list(dict.fromkeys(n.split(".")[0] for n in names))
    assert modules == ["face_nerf_coarse", "face_nerf_fine", "aud_net", "aud_att_net", "ds_aud_net"]
    tr, au = golden("train_step"), golden("audio_nets")
    for tag, mod in (("c", "face_nerf_coarse"), ("f", "face_nerf_fine")):
        ref = [k[len(f"norm:{tag}."):] for k in tr if k.startswith(f"norm:{tag}.")]
        ours = [n[len(mod) + 1:] for n in names if n.startswith(mod + ".")]
        assert len(ref) == 26 and [n for n in ours if n in ref] == ref, mod
        assert [n for n in ours if n not in ref] == ["feature_linear.weight", "feature_linear.bias"]      # unused by the forward: no gradient
    for tag, mod in (("an64", "aud_net"), ("att", "aud_att_net")):
        ref = [k[len(tag) + 1:] for k in au if k.startswith(tag + ".") and k.endswith((".weight", ".bias"))]
        assert [n[len(mod) + 1:] for n in names if n.startswith(mod + ".")] == ref, mod
        assert all(tuple(net.state_dict()[f"{mod}.{k}"].shape) == au[f"{tag}.{k}"].shape for k in ref)


def test_head_tar_interchange_with_reference_adam(M, tmp_path):
    """head.tar both ways (audio_exp_nerf.py:516-525 resume, :584-591 save) with the reference's optimiser, a per-parameter
    torch.optim.Adam over list(network.parameters()) + [latent codes] (:487-489): a checkpoint written by a Network + that optimiser
    loads into a live train.TrainStep with strict keys, IN PLACE (latent codes and weights stay views of the flat Adam buffer), the next
    update equals the per-parameter optimiser's next update bit for bit, and the file TrainStep.save() writes resumes the
    per-parameter optimiser the same way.  Writer and reader are both this project's Network here, so the parameter order that indexes
    the per-parameter state is checked against the reference's by the two tests above, not by this one."""
    from ideal_nerf_b200.train import TrainStep
    torch.manual_seed(0)

    def ref_setup():
        net = M.Network(450, 450, 1200., 0.57, 1.17, 8192, None, 64, 128)
        lat = torch.ones(5, 32)
        lat.requires_grad = True
        tp = list(net.parameters()) + [lat]                                   # :487-489
        return net, lat, tp, torch.optim.Adam(params=tp, lr=3e-4, betas=(0.9, 0.999))

    ref, lat_ref, tp, opt_ref = ref_setup()
    ref.apply(M.init_weights)
    g = torch.Generator().manual_seed(1)

    def fake_grads(params_list):
        gg = torch.Generator().manual_seed(int(torch.randint(1 << 30, (1,), generator=g)))
        grads = [torch.randn(p.shape, generator=gg) * 1e-2 for p in tp]
        for params in params_list:
            for i, (p, gr) in enumerate(zip(params, grads)):
                p.grad = None if 0 <= i - (len(tp) - 3) < 2 else gr.clone()     # ds_aud_net.* never receives a gradient in the reference
    fake_grads([tp]); opt_ref.step()
    fake_grads([tp]); opt_ref.step()
    for gr in opt_ref.param_groups:
        gr["lr"] = 2.9e-4
    p1 = str(tmp_path / "head.tar")
    torch.save({"global_step": 7, "model_state_dict": ref.state_dict(), "optimizer": opt_ref.state_dict(), "latent_codes": lat_ref.data}, p1)

    ours = M.Network(450, 450, 1200., 0.57, 1.17, 8192, None, 64, 128)
    lat = torch.zeros(5, 32)
    ts = TrainStep(ours, lat, ours.args)
    assert ts.load(p1) == 7 and ts.global_step == 7
    assert ts.optimizer.param_groups[0]["lr"] == 2.9e-4
    flat = ts.flat.flat
    for p in ts.flat.params:                                                   # still views of the flat buffer after the load
        assert flat.data_ptr() <= p.data_ptr() < flat.data_ptr() + flat.numel() * 4
    assert all(torch.equal(a, b) for a, b in zip(ref.state_dict().values(), ours.state_dict().values()))      # the weights of the file
    assert torch.equal(lat.data, lat_ref.data)
    before = lat.detach().clone()
    fake_grads([tp, ts.flat.params])
    opt_ref.step()
    ts.flat.gather_grads(); ts.optimizer.step()
    assert not torch.equal(lat.detach(), before), "latent codes must keep training after a resume"
    assert all(torch.equal(p, q) for p, q in zip(tp, ts.flat.params)), "resumed update differs from the reference's"
    # ... and back: the reference's resume code on a file written by TrainStep.save()
    p2 = str(tmp_path / "head2.tar")
    ts.global_step = 8
    ts.save(p2)
    ck = torch.load(p2, weights_only=False)
    assert set(ck) == {"global_step", "model_state_dict", "optimizer", "latent_codes"}
    ref2, lat2, tp2, opt2 = ref_setup()
    ref2.load_state_dict(ck["model_state_dict"])                                # :521
    lat2.data = ck["latent_codes"]                                              # :522
    opt2.load_state_dict(ck["optimizer"])                                       # :524
    fake_grads([tp, tp2])
    opt_ref.step(); opt2.step()
    assert all(torch.equal(p, q) for p, q in zip(tp, tp2))


def test_load_head_checkpoint_copies_latents_in_place(M, tmp_path):
    """ADVICE r1: load_head_checkpoint must not rebind latent_codes.data (TrainStep re-homes it as a view of the flat Adam buffer)."""
    from ideal_nerf_b200 import checkpoint as ck
    from ideal_nerf_b200.train import TrainStep
    net = M.Network(450, 450, 1200., 0.57, 1.17, 8192, None, 64, 128)
    lat = torch.ones(3, 32)
    ts = TrainStep(net, lat, net.args)
    p = str(tmp_path / "h.tar")
    ck.save_head_checkpoint(p, net, None, torch.full((3, 32), 2.0), 5)
    ptr = lat.data_ptr()
    assert ck.load_head_checkpoint(p, net, None, lat) == 5
    assert lat.data_ptr() == ptr and float(lat.detach().mean()) == 2.0
    with pytest.raises(ValueError, match="TrainStep.load"):
        ts.save(p)
        ck.load_head_checkpoint(p, net, torch.optim.Adam([ts.flat.flat]), lat)
