"""CPU-side checks of the torso stage: the argument validation of inerf_head_torso_mse_pair (returns before any device work), what a
train.TorsoTrainStep trains and how its Adam state converts, and checkpoint.load_head_into_torso."""
import pytest
import torch

A16 = 0x10000          # fake device address (never dereferenced: every call below fails before a launch)


@pytest.fixture(scope="module")
def M():
    import ideal_nerf_b200 as m
    m.build()
    return m


def torso_net(M, dim_expr=79, seed=0):
    torch.manual_seed(seed)
    net = M.TorsoNetwork(450, 450, 1200., 0.57, 1.17, 8192, 64, 128, args=M.default_args(dim_aud=64, dim_expr=dim_expr), dim_expr=dim_expr)
    net.apply(M.init_weights)
    return net


def test_head_torso_mse_pair_argument_checks(M):
    L = M.lib()
    f = L.inerf_head_torso_mse_pair
    names = ("head", "head0", "lw", "lw0", "fg", "fg0", "target", "n", "g_lw", "g_lw0", "g_fg", "g_fg0", "loss2")
    ok = dict.fromkeys(names, A16)
    ok["n"] = 5

    def call(**kw):
        a = dict(ok, **kw)
        return f(*[a[k] for k in names], None)

    for k in names:
        if k == "n":
            continue
        assert call(**{k: None}) == -1, k
        assert b"NULL" in L.inerf_last_error()
    assert call(n=0) == -2                                  # at least one ray, like inerf_mse_pair
    assert call(n=-1) == -2
    assert call(n=0, head=None, loss2=None) == -2           # the size is checked before the pointers
    assert b"inerf_head_torso_mse_pair" in L.inerf_last_error()


def test_torso_train_step_trains_exactly_the_torso_pair(M):
    from ideal_nerf_b200.train import TorsoTrainStep
    net = torso_net(M)
    names = [n for n, _ in net.named_parameters()]
    want = [p for n, p in net.named_parameters() if n.startswith(("torso_coarse_nerf.", "torso_fine_nerf."))]
    head_before = {n: p.detach().clone() for n, p in net.named_parameters() if n.startswith("face_nerf_")}
    step = TorsoTrainStep(net, net.args)
    assert len(step.flat.params) == len(want) == 2 * 28 and all(a is b for a, b in zip(step.flat.params, want))
    assert names.index("torso_coarse_nerf.pts_linears.0.weight") < names.index("torso_fine_nerf.pts_linears.0.weight")
    flat = step.flat.flat
    for p in want:                                          # re-homed as views of the one Adam buffer, values kept
        assert flat.data_ptr() <= p.data_ptr() < flat.data_ptr() + flat.numel() * 4
    for n, p in net.named_parameters():
        if n.startswith("face_nerf_"):
            assert not (flat.data_ptr() <= p.data_ptr() < flat.data_ptr() + flat.numel() * 4), n
            assert torch.equal(p, head_before[n])
    with pytest.raises(RuntimeError, match=r"TorsoTrainStep\(cuda_graph=True\) needs CUDA tensors"):
        TorsoTrainStep(torso_net(M), net.args, cuda_graph=True)


def test_torso_optimizer_state_per_parameter_round_trip(M):
    """Two Adam steps on fake gradients: the per-parameter state (one entry per trained parameter, shapes of the parameters) equals that of
    a per-parameter torch.optim.Adam given the same gradients, and loading it into a fresh step restores the flat state exactly."""
    from ideal_nerf_b200.train import TorsoTrainStep
    net, ref = torso_net(M), torso_net(M)
    step = TorsoTrainStep(net, net.args)
    ref_params = [p for n, p in ref.named_parameters() if n.startswith("torso_")]
    opt = torch.optim.Adam(ref_params, lr=net.args.lrate, betas=(0.9, 0.999))
    g = torch.Generator().manual_seed(1)
    for _ in range(2):
        grads = [None if "feature_linear" in n else torch.randn(p.shape, generator=g) * 1e-2
                 for n, p in ref.named_parameters() if n.startswith("torso_")]
        for p, q, gr in zip(step.flat.params, ref_params, grads):
            p.grad = q.grad = None if gr is None else gr.clone()
        step.flat.gather_grads()
        step.optimizer.step()
        opt.step()
    sd, want = step.optimizer_state_dict(), opt.state_dict()
    assert sd["param_groups"][0]["params"] == list(range(len(ref_params)))
    assert set(want["state"]) <= set(sd["state"])
    for i, st in want["state"].items():
        for k in ("exp_avg", "exp_avg_sq"):
            assert sd["state"][i][k].shape == ref_params[i].shape
            assert torch.allclose(sd["state"][i][k], st[k], rtol=1e-6, atol=1e-12), (i, k)
    assert all(torch.allclose(p, q, rtol=0, atol=1e-7) for p, q in zip(step.flat.params, ref_params))
    fresh = TorsoTrainStep(torso_net(M, seed=5), net.args)
    fresh.load_optimizer_state_dict(sd)
    a, b = step.optimizer.state_dict()["state"][0], fresh.optimizer.state_dict()["state"][0]
    assert float(a["step"]) == float(b["step"]) == 2.0
    assert torch.equal(a["exp_avg"], b["exp_avg"]) and torch.equal(a["exp_avg_sq"], b["exp_avg_sq"])
    with pytest.raises(ValueError, match="this TorsoTrainStep has"):
        fresh.load_optimizer_state_dict({"state": {}, "param_groups": [dict(sd["param_groups"][0], params=[0, 1, 2])]})


def test_torso_train_step_save_load_keys(M, tmp_path):
    from ideal_nerf_b200.train import TorsoTrainStep
    net = torso_net(M)
    step = TorsoTrainStep(net, net.args)
    for p in step.flat.params:
        p.grad = torch.full_like(p, 1e-3)
    step.flat.gather_grads(); step.optimizer.step()
    step.global_step = 3
    path = str(tmp_path / "000003_torso.tar")
    step.save(path)
    ck = torch.load(path, weights_only=False)
    assert set(ck) == {"global_step", "model_state_dict", "optimizer"} and ck["global_step"] == 3
    assert list(ck["model_state_dict"]) == list(net.state_dict())
    other = torso_net(M, seed=7)
    s2 = TorsoTrainStep(other, other.args)
    assert s2.load(path) == 3
    assert all(torch.equal(a, b) for a, b in zip(net.state_dict().values(), other.state_dict().values()))
    assert s2.optimizer.param_groups[0]["lr"] == step.optimizer.param_groups[0]["lr"]


def test_load_head_into_torso(M, tmp_path):
    """A head.tar written by save_head_checkpoint loads into the torso network's head pair bit for bit, leaves the torso pair untouched,
    returns the latent codes, and a head trained with another expression width fails before anything is copied."""
    from ideal_nerf_b200 import checkpoint as ck
    torch.manual_seed(3)
    head = M.Network(450, 450, 1200., 0.57, 1.17, 8192, None, 64, 128, args=M.default_args(dim_aud=64, dim_expr=79))
    head.apply(M.init_weights)
    with torch.no_grad():
        for p in head.parameters():
            p.add_(torch.randn(p.shape) * 1e-2)
    lat = torch.randn(6, 32)
    path = str(tmp_path / "head.tar")
    ck.save_head_checkpoint(path, head, None, lat, 100)
    net = torso_net(M)
    torso_before = {k: v.clone() for k, v in net.state_dict().items() if k.startswith("torso_")}
    got = ck.load_head_into_torso(path, net)
    assert torch.equal(got, lat)
    for name in ("face_nerf_coarse", "face_nerf_fine"):
        for k, v in getattr(net, name).state_dict().items():
            assert torch.equal(v, head.state_dict()[f"{name}.{k}"]), (name, k)
    for k, v in net.state_dict().items():
        if k.startswith("torso_"):
            assert torch.equal(v, torso_before[k]), k
    # dim_expr 76 head into the default dim_expr 79 TorsoNetwork: the first-layer widths differ
    head76 = M.Network(450, 450, 1200., 0.57, 1.17, 8192, None, 64, 128, args=M.default_args(dim_aud=64, dim_expr=76))
    p76 = str(tmp_path / "head76.tar")
    ck.save_head_checkpoint(p76, head76, None, lat, 1)
    net2 = torso_net(M)
    before = {k: v.clone() for k, v in net2.state_dict().items()}
    with pytest.raises(ValueError, match=r"face_nerf_coarse\.pts_linears\.0\.weight.*dim_expr"):
        ck.load_head_into_torso(p76, net2)
    assert all(torch.equal(v, before[k]) for k, v in net2.state_dict().items()), "a failed load must copy nothing"
    # a file without the head pair
    torch.save({"global_step": 0, "model_state_dict": {}, "latent_codes": lat}, str(tmp_path / "empty.tar"))
    with pytest.raises(ValueError, match="has no 'face_nerf_coarse"):
        ck.load_head_into_torso(str(tmp_path / "empty.tar"), net2)
