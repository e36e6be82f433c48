"""Data-parallel training as one CUDA graph per rank: train.TrainStep / train.TorsoTrainStep(world=2, cuda_graph=True), the all-reduce
of the flat gradient recorded in each rank's graph.

GPU (two NCCL ranks, skipped below two GPUs): both stages fed from the device datasets on a write_head_subject subject, bf16,
perturb = 0, N_rand = 3072, eight steps on eight frames.  Every rank draws the full batch (sample(k, 0, 1): one draw per step keeps the
ranks' Philox offsets in lock-step) and steps on its band frame.band(3072, rank, 2); against one GPU stepping on the full batch, and
against the eager data-parallel step on the same bands.  Tolerances of test_torso_step_cuda_graph_matches_eager: losses within 2e-4
relative, parameters within 0.75 of the 8 x lr they can have moved (atomic dW sums can flip single Adam updates).

GPU (one NCCL rank): the same data-parallel code path -- rank agreement, the all-reduce captured in the graph -- on a one-rank group,
against the world=1 graph step, so that a one-GPU machine exercises the capture too.

CPU (two gloo ranks): graph mode refuses a gloo group, and train._check_ranks_agree."""
import os
import socket

import pytest
import torch

N_RAND, STEPS, FRAMES = 3072, 8, 8
ROWS = ("rays", "rays_head", "rays_torso", "bc_rgb", "target")          # the per-ray entries of a sample() batch


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _run_ranks(target, args, timeout, n=2):
    """n spawned ranks of target(rank, port, *args, q); returns {rank: what it put on q}.  A rank still running after `timeout` s is
    killed, so a hung collective fails the test instead of outliving it."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=target, args=(r, port) + tuple(args) + (q,)) for r in range(n)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=timeout)
    for p in procs:
        if p.is_alive():
            p.kill()
            p.join()
    assert [p.exitcode for p in procs] == [0] * n
    out = {}
    for _ in procs:
        rank, res = q.get(timeout=10)
        out[rank] = res
    return out


# ------------------------------------------------------------------------------------------------
# CPU: gloo
# ------------------------------------------------------------------------------------------------
def _gloo_rank(rank, port, q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=2)
    import ideal_nerf_b200 as M
    from ideal_nerf_b200.train import TorsoTrainStep, TrainStep, _check_ranks_agree
    res = {}
    net = M.Network(450, 450, 1200., 0.57, 1.17, 8192, None, 64, 128)
    tnet = M.TorsoNetwork(450, 450, 1200., 0.57, 1.17, 8192, 64, 128, args=M.default_args(dim_aud=64, dim_expr=79), dim_expr=79)
    for name, make in (("head", lambda: TrainStep(net, torch.zeros(2, 32), net.args, world=2, cuda_graph=True)),
                       ("torso", lambda: TorsoTrainStep(tnet, tnet.args, world=2, cuda_graph=True))):
        try:
            make()
            res[name] = None
        except ValueError as e:
            res[name] = str(e)
    key = ((1536, 11), (1536, 3), True, 0.0)
    _check_ranks_agree(key)                                                    # equal keys: returns
    try:
        _check_ranks_agree(((1536 + rank, 11),) + key[1:])
        res["differ"] = None
    except RuntimeError as e:
        res["differ"] = str(e)
    _check_ranks_agree(key)                                                    # both ranks raised above: still in step
    q.put((rank, res))
    dist.destroy_process_group()


def test_graph_dp_refuses_gloo_and_ranks_must_agree():
    """cuda_graph=True, world=2 on a gloo group: ValueError naming the backend, from both step classes (before the CUDA-tensor check, so
    on CPU parameters).  _check_ranks_agree returns when the ranks' keys are equal and raises RuntimeError on every rank, naming both
    keys, when they differ."""
    out = _run_ranks(_gloo_rank, (), 120)
    for rank in (0, 1):
        res = out[rank]
        for name in ("head", "torso"):
            assert res[name] is not None and "gloo" in res[name], (rank, name, res[name])
        assert res["differ"] is not None, rank
        assert "(1536, 11)" in res["differ"] and "(1537, 11)" in res["differ"], res["differ"]


# ------------------------------------------------------------------------------------------------
# GPU: two NCCL ranks
# ------------------------------------------------------------------------------------------------
def _args(M, stage):
    from ideal_nerf_b200 import synthetic as S
    common = dict(N_rand=N_RAND, mouth_rays=512, torso_rays=64, sample_rate=0.95, near=S.NEAR, far=S.FAR, dim_aud=64, dim_expr=76,
                  perturb=0., mlp_mode="bf16", lrate_decay=1, nosmo_iters=0)
    if stage == "head":
        return M.default_args(gt_dirs="head_imgs", lrate=3e-4, **common)
    return M.default_args(gt_dirs="com_imgs", lrate=1e-4, **common)


def _setup(M, stage, subject, dev):
    """(dataset, make_net) of a stage on the subject; make_net() returns a fresh network with rank 0's initial weights.  The density
    preset is computed on rank 0 and broadcast, so no rank depends on another rank's fp32 rounding."""
    import torch.distributed as dist
    from ideal_nerf_b200 import synthetic as S
    from ideal_nerf_b200.data import DeviceHeadDataset, DeviceTorsoDataset
    a = _args(M, stage)
    torch.manual_seed(4321)
    if stage == "head":
        ds = DeviceHeadDataset(subject, "aud.npy", "train", a, device=dev)
        net = M.Network(ds.H, ds.W, ds.focal, a.near, a.far, 8192, None, 64, 128, args=a)
    else:
        g = torch.Generator().manual_seed(3)
        aud, lat = torch.randn(FRAMES, 64, generator=g), torch.randn(FRAMES, 32, generator=g)
        ds = DeviceTorsoDataset(subject, "aud.npy", "train", a, aud, lat, device=dev)
        net = M.TorsoNetwork(ds.H, ds.W, ds.focal, a.near, a.far, 1 << 20, 64, 128, args=a, dim_expr=76)
    net.apply(M.init_weights)
    net = net.to(dev)
    M.ops.seed_rng(5, dev, 0)
    b = ds.sample(0)
    if stage == "head":
        with torch.no_grad():
            aud = net.aud_att_net(net.aud_net(b["aud_window"]))
        for m in (net.face_nerf_coarse, net.face_nerf_fine):
            S.normalise_density_(m, b["rays"], aud, b["expr"], torch.ones(32, device=dev))
    else:
        for m in (net.face_nerf_coarse, net.face_nerf_fine):
            S.normalise_density_(m, b["rays_head"], b["aud_feature"], b["expr"], b["latent_code"])
        sig = net.torso_signal(b["aud_feature"], b["pose"])
        for m in (net.torso_coarse_nerf, net.torso_fine_nerf):
            S.normalise_density_(m, b["rays_torso"], sig, None, None)
    sd = net.state_dict()
    for t in sd.values():
        dist.broadcast(t, 0)

    def make_net():
        fresh = M.Network(ds.H, ds.W, ds.focal, a.near, a.far, 8192, None, 64, 128, args=a) if stage == "head" else \
            M.TorsoNetwork(ds.H, ds.W, ds.focal, a.near, a.far, 1 << 20, 64, 128, args=a, dim_expr=76)
        fresh.load_state_dict(sd)
        return fresh.to(dev).train()

    return ds, make_net


def _make_step(stage, net, a, world, graph, dev):
    from ideal_nerf_b200.train import TorsoTrainStep, TrainStep
    if stage == "head":
        return TrainStep(net, torch.ones(FRAMES, 32, device=dev), a, world=world, cuda_graph=graph)
    return TorsoTrainStep(net, a, world=world, cuda_graph=graph)


def _call(stage, step, b, k):
    if stage == "head":
        out = step(b["rays"], b["bc_rgb"], b["target"], None, b["expr"], k, aud_window=b["aud_window"])
        return out, (float(out["img_loss"]), float(out["loss"]))
    out = step(**b)
    return out, (float(out["img_loss"]), float(out["img_loss0"]), float(out["loss"]))


def _dp_rank(rank, port, stage, against, subject, q):
    """One NCCL rank: the graph data-parallel step on its band, and the step it is compared with (rank 0's one-GPU graph step on the
    full batch, or this rank's eager data-parallel step on the same band)."""
    import torch.distributed as dist
    import ideal_nerf_b200 as M
    from ideal_nerf_b200.frame import band
    from ideal_nerf_b200.train import learning_rate
    dev = torch.device("cuda", rank)
    torch.cuda.set_device(dev)
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("nccl", rank=rank, world_size=2, device_id=dev)
    a = _args(M, stage)
    ds, make_net = _setup(M, stage, subject, dev)
    graph_dp = _make_step(stage, make_net(), a, 2, True, dev)
    ref = None
    if against == "eager_dp":
        ref = _make_step(stage, make_net(), a, 2, False, dev)
    elif rank == 0:
        ref = _make_step(stage, make_net(), a, 1, True, dev)
    lo, hi = band(N_RAND, rank, 2)
    M.ops.seed_rng(11, dev, 0)                                                  # the same stream on both ranks
    res = {"graph": [], "ref": [], "lr_err": 0.0}
    for k in range(STEPS):
        b = ds.sample(k, 0, 1)                                                  # the full batch of frame k
        mine = {key: (v[lo:hi] if key in ROWS else v) for key, v in b.items()}
        out, losses = _call(stage, graph_dp, mine, k)
        res["graph"].append(losses)
        res["lr_err"] = max(res["lr_err"], abs(float(out["lr"]) - learning_rate(a, k)))
        if ref is not None:
            res["ref"].append(_call(stage, ref, mine if against == "eager_dp" else b, k)[1])
    torch.cuda.synchronize()
    st = graph_dp._static
    res["captured"] = st["graph"] is not None and graph_dp.global_step == STEPS
    res["capture_mode"] = st.get("capture_mode")
    flat = graph_dp.flat.flat.detach()
    if ref is not None:
        res["param_err"] = float((flat.double() - ref.flat.flat.detach().double()).abs().max())
    every = [torch.empty_like(flat) for _ in range(2)]
    dist.all_gather(every, flat)
    res["ranks_bitwise_equal"] = torch.equal(every[0], every[1])
    q.put((rank, res))
    dist.destroy_process_group()


@pytest.fixture(scope="module")
def subject(tmp_path_factory):
    """A 128 x 128 subject of eight frames with com_imgs: head_imgs are the head stage's targets, com_imgs the torso stage's."""
    from ideal_nerf_b200 import synthetic as S
    d = str(tmp_path_factory.mktemp("dp_subject"))
    S.write_head_subject(d, 128, 128, n_frames=FRAMES, seed=1, torso_rows=12, com_imgs=True)
    return d


def _one_rank(rank, port, subject, q):
    """A one-rank NCCL group: each stage's step built with world=2 takes the data-parallel path (the rank-agreement exchange, the NCCL
    all-reduce recorded in the graph), where an average over one rank leaves the gradient as it is, next to a world=1 graph step on the
    same batches."""
    import torch.distributed as dist
    import ideal_nerf_b200 as M
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("nccl", rank=0, world_size=1, device_id=dev)
    res = {}
    for stage in ("head", "torso"):
        a = _args(M, stage)
        ds, make_net = _setup(M, stage, subject, dev)
        dp, one = _make_step(stage, make_net(), a, 2, True, dev), _make_step(stage, make_net(), a, 1, True, dev)
        M.ops.seed_rng(11, dev, 0)
        curves = ([], [])
        for k in range(STEPS):
            b = ds.sample(k)
            curves[0].append(_call(stage, dp, b, k)[1])
            curves[1].append(_call(stage, one, b, k)[1])
        torch.cuda.synchronize()
        res[stage] = {"curves": curves, "captured": dp._static["graph"] is not None, "capture_mode": dp._static["capture_mode"],
                      "param_err": float((dp.flat.flat.detach().double() - one.flat.flat.detach().double()).abs().max())}
    q.put((rank, res))
    dist.destroy_process_group()


@pytest.mark.gpu
def test_graph_step_records_nccl_all_reduce_on_one_gpu(subject):
    """On one GPU: TrainStep / TorsoTrainStep(world=2, cuda_graph=True) on a one-rank NCCL group capture their graph with the all-reduce
    in it and follow the world=1 graph step over eight steps, to the tolerances of test_graph_dp_matches."""
    out = _run_ranks(_one_rank, (subject,), 300, n=1)[0]
    for stage, lr in (("head", 3e-4), ("torso", 1e-4)):
        res = out[stage]
        print(stage, res["capture_mode"], res["curves"])
        assert res["captured"], stage
        for got, want in zip(*res["curves"]):
            for x, y in zip(got, want):
                assert abs(x - y) <= 2e-4 * abs(y), (stage, res["curves"])
        assert res["param_err"] <= 0.75 * STEPS * lr, (stage, res["param_err"])


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="two NCCL ranks need two GPUs")
@pytest.mark.parametrize("against", ["one_gpu", "eager_dp"])
@pytest.mark.parametrize("stage", ["head", "torso"])
def test_graph_dp_matches(subject, stage, against):
    """TrainStep (stage "head", lr 3e-4) / TorsoTrainStep ("torso", lr 1e-4) with world=2, cuda_graph=True on two NCCL ranks, eight steps:
    the graph is captured on both ranks; the device lr equals learning_rate(args, k); both ranks' flat parameters are bitwise equal;
    against "one_gpu", the mean of the ranks' losses is within 2e-4 relative of a world=1 graph step on the full batch at every step,
    against "eager_dp", every rank's losses are within 2e-4 of the eager world=2 step's on the same band; the parameters within
    0.75 x 8 x lr of the compared run's."""
    out = _run_ranks(_dp_rank, (stage, against, subject), 300)
    lr = 3e-4 if stage == "head" else 1e-4
    print({r: (res["capture_mode"], res["graph"], res["ref"]) for r, res in out.items()})
    for rank, res in out.items():
        assert res["captured"], rank
        assert res["lr_err"] < 1e-10, (rank, res["lr_err"])
        assert res["ranks_bitwise_equal"], rank
    if against == "one_gpu":
        pairs = [([(x + y) / 2 for x, y in zip(g0, g1)], r) for g0, g1, r in zip(out[0]["graph"], out[1]["graph"], out[0]["ref"])]
        errs = [out[0]["param_err"]]
    else:
        pairs = [(g, r) for res in out.values() for g, r in zip(res["graph"], res["ref"])]
        errs = [res["param_err"] for res in out.values()]
    for got, want in pairs:
        for x, y in zip(got, want):
            assert abs(x - y) <= 2e-4 * abs(y), (stage, against, got, want)
    assert max(errs) <= 0.75 * STEPS * lr, (stage, against, errs)
