"""GPU tests of the training driver (ideal_nerf_b200.fit) on a 128 x 128 write_head_subject subject: eight constant-colour train frames,
four val frames (Network.audio_window pads a split correctly from smo_size / 2 frames on), com_imgs for the torso stage; bf16,
N_rand = 1024, perturb = 0.  Every run starts from the same head.tar at global_step 0 (init_weights with the density preset of
synthetic.normalise_density_, so that the rays are neither empty nor opaque), which the driver resumes from like any checkpoint.

Tolerances are those of test_train_step_cuda_graph_matches_eager and test_train_graph_dp (the dW reductions are atomic, so two runs of
the same program agree to float rounding, and Adam's sign-like updates can flip single parameters): losses within 2e-4 relative,
parameters within half of the `steps x lr` they can have moved (0.75 x for the two-rank run)."""
import json
import os
import shutil
import socket

import pytest
import torch

FRAMES, N_RAND, LR = 8, 1024, 3e-4
DEV = "cuda"


def _args(subject, basedir, expname, **over):
    from ideal_nerf_b200 import fit
    from ideal_nerf_b200 import synthetic as S
    a = fit.fit_parser().parse_args([])
    base = dict(datadir=subject, basedir=str(basedir), expname=expname, N_rand=N_RAND, mouth_rays=128, torso_rays=64, sample_rate=0.95,
                near=S.NEAR, far=S.FAR, dim_aud=64, dim_expr=76, perturb=0., mlp_mode="bf16", lrate=LR, nosmo_iters=0, N_iters=1,
                i_print=4, i_weights=0, i_testset=0, i_img=0, gt_dirs="head_imgs")
    base.update(over)
    for k, v in base.items():
        setattr(a, k, v)
    return a


@pytest.fixture(scope="module")
def subject(tmp_path_factory):
    from ideal_nerf_b200 import synthetic as S
    d = str(tmp_path_factory.mktemp("fit_subject"))
    S.write_head_subject(d, 128, 128, n_frames=FRAMES, seed=2, torso_rows=12, constant_rgb=(200, 90, 40), val_frames=4, com_imgs=True)
    return d


@pytest.fixture(scope="module")
def start_tar(subject, tmp_path_factory):
    """head.tar at global_step 0: init_weights (seed 0) with the density preset, an Adam without state."""
    import ideal_nerf_b200 as M
    from ideal_nerf_b200 import synthetic as S
    from ideal_nerf_b200.data import DeviceHeadDataset
    from ideal_nerf_b200.train import TrainStep
    a = _args(subject, "unused", "unused")
    dev = torch.device(DEV, torch.cuda.current_device())
    ds = DeviceHeadDataset(subject, "aud.npy", "train", a, device=dev)
    torch.manual_seed(0)
    net = M.Network(ds.H, ds.W, ds.focal, a.near, a.far, a.chunk, None, 64, 128, args=a)
    net.apply(M.init_weights)
    net = net.to(dev)
    M.ops.seed_rng(5, dev, 0)
    b = ds.sample(0)
    with torch.no_grad():
        aud = net.aud_att_net(net.aud_net(b["aud_window"]))
    for m in (net.face_nerf_coarse, net.face_nerf_fine):
        S.normalise_density_(m, b["rays"], aud, b["expr"], torch.ones(32, device=dev))
    path = str(tmp_path_factory.mktemp("start") / "head.tar")
    TrainStep(net, torch.ones(FRAMES, 32, device=dev), a).save(path)
    return path


def _prepare(args, start_tar):
    d = os.path.join(args.basedir, args.expname)
    os.makedirs(d, exist_ok=True)
    shutil.copy(start_tar, os.path.join(d, "head.tar"))
    return d


def _log(d):
    with open(os.path.join(d, "log.jsonl")) as fp:
        lines = [json.loads(s) for s in fp]
    return [x for x in lines if "train/loss" in x], [x for x in lines if "val/psnr" in x or "val/psnr_torso" in x]


def _max_err(a, b):
    return float((a.detach().double() - b.detach().double()).abs().max())


@pytest.mark.gpu
def test_fit_head_trains_logs_saves_and_validates(subject, start_tar, tmp_path):
    """24 steps (three epochs): the training loss falls; log.jsonl has one line per step with the reference's scalar names, learning
    rates equal to train.learning_rate; head.tar is written at i_weights and at the end with global_step; val scores at every i_testset
    step; one PNG at i_img."""
    from ideal_nerf_b200 import fit
    from ideal_nerf_b200.train import learning_rate
    a = _args(subject, tmp_path, "head", N_iters=3, i_print=4, i_weights=8, i_testset=12, i_img=24, lrate=2e-3)
    d = _prepare(a, start_tar)
    saved = []
    f = fit.HeadFit(a)
    assert f.resumed == os.path.join(d, "head.tar") and f.step.global_step == 0
    for stop in (8, 16, 24):                                  # the checkpoint of each i_weights boundary, read before it is rewritten
        f.run(stop)
        saved.append(torch.load(os.path.join(d, "head.tar"), map_location="cpu", weights_only=False)["global_step"])
    train, val = _log(d)
    print([round(x["train/loss"], 5) for x in train], val)
    assert saved == [8, 16, 24]
    assert [x["step"] for x in train] == list(range(1, 25))
    for x in train:
        assert set(x) == {"step", "train/loss", "train/psnr", "train/learning_rate", "train/latent_code_loss"}
        assert abs(x["train/learning_rate"] - learning_rate(a, x["step"] - 1)) <= 1e-6 * a.lrate
    first = sum(x["train/loss"] for x in train[:4]) / 4
    last = sum(x["train/loss"] for x in train[-4:]) / 4
    assert last < 0.9 * first, (first, last)
    assert [x["step"] for x in val] == [12, 24]
    for x in val:
        assert set(x) == {"step", "val/psnr", "val/psnr_face", "val/psnr_mouth", "val/ssim"}
        assert all(0 < x[k] < 100 for k in ("val/psnr", "val/psnr_face", "val/psnr_mouth")) and -1 <= x["val/ssim"] <= 1
    assert val[1]["val/psnr"] > val[0]["val/psnr"] - 1.0
    assert os.path.isfile(os.path.join(d, "val_000024.png")) and not os.path.exists(os.path.join(d, "val_000012.png"))
    assert sorted(n for n in os.listdir(d) if n.endswith(".tar")) == ["head.tar"]


@pytest.mark.gpu
def test_fit_head_resume_matches_uninterrupted_run(subject, start_tar, tmp_path):
    """16 steps in one run against 8 steps, a restart that resumes from head.tar, 8 more: weights, latent codes and Adam moments agree
    to the graph-vs-eager bound, global_step and the learning rate are equal, and log.jsonl continues without a gap."""
    from ideal_nerf_b200 import fit
    _prepare(_args(subject, tmp_path, "one"), start_tar)
    one = fit.fit_head(_args(subject, tmp_path, "one", N_iters=2, i_print=4, i_weights=8))
    _prepare(_args(subject, tmp_path, "two"), start_tar)
    first = fit.fit_head(_args(subject, tmp_path, "two", N_iters=1, i_print=4, i_weights=8))
    assert first.step.global_step == 8
    del first
    two = fit.fit_head(_args(subject, tmp_path, "two", N_iters=2, i_print=4, i_weights=8))
    assert two.resumed is not None and two.step.global_step == 16 == one.step.global_step
    assert float(two.step._lr_t) == float(one.step._lr_t)
    bound = 0.5 * 16 * LR
    assert _max_err(two.step.flat.flat, one.step.flat.flat) <= bound
    assert _max_err(two.step.latent_codes, one.step.latent_codes) <= bound
    s1, s2 = one.step.optimizer.state[one.step.flat.flat], two.step.optimizer.state[two.step.flat.flat]
    assert float(s1["step"]) == float(s2["step"]) == 16
    for k in ("exp_avg", "exp_avg_sq"):
        scale = float(s1[k].abs().max())
        assert _max_err(s2[k], s1[k]) <= 0.05 * scale, (k, _max_err(s2[k], s1[k]), scale)
    t1, _ = _log(os.path.join(str(tmp_path), "one"))
    t2, _ = _log(os.path.join(str(tmp_path), "two"))
    assert [x["step"] for x in t2] == list(range(1, 17))
    for x, y in zip(t1, t2):
        assert abs(x["train/loss"] - y["train/loss"]) <= 2e-4 * abs(x["train/loss"]), (t1, t2)


@pytest.mark.gpu
def test_fit_head_audio_phases(subject, start_tar, tmp_path):
    """nosmo_iters = 8: during steps 0-7 AudioNet trains and AudioAttNet does not move; from step 8 both train.  The graphed run's losses
    follow an eager TrainStep loop conditioned on Network.audio_feature(auds, i, F, global_step) over the same frames and draws.  A
    TrainStep built without max_graphs still raises when its key changes."""
    import ideal_nerf_b200 as M
    from ideal_nerf_b200 import fit
    from ideal_nerf_b200.train import TrainStep
    a = _args(subject, tmp_path, "phases", N_iters=2, i_print=8, nosmo_iters=8)
    d = _prepare(a, start_tar)
    f = fit.HeadFit(a)
    net = f.step.net

    def snap(m):
        return torch.cat([p.detach().reshape(-1) for p in m.parameters()]).clone()

    aud0, att0 = snap(net.aud_net), snap(net.aud_att_net)
    f.run(8)
    aud8, att8 = snap(net.aud_net), snap(net.aud_att_net)
    assert not torch.equal(aud8, aud0), "AudioNet trains before nosmo_iters"
    assert torch.equal(att8, att0), "AudioAttNet does not move before nosmo_iters"
    f.run()
    assert not torch.equal(snap(net.aud_net), aud8) and not torch.equal(snap(net.aud_att_net), att8), "both train after nosmo_iters"
    assert len(f.step._graphs) == 2 and all(st["graph"] is not None for st in f.step._graphs.values())
    graphed = [x["train/loss"] for x in _log(d)[0]]

    # the eager loop: the same start, frames, Philox seeds (re-seeded where the driver re-seeds: after the log boundary at step 8)
    dev = f.dev
    ds = f.ds
    enet = M.Network(ds.H, ds.W, ds.focal, a.near, a.far, a.chunk, None, 64, 128, args=a).to(dev).train()
    eager = TrainStep(enet, torch.ones(FRAMES, 32, device=dev), a)
    eager.load(start_tar, map_location=dev)
    losses = []
    for g in range(16):
        if g % 8 == 0:
            M.ops.seed_rng(0, dev, fit.RNG_STRIDE * g)
            order = fit.epoch_order(0, g // 8, FRAMES)
        i = int(order[g % 8])
        b = ds.sample(i)
        aud = enet.audio_feature(ds.auds, i, FRAMES, g)
        losses.append(float(eager(b["rays"], b["bc_rgb"], b["target"], aud, b["expr"], i)["loss"]))
    print("graphed", graphed)
    print("eager  ", losses)
    assert len(graphed) == 16
    for x, y in zip(graphed, losses):
        assert abs(x - y) <= 2e-4 * abs(y), (graphed, losses)

    del aud                                          # its autograd graph would keep the eager loop's gradient accumulators alive
    pnet = M.Network(ds.H, ds.W, ds.focal, a.near, a.far, a.chunk, None, 64, 128, args=a).to(dev).train()
    plain = TrainStep(pnet, torch.ones(FRAMES, 32, device=dev), a, cuda_graph=True)
    b = ds.sample(0)
    for _ in range(2):
        plain(b["rays"], b["bc_rgb"], b["target"], None, b["expr"], 0, aud_window=b["aud_window"])
    with pytest.raises(RuntimeError, match="fixed per TrainStep"):
        plain(b["rays"], b["bc_rgb"], b["target"], None, b["expr"], 0, aud_window=b["aud_window"], smooth=False)


@pytest.mark.gpu
def test_fit_steps_between_log_boundaries_do_not_synchronise(subject, start_tar, tmp_path):
    """After the capture, the steps between two i_print boundaries -- an epoch boundary among them, with its permutation upload -- run
    under torch.cuda.set_sync_debug_mode("error"): nothing in them synchronises with the device."""
    from ideal_nerf_b200 import fit
    a = _args(subject, tmp_path, "nosync", N_iters=3, i_print=6)
    d = _prepare(a, start_tar)
    f = fit.HeadFit(a)
    f.run(6)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        f.run(11)                                            # steps 7..11; the second epoch starts at step 9
    finally:
        torch.cuda.set_sync_debug_mode(0)
    f.run(12)
    assert [x["step"] for x in _log(d)[0]] == list(range(1, 13))


@pytest.mark.gpu
def test_fit_torso_trains_the_torso_pair_only(subject, start_tar, tmp_path):
    """fit_torso under a head.tar of fit_head: the head pair stays bit-equal to the head.tar's, the torso pair moves, the torso checkpoint
    is {step:06d}_torso.tar, the log has one line per step and the val scores carry val/psnr_torso."""
    from ideal_nerf_b200 import fit
    ha = _args(subject, tmp_path, "head", N_iters=1, i_print=4)
    hd = _prepare(ha, start_tar)
    fit.fit_head(ha)
    head_tar = os.path.join(hd, "head.tar")
    head_sd = torch.load(head_tar, map_location="cpu", weights_only=False)["model_state_dict"]
    ta = _args(subject, tmp_path, "torso", gt_dirs="com_imgs", N_iters=1, i_print=4, i_testset=8, lrate=1e-4)
    f = fit.TorsoFit(ta, head_tar)
    before = {k: v.detach().clone() for k, v in f.step.net.state_dict().items()}
    f.run()
    after = f.step.net.state_dict()
    for k, v in after.items():
        if k.startswith("face_nerf_"):
            assert torch.equal(v.cpu(), head_sd[k]), k
            assert torch.equal(v, before[k]), k
    moved = [k for k in after if k.startswith("torso_") and not torch.equal(after[k], before[k])]
    assert any(k.startswith("torso_coarse_nerf.") for k in moved) and any(k.startswith("torso_fine_nerf.") for k in moved)
    td = os.path.join(str(tmp_path), "torso")
    assert sorted(n for n in os.listdir(td) if n.endswith(".tar")) == ["000008_torso.tar"]
    train, val = _log(td)
    assert [x["step"] for x in train] == list(range(1, 9))
    assert set(train[0]) == {"step", "train/loss", "train/psnr", "train/learning_rate"}
    assert len(val) == 1 and val[0]["step"] == 8 and 0 < val[0]["val/psnr_torso"] < 100


# ------------------------------------------------------------------------------------------------
# two NCCL ranks
# ------------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _rank(rank, port, args, q):
    import torch.distributed as dist
    from ideal_nerf_b200 import fit
    dev = torch.device("cuda", rank)
    torch.cuda.set_device(dev)
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("nccl", rank=rank, world_size=2, device_id=dev)
    f = fit.fit_head(args, rank, 2)
    q.put((rank, f.step.global_step))
    dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="two NCCL ranks need two GPUs")
def test_fit_head_two_ranks_matches_one_gpu(subject, start_tar, tmp_path):
    """fit_head on two NCCL ranks (each rank steps on its band of every batch) for 8 steps against one GPU on the full batches: the rank-0
    head.tar matches within the two-rank bound of test_train_graph_dp; log.jsonl has each step once and the validation line once, so
    rank 1 wrote nothing."""
    import torch.multiprocessing as mp
    from ideal_nerf_b200 import fit
    kw = dict(N_iters=1, i_print=4, i_testset=8)
    dp, one = _args(subject, tmp_path, "dp", **kw), _args(subject, tmp_path, "one", **kw)
    _prepare(dp, start_tar)
    _prepare(one, start_tar)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_rank, args=(r, port, dp, q)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=600)
    for p in procs:
        if p.is_alive():
            p.kill()
            p.join()
    assert [p.exitcode for p in procs] == [0, 0]
    assert sorted(q.get(timeout=10) for _ in procs) == [(0, 8), (1, 8)]
    fit.fit_head(one)
    ck = [torch.load(os.path.join(str(tmp_path), n, "head.tar"), map_location="cpu", weights_only=False) for n in ("dp", "one")]
    assert ck[0]["global_step"] == ck[1]["global_step"] == 8
    bound = 0.75 * 8 * LR
    for k, v in ck[1]["model_state_dict"].items():
        assert _max_err(ck[0]["model_state_dict"][k], v) <= bound, k
    assert _max_err(ck[0]["latent_codes"], ck[1]["latent_codes"]) <= bound
    train, val = _log(os.path.join(str(tmp_path), "dp"))
    assert [x["step"] for x in train] == list(range(1, 9)) and [x["step"] for x in val] == [8]
