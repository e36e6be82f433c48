"""GPU tests of the torso stage (NeRFs/TorsoNeRF/train_torso.py): the loss kernel inerf_head_torso_mse_pair and train.TorsoTrainStep --
gradients against the CPU oracle, the head-then-torso order of the in-kernel draws, the frozen head, bf16 against fp32 over a real
optimisation, the CUDA-graph mode, resume, and two data-parallel ranks.

The networks are built as in test_gpu_parity.test_head_torso_frame_band_config4: four init_face_nerf presets with normalised density
(the torso neither empty nor opaque), dim_expr 79, the torso conditioned on [aud[:64] | gamma_3(euler) | gamma_3(trans)]."""
import os
import socket

import numpy as np
import pytest
import torch

from oracle import render_oracle as O

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
SEEDS = {"face_nerf_coarse": 21, "face_nerf_fine": 22, "torso_coarse_nerf": 23, "torso_fine_nerf": 24}


@pytest.fixture(scope="module")
def M():
    import ideal_nerf_b200 as m
    assert torch.cuda.is_available(), "-m gpu tests need a GPU"
    m.lib()                                       # raises if the extension is missing: no fallback
    m._lib.check(m.lib().inerf_device_check(), "inerf_device_check")
    return m


def maxabs(a, b):
    return float((a.detach().double().cpu() - b.detach().double().cpu()).abs().max())


def close(a, b, tol, what=""):
    e = maxabs(a, b)
    assert e <= tol, f"{what}: max-abs {e:.3e} > {tol:.1e}"


def bits_equal(a, b):
    a, b = a.detach().cpu().numpy(), b.detach().cpu().numpy()
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def _pose(k=0):
    c2w = O.synthetic_camera()["c2w"].clone()
    c2w[:3, 3] += torch.tensor([0.01 + 0.002 * k, -0.02, 0.001 * k])
    return c2w


def _signal(aud, pose):
    et = O.pose_to_euler_trans(pose[None])
    return torch.cat([aud[:64], O.positional_encoding(et[:, :3], 3).squeeze(0), O.positional_encoding(et[:, 3:], 3).squeeze(0)])


_CACHE = {}


def inputs():
    """Host inputs of one batch (3 072 rays of the synthetic training batch for both pairs) and the four normalised state dicts."""
    if "in" not in _CACHE:
        b = O.synthetic_train_batch(0)
        g = torch.Generator().manual_seed(4)
        aud, expr, lat = b["aud"], torch.randn(79, generator=g), b["latent"]
        pose = _pose()
        sig = _signal(aud, pose)
        sds = {}
        for k, seed in SEEDS.items():
            head = k.startswith("face")
            sd = O.init_face_nerf(seed, 64, 79, 32) if head else O.init_face_nerf(seed, 106, 0, 0)
            sds[k] = O.normalise_density(sd, b["rays"], aud if head else sig, expr if head else None, lat if head else None)
        _CACHE["in"] = dict(rays=b["rays"], bc=b["bc_rgb"], target=b["target"], aud=aud, expr=expr, lat=lat, pose=pose, sig=sig, sds=sds)
    return _CACHE["in"]


def network(M, mode="fp32", torso_seeds=None, **over):
    d = inputs()
    kw = dict(dim_aud=64, dim_expr=79, perturb=0., mlp_mode=mode, lrate=3e-4)
    kw.update(over)
    net = M.TorsoNetwork(450, 450, 1200., O.NEAR, O.FAR, 1 << 20, 64, 128, args=M.default_args(**kw))
    for k, sd in d["sds"].items():
        if torso_seeds is not None and not k.startswith("face"):
            seed = torso_seeds[0] if "coarse" in k else torso_seeds[1]
            sd = O.normalise_density(O.init_face_nerf(seed, 106, 0, 0), d["rays"], d["sig"], None, None)
        getattr(net, k).load_state_dict(sd)
    return net.to(DEV).train()


def dev_inputs(sl=slice(None)):
    d = inputs()
    return (d["rays"][sl].to(DEV), d["rays"][sl].to(DEV), d["bc"][sl].to(DEV), d["target"][sl].to(DEV), d["aud"].to(DEV),
            d["pose"].to(DEV), d["expr"].to(DEV), d["lat"].to(DEV))


# ------------------------------------------------------------------------------------------------
# the kernel
# ------------------------------------------------------------------------------------------------
def _unaligned(shape, gen, lo=0., hi=1.):
    n = int(np.prod(shape))
    return (lo + (hi - lo) * torch.rand(n + 1, device=DEV, generator=gen))[1:].view(shape)      # 4 bytes past a 256-byte boundary


@pytest.mark.parametrize("n", [1, 5, 3072, 100003])
def test_head_torso_mse_pair_kernel(M, n):
    """Against float64 torch and against autograd of ops.mse_pair(ops.head_torso_blend(...)): g_rgb_fg bit for bit, g_last_weight within
    1e-6 of the magnitude of its three terms (the sum order may differ), the losses within 1e-6 relative; unaligned views throughout."""
    ops = M.ops
    gen = torch.Generator(device=DEV).manual_seed(n)
    h, h0, t = _unaligned((n, 3), gen), _unaligned((n, 3), gen), _unaligned((n, 3), gen)
    w, w0 = _unaligned((n,), gen), _unaligned((n,), gen)
    f, f0 = _unaligned((n, 3), gen, -0.2, 0.8), _unaligned((n, 3), gen, -0.2, 0.8)
    assert all(x.data_ptr() % 16 == 4 for x in (h, w, f, t))
    leaves = lambda: [x.detach().clone().requires_grad_(True) for x in (w, w0, f, f0)]
    a = leaves()
    l_ref = ops.mse_pair(ops.head_torso_blend(h, a[0], a[2]), ops.head_torso_blend(h0, a[1], a[3]), t)
    (l_ref[0] + l_ref[1]).backward()
    b = [_unaligned(x.shape, gen) for x in (w, w0, f, f0)]
    for dst, src in zip(b, (w, w0, f, f0)):
        dst.copy_(src)
    b = [x.requires_grad_(True) for x in b]
    l2 = ops.head_torso_mse_pair(h, h0, b[0], b[1], b[2], b[3], t)
    (l2[0] + l2[1]).backward()
    for i in (2, 3):
        assert bits_equal(b[i].grad, a[i].grad), ("g_rgb_fg", i, maxabs(b[i].grad, a[i].grad))
    for i, hh in ((0, h), (1, h0)):
        scale = (a[i + 2].grad.abs() * hh.abs()).sum(-1)
        assert bool(((b[i].grad - a[i].grad).abs() <= 1e-6 * scale + 1e-30).all()), ("g_last_weight", i)
    # float64
    H, H0, T, W, W0, F, F0 = (x.detach().double() for x in (h, h0, t, w, w0, f, f0))
    c, c0 = H * W[:, None] + F - T, H0 * W0[:, None] + F0 - T
    want = torch.stack([(c ** 2).mean(), (c0 ** 2).mean()])
    for k in range(2):
        assert abs(float(l2[k]) - float(want[k])) <= 1e-6 * float(want[k]), ("loss vs float64", k)
        assert abs(float(l2[k]) - float(l_ref[k])) <= 1e-6 * float(l_ref[k]), ("loss vs mse_pair", k)
    g64 = 2 * c / (3 * n)
    close(b[2].grad, g64, 1e-6 * float(g64.abs().max()), "g_rgb_fg vs float64")
    close(b[0].grad, (g64 * H).sum(-1), 1e-6 * float((g64.abs() * H).sum(-1).max()), "g_last_weight vs float64")
    # a head image that requires grad would lose its gradient: refused
    with pytest.raises(ValueError, match="rgb_head"):
        ops.head_torso_mse_pair(h.detach().clone().requires_grad_(True), h0, b[0], b[1], b[2], b[3], t)
    with pytest.raises(ValueError, match="rgb_head"):
        ops.head_torso_mse_pair(h, h0.detach().clone().requires_grad_(True), b[0], b[1], b[2], b[3], t)


# ------------------------------------------------------------------------------------------------
# TorsoTrainStep
# ------------------------------------------------------------------------------------------------
def test_torso_step_grads_match_oracle(M):
    """fp32 mode, perturb = 0, 512 rays: the flat gradient of one step against autograd through the CPU oracle (head rendered without
    grad, torso state dicts requiring grad, loss = MSE of both composites); tolerance as test_train_step_grads_golden."""
    from ideal_nerf_b200.train import TorsoTrainStep
    d = inputs()
    sl = slice(0, 3072, 6)
    net = network(M)
    step = TorsoTrainStep(net, net.args)
    out = step(*dev_inputs(sl), perturb=0.)
    rays, bc, tgt = d["rays"][sl], d["bc"][sl], d["target"][sl]
    with torch.no_grad():
        h = O.render_rays(rays, bc, d["sds"]["face_nerf_coarse"], d["sds"]["face_nerf_fine"], d["aud"], d["expr"], d["lat"], with_fg=True)
    tsd = {k: {n: v.clone().requires_grad_(True) for n, v in d["sds"][k].items()} for k in ("torso_coarse_nerf", "torso_fine_nerf")}
    t = O.render_rays(rays, bc, tsd["torso_coarse_nerf"], tsd["torso_fine_nerf"], d["sig"], None, None, with_fg=True)
    com = O.head_torso_blend(h["rgb_map"], t["last_weight"], t["rgb_map_fg"])
    com0 = O.head_torso_blend(h["rgb0"], t["last_weight0"], t["rgb_map_fg0"])
    l, l0 = torch.mean((com - tgt) ** 2), torch.mean((com0 - tgt) ** 2)
    (l + l0).backward()
    for k, ref in (("img_loss", l), ("img_loss0", l0)):
        assert abs(float(out[k]) - float(ref)) <= 1e-4 * float(ref), (k, float(out[k]), float(ref))
    names = [n for n, _ in net.named_parameters() if n.startswith("torso_")]
    assert len(names) == len(step.flat.gviews)
    checked = 0
    for name, gv in zip(names, step.flat.gviews):
        mod, _, pname = name.partition(".")
        ref = tsd[mod][pname].grad
        if ref is None:
            assert pname.startswith("feature_linear") and not bool(gv.any()), name
            continue
        close(gv, ref, 2e-3 * max(1e-3, float(ref.abs().max())), name)
        checked += 1
    assert checked == 2 * 26


def test_torso_step_draw_order_matches_forward(M):
    """perturb = 1, fp32, the Philox state re-seeded before each: img_loss / img_loss0 of one step equal the MSE of TorsoNetwork.forward's
    two composites to float rounding -- and not the MSE of the same renders drawn torso-first, which pins the head-then-torso order."""
    from ideal_nerf_b200.train import TorsoTrainStep
    ops = M.ops
    sl = slice(0, 1024)
    rays_h, rays_t, bc, tgt, aud, pose, expr, lat = dev_inputs(sl)
    net = network(M)
    ops.seed_rng(1234, DEV, offset=3)
    with torch.no_grad():
        rgb, rgb0 = net(rays_h, rays_t, bc, aud, pose, expr, lat, perturb=1.)
        want = [float(((rgb - tgt) ** 2).mean()), float(((rgb0 - tgt) ** 2).mean())]
        ops.seed_rng(1234, DEV, offset=3)                          # the same draws, torso first
        torso = net.render_pair("torso", rays_t, bc, net.torso_signal(aud, pose), None, None, 1.)
        head = net.render_pair("head", rays_h, bc, aud, expr, lat, 1.)
        swapped = float(((ops.head_torso_blend(head["rgb_map"], torso["last_weight"], torso["rgb_map_fg"]) - tgt) ** 2).mean())
    step = TorsoTrainStep(net, net.args)
    ops.seed_rng(1234, DEV, offset=3)
    out = step(rays_h, rays_t, bc, tgt, aud, pose, expr, lat, perturb=1.)
    got = [float(out["img_loss"]), float(out["img_loss0"])]
    print("forward", want, "step", got, "torso-first", swapped)
    for a, b in zip(got, want):
        assert abs(a - b) <= 1e-5 * b, (got, want)
    assert abs(swapped - want[0]) > 1e-4 * want[0], "the draws do not depend on the order: this check proves nothing"
    assert int(ops.rng_state(DEV)[1].item()) == 3 + 2                # one advance per pair, as forward()


def test_torso_step_freezes_the_head(M):
    """10 bf16 steps: the head pair's parameters are bit-identical, its packed blob is the object built at step 1, and every torso tensor
    except the unused feature_linear has moved."""
    from ideal_nerf_b200.train import TorsoTrainStep
    net = network(M, "bf16")
    head_before = {n: p.detach().clone() for n, p in net.named_parameters() if n.startswith("face_nerf_")}
    torso_before = {n: p.detach().clone() for n, p in net.named_parameters() if n.startswith("torso_")}
    step = TorsoTrainStep(net, net.args)
    args = dev_inputs()
    step(*args, perturb=1.)
    blobs = (net.face_nerf_coarse._packed, net.face_nerf_fine._packed)
    assert all(b is not None for b in blobs)
    for _ in range(9):
        step(*args, perturb=1.)
    torch.cuda.synchronize()
    assert net.face_nerf_coarse._packed is blobs[0] and net.face_nerf_fine._packed is blobs[1]
    for n, p in net.named_parameters():
        if n.startswith("face_nerf_"):
            assert torch.equal(p.detach(), head_before[n]), n
            assert p.grad is None, n
        elif "feature_linear" in n:
            assert torch.equal(p.detach(), torso_before[n]), n
        else:
            assert not torch.equal(p.detach(), torso_before[n]), f"{n} did not move"
    assert step.global_step == 10


def test_torso_bf16_vs_fp32_training_500_steps(M):
    """500 steps of each mode towards the render of a teacher TorsoNetwork (the same head; other torso weights), with the schedule of
    test_bf16_vs_fp32_training_500_steps (the learning rate decaying one decade per 300 steps, perturb = 0): both modes gain >= 1 dB and
    their final PSNR (mean of the last 50 steps) agrees within 0.1 dB.  The run starts at lr 3e-5, not the head test's 3e-4: Adam's
    first update moves every weight by about the learning rate whatever its gradient, and at 3e-4 that first step collapses the density
    of this normalised-density torso for good (PSNR 25.5 -> 22.1 dB, flat for the rest of the run, in both modes alike).  The student
    nearly recovers the teacher here, so the final PSNR is high and bf16 rounding shows in it: at 1e-4 the runs end at 45.66 (fp32) and
    45.53 dB (bf16), at 3e-5 at 41.31 and 41.23 dB."""
    from ideal_nerf_b200.train import TorsoTrainStep
    rays_h, rays_t, bc, _, aud, pose, expr, lat = dev_inputs()
    with torch.no_grad():
        target = network(M).eval()(rays_h, rays_t, bc, aud, pose, expr, lat, perturb=0.)[0]
    curves = {}
    for mode in ("fp32", "bf16"):
        net = network(M, mode, torso_seeds=(33, 34), lrate=3e-5, lrate_decay=0.2)
        step = TorsoTrainStep(net, net.args)
        losses = [step(rays_h, rays_t, bc, target, aud, pose, expr, lat, perturb=0.)["img_loss"] for _ in range(500)]
        curves[mode] = -10. * torch.log10(torch.stack(losses)).cpu()
    p32, p16 = curves["fp32"], curves["bf16"]
    print(f"PSNR step 0: fp32 {float(p32[0]):.3f} bf16 {float(p16[0]):.3f}; last-50 mean: fp32 {float(p32[-50:].mean()):.3f} "
          f"bf16 {float(p16[-50:].mean()):.3f}")
    assert float(p32[-50:].mean()) > float(p32[0]) + 1.0 and float(p16[-50:].mean()) > float(p16[0]) + 1.0
    assert abs(float(p32[-50:].mean()) - float(p16[-50:].mean())) <= 0.1


def test_torso_step_cuda_graph_matches_eager(M):
    """cuda_graph=True against eager over 8 bf16 steps with a different ray batch, pose, audio code and latent code every step: losses
    within 2e-4 relative, parameters within 0.75 of the 8 x lr they can have moved (test_train_step_cuda_graph_matches_eager allows 0.5 of
    it at lr 3e-4, i.e. 1.2e-3: Adam's sign-like updates let float-rounding differences of the atomic dW reductions flip single updates),
    the device learning rate equal to learning_rate(args, k); a shape change raises.  lr 1e-4: at 3e-4 the first update collapses this
    torso's density (see test_torso_bf16_vs_fp32_training_500_steps) and the comparison would be of a diverged run."""
    from ideal_nerf_b200.train import TorsoTrainStep, learning_rate
    d = inputs()
    gen = torch.Generator().manual_seed(8)
    nets, steps = [], []
    for graph in (False, True):
        net = network(M, "bf16", lrate=1e-4, lrate_decay=1)
        nets.append(net)
        steps.append(TorsoTrainStep(net, net.args, cuda_graph=graph))
    curves = [[], []]
    for k in range(8):
        sl = slice(256 * k, 256 * k + 512)
        aud = (d["aud"] + 0.1 * torch.randn(64, generator=gen)).to(DEV)
        lat = (d["lat"] + 0.1 * torch.randn(32, generator=gen)).to(DEV)
        args = (d["rays"][sl].to(DEV), d["rays"][sl].to(DEV), d["bc"][sl].to(DEV), d["target"][sl].to(DEV), aud, _pose(k).to(DEV),
                d["expr"].to(DEV), lat)
        for j in range(2):
            out = steps[j](*args, perturb=0.)
            curves[j].append((float(out["img_loss"]), float(out["img_loss0"]), float(out["loss"])))
            assert abs(float(out["lr"]) - learning_rate(nets[j].args, k)) < 1e-10
    print("eager :", curves[0]); print("graph :", curves[1])
    assert steps[1]._static["graph"] is not None and steps[1].global_step == 8
    for a, c in zip(*curves):
        for x, y in zip(a, c):
            assert abs(x - y) <= 2e-4 * max(1.0, abs(x)), (curves[0], curves[1])
    for (k, p), q in zip(nets[0].state_dict().items(), nets[1].state_dict().values()):
        close(q, p, 0.75 * 8 * 1e-4, f"parameter {k} after 8 steps")
    with pytest.raises(RuntimeError, match="fixed per TorsoTrainStep"):
        steps[1](d["rays"][:100].to(DEV), d["rays"][:100].to(DEV), d["bc"][:100].to(DEV), d["target"][:100].to(DEV), d["aud"].to(DEV),
                 _pose().to(DEV), d["expr"].to(DEV), d["lat"].to(DEV), perturb=0.)


@pytest.mark.parametrize("mode", ["bf16", "fp16x2"])
def test_torso_graph_survives_dropped_head_caches(M, mode, tmp_path):
    """The captured graph reads the head pair's packed blobs through device pointers.  Three graphed and three eager steps; then, on both
    networks, what a validation render between training steps does -- eval(), an inference forward (which packs a new head blob),
    invalidate_packed(), train() -- and torch.cuda.empty_cache(); then one more step each: the graphed step still reads the blobs it
    owns, re-packed from the current head weights, and matches the eager step.  load() after the capture raises and changes nothing."""
    from ideal_nerf_b200.train import TorsoTrainStep
    args = dev_inputs(slice(0, 1024))
    nets = [network(M, mode, lrate=1e-4) for _ in range(2)]
    steps = [TorsoTrainStep(nets[0], nets[0].args), TorsoTrainStep(nets[1], nets[1].args, cuda_graph=True)]
    losses = [[], []]
    for _ in range(3):
        for j in range(2):
            losses[j].append(float(steps[j](*args, perturb=0.)["img_loss"]))
    blobs = steps[1]._static["head_blobs"]
    assert steps[1]._static["graph"] is not None and all(b is not None for b in blobs)
    for net in nets:
        net.eval()
        with torch.no_grad():
            net(*args[:3], *args[4:], perturb=0.)
        for m in net.modules():
            if hasattr(m, "invalidate_packed"):
                m.invalidate_packed()
        net.train()
    torch.cuda.empty_cache()
    for j in range(2):
        losses[j].append(float(steps[j](*args, perturb=0.)["img_loss"]))
    print("eager", losses[0], "graph", losses[1])
    assert nets[1].face_nerf_coarse._packed is blobs[0] and nets[1].face_nerf_fine._packed is blobs[1]
    for a, c in zip(*losses):
        assert abs(a - c) <= 2e-4 * a, losses
    steps[0].save(str(tmp_path / "t.tar"))
    before = {k: v.clone() for k, v in nets[1].state_dict().items()}
    with pytest.raises(RuntimeError, match="after the CUDA graph was captured"):
        steps[1].load(str(tmp_path / "t.tar"))
    assert all(torch.equal(v, before[k]) for k, v in nets[1].state_dict().items())


def test_torso_step_resume(M, tmp_path):
    """5 fp32 steps, save; a fresh network (the head from a head.tar through load_head_into_torso) loads the file; both runs continue
    for 3 steps and their losses agree to float rounding."""
    from ideal_nerf_b200 import checkpoint as ck
    from ideal_nerf_b200.train import TorsoTrainStep
    args = dev_inputs(slice(0, 1024))
    net = network(M)
    step = TorsoTrainStep(net, net.args)
    for _ in range(5):
        step(*args, perturb=0.)
    path = str(tmp_path / "000005_torso.tar")
    step.save(path)
    head = M.Network(450, 450, 1200., O.NEAR, O.FAR, 8192, None, 64, 128, args=M.default_args(dim_aud=64, dim_expr=79))
    head.face_nerf_coarse.load_state_dict(net.face_nerf_coarse.state_dict())
    head.face_nerf_fine.load_state_dict(net.face_nerf_fine.state_dict())
    ck.save_head_checkpoint(str(tmp_path / "head.tar"), head, None, torch.ones(3, 32), 0)
    net2 = network(M, torso_seeds=(51, 52))
    with torch.no_grad():
        for p in list(net2.face_nerf_coarse.parameters()) + list(net2.face_nerf_fine.parameters()):
            p.zero_()
    assert torch.equal(ck.load_head_into_torso(str(tmp_path / "head.tar"), net2), torch.ones(3, 32))
    step2 = TorsoTrainStep(net2, net2.args)
    assert step2.load(path) == 5 and step2.optimizer.param_groups[0]["lr"] == step.optimizer.param_groups[0]["lr"]
    assert all(torch.equal(a, b) for a, b in zip(net.state_dict().values(), net2.state_dict().values()))
    for _ in range(3):
        a, b = step(*args, perturb=0.), step2(*args, perturb=0.)
        assert a["lr"] == b["lr"]
        for k in ("img_loss", "img_loss0"):
            assert abs(float(a[k]) - float(b[k])) <= 1e-5 * float(a[k]), (k, float(a[k]), float(b[k]))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _rank(rank, world, port, q):
    import torch.distributed as dist
    import ideal_nerf_b200 as M
    from ideal_nerf_b200.train import TorsoTrainStep
    global DEV
    DEV = f"cuda:{rank}"
    torch.cuda.set_device(rank)
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("nccl", rank=rank, world_size=world)
    net = network(M, "bf16")
    step = TorsoTrainStep(net, net.args, world=world)
    half = slice(rank * 1536, rank * 1536 + 1536)
    start = step.flat.flat.detach().clone()
    for _ in range(3):
        step(*dev_inputs(half), perturb=0.)
    flat = step.flat.flat.detach().clone()
    every = [torch.empty_like(flat) for _ in range(world)]
    dist.all_gather(every, flat)
    if rank == 0:
        q.put(all(torch.equal(every[0], e) for e in every[1:]) and not torch.equal(every[0], start))
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="two NCCL ranks need two GPUs")
def test_torso_step_two_ranks_stay_identical(M):
    """Two NCCL ranks stepping on different halves of a batch (one all-reduce of the flat gradient per step) keep identical torso
    parameters after 3 steps."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_rank, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=600)
        assert p.exitcode == 0
    assert q.get(timeout=10)
