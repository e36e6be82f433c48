#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native IDEAL-NeRF render_rays path.

    python bench.py --gpus 1 --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --steps K --warmup W     # the reference algorithm on the host CPU cores
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py ... --dump-outputs DIR                     # also write the last timed step's image as DIR/rgb_map.npy

Workload (BASELINE.json configs[1]): one step = one full 450x450 HeadNeRF frame, 202 500 rays,
64 coarse + 128 importance samples (256 FaceNeRF evaluations per ray), random-init FaceNeRF
(dim_aud=64, dim_expr=76, latent 32) with the normalised-density preset, synthetic camera/background/
audio/expression codes (oracle.render_oracle.synthetic_frame).  At N GPUs every step renders a group
of N frames whose rays are block-partitioned across the ranks (each rank renders 1/N of every frame of
the group = 202 500 rays per rank per step: weak scaling) and the rendered bands are gathered on rank 0
over NCCL.  Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H = W = 450
N_RAYS = H * W
S1, S_IMP = 64, 128
FLOP_PER_POINT_FWD = 1_121_280           # SURVEY.md 8d: 560 640 MAC, conditioning folded, K unpadded
METRIC = "rays/sec render (64+128 samples), 450x450 frame"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


def mlp_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of the MLP kernel, mean per launch over the coarse and the fine pass, from the
    committed ncu --set full capture (profiles/); None when the summary is absent."""
    p = os.path.join(ROOT, "profiles", "r03_mlp_traffic.json")
    if not os.path.exists(p):
        return None
    d = json.load(open(p))["dram_bytes_per_launch"]
    return sum(d.values()) / len(d)


class ClockSampler(threading.Thread):
    """SM clock / throttle reasons during the timed region (B200_PROFILING.md recipe): NVML polled every 10 ms through pynvml when it
    loads (the timed region of a default run is a quarter of a second), else one nvidia-smi query per 0.2 s."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    BITS = (("sw_power_cap", 0x4), ("hw_slowdown", 0x8), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40))

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_evt = index, [], threading.Event()
        self.nvml = self.handle = None
        try:
            import pynvml
            pynvml.nvmlInit()
            try:
                uuid = str(torch.cuda.get_device_properties(index).uuid)
                self.handle = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
            except Exception:
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _poll_nvml(self):
        n, h = self.nvml, self.handle
        sm = n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM)
        mx = n.nvmlDeviceGetMaxClockInfo(h, n.NVML_CLOCK_SM)
        mask = n.nvmlDeviceGetCurrentClocksThrottleReasons(h)
        self.rows.append([str(sm), str(mx), ""] + ["Active" if mask & b else "Not Active" for _, b in
                                                   (self.BITS[1], self.BITS[3], self.BITS[2], self.BITS[0])])

    def run(self):
        while not self._stop_evt.is_set():
            try:
                if self.nvml is not None:
                    self._poll_nvml()
                else:
                    out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                    f = [x.strip() for x in out.strip().split(",")]
                    if len(f) >= 7:
                        self.rows.append(f)
            except Exception:
                if self.nvml is not None:
                    self.nvml = None              # fall back to nvidia-smi for the rest of the run
            self._stop_evt.wait(0.01 if self.nvml is not None else 0.2)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=6)
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace('.', '', 1).isdigit())
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        mx = [float(r[1]) for r in self.rows if r[1].replace('.', '', 1).isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


# ------------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the oracle port of the reference algorithm on the host cores
# ------------------------------------------------------------------------------------------------
def _reference_available():
    from oracle import ref_import
    return ref_import.available()


def cpu_reference_rays_per_s(n_rays, steps, warmup):
    """The reference's own Network.render_rays (oracle/_ref: the verbatim copy oracle/make_ref.py made, or /root/reference in the build
    container) on the host cores; the oracle port when neither exists.  Returns (rays/s, s per run, threads, kind)."""
    from oracle import render_oracle as O
    torch.set_num_threads(os.cpu_count())
    fr = O.synthetic_frame(0)
    c, f = O.init_face_nerf(1), O.init_face_nerf(2)
    sub = torch.arange(0, N_RAYS, N_RAYS // n_rays)[:n_rays]
    rays, bc = fr["rays"][sub].contiguous(), fr["bc_rgb"][sub].contiguous()
    c = O.normalise_density(c, rays, fr["aud"], fr["expr"], fr["latent"])
    f = O.normalise_density(f, rays, fr["aud"], fr["expr"], fr["latent"])
    kind = "port"
    run = lambda: O.render_rays(rays, bc, c, f, fr["aud"], fr["expr"], fr["latent"])
    if _reference_available():
        from oracle import ref_import
        head = ref_import.import_head(perturb=1.0, force_cpu=True)          # unmodified reference, its hard-coded .cuda() kept on the host
        net = head.Network(H, W, 1200., O.NEAR, O.FAR, 8192, None, S1, S_IMP)
        net.face_nerf_coarse.load_state_dict(c)
        net.face_nerf_fine.load_state_dict(f)
        kind = "reference"
        run = lambda: net.render_rays(rays, bc, fr["aud"], None, fr["latent"], fr["expr"], perturb=1.0)
    ts = []
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            run()
            if i >= warmup:
                ts.append(time.perf_counter() - t0)
    dt = sum(ts) / len(ts)
    return n_rays / dt, dt, torch.get_num_threads(), kind


def reference_gpu_rays_per_s():
    """`--impl reference-gpu` (run as a subprocess of the product arm: the reference's import sets process-wide defaults): the UNMODIFIED
    reference renderer in stock PyTorch eager fp32 on cuda:0, set up the way its own __main__ does (set_default_tensor_type, :598) -- one
    450x450 frame in 25 chunks of 8192 rays through Network.batchify_rays.  The honest same-box comparison next to the CPU figure."""
    from oracle import render_oracle as O, ref_import
    fr = O.synthetic_frame(0)
    c, f = O.init_face_nerf(1), O.init_face_nerf(2)
    kind = "reference" if ref_import.available() else "port"
    dev = torch.device("cuda", 0)
    if kind == "reference":
        torch.set_default_tensor_type('torch.cuda.FloatTensor')
        head = ref_import.import_head(perturb=1.0)
        net = head.Network(H, W, 1200., O.NEAR, O.FAR, 8192, None, S1, S_IMP)
        net.face_nerf_coarse.load_state_dict(c)
        net.face_nerf_fine.load_state_dict(f)
        net = net.to(dev)
        to = lambda t: t.to(dev)
        rays, bc, aud, expr, lat = to(fr["rays"]), to(fr["bc_rgb"]), to(fr["aud"]), to(fr["expr"]), to(fr["latent"])
        frame = lambda: net.batchify_rays(rays, bc, aud, None, lat, expr, chunk=8192)       # perturb = args.perturb, captured at import (:298)
    else:
        to = lambda t: t.to(dev)
        c, f = {k: to(v) for k, v in c.items()}, {k: to(v) for k, v in f.items()}
        rays, bc, aud, expr, lat = to(fr["rays"]), to(fr["bc_rgb"]), to(fr["aud"]), to(fr["expr"]), to(fr["latent"])

        def frame():
            for i in range(0, N_RAYS, 8192):
                O.render_rays(rays[i:i + 8192], bc[i:i + 8192], c, f, aud, expr, lat)
    with torch.no_grad():
        frame()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(2):
            frame()
        e1.record()
        torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / 2
    return {"value": N_RAYS / (ms * 1e-3), "unit": "rays/s", "ms_per_frame": ms, "kind": kind,
            "sample": f"full 202500-ray frame in 25 chunks of 8192 (batchify_rays), 1 warm-up + 2 timed frames, torch {torch.__version__} eager "
                      f"fp32 (allow_tf32={torch.backends.cuda.matmul.allow_tf32}) on the same GPU"}


def run_sub(extra, timeout=900):
    """Run another arm of this script in a fresh interpreter and return its JSON line (None on failure)."""
    try:
        r = subprocess.run([sys.executable, os.path.abspath(__file__)] + extra, capture_output=True, text=True, timeout=timeout,
                           env={k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")})
        lines = [l for l in r.stdout.splitlines() if l.strip().startswith("{")]
        return json.loads(lines[-1]) if r.returncode == 0 and lines else {"error": (r.stderr or r.stdout)[-300:]}
    except Exception as e:            # noqa: BLE001 -- a failed baseline leg must not lose the product line
        return {"error": repr(e)[:300]}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.impl == "reference-gpu":
        emit(dict(reference_gpu_rays_per_s(), impl="reference-gpu"))
        return
    n = args.ref_rays
    v, dt, cores, kind = cpu_reference_rays_per_s(n, args.steps, max(1, args.warmup))
    what = "the reference's own Network.render_rays (oracle/_ref)" if kind == "reference" else "oracle port of the reference algorithm"
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "rays/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"HeadNeRF 450x450 frame render (coarse 64 + fine 192 samples), {what} on the host CPU",
                       "sample": f"{n} rays of the frame per step", "perturb": 1.0, "mlp_mode": "fp32 (torch CPU)"},
            "cpu_baseline": {"value": v, "unit": "rays/s", "cores": cores, "kind": kind,
                             "sample": f"{n} of 202500 frame rays per step ({dt:.2f} s), perturb=1, torch {torch.__version__} fp32, "
                                       f"{torch.backends.cpu.get_cpu_capability()}"},
            "e2e": {"value": v, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


# ------------------------------------------------------------------------------------------------
# this repo's arm
# ------------------------------------------------------------------------------------------------
def build_network(mode, dev):
    import ideal_nerf_b200 as M
    from ideal_nerf_b200 import synthetic as S, ops
    cam, fr = S.camera(), S.frame_inputs(0)
    a = M.default_args(dim_aud=64, dim_expr=76, perturb=1.0, mlp_mode=mode, N_samples=S1, N_importance=S_IMP,
                       near=S.NEAR, far=S.FAR)
    net = M.Network(H, W, cam["focal"], S.NEAR, S.FAR, 1 << 20, None, S1, S_IMP, args=a)
    torch.manual_seed(1234)
    net.apply(M.init_weights)                       # xavier-uniform, bias 0.01 (audio_exp_nerf.py:442-448)
    net = net.to(dev).eval()
    rays = ops.get_rays_packed(H, W, cam["focal"], cam["c2w"].to(dev), S.NEAR, S.FAR)[::197].contiguous()
    for fn in (net.face_nerf_coarse, net.face_nerf_fine):
        S.normalise_density_(fn, rays, fr["aud"].to(dev), fr["expr"].to(dev), fr["latent"].to(dev))
    return M, net, fr, cam


def composite_standalone(M, dev, n_rays, reps=20):
    """raw2outputs alone on frame-sized resident tensors (S = 64 then S = 192), `reps` back-to-back launches per CUDA-event pair:
    the inputs of one launch (207 / 622 MB of raw) exceed L2, so every launch streams from HBM, and the per-launch event overhead
    that dominates the in-step figure (0.1 ms kernels) is amortised.  Returns (algorithmic bytes, ms) summed over both shapes."""
    from ideal_nerf_b200 import ops
    g = torch.Generator(device=dev).manual_seed(11)
    tot_bytes, tot_ms = 0.0, 0.0
    d = torch.randn(n_rays, 3, device=dev, generator=g)
    bc = torch.rand(n_rays, 3, device=dev, generator=g)
    for s in (S1, S1 + S_IMP):
        raw = torch.randn(n_rays, s, 4, device=dev, generator=g)
        z = torch.sort(torch.rand(n_rays, s, device=dev, generator=g), -1)[0]
        for _ in range(3):
            ops.composite(raw, z, d, bc)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            ops.composite(raw, z, d, bc)
        e1.record()
        torch.cuda.synchronize()
        tot_ms += e0.elapsed_time(e1) / reps
        tot_bytes += n_rays * (24 * s + 48)
    return tot_bytes, tot_ms


def train_step_bench(M, dev, steps, mode="bf16", rank=0, world=1, cuda_graph=False):
    """BASELINE.json config 3: N_rand=3072 rays (64+128 samples), loss of audio_exp_nerf.py:540-548, backward through
    compositing + both FaceNeRFs + AudioNet / AudioAttNet (the audio code is computed from an 8-frame DeepSpeech window inside the step,
    :241-266), Adam(lr=3e-4) step and learning-rate schedule -- train.TrainStep, the repo's public training call.
    mode: bf16 = tcgen05 forward-with-save + chain + dW kernels; fp32 = FFMA.  cuda_graph: the whole iteration as one graph launch.
    world > 1: data parallel, weak scaling -- every rank takes its own 3072 rays through identical weights, one NCCL all-reduce of the
    flat gradient (train.FlatParams.gather_grads, the reference's nn.DataParallel backward) before the optimiser step; time = max over ranks."""
    import torch.distributed as dist
    from ideal_nerf_b200 import synthetic as S, ops
    from ideal_nerf_b200 import train as T
    cam, fr = S.camera(), S.frame_inputs(0)
    a = M.default_args(dim_aud=64, dim_expr=76, perturb=1.0, mlp_mode=mode, N_samples=S1, N_importance=S_IMP, lrate=3e-4, nosmo_iters=0)
    net = M.Network(H, W, cam["focal"], S.NEAR, S.FAR, 8192, None, S1, S_IMP, args=a)
    torch.manual_seed(4321)
    net.apply(M.init_weights)
    net = net.to(dev).train()
    g = torch.Generator().manual_seed(5 + rank)
    idx = torch.randperm(N_RAYS, generator=g)[:3072].to(dev)
    rays = ops.get_rays_packed(H, W, cam["focal"], cam["c2w"].to(dev), S.NEAR, S.FAR)[idx].contiguous()
    bc, tgt = fr["bc_rgb"].to(dev)[idx].contiguous(), torch.rand(3072, 3, generator=g).to(dev)
    expr = fr["expr"].to(dev)
    auds = torch.randn(40, 16, 29, generator=torch.Generator().manual_seed(6)).to(dev)       # synthetic DeepSpeech windows, 40 frames
    lat = torch.ones(40, 32, device=dev)
    ts = T.TrainStep(net, lat, a, world=world, cuda_graph=cuda_graph)
    win = net.audio_window(auds, 17, 40)

    def step():
        return ts(rays, bc, tgt, None, expr, 17, aud_window=win)

    for _ in range(3):
        step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    h0 = time.perf_counter()
    e0.record()
    for _ in range(steps):
        out = step()
    e1.record()
    host_ms = (time.perf_counter() - h0) * 1e3 / steps            # host time to ENQUEUE a step (no synchronisation inside)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / steps], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    res = {"rays_per_s": 3072 * world / (ms * 1e-3), "ms_per_step": ms, "host_ms_per_step": host_ms, "n_rand": 3072 * world, "n_gpus": world,
           "mlp_mode": mode, "cuda_graph": bool(cuda_graph), "optimizer": "Adam lr=3e-4 (one flat tensor), lr schedule of :554-558",
           "trains": "face_nerf_coarse, face_nerf_fine, aud_net, aud_att_net, latent_codes[index]", "loss": float(out["loss"])}
    if not cuda_graph:
        # per-kernel breakdown in a second pass: an event pair around each launch of a ~4 ms step would cost the step ~4 %
        ops.LAUNCHES["count"] = 0
        with ops.kernel_timing() as kt:
            for _ in range(steps):
                step()
            torch.cuda.synchronize()
        kms = {k: v[1] / steps for k, v in kt.summary().items()}
        res["gpu_launches_per_step"] = ops.LAUNCHES["count"] / steps
        res["kernels_ms_per_step"] = {k: round(v, 3) for k, v in kms.items()}
        if mode == "bf16":
            # The three training kernels exchange their operands through HBM (DESIGN.md 4.2), so HBM bounds them.  Algorithmic bytes per
            # 128-point tile: forward writes 40 activation images (16 KB) + 76 mask words x 128 rows; the chain reads the masks and writes
            # 39 delta images; dW reads every activation and delta image once.
            tiles = 3072 * (S1 + S1 + S_IMP) // 128
            per_tile = (40 + 39 + 79) * 16384 + 2 * 76 * 512
            t_k = (kms.get("inerf_mlp_fwd_train", 0.0) + kms.get("inerf_mlp_bwd", 0.0)) * 1e-3
            pk, pk_kind = peaks()
            if t_k > 0:
                ach = tiles * per_tile / t_k / 1e9
                res["roofline"] = {"bound": "hbm", "kernels": "inerf_mlp_fwd_train + inerf_mlp_bwd (chain + dW)", "achieved": ach, "peak": pk["hbm_gbs"],
                                   "unit": "GB/s", "frac": ach / pk["hbm_gbs"], "bytes_per_step": tiles * per_tile, "peak_kind": f"HBM copy, {pk_kind}"}
            flops = 3072 * (S1 + S1 + S_IMP) * 3_292_416           # SURVEY.md 8d: fwd + bwd, 1 646 208 MAC per point
            res["tensor_frac_of_sustained"] = flops / (ms * 1e-3) / 1e12 / pk["bf16_tflops_sustained"]
    return res


def sampling_standalone(M, dev, n_rays, reps=20):
    """The two sampling kernels alone on frame-sized resident tensors (perturb > 0 forms: stratified depths + importance sampling with
    in-kernel draws), `reps` back-to-back launches per event pair.  Algorithmic bytes per ray (SURVEY.md 8d): coarse 44 in + 256 out;
    sample_pdf + merge 512 in (z, weights) + 768 (merged z) + 4 (z_std) out -- the draws and z_samples never touch HBM."""
    from ideal_nerf_b200 import ops, synthetic as S
    cam = S.camera()
    rays = ops.get_rays_packed(H, W, cam["focal"], cam["c2w"].to(dev), S.NEAR, S.FAR)[:n_rays].contiguous()
    g = torch.Generator(device=dev).manual_seed(12)
    w = torch.rand(n_rays, S1, device=dev, generator=g) ** 4
    st = ops.rng_state(dev)
    z = ops.sample_coarse_rng(rays, S1, st, advance=False)
    out = {}
    for name, fn, nbytes in (("inerf_sample_coarse_rng", lambda: ops.sample_coarse_rng(rays, S1, st, advance=False), 44 + 4 * S1),
                             ("inerf_importance_sample_rng", lambda: ops.importance_sample_rng(z, w, S_IMP, st, advance=False),
                              8 * S1 + 4 * (S1 + S_IMP) + 4)):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        out[name] = {"ms": ms, "bytes": n_rays * nbytes, "gbs": n_rays * nbytes / (ms * 1e-3) / 1e9}
    return out


def fused_stage_rooflines(net, dev, res, peak_gbs, reps=7):
    """The three small kernels of the shipped path (inerf_render_rays_fused) on the benchmark frame: device time between CUDA events the
    measurement twin of the entry records around its five stages (inerf_debug_render_stage_ms), median over `reps` frames.  Algorithmic
    bytes per ray (SURVEY.md 8d, 64 + 128 samples): set-up 44 (rays) + 256 (z) out; coarse raw2outputs + sampling 1 024 (raw) + 256 (z) +
    44 + 12 (ray, background) in, 768 (merged z) + 28 (maps, z_std) out; final raw2outputs 3 072 + 768 + 56 in, 28 out."""
    from ideal_nerf_b200 import ops
    a = net.args
    gen = dict(H=H, W=W, focal=net.focal, cx=W * .5, cy=H * .5, near=net.near, far=net.far, c2w=res["pose"][:3, :4], first=0, count=N_RAYS)
    cond = (res["aud"], res["expr"], res["latent"])
    ms = []
    with torch.no_grad():
        for i in range(reps + 2):
            out = []
            ops.render_rays_fused(net.face_nerf_coarse, net.face_nerf_fine, cond, cond, res["bc"], a.N_samples, a.N_importance, 1.0, gen=gen,
                                  stage_ms=out)
            if i >= 2:
                ms.append(out[0])
    med = [sorted(m[k] for m in ms)[len(ms) // 2] for k in range(5)]
    nbytes = {"render_setup (2 folds + rays + coarse depths)": (0, 300), "composite_sample_64_128 (coarse raw2outputs + sampler)": (2, 2132),
              "composite_final (fine raw2outputs, flags, rng)": (4, 3924)}
    out = {"stage_ms": {"setup": med[0], "mlp_coarse": med[1], "composite_sample": med[2], "mlp_fine": med[3], "composite_final": med[4]},
           "how": "inerf_debug_render_stage_ms: CUDA events between the five launches of one fused call, median of %d frames" % reps,
           "kernels": {}}
    for name, (k, b) in nbytes.items():
        gbs = N_RAYS * b / (med[k] * 1e-3) / 1e9
        out["kernels"][name] = {"ms": med[k], "bytes": N_RAYS * b, "achieved": gbs, "frac": gbs / peak_gbs}
    return out


def build_torso_network(mode, dev):
    """BASELINE.json config 4: head + torso renderer (train_torso.py:186), random init + density preset on all four FaceNeRFs."""
    import ideal_nerf_b200 as M
    from ideal_nerf_b200 import synthetic as S, ops
    cam, fr = S.camera(), S.frame_inputs(0)
    a = M.default_args(dim_aud=64, dim_expr=79, perturb=1.0, mlp_mode=mode, N_samples=S1, N_importance=S_IMP, near=S.NEAR, far=S.FAR)
    net = M.TorsoNetwork(H, W, cam["focal"], S.NEAR, S.FAR, 1 << 20, S1, S_IMP, args=a, dim_expr=79)
    torch.manual_seed(77)
    net.apply(M.init_weights)
    net = net.to(dev).eval()
    g = torch.Generator().manual_seed(3)
    expr = torch.randn(79, generator=g).to(dev)
    aud, lat, pose = fr["aud"].to(dev), fr["latent"].to(dev), fr["pose"].to(dev)
    rays = ops.get_rays_packed(H, W, cam["focal"], cam["c2w"].to(dev), S.NEAR, S.FAR)
    sub = rays[::197].contiguous()
    with torch.no_grad():
        sig = net.torso_signal(aud, pose)
        for fn in (net.face_nerf_coarse, net.face_nerf_fine):
            S.normalise_density_(fn, sub, aud, expr, lat)
        for fn in (net.torso_coarse_nerf, net.torso_fine_nerf):
            S.normalise_density_(fn, sub, sig, None, None)
    return net, rays, fr["bc_rgb"].to(dev), aud, pose, expr, lat


def run_ours(args):
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    M, net, fr, cam = build_network(args.mode, dev)
    from ideal_nerf_b200 import ops, synthetic as S
    from ideal_nerf_b200.frame import FrameRenderer, band, render_video
    M._lib.check(M.lib().inerf_device_check(), "inerf_device_check")
    fr_r = FrameRenderer(net, rank, world)

    # ---- inputs: pinned host copies (e2e) and resident device copies (value) ----------------------
    host = {"pose": fr["pose"].pin_memory(), "aud": fr["aud"].pin_memory(), "expr": fr["expr"].pin_memory(),
            "latent": fr["latent"].pin_memory(), "bc": fr["bc_rgb"].pin_memory()}
    res = {k: v.to(dev) for k, v in host.items()}
    frames = world                                   # frames per step (weak scaling: 202 500 rays per rank per step)
    lo, hi = band(N_RAYS, rank, world)

    last = {}

    @torch.no_grad()
    def step_resident():
        """`frames` frames, each ray-sharded over the ranks; the band all-gather of frame i overlaps the kernels of frame i+1."""
        hs = [fr_r.render_frame(res["pose"], res["aud"], res["expr"], res["latent"], res["bc"], perturb=1.0, async_op=True)
              for _ in range(frames)]
        last["rgb_map"] = [h.wait() for h in hs][-1]
        return last["rgb_map"]

    out_h = torch.empty((N_RAYS, 3)).pin_memory()
    h2d = sum(host[k].numel() * 4 for k in host)

    @torch.no_grad()
    def step_e2e():
        """Public API with HOST buffers: H2D of the frame's inputs, render, gather, D2H of the image."""
        for _ in range(frames):
            d = {k: v.to(dev, non_blocking=True) for k, v in host.items()}
            if world == 1:
                rgb = net.render_dynamic_face(H, W, net.focal, d["expr"], d["pose"], d["latent"], render_poses=d["pose"][:3, :4],
                                              chunk=1 << 20, near=net.near, far=net.far, bc_rgb=d["bc"].reshape(H, W, 3),
                                              aud_para=d["aud"], perturb=1.0)[0].reshape(-1, 3)
            else:
                rgb = fr_r.render_frame(d["pose"], d["aud"], d["expr"], d["latent"], d["bc"], perturb=1.0)
            if rank == 0:
                out_h.copy_(rgb, non_blocking=True)
        torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    for _ in range(max(3, args.warmup)):
        step_resident()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    ops.LAUNCHES["count"] = 0
    total_ms = timed(step_resident, args.steps)          # the headline: no per-kernel events inside this region
    launches = ops.LAUNCHES["count"]
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        # the image the last timed step returned, before the passes below reuse its buffers; with the same arguments the inputs, the
        # weights and the Philox seed / offsets are the same in every run, so two builds can be compared output for output
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "rgb_map.npy"), last["rgb_map"].float().cpu().numpy())
    # second, identical pass with a CUDA-event pair around every launch (on the launching stream) for the roofline / breakdown; under
    # kernel_timing the renderer takes the stage-by-stage entry points (one event pair per kernel), so that path gets its own warm-up
    with ops.kernel_timing():
        step_resident()
    with ops.kernel_timing() as kt:
        timed_ms_events = timed(step_resident, args.steps)
    ksum = kt.summary()

    for _ in range(2):
        step_e2e()
    t_e2e = timed(step_e2e, args.steps)

    rays_per_step = N_RAYS * frames                   # all ranks together
    value = rays_per_step * args.steps / (total_ms * 1e-3)
    e2e_value = rays_per_step * args.steps / (t_e2e * 1e-3)

    # ---- config 5: eval video, per-frame audio / expression codes, rays of EVERY frame sharded over the ranks -----------------------
    video = None
    if args.video_frames > 0:
        nf = args.video_frames
        aud_v, expr_v = S.video_codes(nf, 0)
        aud_v, expr_v = aud_v.to(dev), expr_v.to(dev)
        seq = [(res["pose"], aud_v[i], expr_v[i]) for i in range(nf)]
        with torch.no_grad():
            render_video(fr_r, seq[:4], res["latent"], res["bc"], perturb=0.)
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            vid = render_video(fr_r, seq, res["latent"], res["bc"], perturb=0.)          # eval: perturb = 0 (eval_aud_exp_nerf.py)
            e1.record()
            barrier()
            ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            v_ms = float(ms.item())
            # latency of ONE frame: inputs resident, render -> gather -> to8b -> pinned host copy, a synchronise per frame
            lat_ms = []
            one = torch.empty((H, W, 3), dtype=torch.uint8).pin_memory()
            for i in range(12):
                barrier()
                t0 = time.perf_counter()
                pose_i, aud_i, expr_i = seq[i]
                rgb = fr_r.render_frame(pose_i, aud_i, expr_i, res["latent"], res["bc"], 0.)
                if rank == 0:
                    one.copy_(ops.to8b(rgb).reshape(H, W, 3), non_blocking=True)
                torch.cuda.synchronize()
                lat_ms.append((time.perf_counter() - t0) * 1e3)
            lat = torch.tensor(sorted(lat_ms[2:])[len(lat_ms[2:]) // 2], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(lat, op=dist.ReduceOp.MAX)
        video = {"frames": nf, "ms_total": v_ms, "fps": nf / (v_ms * 1e-3), "rays_per_s": nf * N_RAYS / (v_ms * 1e-3),
                 "ms_per_frame": v_ms / nf, "latency_ms_per_frame": float(lat.item()), "perturb": 0.0,
                 "codes": "seeded Gaussian random walk of aud (64) / expr (76), sigma 0.1 per frame; pose fixed",
                 "sharding": f"rays of every frame block-partitioned over {world} GPU(s), one all-gather per frame overlapped with the next frame",
                 "output": "uint8 frames in one pinned host array (to8b on device)",
                 "checksum": int(vid.to(torch.int64).sum()) if rank == 0 else None}

    train_bf16 = None if args.no_train else train_step_bench(M, dev, 5, "bf16", rank, world)      # every rank takes part (gradient all-reduce)

    if rank == 0:
        pk, pk_kind = peaks()
        n_mlp, mlp_ms = ksum.get("inerf_mlp_fwd", (0, 0.0))
        # dominant kernel: FaceNeRF forward.  Algorithmic FLOPs of the launches in the (second) timed region / their event time.
        pts_per_step_rank = (hi - lo) * (S1 + S1 + S_IMP) * frames
        mlp_flops = pts_per_step_rank * args.steps * FLOP_PER_POINT_FWD
        achieved = mlp_flops / (mlp_ms * 1e-3) / 1e12 if mlp_ms > 0 else None
        peak = pk["bf16_tflops_sustained"]
        with torch.no_grad():
            sa_bytes, sa_ms = composite_standalone(M, dev, N_RAYS)      # always frame-sized: inputs larger than L2
            samp = sampling_standalone(M, dev, N_RAYS)
            fused_small = fused_stage_rooflines(net, dev, res, pk["hbm_gbs"]) if world == 1 else None
        line = {
            "metric": METRIC, "value": value, "unit": "rays/s", "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if args.mode == "fp32" else "bf16", "data": "synthetic",
            "config": {"workload": "HeadNeRF full 450x450 frame render (coarse 64 + fine 192 samples), FaceNeRF dim_aud=64 dim_expr=76",
                       "frames_per_step": frames, "rays_per_rank_per_step": (hi - lo) * frames, "mlp_mode": args.mode,
                       "perturb": 1.0, "rng": "in-kernel Philox4x32-10 (stratified jitter + importance draws)",
                       "entry": "inerf_render_rays_fused: one C call and 5 kernel launches per render_rays (set-up, coarse FaceNeRF, "
                                "compositor + sampler, fine FaceNeRF, final compositor)",
                       "l2": "inputs larger than L2 (raw 207+622 MB per frame pass)",
                       "parallelism": f"rays block-partitioned over {world} GPU(s), one NCCL all-gather of the bands per frame"},
            "e2e": {"value": e2e_value, "unit": "rays/s", "h2d_bytes_per_step": h2d * frames,
                    "d2h_bytes_per_step": N_RAYS * 3 * 4 * frames, "ms_per_step": t_e2e / args.steps},
            "gpu_launches": launches,
            "clocks": clocks,
            "roofline": {"bound": "tensor", "kernel": "inerf_mlp_fwd", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                         "frac": (achieved / peak) if achieved else None, "traffic": mlp_traffic(),
                         "peak_kind": f"bf16 dense sustained, {pk_kind}", "launches": n_mlp, "kernel_ms_total": mlp_ms,
                         "share_of_step": mlp_ms / timed_ms_events if timed_ms_events else None,
                         "how": "second pass of the same steps through the stage-by-stage entry points with a CUDA-event pair around every launch "
                                "(the same FaceNeRF kernel); `value` is the event-free pass through inerf_render_rays_fused"},
            "roofline_composite": {"bound": "hbm", "kernel": "inerf_composite_fwd",
                                   "achieved": sa_bytes / (sa_ms * 1e-3) / 1e9, "peak": pk["hbm_gbs"], "unit": "GB/s",
                                   "frac": sa_bytes / (sa_ms * 1e-3) / 1e9 / pk["hbm_gbs"],
                                   "how": "stand-alone, 20 back-to-back launches per event pair on frame-sized resident inputs (S=64 and S=192)"},
            "roofline_sampling": {"bound": "hbm", "peak": pk["hbm_gbs"], "unit": "GB/s",
                                  "kernels": {k: {"achieved": v["gbs"], "frac": v["gbs"] / pk["hbm_gbs"], "ms": v["ms"], "bytes": v["bytes"]}
                                              for k, v in samp.items()},
                                  "how": "stand-alone on 202 500 rays, 20 back-to-back launches per event pair"},
            "kernels_ms": {k: round(v[1], 3) for k, v in ksum.items()},
        }
        if fused_small is not None:
            line["roofline_fused_small"] = fused_small
        if video is not None:
            line["config5_video"] = video
        if train_bf16 is not None:
            line["train_step"] = train_bf16
            if world == 1:
                line["train_step_graph"] = train_step_bench(M, dev, 20, "bf16", cuda_graph=True)
        if world == 1 and not args.no_extra:
            line.update(extra_single_gpu(M, net, dev, res, args))
        if world == 1 and not args.no_train:
            line["train_step_fp32"] = train_step_bench(M, dev, 3, "fp32")
        if world == 1 and not args.no_cpu_baseline:
            ref = run_sub(["--impl", "reference", "--steps", "2", "--warmup", "1", "--ref-rays", "3072"])
            if ref and "cpu_baseline" in ref:
                line["cpu_baseline"] = ref["cpu_baseline"]
            else:                                              # the subprocess failed: time the port in-process instead
                v, dt, cores, kind = cpu_reference_rays_per_s(3072, 2, 1)
                line["cpu_baseline"] = {"value": v, "unit": "rays/s", "cores": cores, "kind": kind, "sample": f"3072 of 202500 frame rays ({dt:.2f} s per run)",
                                        "note": str(ref)[:200]}
            line["torch_gpu_baseline"] = run_sub(["--impl", "reference-gpu"])
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def extra_single_gpu(M, net, dev, res, args):
    """Extra keys measured on one GPU: the fp32-gate mode's frame rate, bf16-vs-fp32 render parity on the benchmark frame, and
    BASELINE.json config 4 (head + torso composited frame)."""
    from ideal_nerf_b200 import ops
    out = {}

    def time_frames(fn, n):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    with torch.no_grad():
        rays = ops.get_rays_packed(H, W, net.focal, res["pose"][:3, :4], net.near, net.far)
        render = lambda p: net.render_rays(rays, res["bc"], res["aud"], None, res["latent"], res["expr"], perturb=p)
        # parity of the benchmark mode on the benchmark frame (perturb = 0 so both modes see the same depths): bf16 vs the fp32 kernels
        mode0 = args.mode
        r_fast = render(0.)
        net.set_mlp_mode("fp32")
        r32 = render(0.)
        ms32 = time_frames(lambda: render(1.0), 1)
        net.set_mlp_mode(mode0)
        mse = float(torch.mean((r_fast["rgb_map"] - r32["rgb_map"]) ** 2))
        out["parity"] = {"against": "this repo's fp32 (FFMA) kernels on the same 202 500-ray frame, perturb=0 (the fp32 kernels are checked "
                                    "against the reference's outputs at <= 1e-3 in tests/test_gpu_parity.py)",
                         "psnr_db": float(-10. * torch.log10(torch.tensor(mse))) if mse > 0 else None,
                         "max_abs": float((r_fast["rgb_map"] - r32["rgb_map"]).abs().max()),
                         "acc_max_abs": float((r_fast["acc_map"] - r32["acc_map"]).abs().max())}
        out["render_fp32"] = {"rays_per_s": N_RAYS / (ms32 * 1e-3), "ms_per_frame": ms32, "mlp_mode": "fp32 (FFMA, the <= 1e-3 max-abs mode)",
                              "frames": 1}
        # the fp32-gate TENSOR-CORE mode (fp16 hi/lo operand pairs, 3 MMA passes): frame rate + agreement with the FFMA kernels
        net.set_mlp_mode("fp16x2")
        rx = render(0.)
        msx = time_frames(lambda: render(1.0), 5)
        net.set_mlp_mode(mode0)
        pk, _ = peaks()
        out["render_fp16x2"] = {"rays_per_s": N_RAYS / (msx * 1e-3), "ms_per_frame": msx,
                                "mlp_mode": "fp16x2 (tcgen05, fp16 hi/lo operands, hi.hi + lo.hi + hi.lo, fp32 accumulate): the <= 1e-3 max-abs mode on tensor cores",
                                "max_abs_vs_fp32_kernels": float((rx["rgb_map"] - r32["rgb_map"]).abs().max()),
                                "tensor_frac_of_sustained": 3 * N_RAYS * (S1 + S1 + S_IMP) * FLOP_PER_POINT_FWD / (msx * 1e-3) / 1e12 / pk["bf16_tflops_sustained"],
                                "note": "tensor_frac counts the three MMA passes this mode issues per algorithmic product"}
        # config 4: head + torso composited frame with background blending (test_torso.py:516-523)
        tn, trays, bc, aud, pose, expr, lat = build_torso_network(args.mode, dev)
        step = lambda: tn(trays, trays, bc, aud, pose, expr, lat, perturb=1.0)
        for _ in range(2):
            step()
        ops.LAUNCHES["count"] = 0
        ms4 = time_frames(step, max(3, args.steps // 2))
        out["config4_head_torso"] = {"rays_per_s": N_RAYS / (ms4 * 1e-3), "ms_per_frame": ms4, "mlp_mode": args.mode,
                                     "point_evals_per_ray": 2 * (S1 + S1 + S_IMP),
                                     "workload": "HeadNeRF + TorsoNeRF 450x450 frame: two coarse+fine FaceNeRF pairs (torso cond 106 = aud 64 + "
                                                 "gamma_3(euler) 21 + gamma_3(trans) 21), rgb = rgb_head * last_weight_torso + rgb_fg_torso",
                                     "perturb": 1.0}
    return out


_RESULT_OUT = None


def emit(line):
    """The ONE JSON line of the contract, on the process's original stdout."""
    out = _RESULT_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    # Libraries print to fd 1 as well (NCCL's version banner on the first collective, for one): keep a private handle on the original
    # stdout for the result line and point fd 1 at stderr, so that stdout carries exactly one line whatever else talks.
    global _RESULT_OUT
    sys.stdout.flush()
    _RESULT_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", type=str, default="ours", choices=["ours", "reference", "reference-gpu"])
    ap.add_argument("--ref-rays", dest="ref_rays", type=int, default=2048, help="rays per step of the reference arm (bounded sample)")
    ap.add_argument("--video-frames", dest="video_frames", type=int, default=200)
    ap.add_argument("--mode", type=str, default=os.environ.get("INERF_BENCH_MODE", "bf16"), choices=["fp32", "bf16"])
    ap.add_argument("--no-cpu-baseline", dest="no_cpu_baseline", action="store_true")
    ap.add_argument("--no-train", dest="no_train", action="store_true")
    ap.add_argument("--no-extra", dest="no_extra", action="store_true", help="skip the fp32-mode render, parity and config-4 keys")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR",
                    help="write the image the last timed step rendered to DIR/rgb_map.npy ((202500, 3) float32, --impl ours)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl in ("reference", "reference-gpu"):
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
