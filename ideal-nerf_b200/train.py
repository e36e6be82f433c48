"""The optimisation step around render_rays, NeRFs/HeadNeRF/train/audio_exp_nerf.py:529-558 (SURVEY.md 8f-2): loss, backward, Adam, the
exponential learning-rate schedule and (multi-GPU) the gradient all-reduce, with the reference's hyper-parameter names.

    loss = mse(rgb, target) + mse(rgb0, target) + 10 * lc_weight * ||latent_code||_2            (:540-548)
    new_lrate = lrate * 0.1 ** (global_step / (lrate_decay * 1500))                             (:554-558)

The two image losses and their gradients come from one kernel (ops.mse_pair).  Adam is torch's fused implementation run on ONE tensor:
FlatParams re-homes every parameter as a view of a single buffer, so the optimiser step is one bandwidth-bound launch (~20 us for the
2.9 M parameters of two FaceNeRFs) instead of a multi-tensor sweep over 53 small tensors (~150 us), and the data-parallel all-reduce
runs on the flat gradient directly.  Adam is element-wise, so the result equals the per-parameter optimiser of the reference."""
import torch
import torch.distributed as dist

from . import ops


class FlatParams:
    """Parameters (and their gradients) as views of one flat buffer each.  Every view starts on a 256-byte boundary (the kernels read
    weights with vector loads).  `flat` is the single nn.Parameter the optimiser sees; `gather_grads()` copies the .grad tensors autograd
    produced into the flat gradient with one multi-tensor launch (parameters without a gradient contribute zeros = no update)."""
    ALIGN = 64      # floats

    def __init__(self, params):
        self.params = [p for p in params]
        if not self.params:
            raise ValueError("FlatParams: no parameters")
        dev, dt = self.params[0].device, self.params[0].dtype
        offs, o = [], 0
        self.offsets = offs
        for p in self.params:
            if p.device != dev or p.dtype != dt:
                raise ValueError("FlatParams: parameters must share device and dtype")
            offs.append(o)
            o += (p.numel() + self.ALIGN - 1) // self.ALIGN * self.ALIGN
        self.flat = torch.nn.Parameter(torch.zeros(o, device=dev, dtype=dt))
        self.grad = torch.zeros(o, device=dev, dtype=dt)
        self.flat.grad = self.grad
        self.gviews = []
        with torch.no_grad():
            for p, off in zip(self.params, offs):
                v = self.flat.data[off:off + p.numel()].view(p.shape)
                v.copy_(p.data)
                p.data = v
                self.gviews.append(self.grad[off:off + p.numel()].view(p.shape))

    def gather_grads(self, world=1, group=None):
        have = [(gv, p.grad) for gv, p in zip(self.gviews, self.params) if p.grad is not None]
        none = [gv for gv, p in zip(self.gviews, self.params) if p.grad is None]
        if none:
            torch._foreach_zero_(none)
        if have:
            torch._foreach_copy_([h[0] for h in have], [h[1] for h in have])
        if world > 1:      # the reference's nn.DataParallel backward (distribute_nerf.py:423) as one all-reduce of the flat gradient
            if dist.get_backend(group) == "nccl":
                dist.all_reduce(self.grad, op=dist.ReduceOp.AVG, group=group)
            else:
                dist.all_reduce(self.grad, op=dist.ReduceOp.SUM, group=group)
                self.grad.div_(world)
        self.flat.grad = self.grad


def head_loss(ret, target, latent_code, lc_weight):
    """Returns (loss, img_loss, latent_code_loss) as the reference logs them."""
    l2 = ops.mse_pair(ret["rgb_map"], ret["rgb0"], target)
    latent_loss = torch.norm(latent_code) * lc_weight
    return l2[0] + l2[1] + latent_loss * 10, l2[0], latent_loss


def learning_rate(args, global_step):
    return args.lrate * (0.1 ** (global_step / (args.lrate_decay * 1500)))


class _AdamStep:
    """What TrainStep and TorsoTrainStep share: the trained parameters as one FlatParams buffer under ONE Adam (torch's fused kernel;
    with cuda_graph=True its capturable form, the learning rate and the step count held in device tensors), the learning-rate schedule,
    the conversion of that Adam's state to and from the reference's per-parameter layout, and the capture / replay bookkeeping of the
    CUDA-graph mode.  Subclasses name what a captured graph fixes in _FIXED."""
    _FIXED = "batch shapes and perturb"

    def __init__(self, params, args, world, group, cuda_graph):
        self.args, self.world, self.group = args, world, group
        self.flat = FlatParams(params)
        self.cuda_graph = bool(cuda_graph)
        self._static = None
        name = type(self).__name__
        on_cuda = self.flat.flat.is_cuda
        if self.cuda_graph:
            if not on_cuda:
                raise RuntimeError(f"{name}(cuda_graph=True) needs CUDA tensors")
            if world > 1:
                raise NotImplementedError("cuda_graph=True is built for one process per model replica without a gradient all-reduce")
            dev = self.flat.flat.device
            self._lr_t = torch.tensor(float(args.lrate), device=dev)          # the learning rate and the step count live on the device
            self._gs_t = torch.zeros((), device=dev)
            self.optimizer = torch.optim.Adam([self.flat.flat], lr=self._lr_t, betas=(0.9, 0.999), fused=True, capturable=True)
        else:
            self.optimizer = torch.optim.Adam([self.flat.flat], lr=args.lrate, betas=(0.9, 0.999), fused=on_cuda)
        self.global_step = 0

    # -- checkpoint interchange with the reference's per-parameter Adam -----------------------------------------------------------
    def optimizer_state_dict(self):
        """Adam state in the layout a per-parameter torch.optim.Adam over the trained parameters writes: one entry per parameter."""
        sd = self.optimizer.state_dict()
        st = sd["state"].get(0)
        state = {}
        if st:
            for i, (p, off) in enumerate(zip(self.flat.params, self.flat.offsets)):
                n = p.numel()
                state[i] = {"step": st["step"].detach().clone().cpu(), "exp_avg": st["exp_avg"][off:off + n].view(p.shape).clone(),
                            "exp_avg_sq": st["exp_avg_sq"][off:off + n].view(p.shape).clone()}
        group = {k: v for k, v in sd["param_groups"][0].items() if k != "params"}
        group.update(fused=None, foreach=None, params=list(range(len(self.flat.params))))
        return {"state": state, "param_groups": [group]}

    def load_optimizer_state_dict(self, sd):
        """Accepts the per-parameter layout above (the reference's head.tar) or this class's own flat one-parameter layout."""
        n_par = len(self.flat.params)
        ids = sd["param_groups"][0]["params"]
        if len(ids) == 1 and n_par != 1:
            self.optimizer.load_state_dict(sd)
            return
        if len(ids) != n_par:
            raise ValueError(f"optimizer state has {len(ids)} parameters, this {type(self).__name__} has {n_par}")
        flat = self.flat.flat
        exp_avg, exp_avg_sq = torch.zeros_like(flat.data), torch.zeros_like(flat.data)
        step = None
        for i, (p, off) in enumerate(zip(self.flat.params, self.flat.offsets)):
            st = sd["state"].get(ids[i])
            if not st:                                   # a parameter that never received a gradient has no state in the reference
                continue
            if tuple(st["exp_avg"].shape) != tuple(p.shape):
                raise ValueError(f"optimizer state of parameter {i} has shape {tuple(st['exp_avg'].shape)}, expected {tuple(p.shape)}")
            n = p.numel()
            exp_avg[off:off + n].copy_(st["exp_avg"].reshape(-1))
            exp_avg_sq[off:off + n].copy_(st["exp_avg_sq"].reshape(-1))
            s = float(st["step"])
            step = s if step is None else max(step, s)
        group = {k: v for k, v in self.optimizer.state_dict()["param_groups"][0].items()}
        for k in ("lr", "betas", "eps", "weight_decay", "amsgrad"):
            if k in sd["param_groups"][0]:
                group[k] = sd["param_groups"][0][k]
        state = {} if step is None else {0: {"step": torch.tensor(step, dtype=torch.float32), "exp_avg": exp_avg, "exp_avg_sq": exp_avg_sq}}
        self.optimizer.load_state_dict({"state": state, "param_groups": [group]})

    def _check_loadable(self):
        """load() replaces weights the captured graph reads: it is refused, before anything is changed, once the graph exists."""
        if self.cuda_graph and self._static is not None and self._static["graph"] is not None:
            name = type(self).__name__
            raise RuntimeError(f"{name}.load() after the CUDA graph was captured: load before the first graphed step")

    def _load_schedule(self, ckpt):
        """global_step, the Adam state and the learning rate of a checkpoint whose weights were just loaded."""
        self.global_step = int(ckpt.get("global_step", 0))
        if ckpt.get("optimizer") is not None:
            self.load_optimizer_state_dict(ckpt["optimizer"])              # carries the learning rate the schedule had reached (:554-558)
        else:
            for g in self.optimizer.param_groups:                          # the lr in force at step k is the one set after step k-1
                g["lr"] = learning_rate(self.args, self.global_step - 1) if self.global_step > 0 else self.args.lrate
        if self.cuda_graph:                                                # keep the device-resident schedule state the graph reads
            for g in self.optimizer.param_groups:
                self._lr_t.fill_(float(g["lr"]))
                g["lr"] = self._lr_t
            self._gs_t.fill_(float(self.global_step))

    def _update(self, loss, nets):
        """Backward, gradient gather (+ all-reduce), Adam, and the packed-weight caches of the trained FaceNeRFs dropped."""
        loss.backward()
        self.flat.gather_grads(self.world, self.group)
        self.optimizer.step()
        for m in nets:                                                     # fused Adam does not bump parameter versions
            m.invalidate_packed()

    def _advance_lr(self):
        """Eager mode, after an update: the learning rate of the next step (:554-558)."""
        lr = learning_rate(self.args, self.global_step)
        for g in self.optimizer.param_groups:
            g["lr"] = lr
        self.global_step += 1
        return lr

    def _graph_step(self, key, make_static, fill, body):
        """One call of the CUDA-graph mode.  `key` is what a captured graph fixes; make_static() returns the static input buffers,
        fill(st) copies this call's inputs into them, body(st) is the iteration (its tensors are the outputs the replays refresh).  The
        learning-rate schedule runs on the device after body.  The first call runs eagerly (it initialises Adam's state and the kernels'
        per-device constants), the second call captures, every later call replays."""
        if self._static is None or self._static["key"] != key:
            if self._static is not None:
                name = type(self).__name__
                raise RuntimeError(f"{name}(cuda_graph=True) was captured for {self._static['key']}, got {key}: {self._FIXED} are fixed "
                                   f"per {name}")
            self._static = dict(make_static(), key=key, graph=None, out=None, calls=0)
        st = self._static
        fill(st)

        def run():
            out = body(st)
            # new_lrate = lrate * 0.1 ** (global_step / (lrate_decay * 1500)); global_step += 1      (:554-558), on the device
            self._lr_t.copy_(self.args.lrate * torch.pow(0.1, self._gs_t / (self.args.lrate_decay * 1500)))
            self._gs_t.add_(1.0)
            return out

        if st["calls"] == 0:
            st["out"] = run()                                        # eager: lazy initialisations happen here
        else:
            if st["graph"] is None:
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    st["out"] = run()
                st["graph"] = g
            st["graph"].replay()
        st["calls"] += 1
        self.global_step += 1
        return st["out"]


class TrainStep(_AdamStep):
    """One call = one iteration of the reference's inner loop for a ray batch already on the device.

    The optimiser is ONE Adam over the flat buffer; `optimizer_state_dict()` / `load_optimizer_state_dict()` convert to and from the
    reference's per-parameter Adam state (params = list(network.parameters()) + [latent_codes], audio_exp_nerf.py:487-493) so the
    'optimizer' entry of head.tar moves both ways; `save()` / `load()` write and resume the reference's checkpoint (:516-525, :584-591)."""
    _FIXED = "batch shapes, the aud_window / aud_feature choice and perturb"

    def __init__(self, network, latent_codes, args, world=1, group=None, cuda_graph=False):
        self.net, self.latent_codes = network, latent_codes
        latent_codes.requires_grad_(True)
        super().__init__(list(network.parameters()) + [latent_codes], args, world, group, cuda_graph)

    def save(self, path):
        """head.tar as the reference writes it (audio_exp_nerf.py:584-591), loadable by the reference's resume code (:516-525)."""
        torch.save({"global_step": int(self.global_step), "model_state_dict": self.net.state_dict(),
                    "optimizer": self.optimizer_state_dict(), "latent_codes": self.latent_codes.data.clone()}, path)

    def load(self, path, map_location=None):
        """Resume from a head.tar written by the reference or by save(): weights and latent codes are copied IN PLACE (they are views of
        the flat Adam buffer), the Adam moments are scattered into the flat state, global_step and the learning rate are restored."""
        self._check_loadable()
        ckpt = torch.load(path, map_location=map_location, weights_only=False)
        self.net.load_state_dict(ckpt["model_state_dict"])                 # nn.Module.load_state_dict copies in place
        with torch.no_grad():
            self.latent_codes.data.copy_(ckpt["latent_codes"].to(self.latent_codes.device))
        self._load_schedule(ckpt)
        for m in self.net.modules():
            if hasattr(m, "invalidate_packed"):
                m.invalidate_packed()
        return self.global_step

    def __call__(self, rays, bc_rgb, target, aud_feature, expr, index, perturb=None, aud_window=None):
        """aud_feature: the (dim_aud,) audio code (a constant, or a tensor with a graph into the conditioning nets); or pass
        aud_window = the (smo_size, 16, 29) DeepSpeech window (Network.audio_window) and the code is computed -- and the two
        conditioning nets are trained -- inside the step, as the reference's forward does (audio_exp_nerf.py:241-266)."""
        perturb = self.args.perturb if perturb is None else perturb
        if self.cuda_graph:
            return self._graphed(rays, bc_rgb, target, aud_feature, expr, index, perturb, aud_window)
        latent_code = self.latent_codes[index]
        if aud_window is not None:
            aud_feature = self.net.aud_att_net(self.net.aud_net(aud_window))
        loss, img_loss, latent_loss = self._body(rays, bc_rgb, target, aud_feature, expr, latent_code, perturb)
        lr = self._advance_lr()
        return {"loss": loss.detach(), "img_loss": img_loss.detach(), "latent_code_loss": latent_loss.detach(), "lr": lr}

    def _body(self, rays, bc_rgb, target, aud_feature, expr, latent_code, perturb):
        """Forward, loss, backward, gradient gather (+ all-reduce), Adam: everything between two learning-rate updates."""
        for p in self.flat.params:
            p.grad = None
        ret = self.net.render_rays(rays, bc_rgb, aud_feature, None, latent_code, expr, perturb=perturb)
        loss, img_loss, latent_loss = head_loss(ret, target, latent_code, self.args.lc_weight)
        self._update(loss, (self.net.face_nerf_coarse, self.net.face_nerf_fine))
        return loss, img_loss, latent_loss

    # -- CUDA-graph mode (SURVEY.md 8f-2) ------------------------------------------------------------------------------------------
    def _graphed(self, rays, bc_rgb, target, aud_feature, expr, index, perturb, aud_window):
        """The whole iteration -- conditioning nets, both render passes, loss, backward, gradient gather, Adam, learning-rate schedule, RNG
        offset -- as ONE cudaGraphLaunch.  Inputs are copied into static buffers; the latent-code row is selected on the device from a
        one-element index tensor; the learning rate and Adam's step count live in device tensors updated inside the graph; the
        stochastic draws come from the in-kernel Philox stream whose offset the graph advances."""
        dev = self.flat.flat.device
        use_win = aud_window is not None
        aud_src = aud_window if use_win else aud_feature
        key = (tuple(rays.shape), tuple(bc_rgb.shape), use_win, float(perturb))

        def make_static():
            return {"rays": torch.empty_like(rays), "bc": torch.empty_like(bc_rgb), "target": torch.empty_like(target),
                    "aud": torch.empty_like(aud_src.detach()), "expr": torch.empty_like(expr),
                    "idx": torch.zeros((1,), dtype=torch.int64, device=dev)}

        def fill(st):
            st["rays"].copy_(rays, non_blocking=True); st["bc"].copy_(bc_rgb, non_blocking=True); st["target"].copy_(target, non_blocking=True)
            st["aud"].copy_(aud_src.detach(), non_blocking=True); st["expr"].copy_(expr, non_blocking=True)
            if torch.is_tensor(index):
                st["idx"].copy_(index.reshape(1), non_blocking=True)
            else:
                st["idx"].fill_(int(index))

        def body(st):
            latent_code = self.latent_codes.index_select(0, st["idx"]).squeeze(0)
            aud = self.net.aud_att_net(self.net.aud_net(st["aud"])) if use_win else st["aud"]
            loss, img_loss, latent_loss = self._body(st["rays"], st["bc"], st["target"], aud, st["expr"], latent_code, perturb)
            return loss.detach(), img_loss.detach(), latent_loss.detach()

        loss, img_loss, latent_loss = self._graph_step(key, make_static, fill, body)
        return {"loss": loss, "img_loss": img_loss, "latent_code_loss": latent_loss, "lr": self._lr_t}


class TorsoTrainStep(_AdamStep):
    """One iteration of the torso stage (NeRFs/TorsoNeRF/train_torso.py) for ray batches already on the device: the head pair renders
    the head image, the torso pair renders the torso over it, and only the torso pair learns.

        step(rays_head, rays_torso, bc_rgb, target, aud_feature, pose, expr, latent_code, perturb=None)
            -> {"loss", "img_loss", "img_loss0", "lr"}

    takes TorsoNetwork.forward's arguments plus `target`, and runs, in this order: the head pair through render_pair("head", ...) under
    torch.no_grad() (the fused inference entry, as forward() does); the torso pair with autograd on torso_signal(aud_feature.detach(),
    pose) -- head first, then torso, so the in-kernel Philox draws come in forward()'s order; ops.head_torso_mse_pair on the two
    composites rgb_head * last_weight + rgb_map_fg (fine and coarse); loss = img_loss + img_loss0; backward; FlatParams.gather_grads
    (the all-reduce when world > 1); fused Adam; invalidate_packed() on the two torso nets; the learning rate of learning_rate(args, k).

    * Trained: torso_coarse_nerf and torso_fine_nerf, in TorsoNetwork.parameters() order; their unused feature_linear gets a zero
      gradient, as in TrainStep.
    * Frozen: the head pair and the conditioning.  The head's packed weight blobs are built once and reused every step.
    * Audio: TorsoNetwork has no audio nets, so aud_feature is an input (the head stage's Network.audio_feature); the torso stage does
      not train them.
    * The loss follows the two composites TorsoNetwork.forward restates (train_torso.py:247-271) and the schedule is the head stage's
      (audio_exp_nerf.py:554-558).  The reference's train_torso.py was not available when this was written, so its own loss and
      schedule lines were not re-read: that they are the same is not verified.
    * cuda_graph=True works as in TrainStep: the first call runs eagerly, the second captures, later calls replay.  The inputs are copied
      into static buffers (pose, aud_feature, expr and latent_code included; torso_signal is computed inside the graph), the learning
      rate and Adam's step count are device tensors, batch shapes and perturb are fixed per step (a change raises), and world == 1.
      The step owns the head pair's packed blobs the graph reads; when the nets' caches were dropped (train() / eval(),
      invalidate_packed(), checkpoint.load_head_into_torso) the next call re-packs the current head weights into that same memory.
      load() after the capture raises before it changes anything.

    save() / load() write and read {'global_step', 'model_state_dict': torso_network.state_dict(), 'optimizer': the per-parameter Adam
    state over the trained parameters}, the key set and per-parameter layout of head.tar.  Whether that equals the reference's
    {:06d}_torso.tar (train_torso.py:565-572) is not verified."""

    def __init__(self, torso_network, args, world=1, group=None, cuda_graph=False):
        self.net = torso_network
        self.trained = (torso_network.torso_coarse_nerf, torso_network.torso_fine_nerf)
        mine = {id(p) for m in self.trained for p in m.parameters()}
        super().__init__([p for p in torso_network.parameters() if id(p) in mine], args, world, group, cuda_graph)

    def save(self, path):
        torch.save({"global_step": int(self.global_step), "model_state_dict": self.net.state_dict(),
                    "optimizer": self.optimizer_state_dict()}, path)

    def load(self, path, map_location=None):
        """Resume from a file written by save(): weights copied IN PLACE (the torso weights are views of the flat Adam buffer), the Adam
        moments scattered into the flat state, global_step and the learning rate restored, every packed-weight cache dropped."""
        self._check_loadable()
        ckpt = torch.load(path, map_location=map_location, weights_only=False)
        self.net.load_state_dict(ckpt["model_state_dict"])
        self._load_schedule(ckpt)
        for m in self.net.modules():
            if hasattr(m, "invalidate_packed"):
                m.invalidate_packed()
        return self.global_step

    def __call__(self, rays_head, rays_torso, bc_rgb, target, aud_feature, pose, expr, latent_code, perturb=None):
        perturb = self.args.perturb if perturb is None else perturb
        if self.cuda_graph:
            return self._graphed(rays_head, rays_torso, bc_rgb, target, aud_feature, pose, expr, latent_code, perturb)
        loss, l2 = self._body(rays_head, rays_torso, bc_rgb, target, aud_feature, pose, expr, latent_code, perturb)
        lr = self._advance_lr()
        return {"loss": loss.detach(), "img_loss": l2[0], "img_loss0": l2[1], "lr": lr}

    def _body(self, rays_head, rays_torso, bc_rgb, target, aud_feature, pose, expr, latent_code, perturb):
        for p in self.flat.params:
            p.grad = None
        net = self.net
        with torch.no_grad():
            head = net.render_pair("head", rays_head, bc_rgb, aud_feature, expr, latent_code, perturb)
        torso = net.render_pair("torso", rays_torso, bc_rgb, net.torso_signal(aud_feature.detach(), pose), None, None, perturb)
        l2 = ops.head_torso_mse_pair(head["rgb_map"], head["rgb0"], torso["last_weight"], torso["last_weight0"], torso["rgb_map_fg"],
                                     torso["rgb_map_fg0"], target)
        loss = l2[0] + l2[1]
        self._update(loss, self.trained)
        return loss, l2.detach()

    def _graphed(self, rays_head, rays_torso, bc_rgb, target, aud_feature, pose, expr, latent_code, perturb):
        ins = {"rays_h": rays_head, "rays_t": rays_torso, "bc": bc_rgb, "target": target, "aud": aud_feature, "pose": pose, "expr": expr,
               "latent": latent_code}
        key = tuple(tuple(t.shape) for t in ins.values()) + (float(perturb),)

        heads = (self.net.face_nerf_coarse, self.net.face_nerf_fine)

        def make_static():
            st = {k: torch.empty_like(t.detach()) for k, t in ins.items()}
            # the head pair's packed weights (None in fp32 mode), owned here: the graph holds their device pointers, and the nets' own
            # caches may be dropped (train() / eval(), invalidate_packed(), load_head_into_torso) while the graph lives
            st["head_blobs"] = [m.packed_weights(m.kernel_params()) for m in heads]
            return st

        def fill(st):
            for k, t in ins.items():
                st[k].copy_(t.detach(), non_blocking=True)
            for m, blob in zip(heads, st["head_blobs"]):                   # re-packed into the same memory when the cache was dropped
                if blob is not None:
                    m.packed_weights(m.kernel_params(), out=blob)

        def body(st):
            loss, l2 = self._body(st["rays_h"], st["rays_t"], st["bc"], st["target"], st["aud"], st["pose"], st["expr"], st["latent"],
                                  perturb)
            return loss.detach(), l2

        loss, l2 = self._graph_step(key, make_static, fill, body)
        return {"loss": loss, "img_loss": l2[0], "img_loss0": l2[1], "lr": self._lr_t}
