"""Checkpoint formats of the reference's HeadNeRF training script, read and written with the same dictionary keys so files move both ways
(the 'optimizer' entry too: train.TrainStep.save / load convert between its flat Adam and the reference's per-parameter state).

* head.tar (NeRFs/HeadNeRF/train/audio_exp_nerf.py:584-591 save, :518-525 resume):
      {'global_step', 'model_state_dict' (Network.state_dict(): face_nerf_coarse.*, face_nerf_fine.*, aud_net.*, aud_att_net.*,
       ds_aud_net.*), 'optimizer', 'latent_codes' (n_frames, 32)}
* fine-tune source (--ft_path, :498-514): {'network_fn_state_dict', 'network_fine_state_dict', 'network_audnet_state_dict',
      'network_audattnet_state_dict'}; the reference drops pts_linears.0 / pts_linears.5 / views_linears.0 weights (their input
      widths depend on dim_aud / dim_expr) and loads the rest with strict=False.
* the start of the torso stage (NeRFs/TorsoNeRF/train_torso.py): load_head_into_torso copies a head.tar's head pair into a TorsoNetwork;
      train.TorsoTrainStep.save / load write and resume the torso stage itself.
Pure host I/O: nothing here launches a kernel."""
import torch

_FT_DROPPED = ("pts_linears.0.weight", "pts_linears.5.weight", "views_linears.0.weight")


def save_head_checkpoint(path, network, optimizer, latent_codes, global_step):
    """audio_exp_nerf.py:584-591."""
    torch.save({"global_step": int(global_step), "model_state_dict": network.state_dict(),
                "optimizer": optimizer.state_dict() if optimizer is not None else None,
                "latent_codes": latent_codes.data if hasattr(latent_codes, "data") else latent_codes}, path)


def load_head_checkpoint(path, network, optimizer=None, latent_codes=None, map_location=None, strict=True):
    """audio_exp_nerf.py:518-525.  Returns global_step.  Weights written by the reference load unchanged (same keys).

    The latent codes are copied IN PLACE (the reference rebinds `latent_codes.data`, :522; here the tensor may be a view of
    train.FlatParams' flat Adam buffer and must stay one).  `optimizer` is a per-parameter torch.optim.Adam like the reference's; to
    resume a train.TrainStep (one flat Adam) use TrainStep.load(path), which also restores global_step and the learning rate."""
    ckpt = torch.load(path, map_location=map_location, weights_only=False)
    network.load_state_dict(ckpt["model_state_dict"], strict=strict)
    if latent_codes is not None and ckpt.get("latent_codes") is not None:
        with torch.no_grad():
            latent_codes.data.copy_(ckpt["latent_codes"].to(latent_codes.device))
    if optimizer is not None and ckpt.get("optimizer") is not None:
        n_saved = sum(len(g["params"]) for g in ckpt["optimizer"]["param_groups"])
        n_have = sum(len(g["params"]) for g in optimizer.param_groups)
        if n_saved != n_have:
            raise ValueError(f"checkpoint optimiser state covers {n_saved} parameters, the given optimiser {n_have}: "
                             "use train.TrainStep.load(path) for the flat-buffer Adam")
        optimizer.load_state_dict(ckpt["optimizer"])
    for m in network.modules():
        if hasattr(m, "invalidate_packed"):
            m.invalidate_packed()
    return int(ckpt.get("global_step", 0))


def load_finetune_checkpoint(path, network, map_location=None):
    """audio_exp_nerf.py:498-514 (--ft_path)."""
    ckpt = torch.load(path, map_location=map_location, weights_only=False)
    coarse, fine = dict(ckpt["network_fn_state_dict"]), dict(ckpt["network_fine_state_dict"])
    for k in _FT_DROPPED:
        coarse.pop(k, None)
        fine.pop(k, None)
    network.face_nerf_coarse.load_state_dict(coarse, strict=False)
    network.face_nerf_fine.load_state_dict(fine, strict=False)
    if "network_audnet_state_dict" in ckpt:
        network.aud_net.load_state_dict(ckpt["network_audnet_state_dict"], strict=False)
    if "network_audattnet_state_dict" in ckpt:
        network.aud_att_net.load_state_dict(ckpt["network_audattnet_state_dict"], strict=False)
    return 0


def load_head_into_torso(path, torso_network, map_location=None):
    """The start of the torso stage: copy the head pair of a head.tar (the reference's keys, as load_head_checkpoint reads them) into
    torso_network.face_nerf_coarse / face_nerf_fine, in place.  The torso pair is left alone and the head pair's packed weight blobs are
    dropped.  Returns the head's latent codes (n_frames, 32), or None when the file has none.

    Every key of the head pair must be present with this network's shape; otherwise ValueError names the key and both shapes before
    anything is copied.  TorsoNetwork defaults to dim_expr=79, so a head trained with another expression width fails here."""
    ckpt = torch.load(path, map_location=map_location, weights_only=False)
    sd = ckpt["model_state_dict"]
    pairs = []
    for name in ("face_nerf_coarse", "face_nerf_fine"):
        for k, v in getattr(torso_network, name).state_dict().items():
            key = f"{name}.{k}"
            if key not in sd:
                raise ValueError(f"load_head_into_torso: {path} has no '{key}': not a head.tar of the reference's Network")
            if tuple(sd[key].shape) != tuple(v.shape):
                raise ValueError(f"load_head_into_torso: '{key}' is {tuple(sd[key].shape)} in {path} but {tuple(v.shape)} in this "
                                 "TorsoNetwork: the head was trained with other conditioning widths (dim_aud / dim_expr / dim_latent; "
                                 "TorsoNetwork(dim_expr=...) must match the head's)")
            pairs.append((v, sd[key]))
    with torch.no_grad():
        for dst, src in pairs:
            dst.copy_(src.to(dst.device))
    for m in (torso_network.face_nerf_coarse, torso_network.face_nerf_fine):
        m.invalidate_packed()
    return ckpt.get("latent_codes")
