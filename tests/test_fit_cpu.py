"""CPU tests of the training driver (ideal_nerf_b200.fit): flag and config-file parsing, checkpoint naming and the choice of the
checkpoint to resume from, the per-epoch frame permutation, the schedule of boundary steps, and TrainStep's graph-only options."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_config_file_and_flags(tmp_path):
    """--config key = value lines fill the reference's flags and the trainer's own; the command line wins over the file."""
    from ideal_nerf_b200 import fit
    cfg = tmp_path / "subject.txt"
    cfg.write_text("expname = obama_head\nbasedir = ./logs\ndatadir = ./dataset/Obama  # the subject\nN_iters = 3\nnosmo_iters = 5\n"
                   "i_print = 7\nno_reload = True\nstage = torso\nseed = 9\nmlp_mode = bf16\n")
    a = fit.fit_parser().parse_args(["--config", str(cfg), "--N_iters", "4", "--head_ckpt", "h.tar"])
    assert (a.expname, a.basedir, a.datadir) == ("obama_head", "./logs", "./dataset/Obama")
    assert (a.N_iters, a.nosmo_iters, a.i_print, a.no_reload, a.stage, a.seed, a.mlp_mode) == (4, 5, 7, True, "torso", 9, "bf16")
    assert a.head_ckpt == "h.tar"
    assert fit.run_dir(a) == os.path.join("./logs", "obama_head")
    d = fit.fit_parser().parse_args([])
    assert (d.stage, d.seed, d.head_ckpt, d.no_reload, d.i_weights, d.i_testset) == ("head", 0, None, False, 5000, 1000)
    with pytest.raises(SystemExit):
        fit.fit_parser().parse_args(["--stage", "neck"])


def test_cli_needs_a_run_directory_and_a_head_for_the_torso():
    from ideal_nerf_b200 import fit
    with pytest.raises(SystemExit, match="basedir"):
        fit.main([])
    with pytest.raises(SystemExit, match="head_ckpt"):
        fit.main(["--basedir", "b", "--expname", "e", "--stage", "torso"])


def test_checkpoint_names_and_latest(tmp_path):
    """head.tar (one file, rewritten) for the head, {step:06d}_torso.tar for the torso; the latest is the naturally sorted last file with
    the stage's suffix, so 10 sorts after 9 without zero padding and a half-written .tmp file is never picked."""
    from ideal_nerf_b200 import fit
    assert fit.checkpoint_name("head", 1234) == "head.tar"
    assert fit.checkpoint_name("torso", 1234) == "001234_torso.tar"
    assert fit.latest_checkpoint(str(tmp_path / "missing")) is None
    assert fit.latest_checkpoint(str(tmp_path)) is None
    for name in ("000020_torso.tar", "000100_torso.tar", "000099_torso.tar", "head.tar", "000200_torso.tar.tmp", "log.jsonl"):
        (tmp_path / name).write_bytes(b"")
    assert fit.latest_checkpoint(str(tmp_path), "_torso.tar") == str(tmp_path / "000100_torso.tar")
    assert fit.latest_checkpoint(str(tmp_path), ".tar") == str(tmp_path / "head.tar")
    nat = tmp_path / "nat"
    nat.mkdir()
    for name in ("9_torso.tar", "10_torso.tar", "2_torso.tar"):
        (nat / name).write_bytes(b"")
    assert fit.latest_checkpoint(str(nat), "_torso.tar") == str(nat / "10_torso.tar")


def test_epoch_permutation_is_the_same_in_every_process():
    """epoch_order is a permutation that depends on (seed, epoch) only: two separate interpreters (two ranks) get the same frames in the
    same order; another epoch or another seed gives another order."""
    from ideal_nerf_b200 import fit
    code = ("import sys; sys.path.insert(0, %r); import numpy as np; from ideal_nerf_b200 import fit; "
            "np.random.seed(int(sys.argv[1])); print(fit.epoch_order(3, 7, 50).tolist())" % ROOT)
    outs = [subprocess.run([sys.executable, "-c", code, str(r)], capture_output=True, text=True, check=True).stdout for r in (0, 1)]
    assert outs[0] == outs[1]
    p = fit.epoch_order(3, 7, 50)
    assert p.dtype == np.int64 and sorted(p.tolist()) == list(range(50))
    assert str(p.tolist()) == outs[0].strip()
    assert not np.array_equal(p, fit.epoch_order(3, 8, 50)) and not np.array_equal(p, fit.epoch_order(4, 7, 50))


def test_event_schedule():
    """Log every i_print steps and after the last, save every i_weights steps and after the last, validate every i_testset steps and
    write the image every i_img steps; a zero interval switches its event off."""
    from types import SimpleNamespace
    from ideal_nerf_b200 import fit
    a = SimpleNamespace(i_print=3, i_weights=5, i_testset=4, i_img=0)
    ev = {s: fit.events(s, a, 10) for s in range(1, 11)}
    assert [s for s, e in ev.items() if e["log"]] == [3, 6, 9, 10]
    assert [s for s, e in ev.items() if e["save"]] == [5, 10]
    assert [s for s, e in ev.items() if e["val"]] == [4, 8]
    assert [s for s, e in ev.items() if e["img"]] == []
    b = SimpleNamespace(i_print=1, i_weights=0, i_testset=0, i_img=2)
    ev = {s: fit.events(s, b, 4) for s in range(1, 5)}
    assert all(e["log"] for e in ev.values())
    assert [s for s, e in ev.items() if e["save"]] == [4]
    assert [s for s, e in ev.items() if e["img"]] == [2, 4]


def test_graph_options_need_graph_mode():
    """max_graphs and log_rows belong to the CUDA-graph mode: asking for them on an eager step raises before anything runs."""
    import torch
    import ideal_nerf_b200 as M
    from ideal_nerf_b200.train import TorsoTrainStep, TrainStep
    net = M.Network(450, 450, 1200., 0.57, 1.17, 8192, None, 64, 128)
    with pytest.raises(ValueError, match="cuda_graph=True"):
        TrainStep(net, torch.zeros(2, 32), net.args, max_graphs=2)
    with pytest.raises(ValueError, match="cuda_graph=True"):
        TrainStep(net, torch.zeros(2, 32), net.args, log_rows=10)
    with pytest.raises(ValueError, match="max_graphs"):
        TrainStep(net, torch.zeros(2, 32), net.args, max_graphs=0)
    tnet = M.TorsoNetwork(450, 450, 1200., 0.57, 1.17, 8192, 64, 128, args=M.default_args(dim_aud=64, dim_expr=79), dim_expr=79)
    with pytest.raises(ValueError, match="cuda_graph=True"):
        TorsoTrainStep(tnet, tnet.args, log_rows=10)
    assert TrainStep.LOG_COLUMNS == ("loss", "img_loss", "latent_code_loss", "psnr", "lr")
    assert TorsoTrainStep.LOG_COLUMNS == ("loss", "img_loss", "img_loss0", "psnr", "lr")
