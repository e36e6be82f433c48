"""CPU-side checks of the head + torso video path: the argument validation of inerf_head_torso_to8b, which returns before any device
work, and a world-size-2 gloo run of the uint8 band gather of render_head_torso_video (the render kernels themselves are GPU-only)."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

A16 = 0x10000          # fake device address (never dereferenced: every call below fails or returns before a launch)


@pytest.fixture(scope="module")
def L():
    import ideal_nerf_b200 as m
    m.build()
    return m.lib()


def test_head_torso_to8b_argument_checks(L):
    f = L.inerf_head_torso_to8b
    ok = dict(head=A16, lw=A16, fg=A16, n=5, out=A16, rgb=A16)

    def call(**kw):
        a = dict(ok, **kw)
        return f(a["head"], a["lw"], a["fg"], a["n"], a["out"], a["rgb"], None)

    for k in ("head", "lw", "fg", "out"):
        assert call(**{k: None}) == -1, k
        assert b"NULL" in L.inerf_last_error()
    assert call(n=-1) == -2
    assert call(n=-1, head=None) == -2                     # the size is checked first
    assert call(n=1 << 62) == -2                           # more rays than one launch covers
    assert call(n=0) == 0                                  # nothing to do: no pointer is needed
    assert call(n=0, head=None, lw=None, fg=None, out=None, rgb=None) == 0


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, n_rays, q):
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from ideal_nerf_b200.frame import HeadTorsoFrameRenderer, band
    lo, hi = band(n_rays, rank, world)
    full = (torch.arange(n_rays * 3) * 7 % 256).to(torch.uint8).reshape(n_rays, 3)        # the "to8b bytes" of a frame
    fr = HeadTorsoFrameRenderer(network=None, torso_pose=None, rank=rank, world=world)
    out = fr.gather_image(full[lo:hi].clone(), n_rays)
    ok = out.dtype == torch.uint8 and bool(torch.equal(out, full))
    # the double-buffered form render_head_torso_video uses: each gather consumed one frame late
    frame = lambda k: (full.to(torch.int32) + k).remainder(256).to(torch.uint8)
    hs = [fr.gather_image(frame(k)[lo:hi].clone(), n_rays, async_op=True) for k in range(2)]
    for k in range(2, 5):
        ok = ok and bool(torch.equal(hs[k - 2].wait(), frame(k - 2)))
        hs.append(fr.gather_image(frame(k)[lo:hi].clone(), n_rays, async_op=True))
    ok = ok and bool(torch.equal(hs[3].wait(), frame(3))) and bool(torch.equal(hs[4].wait(), frame(4)))
    # an fp32 gather on the same renderer (render_frame) keeps its own buffers: the byte images above are not touched by it
    img = torch.arange(n_rays * 3, dtype=torch.float32).reshape(n_rays, 3)
    ok = ok and bool(torch.equal(fr.gather_image(img[lo:hi].clone(), n_rays), img))
    ok = ok and bool(torch.equal(hs[4].wait(), frame(4)))
    if rank == 0:
        q.put((tuple(out.shape), ok))
    else:
        assert ok
    dist.destroy_process_group()


def test_gather_u8_bands_world2_gloo():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    for n_rays in (202500, 11):           # even split, and a ragged tail (6 + 5)
        port = _free_port()
        procs = [ctx.Process(target=_worker, args=(r, 2, port, n_rays, q)) for r in range(2)]
        for p in procs:
            p.start()
        for p in procs:
            p.join(timeout=120)
            assert p.exitcode == 0
        shape, ok = q.get(timeout=10)
        assert shape == (n_rays, 3) and ok
