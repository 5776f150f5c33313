"""world_size-2 (and 3) runs of the N>1 path's HOST logic on CPU with the gloo backend: tile ownership,
dense packing order, the padded gather and the re-assembly on rank 0.  The renderer in these processes
is the checker (there is no GPU here); what is under test is raytracerwin_b200.tiles."""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import scenes
from conftest import ROOT, bits


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, W, H, T, data_dir, out_path):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import raytracerwin_b200 as rt
    from raytracerwin_b200 import tiles
    from oracle.bindings import PortOracle
    sc = rt.Scene(scenes.deterministic_mix(data_dir))
    kw = dict(mode=rt.RT_MODE_PATH, max_bounce=4, antialias=0, traverse=rt.RT_TRAVERSE_EXACT)
    p = rt.make_params(W, H, tile_size=T, tile_count=world, tile_rank=rank, **kw)
    part = PortOracle().render(sc.desc, p)["accum"].reshape(-1, 4)
    counts = [rt.owned_pixels(W, H, T, world, r) for r in range(world)]
    assert counts[rank] == tiles.owned_count(W, H, T, world, rank)
    idx = tiles.dense_index(W, H, T, world, rank)
    assert len(idx) == counts[rank]
    # a rank touched exactly its own pixels
    touched = np.nonzero(part[:, 3] > 0)[0]
    assert np.array_equal(np.sort(idx), touched)
    send = torch.zeros((max(counts), 4), dtype=torch.float32)
    send[:counts[rank]] = torch.from_numpy(part[idx])
    recv = tiles.gather_owned(dist, send, counts, rank, world, dst=0)
    if rank == 0:
        frame = np.zeros((W * H, 4), np.float32)
        for r in range(world):
            frame[tiles.dense_index(W, H, T, world, r)] = recv[r][:counts[r]].numpy()
        np.save(out_path, frame.reshape(H, W, 4))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("world,W,H,T", [(2, 150, 70, 32), (3, 97, 61, 16)])
def test_tile_sharded_render_reassembles(tmp_path, rt, port, data_dir, world, W, H, T):
    out = str(tmp_path / "frame.npy")
    mp.spawn(_worker, args=(world, _free_port(), W, H, T, data_dir, out), nprocs=world, join=True)
    frame = np.load(out)
    sc = rt.Scene(scenes.deterministic_mix(data_dir))
    whole = port.render(sc.desc, rt.make_params(W, H, mode=rt.RT_MODE_PATH, max_bounce=4, antialias=0,
                                                traverse=rt.RT_TRAVERSE_EXACT))["accum"]
    np.testing.assert_array_equal(bits(frame), bits(whole))


def _shared_frame_worker(rank, world, port, W, H, T, data_dir, name, out_path):
    """The N > 1 end-to-end host logic of bench.py: every rank attaches ONE shared host frame and puts its own tiles
    into it (on the GPU box rt_gpu_deliver_owned writes them over PCIe; here the checker's pixels are copied in)."""
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import bench
    import raytracerwin_b200 as rt
    from raytracerwin_b200 import tiles
    from oracle.bindings import PortOracle
    npix = W * H
    frame = bench.SharedFrame(name, npix, True) if rank == 0 else None
    dist.barrier()
    if rank != 0:
        frame = bench.SharedFrame(name, npix, False)
    sc = rt.Scene(scenes.deterministic_mix(data_dir))
    p = rt.make_params(W, H, mode=rt.RT_MODE_PATH, max_bounce=4, antialias=0, traverse=rt.RT_TRAVERSE_EXACT,
                       tile_size=T, tile_count=world, tile_rank=rank)
    o = PortOracle().render(sc.desc, p, want_display=True)
    idx = tiles.dense_index(W, H, T, world, rank)
    frame.accum[idx] = o["accum"].reshape(-1, 4)[idx]
    frame.display[idx] = o["display"].reshape(-1)[idx]
    dist.barrier()
    if rank == 0:
        np.savez(out_path, accum=frame.accum.reshape(H, W, 4).copy(), display=frame.display.reshape(H, W).copy())
    dist.barrier()
    frame.close(unlink=(rank == 0))
    dist.destroy_process_group()


def test_shared_host_frame_assembled_by_two_ranks(tmp_path, rt, port, data_dir):
    W, H, T, world = 150, 70, 32, 2
    out = str(tmp_path / "frame.npz")
    mp.spawn(_shared_frame_worker, args=(world, _free_port(), W, H, T, data_dir, f"rtb200_test_{os.getpid()}", out), nprocs=world, join=True)
    got = np.load(out)
    sc = rt.Scene(scenes.deterministic_mix(data_dir))
    whole = port.render(sc.desc, rt.make_params(W, H, mode=rt.RT_MODE_PATH, max_bounce=4, antialias=0,
                                                traverse=rt.RT_TRAVERSE_EXACT), want_display=True)
    np.testing.assert_array_equal(bits(got["accum"]), bits(whole["accum"]))
    np.testing.assert_array_equal(got["display"], whole["display"])


def test_dense_index_is_a_partition():
    from raytracerwin_b200 import tiles
    for (W, H, T, n) in ((150, 70, 32, 3), (64, 64, 32, 4), (33, 17, 8, 5), (1920, 1080, 32, 8)):
        allidx = np.concatenate([tiles.dense_index(W, H, T, n, r) for r in range(n)])
        assert len(allidx) == W * H and np.array_equal(np.sort(allidx), np.arange(W * H))
    assert np.array_equal(tiles.dense_index(5, 3, 0, 1, 0), np.arange(15))
