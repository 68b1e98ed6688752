"""CPU, world_size 2, gloo: the N>1 path of the frame / voxel-slab sharding (no data-path collective; one all_gather)."""

import os
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import ROOT


def _worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    from ide3d_b200 import dist as idist
    from oracle.backend import cpu_reference_ops
    from ide3d_b200.training.triplane import TriPlaneGenerator
    r, w, dev = idist.init_from_env(backend='gloo')
    assert (r, w) == (rank, world) and dev.type == 'cpu'
    torch.manual_seed(0)                                   # identical replicas on every rank
    G = TriPlaneGenerator(z_dim=16, w_dim=16, img_resolution=32, plane_resolution=16, render_size=8, channel_base=256,
                          channel_max=16, sr_channels=(8, 8), mapping_kwargs=dict(num_layers=1)).eval().requires_grad_(False)
    F = 5                                                  # odd on purpose: ragged shard
    z = torch.randn(F, 16)
    c = torch.tensor([1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 2.7, 0, 0, 0, 1, 4.2647, 0, 0.5, 0, 4.2647, 0.5, 0, 0, 1.]).repeat(F, 1)
    with cpu_reference_ops():
        ws = G.mapping(z, c)
        frames = idist.render_frames_sharded(G, ws, c, rank, world, batch=2, num_steps=6, perturb=None)
        single = idist.render_frames_sharded(G, ws, c, 0, 1, batch=8, num_steps=6, perturb=None)
        # streaming variant (the e2e leg of bench.py): F multiple of world * batch, result on the host of rank 0 only
        streamed = idist.stream_frames_sharded(G, ws[:4], c[:4], rank, world, batch=2, num_steps=6, perturb=None)
        sdiff = int((streamed.int() - single[:4].int()).abs().max()) if rank == 0 else (0 if streamed is None else 99)
        # the shared-memory transport (default on CUDA boxes): every rank writes its own frames into one /dev/shm buffer
        shm = idist.stream_frames_sharded(G, ws[:4], c[:4], rank, world, batch=2, transport='shm', num_steps=6, perturb=None)
        sdiff = max(sdiff, int((shm.int() - single[:4].int()).abs().max()) if rank == 0 else (0 if shm is None else 99))
    # voxel slabs: every rank fills its contiguous slab of a fake sigma volume, one all_gather restores the volume
    total = 4 ** 3 + 1
    first, count = idist.slab_range(total, rank, world)
    local = torch.arange(first, first + count, dtype=torch.float32)[None]
    vol = idist.all_gather_slabs(local, total, world)
    # different batch compositions may pick different CPU conv algorithms: allow one uint8 level
    diff = int((frames.int() - single.int()).abs().max())
    q.put((rank, frames.shape, max(diff, sdiff), bool(torch.equal(vol[0], torch.arange(total, dtype=torch.float32)))))
    dist.barrier()
    dist.destroy_process_group()


def test_shard_helpers():
    from ide3d_b200 import dist as idist
    assert idist.shard_indices(7, 1, 3) == [1, 4]
    cover = sorted(i for r in range(3) for i in idist.shard_indices(7, r, 3))
    assert cover == list(range(7))
    spans = [idist.slab_range(10, r, 4) for r in range(4)]
    assert spans == [(0, 3), (3, 3), (6, 2), (8, 2)]


@pytest.mark.timeout(300)
def test_two_rank_gloo_frame_and_slab_gather(monkeypatch):
    # the ranks stay on the CPU on a GPU machine too: init_from_env would bind rank r to cuda:r, which a one-GPU machine lacks
    monkeypatch.setenv('CUDA_VISIBLE_DEVICES', '')
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    try:
        res = [q.get(timeout=240) for _ in procs]
        for p in procs:
            p.join(timeout=60)
    finally:
        for p in procs:                                  # a rank whose peer died waits in the rendezvous: do not leave it behind
            if p.is_alive():
                p.kill()
                p.join()
    for p in procs:
        assert p.exitcode == 0
    for rank, shape, diff, same_vol in res:
        assert tuple(shape) == (5, 3, 32, 32) and diff <= 1 and same_vol, (rank, shape, diff, same_vol)
