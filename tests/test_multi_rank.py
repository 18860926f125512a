"""CPU test of the N>1 path: world_size-2 gloo processes take their share of the tile queue from the host C dispatcher
(libcrhost.so takeRankTiles — the code a torchrun rank of bench.py runs), "render" those tiles with the CPU oracle (test
infrastructure standing in for the GPU) and gather the packed tiles on rank 0 (gloo here, the C NCCL gather on GPUs): the
frame must be bit-identical to a single-rank render, and the ranks' shares must partition the tile queue."""
import os
import socket
import subprocess
import sys

import numpy as np

from conftest import ROOT, GOLDEN

WORKER = r'''
import os, sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, os.path.join(sys.argv[1], "c-ray_b200")); sys.path.insert(0, os.path.join(sys.argv[1], "tests"))
import shard, crhost, oracle_lib as O
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo")
sc = O.OracleScene(sys.argv[2])
W, H = sc.W, sc.H
R = crhost.Renderer(sys.argv[2], tile=16)                      # the C dispatcher: tile grid, order, rank assignment
mine, owner, every = R.rank_tiles(rank, world)
assert len(every) == len(owner) and sorted(map(tuple, mine.tolist())) == sorted(tuple(every[k]) for k in range(len(every)) if owner[k] == rank)
fb = np.zeros((H, W, 3), dtype=np.float32)
for r in mine:
    sc.render(threads=1, tile=tuple(int(v) for v in r), rgb=fb)
t = torch.from_numpy(fb)
share = [[tuple(int(v) for v in every[k]) for k in range(len(every)) if owner[k] == q] for q in range(world)]
pad = max(sum((x1 - x0) * (y1 - y0) * 3 for x0, y0, x1, y1 in s) for s in share)
buf = torch.zeros(pad)
p = shard.pack(t, share[rank])
buf[:p.numel()] = p
outs = [torch.empty(pad) for _ in range(world)] if rank == 0 else None
dist.gather(buf, outs, dst=0)
if rank == 0:
    for q in range(1, world):
        shard.unpack_into(t, share[q], outs[q])
    t.numpy().tofile(sys.argv[3])
dist.barrier()
dist.destroy_process_group()
'''


def free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def test_two_ranks_reassemble_the_frame(tmp_path):
    scene = os.path.join(GOLDEN, "g_nodes.crscene")
    out = str(tmp_path / "frame.f32")
    w = tmp_path / "worker.py"
    w.write_text(WORKER)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(free_port()), str(w), ROOT, scene, out]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-3000:]
    got = np.fromfile(out, dtype=np.float32)
    ref = np.fromfile(os.path.join(GOLDEN, "g_nodes.f32"), dtype=np.float32)
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))


def test_shard_helpers():
    sys.path.insert(0, os.path.join(ROOT, "c-ray_b200"))
    import torch
    import shard
    W, H, t = 50, 35, 16
    rects = shard.tiles_of(W, H, t)
    assert len(rects) == 4 * 3
    for world in (1, 2, 3, 8):
        parts = [shard.rank_rects(W, H, t, r, world) for r in range(world)]
        assert sorted(sum(parts, [])) == sorted(rects)
    fb = torch.arange(H * W * 3, dtype=torch.float32).view(H, W, 3)
    flat = shard.pack(fb, rects[::2])
    fb2 = torch.zeros_like(fb)
    shard.unpack_into(fb2, rects[::2], flat)
    for r in rects[::2]:
        assert torch.equal(shard.rect_view(fb2, r), shard.rect_view(fb, r))
    assert shard.rect_view(fb, (0, 0, 16, 16)).shape == (16, 16, 3) and shard.rect_view(fb, (48, 32, 50, 35)).shape == (3, 2, 3)


def test_gather_index_path_equals_tile_by_tile_copies():
    """gather_to_rank0 packs/unpacks with one index_select / index_copy_ per rank; same bytes as copying tile by tile."""
    import torch
    import shard
    W, H, t, world = 200, 117, 32, 3
    fb = torch.arange(H * W * 3, dtype=torch.float32).view(H, W, 3)
    idx = shard._pixel_indices(W, H, t, world, fb.device)
    assert sum(int(i.numel()) for i in idx) == W * H
    for r in range(world):
        rects = shard.rank_rects(W, H, t, r, world)
        a = shard.pack(fb, rects)
        b = fb.view(-1, 3).index_select(0, idx[r]).reshape(-1)
        assert torch.equal(a, b)
        x, y = torch.zeros_like(fb), torch.zeros_like(fb)
        shard.unpack_into(x, rects, a)
        y.view(-1, 3).index_copy_(0, idx[r], b.view(-1, 3))
        assert torch.equal(x, y)


def test_rank_placement_balances_the_rays_of_the_headline_scene(bundled_scene):
    """Static tile placement must spread the WORK, not just the tile count.  Dealing tiles by queue position (k % world) looks
    neutral but, under c-ray's default "fromMiddle" order, hands one rank every tile left of the image centre: on hdr.json the odd
    positions carry ~12% more rays (that was 0.88 instead of ~0.97 strong-scaling efficiency on 8 B200).  The spatial interleave of
    takeRankTiles (tile (tx, ty) -> rank (tx + 5 ty) % world) must stay within a few percent; rays per tile counted by the oracle
    on the 1080p tile grid at quarter resolution."""
    import pytest
    import crhost
    import oracle_lib as O
    from conftest import NO_BUNDLED
    scene = bundled_scene("hdr")
    if scene is None:
        pytest.skip(NO_BUNDLED)
    W, H, T = 480, 270, 16                                  # the 30 x 17 tile grid of 1920x1080 in 64x64 tiles
    R = crhost.Renderer(scene, W, H, 2, 32, gpus=1, tile=T, quiet=True)
    o = O.OracleScene(scene, W, H, 2, 32)
    _, _, every = R.rank_tiles(0, 1)
    rays = np.array([o.render(threads=8, tile=tuple(int(v) for v in r), count=True)[1]["rays"] for r in every], dtype=np.float64)
    for world in (2, 4, 8):
        _, owner, _ = R.rank_tiles(0, world)
        share = np.array([rays[owner == q].sum() for q in range(world)])
        assert np.bincount(owner, minlength=world).min() > 0
        assert share.max() / share.mean() < 1.06, (world, share / share.mean())
        by_position = np.array([rays[q::world].sum() for q in range(world)])
        assert by_position.max() / by_position.mean() > 1.08          # the trap this test documents
    o.close()
    R.close()
