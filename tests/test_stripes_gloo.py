"""N>1 host logic on CPU: world_size-2 (and 3) `gloo` process groups render bin-row stripes of one frame
(with the CPU oracle standing in for the per-rank renderer) and all-gather them; the result must equal the
single-rank frame. Exercises vello_b200.stripes (the partition bench.py uses under torchrun) and the stripe window."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from vello_b200 import scenes
from vello_b200.encoding import BLACK, resolve
from vello_b200.stripes import assemble, n_bin_rows, stripe_for, stripe_pixel_rows


def test_partition_properties():
    for height in (1, 255, 256, 257, 1000, 4096, 16384):
        for world in (1, 2, 3, 4, 8, 16):
            ranges = [stripe_for(r, world, height) for r in range(world)]
            assert ranges[0][0] == 0 and ranges[-1][1] == n_bin_rows(height)
            for a, b in zip(ranges, ranges[1:]):
                assert a[1] == b[0]
            sizes = [b - a for a, b in ranges]
            assert max(sizes) - min(sizes) <= 1
            assert sum(stripe_pixel_rows(r, height)[1] - stripe_pixel_rows(r, height)[0] for r in ranges) == height


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, w, h, aa, out_path):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from oracle.vbo import Oracle
    packed = resolve(scenes.paris_like(400, h, seed=5).encoding)
    br = stripe_for(rank, world, h)
    img = Oracle().render(packed, w, h, BLACK.premul_rgba8_u32(), aa, bin_rows=br if br[1] > br[0] else (0, 0))
    r0, r1 = stripe_pixel_rows(br, h)
    mine = torch.from_numpy(np.ascontiguousarray(img[r0:r1] if br[1] > br[0] else img[:0]))
    sizes = [torch.zeros(1, dtype=torch.int64) for _ in range(world)]
    dist.all_gather(sizes, torch.tensor([mine.shape[0]], dtype=torch.int64))
    mx = int(max(s.item() for s in sizes))
    pad = torch.zeros((mx, w, 4), dtype=torch.uint8)
    pad[: mine.shape[0]] = mine
    gathered = [torch.zeros((mx, w, 4), dtype=torch.uint8) for _ in range(world)]
    dist.all_gather(gathered, pad)
    t = torch.tensor([float(rank + 1)])
    dist.all_reduce(t, op=dist.ReduceOp.MAX)  # the max-over-ranks timing reduction bench.py uses
    if rank == 0:
        assert t.item() == world
        frame = assemble([g[: int(s.item())].numpy() for g, s in zip(gathered, sizes)])
        np.save(out_path, frame)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_stripes_over_gloo(tmp_path, world):
    from oracle.vbo import Oracle
    w, h, aa = 300, 700, 2
    out = str(tmp_path / "frame.npy")
    mp.spawn(_worker, args=(world, _free_port(), w, h, aa, out), nprocs=world, join=True)
    packed = resolve(scenes.paris_like(400, h, seed=5).encoding)
    full = Oracle().render(packed, w, h, BLACK.premul_rgba8_u32(), aa)
    assert np.array_equal(np.load(out), full)


def test_tile_row_bounds_and_rebalance():
    """The cost-balanced tile-row split (vello_b200.stripes.rebalance == group_rebalance in vb_group.cu): boundaries stay
    monotone with at least one row per stripe, move towards the slower stripes, stop inside the tolerance, and converge on a
    synthetic cost profile."""
    from vello_b200.stripes import even_tile_bounds, n_tile_rows, rebalance
    for h in (16, 100, 1080, 4096, 16384):
        for w in (1, 2, 3, 8):
            b = even_tile_bounds(w, h)
            assert b[0] == 0 and b[-1] == n_tile_rows(h) and all(x <= y for x, y in zip(b, b[1:]))
    b = even_tile_bounds(8, 4096)
    assert rebalance(b, [1.0] * 8) == b                       # balanced: unchanged
    assert rebalance(b, [1.0, 1.02, 0.99, 1.0, 1.01, 1.0, 0.98, 1.0]) == b   # inside the 6 % tolerance
    assert rebalance(b, [0.0] * 8) == b                       # no measurement yet
    nb = rebalance(b, [2.0, 1.0, 1.0, 1.0, 1.0, 1.0, 1.0, 1.0])
    assert nb[1] < b[1] and nb[0] == 0 and nb[-1] == b[-1] and all(x < y for x, y in zip(nb, nb[1:]))
    # a cost density that falls linearly over the rows: iterate with the "true" cost of each stripe
    import numpy as np
    dens = np.linspace(3.0, 1.0, 256)
    cum = np.concatenate([[0.0], np.cumsum(dens)])
    b = even_tile_bounds(8, 4096)
    for _ in range(40):
        ms = [float(cum[b[i + 1]] - cum[b[i]]) for i in range(8)]
        nb = rebalance(b, ms)
        if nb == b:
            break
        b = nb
    ms = [float(cum[b[i + 1]] - cum[b[i]]) for i in range(8)]
    assert (max(ms) - min(ms)) / (sum(ms) / 8) < 0.12
    # tiny frames: more stripes than rows cannot be balanced and are returned unchanged
    assert rebalance([0, 1, 1, 2], [1.0, 0.0, 1.0]) == [0, 1, 1, 2]
