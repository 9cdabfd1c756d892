"""Bin-row stripe partition of one frame across ranks (SURVEY.md section 8e, DESIGN.md section 6).

The path shards by bin rows (256-px stripes): backdrop only propagates left-to-right inside a tile row, tiles, PTCL
and segments are per tile, so horizontal stripes need NO data-path collective. Each rank renders
`bin_rows = stripe_for(rank, world, height)`; concatenating the stripes in rank order is the full frame.
"""
from __future__ import annotations

from typing import List, Tuple

import numpy as np

BIN_PX = 256  # 16 tiles x 16 px


def n_bin_rows(height: int) -> int:
    return (height + BIN_PX - 1) // BIN_PX


def stripe_for(rank: int, world: int, height: int) -> Tuple[int, int]:
    """Contiguous, as-even-as-possible bin-row range [b0, b1) of `rank`. Ranks beyond the number of bin rows
    get an empty range (b0 == b1)."""
    n = n_bin_rows(height)
    base, rem = divmod(n, world)
    b0 = rank * base + min(rank, rem)
    b1 = b0 + base + (1 if rank < rem else 0)
    return b0, b1


def stripe_pixel_rows(bin_rows: Tuple[int, int], height: int) -> Tuple[int, int]:
    return min(bin_rows[0] * BIN_PX, height), min(bin_rows[1] * BIN_PX, height)


def assemble(stripes: List[np.ndarray]) -> np.ndarray:
    """Concatenate per-rank stripes (rank order) into the frame; empty stripes are skipped."""
    parts = [s for s in stripes if s.shape[0] > 0]
    return np.concatenate(parts, axis=0)


# ---- tile-row stripes with cost balancing (the multi-GPU split of vb_group and bench.py) -----------------------------------
TILE_PX = 16


def n_tile_rows(height: int) -> int:
    return (height + TILE_PX - 1) // TILE_PX


def even_tile_bounds(world: int, height: int) -> List[int]:
    """world + 1 tile-row boundaries, stripes as even as possible."""
    ht = n_tile_rows(height)
    return [ht * i // world for i in range(world + 1)]


def rebalance(bounds: List[int], ms: List[float], damping: float = 0.5, tolerance: float = 0.06) -> List[int]:
    """New boundaries from the device times of the last frame (same rule as group_rebalance in vb_group.cu): the cost of a
    stripe is assumed to be spread evenly over its tile rows, the boundaries move (damped) to where the cumulative cost
    crosses k/n of the total; every stripe keeps at least one tile row. Unchanged when the times agree within `tolerance`."""
    n = len(ms)
    ht = bounds[-1]
    if n < 2 or ht < n or any(not (m > 0.0) for m in ms):
        return list(bounds)
    total = float(sum(ms))
    if max(ms) - min(ms) < tolerance * (total / n):
        return list(bounds)
    nb = [0] * (n + 1)
    nb[n] = ht
    seg, acc = 0, 0.0
    for k in range(1, n):
        want = total * k / n
        while seg + 1 < n and acc + ms[seg] < want:
            acc += ms[seg]
            seg += 1
        rows = bounds[seg + 1] - bounds[seg]
        frac = (want - acc) / ms[seg] if ms[seg] > 0 else 0.0
        ideal = bounds[seg] + rows * frac
        nb[k] = int((1.0 - damping) * bounds[k] + damping * ideal + 0.5)
    for k in range(1, n):
        nb[k] = max(nb[k], nb[k - 1] + 1)
    for k in range(n - 1, 0, -1):
        nb[k] = min(nb[k], nb[k + 1] - 1)
    return nb
