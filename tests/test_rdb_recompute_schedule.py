"""CPU: the barrier protocol of the conv4-only form of the fused conv4 + conv5 kernel (csrc/conv3x3_rdb.cuh:
conv3x3_rdb_kernel<4, 2, PAIR, true>, the recompute of a dense block's x4 in a memory-efficient backward), restated in
tools/rdb_protocol_sim.py -- no GPU.

The producer loads conv4's chunks only, conv5's issuer and epilogue group do nothing and conv4's epilogue writes no map
rows.  The protocol must still run to the end, every wait in the phase it means: single CTAs with the launcher's 8
stages, CTA pairs with 16, at batch 1 (an odd column count: rank 1's last column is a phantom), 16 and 64 at 416^2.
"""
import os
import sys

import pytest

from test_rdb_pair_schedule import pair_grid, pair_pieces
from test_rdb_schedule import cta_pieces, tiles_x

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
from rdb_protocol_sim import simulate, simulate_pair  # noqa: E402

NL, G = 2, 4
CASES = [(1, 416, 416), (16, 416, 416), (64, 416, 416), (3, 8, 200), (2, 18, 64)]


@pytest.mark.parametrize("batch,height,width", CASES)
def test_conv4_only_single_cta_protocol(batch, height, width):
    band_h = height // 2
    grid = min(148, batch * tiles_x(width, NL) * band_h)
    for cta in sorted(set([0, 1, grid // 2, grid - 1])):
        ok, info = simulate(NL, G, cta_pieces(cta, grid, batch, band_h, width, NL), 8, first_only=True)
        assert ok, (cta, info)


@pytest.mark.parametrize("batch,height,width", CASES)
def test_conv4_only_pair_protocol(batch, height, width):
    band_h = height // 2
    grid = pair_grid(batch, band_h, width, NL)
    pairs = grid // 2
    for u in sorted(set([0, 1, pairs // 2, pairs - 1])):
        pcs = [pair_pieces(2 * u + rank, grid, batch, band_h, width, NL) for rank in (0, 1)]
        ok, info = simulate_pair(G, pcs, 16, first_only=True)
        assert ok, (u, info)


def test_batch_one_pairs_have_a_phantom_column():
    grid = pair_grid(1, 208, 416, NL)
    last = pair_pieces(grid - 1, grid, 1, 208, 416, NL)
    assert any(pc["phantom"] for pc in last)
