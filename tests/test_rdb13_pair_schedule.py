"""CPU: the CTA-pair form of the fused conv1..conv3 kernel (csrc/conv3x3_rdb.cuh: RdbSched<3, true> and the x0 ring),
restated in Python -- no GPU.

* both CTAs of a pair take identical walks over three layers, and every row of every real column is stored once;
* the barrier protocol of the x0 ring (tools/rdb_protocol_sim.py, simulate_pair with nl = 3) runs to the end without
  a deadlock, every wait in the phase it means (the later layers skip the slots of a piece's edge rows) and every
  issuer finding the row it expects in its slot -- with the launcher's 11 slots and with its minimum of 4.
"""
import os
import sys

import pytest

from test_rdb_pair_schedule import pair_grid, pair_pieces
from test_rdb_schedule import tiles_x, walk, walk_reference

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
from rdb_protocol_sim import simulate_pair  # noqa: E402

NL = 3
CASES = [(b, h, w) for b in (1, 3, 64) for h in (8, 40, 416) for w in (416, 201)] + [(2, 36, 64), (5, 66, 131)]


@pytest.mark.parametrize("batch,height,width", CASES)
def test_both_ranks_take_identical_three_layer_walks(batch, height, width):
    band_h = height // 2
    grid = pair_grid(batch, band_h, width, NL)
    for unit in sorted(set([0, 1, grid // 4, grid // 2 - 1])):
        p0 = pair_pieces(2 * unit, grid, batch, band_h, width, NL)
        p1 = pair_pieces(2 * unit + 1, grid, batch, band_h, width, NL)
        assert [(p["ra"], p["rb"]) for p in p0] == [(p["ra"], p["rb"]) for p in p1]
        w0 = list(walk(p0, NL))
        assert w0 == list(walk(p1, NL)) == list(walk_reference(p0, NL))


@pytest.mark.parametrize("batch,height,width", CASES)
def test_every_row_of_every_real_column_is_stored_once(batch, height, width):
    band_h = height // 2
    grid = pair_grid(batch, band_h, width, NL)
    stored = set()
    for cta in range(grid):
        for pc in pair_pieces(cta, grid, batch, band_h, width, NL):
            if pc["own_hi"] <= pc["own_lo"]:
                assert pc["phantom"] and cta % 2 == 1
                continue
            for row in range(pc["ra"], pc["rb"]):
                key = (pc["b"], pc["t"], row)
                assert key not in stored, (key, cta)
                stored.add(key)
    assert len(stored) == batch * tiles_x(width, NL) * band_h


@pytest.mark.parametrize("batch,band_h,width,grid", [(1, 4, 416, 148), (3, 20, 201, 148), (1, 208, 416, 148),
                                                      (3, 4, 416, 4), (2, 9, 64, 26), (5, 33, 131, 12)])
@pytest.mark.parametrize("xring", [11, 4])
def test_x0_ring_protocol(batch, band_h, width, grid, xring):
    pairs = min(grid // 2, (batch * tiles_x(width, NL) + 1) // 2 * band_h)
    for u in sorted(set([0, 1, pairs // 2, pairs - 1])):
        pcs = [pair_pieces(2 * u + rank, 2 * pairs, batch, band_h, width, NL) for rank in (0, 1)]
        ok, info = simulate_pair(1, pcs, xring, nl=NL)
        assert ok, info
