"""CPU: the work split of the CTA-pair form of the fused conv4 + conv5 kernel (csrc/conv3x3_rdb.cuh:
RdbSched<NL, true>), restated in Python -- no GPU.

* both CTAs of a pair take identical walks (the leader's MMAs address both CTAs' stages and map rows with one set of
  ids, so the same pieces, rows and flush steps in the same order);
* every row of every real column is stored exactly once over all pairs;
* with an odd column count rank 1's last column is a phantom that stores nothing.
"""
import pytest

from test_rdb_schedule import piece, tiles_x, walk, walk_reference


def pair_pieces(cta, grid, batch, band_h, width, nl):
    """RdbSched<NL, true>::init / get for CTA `cta` of a grid of `grid` CTAs (clusters of two: rank = cta % 2)."""
    rank, unit, nunits = cta % 2, cta // 2, grid // 2
    ntx = tiles_x(width, nl)
    ncols = batch * ntx
    total = (ncols + 1) // 2 * band_h
    t0, t1 = total * unit // nunits, total * (unit + 1) // nunits
    if t1 <= t0:
        return []
    c0 = t0 // band_h
    out = []
    for i in range((t1 - 1) // band_h - c0 + 1):
        pcol = c0 + i
        col = 2 * pcol + rank
        phantom = col >= ncols
        pc = piece(ncols - 1 if phantom else col, 0, 0, band_h, ntx, width, nl)  # (b, tile, pixels of the column)
        base = pcol * band_h
        pc["ra"], pc["rb"] = max(t0 - base, 0), min(t1 - base, band_h)
        if phantom:
            pc["own_hi"] = pc["own_lo"]
        pc["phantom"] = phantom
        out.append(pc)
    return out


def pair_grid(batch, band_h, width, nl, sms=148):
    """the launcher's grid: as many pairs as fit (74 on 148 SMs), no more than there are pair-column rows"""
    ncols = batch * tiles_x(width, nl)
    return 2 * min(sms // 2, (ncols + 1) // 2 * band_h)


CASES = [(b, h, w) for b in (1, 3, 64) for h in (8, 40, 416) for w in (416, 200)] + [(2, 18, 64), (5, 66, 130)]


@pytest.mark.parametrize("batch,height,width", CASES)
def test_both_ranks_take_identical_walks(batch, height, width):
    nl, band_h = 2, height // 2
    grid = pair_grid(batch, band_h, width, nl)
    for unit in sorted(set([0, 1, grid // 4, grid // 2 - 1])):
        p0 = pair_pieces(2 * unit, grid, batch, band_h, width, nl)
        p1 = pair_pieces(2 * unit + 1, grid, batch, band_h, width, nl)
        assert [(p["ra"], p["rb"]) for p in p0] == [(p["ra"], p["rb"]) for p in p1]
        w0, w1 = list(walk(p0, nl)), list(walk(p1, nl))
        assert w0 == w1
        assert w0 == list(walk_reference(p0, nl))


@pytest.mark.parametrize("batch,height,width", CASES)
def test_every_row_of_every_real_column_is_stored_once(batch, height, width):
    nl, band_h = 2, height // 2
    ntx = tiles_x(width, nl)
    grid = pair_grid(batch, band_h, width, nl)
    stored = {}
    for cta in range(grid):
        for pc in pair_pieces(cta, grid, batch, band_h, width, nl):
            if pc["own_hi"] <= pc["own_lo"]:
                continue
            for row in range(pc["ra"], pc["rb"]):
                key = (pc["b"], pc["t"], row)
                assert key not in stored, (key, cta, stored.get(key))
                stored[key] = cta
    assert len(stored) == batch * ntx * band_h


@pytest.mark.parametrize("batch,height,width", CASES)
def test_the_phantom_column_stores_nothing(batch, height, width):
    nl, band_h = 2, height // 2
    ncols = batch * tiles_x(width, nl)
    grid = pair_grid(batch, band_h, width, nl)
    phantoms = [(cta, pc) for cta in range(grid) for pc in pair_pieces(cta, grid, batch, band_h, width, nl) if pc["phantom"]]
    if ncols % 2 == 0:
        assert not phantoms
        return
    assert phantoms
    for cta, pc in phantoms:
        assert cta % 2 == 1  # rank 1, on the last pair-column, owning no pixel, at in-bounds coordinates
        assert pc["b"] == batch - 1 and pc["own_lo"] == pc["own_hi"] and 0 <= pc["x0"] < width


def test_batch_one_has_an_odd_column_count():
    assert tiles_x(416, 2) == 7  # batch 1 at the bench's size: 4 pair-columns, the last one half phantom
