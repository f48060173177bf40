"""GPU: conv4 + conv5 of the fused dense block as CTA pairs (csrc/conv3x3_rdb.cuh, PAIR) against the single-CTA
kernel.  The pair only changes who issues the MMAs and where the weights sit, not the order of any sum, so every
output must have the same bits: with and without the RRDB-closing residuals, with r2 aliasing the output (as the
inference ring passes it), with and without SKIP_DEAD_STORES (x4 stored for the training backward), at odd column
counts (rank 1's phantom column), and batch invariant."""
import pytest
import torch

from xmm_superres_denoise_b200 import ops

pytestmark = pytest.mark.gpu

F32 = 32


@pytest.fixture(scope="module")
def dev():
    from xmm_superres_denoise_b200 import _lib

    _lib.check(_lib.load().xmm_check_device())
    return torch.device("cuda:0")


def _block(dev, seed):
    from xmm_superres_denoise_b200.engine import WeightArena, _Blob, _Segment

    f = F32
    g = torch.Generator().manual_seed(seed)
    ws = [(torch.randn(f, k * f, 3, 3, generator=g) * 0.05).to(dev) for k in range(1, 6)]
    bs = [(torch.randn(f, generator=g) * 0.1).to(dev) for _ in range(5)]
    arena = WeightArena()
    for k in range(1, 6):
        seg = [_Segment(ws[k - 1], k * f, 0, 0, 0, 0, k * f, 1.0)]
        arena.add(_Blob(f"c{k}", f, 32, k, seg, bs[k - 1]))
        arena.add(_Blob(f"c{k}.row", f, 32, k, seg, bs[k - 1], tap_order=1))
    arena.ensure(dev)
    return arena


def _run(arena, x0, xr, third, alias, mode):
    """One dense block; returns (feature buffer, output).  alias: r2 is the output buffer itself (holding xr)."""
    f = F32
    b, h, w, _ = x0.shape
    buf = torch.full((b, h, w, 5 * f), -7.0, dtype=torch.bfloat16, device=x0.device)
    buf[..., :f] = x0
    nxt = xr.clone() if alias else torch.full((b, h, w, f), 5.0, dtype=torch.bfloat16, device=x0.device)
    layers = [((buf, 0, k * f, arena.ptr(f"c{k}"), 32, f, buf, k * f), dict(lrelu=0.2, wblob_row=arena.ptr(f"c{k}.row")))
              for k in range(1, 5)]
    kw = dict(s0=0.04, r1=buf, r1_coff=0, s1=0.2, r2=nxt if alias else xr, r2_coff=0, s2=1.0) if third else \
        dict(s0=0.2, r1=buf, r1_coff=0, s1=1.0)
    layers.append(((buf, 0, 5 * f, arena.ptr("c5"), 32, f, nxt, 0), dict(wblob_row=arena.ptr("c5.row"), **kw)))
    ops.conv3x3_chain(layers, mode)
    torch.cuda.synchronize()
    return buf, nxt


@pytest.mark.parametrize("b,h,w,third,alias", [(1, 8, 416, True, True), (1, 416, 416, False, False),
                                               (3, 40, 200, True, False), (3, 416, 130, True, True),
                                               (3, 8, 70, False, False), (64, 40, 200, False, False),
                                               (64, 416, 416, True, True)])
def test_pair_is_bit_identical_to_single_ctas(dev, b, h, w, third, alias):
    arena = _block(dev, 11 * b + h + w)
    g = torch.Generator().manual_seed(b + h + w)
    x0 = torch.randn(b, h, w, F32, generator=g).to(torch.bfloat16).to(dev)
    xr = torch.randn(b, h, w, F32, generator=g).to(torch.bfloat16).to(dev)
    for skip in (0, ops.CHAIN_SKIP_DEAD_STORES):
        single = _run(arena, x0, xr, third, alias, ops.CHAIN_FUSED | skip | ops.CHAIN_RDB_SINGLE)
        pair = _run(arena, x0, xr, third, alias, ops.CHAIN_FUSED | skip | ops.CHAIN_RDB_PAIR)
        assert torch.equal(pair[1], single[1]), "block output"
        assert torch.equal(pair[0], single[0]), "feature maps (x4 stored unless SKIP_DEAD_STORES)"
        if skip:
            assert torch.all(pair[0][..., 4 * F32:] == -7.0)  # x4 never left the SM
        else:
            assert not torch.all(pair[0][..., 4 * F32:] == -7.0)


def test_pair_is_batch_invariant(dev):
    b, h, w = 6, 64, 200  # 24 columns; alone: 4 columns (no phantom), batches of 3 / 5: odd column counts
    arena = _block(dev, 5)
    g = torch.Generator().manual_seed(5)
    x0 = torch.randn(b, h, w, F32, generator=g).to(torch.bfloat16).to(dev)
    xr = torch.randn(b, h, w, F32, generator=g).to(torch.bfloat16).to(dev)
    mode = ops.CHAIN_FUSED | ops.CHAIN_RDB_PAIR
    full = _run(arena, x0, xr, True, True, mode)
    for sel in ([0], [4], [1, 2, 3], [0, 1, 2, 3, 5]):
        part = _run(arena, x0[sel], xr[sel], True, True, mode)
        assert torch.equal(part[0], full[0][sel]) and torch.equal(part[1], full[1][sel]), sel


def test_pair_flags_are_exclusive(dev):
    arena = _block(dev, 3)
    x0 = torch.zeros(1, 8, 16, F32, dtype=torch.bfloat16, device=dev)
    auto = _run(arena, x0, x0, False, False, ops.CHAIN_AUTO | ops.CHAIN_RDB_PAIR)
    assert torch.equal(auto[1], _run(arena, x0, x0, False, False, ops.CHAIN_FUSED | ops.CHAIN_RDB_SINGLE)[1])
    with pytest.raises(RuntimeError, match="at most one"):
        _run(arena, x0, x0, False, False, ops.CHAIN_FUSED | ops.CHAIN_RDB_PAIR | ops.CHAIN_RDB_SINGLE)
