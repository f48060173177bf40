"""GPU: conv1..conv3 of the fused dense block as CTA pairs with the x0 ring (csrc/conv3x3_rdb.cuh, kRdbXRing) against
the single-CTA kernel.  x1..x3 come from that kernel alone, so comparing them compares the two forms of it; the pair
keeps every layer's K order, so every bit must be the same.  Band heights 4, 18, 20 and 208 (H/2 a multiple of 3 or
not: the band-seam rows), odd widths, batch 1 (an odd column count: rank 1's phantom column), x4 stored or skipped,
batch invariance, and the XMM_RDB_PAIR bit mask (bit 0 conv1..conv3, bit 1 conv4..conv5)."""
import os
import subprocess
import sys

import pytest
import torch

from test_gpu_rdb_pair import F32, _block, _run
from xmm_superres_denoise_b200 import ops

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def dev():
    from xmm_superres_denoise_b200 import _lib

    _lib.check(_lib.load().xmm_check_device())
    return torch.device("cuda:0")


def _inputs(dev, b, h, w, seed):
    g = torch.Generator().manual_seed(seed)
    x0 = torch.randn(b, h, w, F32, generator=g).to(torch.bfloat16).to(dev)
    xr = torch.randn(b, h, w, F32, generator=g).to(torch.bfloat16).to(dev)
    return x0, xr


@pytest.mark.parametrize("b,h,w", [(1, 8, 416), (1, 40, 131), (1, 416, 416), (3, 8, 201), (3, 36, 64), (3, 416, 131),
                                   (64, 40, 200), (64, 416, 416)])
def test_conv1_to_conv3_pair_is_bit_identical_to_single_ctas(dev, b, h, w):
    arena = _block(dev, 7 * b + h + w)
    x0, xr = _inputs(dev, b, h, w, b * h + w)
    for skip in (0, ops.CHAIN_SKIP_DEAD_STORES):
        single = _run(arena, x0, xr, True, True, ops.CHAIN_FUSED | skip | ops.CHAIN_RDB_SINGLE)
        pair = _run(arena, x0, xr, True, True, ops.CHAIN_FUSED | skip | ops.CHAIN_RDB_PAIR)
        for k in (1, 2, 3):
            sl = slice(k * F32, (k + 1) * F32)
            assert torch.equal(pair[0][..., sl], single[0][..., sl]), f"x{k}"
            assert not torch.all(pair[0][..., sl] == -7.0), f"x{k} stored"
        assert torch.equal(pair[0], single[0]) and torch.equal(pair[1], single[1]), "x4 and the block output"


def test_conv1_to_conv3_pair_is_batch_invariant(dev):
    b, h, w = 5, 40, 131  # 10 columns; alone: 2 columns, batches of 3: an odd column count
    arena = _block(dev, 9)
    x0, xr = _inputs(dev, b, h, w, 9)
    mode = ops.CHAIN_FUSED | ops.CHAIN_RDB_PAIR
    full = _run(arena, x0, xr, True, True, mode)
    for sel in ([0], [3], [1, 2, 4], [0, 1, 2, 3]):
        part = _run(arena, x0[sel], xr[sel], True, True, mode)
        assert torch.equal(part[0], full[0][sel]) and torch.equal(part[1], full[1][sel]), sel


_MASK_SCRIPT = r"""
import sys, torch
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[1] + "/tests")
from test_gpu_rdb_pair import _block, _run
from xmm_superres_denoise_b200 import ops
dev = torch.device("cuda:0")
arena = _block(dev, 4)
g = torch.Generator().manual_seed(4)
x0 = torch.randn(3, 40, 131, 32, generator=g).to(torch.bfloat16).to(dev)
xr = torch.randn(3, 40, 131, 32, generator=g).to(torch.bfloat16).to(dev)
auto = _run(arena, x0, xr, True, True, ops.CHAIN_FUSED)
single = _run(arena, x0, xr, True, True, ops.CHAIN_FUSED | ops.CHAIN_RDB_SINGLE)
print("EQUAL" if torch.equal(auto[0], single[0]) and torch.equal(auto[1], single[1]) else "DIFFERENT")
"""


@pytest.mark.parametrize("mask", ["0", "1", "2", "3"])
def test_pair_mask_selects_the_kernels(dev, mask):
    env = dict(os.environ, XMM_RDB_PAIR=mask)
    out = subprocess.run([sys.executable, "-c", _MASK_SCRIPT, ROOT], env=env, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    assert out.stdout.strip().splitlines()[-1] == "EQUAL"
