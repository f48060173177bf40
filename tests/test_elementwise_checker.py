"""CPU: the per-element checker of tests/helpers.py (`assert_bf16_elementwise`) and its constants.  Correctly rounded
results -- float64 references rounded the way the kernels round -- must pass; each of the local faults a fused or
tiled kernel can make must fail, although every one of them moves the whole-tensor relative L2 by less than the
4e-3 / 6e-3 bars of whole-tensor checks.  These tests fix the constants (helpers.C_*) that the GPU tests use."""
import pytest
import torch
import torch.nn.functional as F

from helpers import C_FIRST, C_LAST, C_TC, REL_LAST, abs_conv, assert_bf16_elementwise, ref_conv, rel_l2, ulp_bf16


def _bf16(t):
    """fp32 result -> bf16, round to nearest even (the kernels' epilogue store)."""
    return t.float().to(torch.bfloat16).double()


@pytest.fixture(scope="module")
def layer():
    """A Cin-128 dense-block layer (conv4) on a 2-tile, 2-band image: bf16 operands, float64 reference."""
    g = torch.Generator().manual_seed(1)
    x = torch.randn(1, 128, 40, 130, generator=g).to(torch.bfloat16).double()
    w = (torch.randn(32, 128, 3, 3, generator=g) * 0.05).to(torch.bfloat16).double()
    b = torch.randn(32, generator=g) * 0.1
    ref = F.leaky_relu(ref_conv(x, w, b), 0.2)
    return x, w, b, ref, abs_conv(x, w, b)


def _mutant(x, w, b):
    return _bf16(F.leaky_relu(ref_conv(x, w, b), 0.2))


def test_checker_accepts_correctly_rounded_layers(layer):
    x, w, b, ref, S = layer
    r = assert_bf16_elementwise(_bf16(ref), ref, S, C_TC, what="f64 rounded to bf16")
    # fp32 accumulation in another order (CPU conv2d), then the bf16 store
    f32 = _bf16(F.leaky_relu(F.conv2d(x.float(), w.float(), b.float(), padding=1), 0.2))
    r32 = assert_bf16_elementwise(f32, ref, S, C_TC, what="fp32 accumulation")
    print(f"correct rounding: max |err|/bound {r:.3f}, fp32 accumulation {r32:.3f}")
    assert r <= 0.5 + 1e-9  # half an ulp of rounding, the other half and c*S are margin


def test_checker_accepts_block_output_with_residuals(layer):
    """conv5 of the RRDB-closing block: s0 * (conv + b) + s1 * x0 + s2 * xr, fp32 epilogue, one bf16 store."""
    x, w, b, _, _ = layer
    g = torch.Generator().manual_seed(2)
    x0 = torch.randn(1, 32, 40, 130, generator=g).to(torch.bfloat16).double()
    xr = torch.randn(1, 32, 40, 130, generator=g).to(torch.bfloat16).double()
    for s0, s1, s2 in ((0.2, 1.0, 0.0), (0.04, 0.2, 1.0)):
        ref = s0 * ref_conv(x, w, b) + s1 * x0 + s2 * xr
        acc = F.conv2d(x.float(), w.float(), b.float(), padding=1)
        got = _bf16(s0 * acc + s1 * x0.float() + s2 * xr.float())
        assert_bf16_elementwise(got, ref, abs_conv(x, w, b), C_TC, lip=s0, what=f"s0 {s0}")


def test_checker_reports_the_worst_element(layer):
    x, w, b, ref, S = layer
    got = _bf16(ref)
    got[0, 5, 17, 99] += 0.5
    with pytest.raises(AssertionError, match=r"1 of .* worst at \(b, y, x, c\) = \(0, 17, 99, 5\)"):
        assert_bf16_elementwise(got, ref, S, C_TC, what="planted")
    got[0, 5, 17, 99] = float("nan")
    with pytest.raises(AssertionError, match=r"\(0, 17, 99, 5\)"):
        assert_bf16_elementwise(got, ref, S, C_TC, what="nan")


def _rejected(got, ref, S, c, **kw):
    """The checker must fail; returns (max |err|/bound, message)."""
    with pytest.raises(AssertionError) as e:
        assert_bf16_elementwise(got, ref, S, c, **kw)
    msg = str(e.value)
    rmax = float(msg.rsplit("= ", 1)[1])
    return rmax, msg


def test_rejects_missing_chunk_tap_in_a_seam_column(layer):
    """One 32-channel K chunk's dx = -1 tap missing in column 61 (the first column of `<1,3>`'s second tile)."""
    x, w, b, ref, S = layer
    wm = w.clone()
    wm[:, 32:64, :, 0] = 0
    got = _bf16(ref)
    got[..., 61] = _mutant(x, wm, b)[..., 61]
    col = (got[..., 61] - ref[..., 61]).abs() / (ulp_bf16(ref[..., 61]) + C_TC * S[..., 61])
    rmax, _ = _rejected(got, ref, S, C_TC, what="chunk tap")
    print(f"chunk-tap mutation: max ratio {rmax:.1f}, {100 * float((col > 1).double().mean()):.0f} % of the column over, "
          f"rel-L2 {rel_l2(got, ref):.1e}")
    assert float((col > 1).double().mean()) > 0.9


def test_rejects_zero_halo_row_at_the_band_seam(layer):
    """Row H/2 - 1 computed with its halo row H/2 (the other band's first row) read as zero."""
    x, w, b, ref, S = layer
    h2 = x.shape[2] // 2
    xz = x.clone()
    xz[:, :, h2] = 0
    got = _bf16(ref)
    got[:, :, h2 - 1] = _mutant(xz, w, b)[:, :, h2 - 1]
    rmax, _ = _rejected(got, ref, S, C_TC, what="halo row")
    print(f"halo-row mutation: max ratio {rmax:.1f}, rel-L2 {rel_l2(got, ref):.1e}")


def test_rejects_one_pixel_shift_of_a_k_chunk_in_one_tile(layer):
    """Channels 64..95 read one pixel to the right in the tile of columns 61..119, rows 0..19 only."""
    x, w, b, ref, S = layer
    xs = x.clone()
    xs[:, 64:96] = torch.roll(x[:, 64:96], -1, dims=3)
    got = _bf16(ref)
    got[:, :, :20, 61:120] = _mutant(xs, w, b)[:, :, :20, 61:120]
    rmax, _ = _rejected(got, ref, S, C_TC, what="chunk shift")
    print(f"K-chunk shift mutation: max ratio {rmax:.1f}, rel-L2 {rel_l2(got, ref):.1e}")


@pytest.mark.parametrize("nf", [32, 64])
def test_conv_last_split_weights_pass_and_hi_half_alone_fails(nf):
    """conv_last on the tensor cores: fp32 weights as bf16 hi + lo halves against the fp32-weight reference (fp32
    output, so fp32's ulp).  hi + lo passes; hi alone fails per element and on rel-L2."""
    g = torch.Generator().manual_seed(nf)
    x = torch.randn(2, nf, 64, 48, generator=g).to(torch.bfloat16).double()
    w = torch.randn(3, nf, 3, 3, generator=g) * 0.05
    b = torch.randn(3, generator=g) * 0.1
    ref, S = ref_conv(x, w, b), abs_conv(x, w, b)
    hi = w.to(torch.bfloat16).float()
    lo = (w - hi).to(torch.bfloat16).float()
    split = ref_conv(x, hi.double() + lo.double(), b).float()
    r = assert_bf16_elementwise(split, ref, S, C_LAST, mant_bits=23, what="hi + lo")
    rl = rel_l2(split, ref)
    hi_only = ref_conv(x, hi, b).float()
    rmax, _ = _rejected(hi_only, ref, S, C_LAST, mant_bits=23, what="hi only")
    print(f"conv_last F={nf}: hi+lo max ratio {r:.3f} rel-L2 {rl:.1e}; hi only max ratio {rmax:.1f} "
          f"rel-L2 {rel_l2(hi_only, ref):.1e}")
    assert rl < REL_LAST < rel_l2(hi_only, ref)


@pytest.mark.parametrize("cin", [1, 4])
def test_conv_first_fp32_weights_pass_and_bf16_weights_fail(cin):
    """conv_first: fp32 image, fp32 weights, <= 36 fp32 FMAs, one bf16 store (c = 2^-18); bf16-rounded weights fail."""
    g = torch.Generator().manual_seed(cin)
    x = torch.rand(2, cin, 37, 29, generator=g) * 2 - 0.5
    w = torch.randn(32, cin, 3, 3, generator=g) * 0.3
    b = torch.randn(32, generator=g) * 0.1
    ref, S = ref_conv(x, w, b), abs_conv(x, w, b)
    r = assert_bf16_elementwise(_bf16(F.conv2d(x, w, b, padding=1)), ref, S, C_FIRST, what="fp32 weights")
    bad = _bf16(F.conv2d(x, w.to(torch.bfloat16).float(), b, padding=1))
    rmax, _ = _rejected(bad, ref, S, C_FIRST, what="bf16 weights")
    print(f"conv_first cin={cin}: fp32 weights max ratio {r:.3f}; bf16 weights max ratio {rmax:.1f}")
