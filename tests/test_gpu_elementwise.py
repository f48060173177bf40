"""GPU: the inference kernels element by element against float64 references (helpers.assert_bf16_elementwise), at the
shapes where their tiles, bands, pieces, CTA pairs and channel windows meet.  Each check feeds the reference the
operands the kernel itself read (for a fused dense block: x1..x4 as the kernel stored them), so rounding does not
compound and every element can be held to its own bound.  Every case prints its largest |err| / bound."""
import pytest
import torch
import torch.nn.functional as F

from helpers import C_FIRST, C_LAST, C_TC, REL_LAST, abs_conv, assert_bf16_elementwise, ref_conv, rel_l2, ulp_bf16
from xmm_superres_denoise_b200 import ops

pytestmark = pytest.mark.gpu

F32 = 32


@pytest.fixture(scope="module")
def dev():
    from xmm_superres_denoise_b200 import _lib

    _lib.check(_lib.load().xmm_check_device())
    return torch.device("cuda:0")


def _nchw(t):
    return t.permute(0, 3, 1, 2)


def _report(what, r):
    print(f"{what}: max |err|/bound = {r:.3f}")
    return r


def _randn(shape, dev, seed, scale=1.0):
    g = torch.Generator(device=dev).manual_seed(seed)
    return (torch.randn(shape, generator=g, device=dev) * scale)


# ------------------------------------------------------------------------------ fused dense block (conv3x3_rdb.cuh)
# Tile origins: <1,3> 0, 61, 120, ...; <4,2> 0, 62, 123, ...  Bands: rows [0, H/2) and [H/2, H).
RDB_SHAPES = [
    (1, 8, 9),         # narrower than one tile, 4-row bands
    (1, 18, 63),       # exactly one tile, odd band height 9
    (1, 16, 64),       # the second tile owns 3 px (<1,3>) / 2 px (<4,2>)
    (2, 40, 122),      # <1,3>: 2 tiles
    (2, 40, 123),      # <1,3>: 3 tiles
    (2, 40, 124),      # <4,2>: 2 tiles
    (2, 40, 125),      # <4,2>: 3 tiles
    (3, 416, 130),     # 9 columns: rank 1's phantom column
    (1, 416, 416),     # ~10 rows per CTA: piece boundaries in y throughout, band seam at 208
    (64, 416, 416),    # the benchmark's dispatch (images 0, 37, 63 checked)
]
RDB_VARIANTS = ["plain", "third", "third_alias"]  # RRDB-closing block with both residuals; r2 is the output buffer


def _rdb_weights(dev, seed):
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
    return arena, ws, bs


def _rdb_run(arena, x0, xr, variant, mode):
    f = F32
    b, h, w, _ = x0.shape
    buf = torch.full((b, h, w, 5 * f), -7.0, dtype=torch.bfloat16, device=x0.device)
    buf[..., :f] = x0
    alias = variant == "third_alias"
    nxt = xr.clone() if alias else torch.full((b, h, w, f), 5.0, dtype=torch.bfloat16, device=x0.device)
    layers = [((buf, 0, k * f, arena.ptr(f"c{k}"), 32, f, buf, k * f), dict(lrelu=0.2, wblob_row=arena.ptr(f"c{k}.row")))
              for k in range(1, 5)]
    kw = dict(s0=0.2, r1=buf, r1_coff=0, s1=1.0) if variant == "plain" else \
        dict(s0=0.04, r1=buf, r1_coff=0, s1=0.2, r2=nxt if alias else xr, r2_coff=0, s2=1.0)
    layers.append(((buf, 0, 5 * f, arena.ptr("c5"), 32, f, nxt, 0), dict(wblob_row=arena.ptr("c5.row"), **kw)))
    ops.conv3x3_chain(layers, mode)
    torch.cuda.synchronize()
    return buf, nxt


# Maps a layer reads across the band seam from the other band's recompute, not from what was stored: conv2 / conv3
# read x1 / x1..x2 (conv1..conv3 in one kernel), conv5 reads x4 (conv4..conv5); x0..x3 of conv4 come from memory.
_RECOMPUTED = {2: (1, 2), 3: (1, 3), 5: (4, 5)}


def _seam_slack(feats, wq, k, band_h):
    """Allowance for the two seam rows (H/2 - 1, H/2) of layer k: the halo row a band recomputes from the other band's
    rows gets its accumulator-slot split from the BAND-LOCAL row index mod 3 (conv3x3_rdb.cuh, "Accumulators"), so
    unless H/2 is a multiple of 3 it may differ from the stored map in the last bit.  Allow each recomputed input
    value two bf16 ulps (its own rounding plus what its recomputed inputs carried) where it enters a seam row."""
    if k not in _RECOMPUTED or band_h % 3 == 0:
        return None
    lo, hi = _RECOMPUTED[k]
    u = torch.zeros_like(feats[:, :k * F32])
    rows = slice(band_h - 1, band_h + 1)
    u[:, lo * F32:hi * F32, rows] = 2 * ulp_bf16(feats[:, lo * F32:hi * F32, rows])
    slack = F.conv2d(u, wq.double().abs(), padding=1)
    keep = torch.zeros_like(slack)
    keep[:, :, rows] = 1.0
    return slack * keep


def _rdb_check(tag, buf, out, x0, xr, ws, bs, variant):
    """x1..x4 against lrelu(conv(buf[..., :kF] as stored) + b_k); the output against s0 (conv5 + b5) + s1 x0 + s2 xr."""
    f = F32
    feats = _nchw(buf).double()
    band_h = feats.shape[2] // 2
    worst = 0.0
    for k in range(1, 6):
        xin = feats[:, :k * f]
        wq = ws[k - 1].to(torch.bfloat16)
        y, S = ref_conv(xin, wq, bs[k - 1]), abs_conv(xin, wq, bs[k - 1])
        extra = _seam_slack(feats, wq, k, band_h)
        if k < 5:
            r = assert_bf16_elementwise(feats[:, k * f:(k + 1) * f], F.leaky_relu(y, 0.2), S, C_TC, what=f"{tag} x{k}",
                                        extra=extra)
        else:
            s0, s1, s2 = (0.2, 1.0, 0.0) if variant == "plain" else (0.04, 0.2, 1.0)
            want = s0 * y + s1 * _nchw(x0).double() + s2 * _nchw(xr).double()
            r = assert_bf16_elementwise(_nchw(out), want, S, C_TC, lip=s0, what=f"{tag} out", extra=extra)
        worst = max(worst, r)
    return worst


@pytest.mark.parametrize("variant", RDB_VARIANTS)
@pytest.mark.parametrize("b,h,w", RDB_SHAPES)
def test_fused_dense_block_per_element(dev, b, h, w, variant):
    arena, ws, bs = _rdb_weights(dev, 13 * b + h + w)
    x0 = _randn((b, h, w, F32), dev, b + h + w).to(torch.bfloat16)
    xr = _randn((b, h, w, F32), dev, b + h + w + 1).to(torch.bfloat16)
    sel = [0, 37, 63] if b == 64 else list(range(b))
    checked = None
    for form, flag in (("single", ops.CHAIN_RDB_SINGLE), ("pair", ops.CHAIN_RDB_PAIR)):
        buf, out = _rdb_run(arena, x0, xr, variant, ops.CHAIN_FUSED | flag)
        assert torch.equal(buf[..., :F32], x0)  # the block's input window is read, never written
        buf, out = buf[sel], out[sel]
        if checked is not None and torch.equal(buf, checked[0]) and torch.equal(out, checked[1]):
            print(f"rdb {b}x{h}x{w} {variant} {form}: bits equal to single")  # same operands, same bound
            continue
        r = _rdb_check(f"rdb {b}x{h}x{w} {variant} {form}", buf, out, x0[sel], xr[sel], ws, bs, variant)
        _report(f"rdb {b}x{h}x{w} {variant} {form}", r)
        checked = (buf, out)


# ------------------------------------------------------------------------------ conv_last (tensor cores / CUDA cores)
def _engine(dev, kind, cin, cout, nf, seed, scale=None):
    """An RRDBEngine (nb = 1) over a generator with seeded weights; its weight arena packed on `dev`."""
    from xmm_superres_denoise_b200.engine import RRDBEngine
    from xmm_superres_denoise_b200.models import GeneratorRRDB_DN, GeneratorRRDB_SR

    torch.manual_seed(seed)
    gen = GeneratorRRDB_DN(cin, cout, nf, 1) if kind == "dn" else GeneratorRRDB_SR(cin, cout, nf, 1, num_upsample=1)
    if scale is not None:
        with torch.no_grad():
            gen.conv_last.weight.normal_(0.0, scale)
            gen.conv_last.bias.normal_(0.0, 0.1)
    gen = gen.to(dev).eval()
    eng = RRDBEngine(gen, kind)
    eng.arena.ensure(dev)
    return gen, eng


@pytest.mark.parametrize("cout", [1, 2, 3, 4])
@pytest.mark.parametrize("nf", [32, 64])
def test_conv_last_per_element(dev, nf, cout):
    """Un-clamped output (`pre`) against float64 with the fp32 weights, per element (fp32 ulp + 2^-14 S) and on
    rel-L2; `out` is clamp(pre).  Both paths; with and without the DN residual; an input channel window."""
    gen, eng = _engine(dev, "dn", 1, cout, nf, 100 * nf + cout, scale=0.05)
    wt, bias = gen.conv_last.weight, gen.conv_last.bias
    wblob = eng._last_ptr()
    assert wblob is not None
    for b, h, w, in_coff, with_res in ((3, 37, 29, 32, True), (1, 832, 832, 0, False), (1, 832, 832, 0, True)):
        x = _randn((b, h, w, nf + in_coff), dev, b + h + cout).to(torch.bfloat16)
        res = torch.rand(b, cout, h, w, device=dev, generator=torch.Generator(device=dev).manual_seed(h)) \
            if with_res else None
        xin = _nchw(x[..., in_coff:in_coff + nf]).double()
        want, S = ref_conv(xin, wt, bias), abs_conv(xin, wt, bias)
        if with_res:
            want, S = want + res.double(), S + res.double().abs()
        for path, ptr in (("tensor cores", wblob), ("cuda cores", None)):
            out = torch.full((b, cout, h, w), 9.0, device=dev)
            pre = torch.full((b, cout, h, w), 9.0, device=dev)
            ops.conv_last(x, in_coff, wt, bias, out, residual=res, pre=pre, clamp=True, wblob_ptr=ptr)
            torch.cuda.synchronize()
            tag = f"conv_last F={nf} cout={cout} {b}x{h}x{w} coff {in_coff} res {int(with_res)} {path}"
            r = assert_bf16_elementwise(pre, want, S, C_LAST, mant_bits=23, what=tag)
            rl = rel_l2(pre, want)
            _report(f"{tag} (rel-L2 {rl:.1e})", r)
            assert rl < REL_LAST, tag
            assert torch.equal(out, pre.clamp(0.0, 1.0)), tag


# ------------------------------------------------------------------------------ conv_first
@pytest.mark.parametrize("cin", [1, 2, 3, 4])
@pytest.mark.parametrize("nf", [32, 64])
def test_conv_first_per_element(dev, nf, cin):
    """fp32 NCHW image -> bf16 NHWC features in channel windows (out at 32 of 160, out2 at 64 of 160): <= 36 fp32
    FMAs and one rounding, so c = 2^-18; out2 has the bits of out; channels outside the windows stay untouched."""
    g = torch.Generator().manual_seed(nf + cin)
    wt = (torch.randn(nf, cin, 3, 3, generator=g) * 0.3).to(dev)
    bias = (torch.randn(nf, generator=g) * 0.1).to(dev)
    for b, h, w in ((3, 37, 29), (2, 416, 416)):  # 3219 pixels: not a multiple of the 128-pixel block
        x = torch.rand(b, cin, h, w, device=dev, generator=torch.Generator(device=dev).manual_seed(h)) * 2 - 0.5
        out = torch.full((b, h, w, 160), 3.0, dtype=torch.bfloat16, device=dev)
        out2 = torch.full((b, h, w, 160), -3.0, dtype=torch.bfloat16, device=dev)
        ops.conv_first(x, wt, bias, out, 32, out2=out2, out2_coff=64)
        torch.cuda.synchronize()
        tag = f"conv_first F={nf} cin={cin} {b}x{h}x{w}"
        r = assert_bf16_elementwise(_nchw(out[..., 32:32 + nf]), ref_conv(x, wt, bias), abs_conv(x, wt, bias), C_FIRST,
                                    what=tag)
        _report(tag, r)
        assert torch.equal(out2[..., 64:64 + nf], out[..., 32:32 + nf])
        assert torch.all(out[..., :32] == 3.0) and torch.all(out[..., 32 + nf:] == 3.0)
        assert torch.all(out2[..., :64] == -3.0) and torch.all(out2[..., 64 + nf:] == -3.0)


# ------------------------------------------------------------------------------ trunk / upsampling / HRconv / F=64 parts
@pytest.mark.parametrize("nf", [32, 64])
def test_engine_layers_per_element(dev, nf):
    """The remaining layers of SR-2x inference through RRDBEngine's own plans (packing, perm = 1, output-row parts),
    launched as _forward_inference_eager launches them: trunk conv (row-hop at H = 416, r1 = fea), the upsampling conv
    (PixelShuffle store, LeakyReLU 0.01; F=64: two 128-row parts into windows n0/4), HRconv at 832^2; at F=64 also
    conv5 of a dense block (Cin 320) as 32-row parts."""
    gen, eng = _engine(dev, "sr", 1, 1, nf, 7 + nf)
    b, h, w = 1, 416, 416

    def check(tag, name, conv, inp, in_coff, cin, out, want_fn, lip=1.0, **kw):
        eng._run(eng._conv(name, inp, in_coff, cin, out, 0, **kw))
        torch.cuda.synchronize()
        xin = _nchw(inp[..., in_coff:in_coff + cin]).double()
        wq = conv.weight.to(torch.bfloat16)
        y, S = ref_conv(xin, wq, conv.bias), abs_conv(xin, wq, conv.bias)
        want, S = want_fn(y, S)
        r = assert_bf16_elementwise(_nchw(out), want, S, C_TC, lip=lip, what=f"{tag} F={nf}")
        _report(f"{tag} F={nf} ({len(eng.plans[name])} launch(es))", r)

    last = _randn((b, h, w, 5 * nf), dev, 1).to(torch.bfloat16)
    fea = _randn((b, h, w, nf), dev, 2).to(torch.bfloat16)
    trunk = torch.empty(b, h, w, nf, dtype=torch.bfloat16, device=dev)
    check("trunk", "f.trunk", gen.trunk_conv, last, 0, nf, trunk, lambda y, S: (y + _nchw(fea).double(), S),
          s0=1.0, r1=fea, r1_coff=0, s1=1.0)
    up = torch.empty(b, 2 * h, 2 * w, nf, dtype=torch.bfloat16, device=dev)
    check("upsampling", "f.up0", gen.upsampling[0], trunk, 0, nf, up,
          lambda y, S: (F.pixel_shuffle(F.leaky_relu(y, 0.01), 2), F.pixel_shuffle(S, 2)), lrelu=0.01, pixel_shuffle=1)
    hr = torch.empty_like(up)
    check("HRconv", "f.hr", gen.HRconv, up, 0, nf, hr, lambda y, S: (F.leaky_relu(y, 0.2), S), lrelu=0.2)
    if nf == 64:
        rdb = gen.rrdb[0].RDB1
        out = torch.empty(b, h, w, nf, dtype=torch.bfloat16, device=dev)
        assert len(eng.plans["f.0.0.5"]) == 2
        check("dense conv5 (Cin 320)", "f.0.0.5", rdb.conv5, last, 0, 5 * nf, out,
              lambda y, S: (0.2 * y + _nchw(last[..., :nf]).double(), S), lip=0.2,
              s0=0.2, r1=last, r1_coff=0, s1=1.0)
