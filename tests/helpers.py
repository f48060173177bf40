"""Shared helpers for the parity tests (tolerances are the ones BASELINE.json's north_star states)."""
from __future__ import annotations

import os

import numpy as np
import torch
import torch.nn.functional as F

# bf16 compute: per-pixel relative L2 <= 1e-2; loss / gradient relative error <= 1e-2
REL_L2_BF16 = 1e-2
GRAD_REL = 1e-2
PSNR_DELTA_DB = 0.05

# per-element bounds (assert_bf16_elementwise): c of |got - ref| <= ulp(ref) + lip * c * S, fixed by
# tests/test_elementwise_checker.py (correct rounding passes, every local fault there fails)
C_TC = 2.0 ** -16     # tensor-core 3x3 layers: bf16 operands, fp32 accumulation, bf16 output
C_LAST = 2.0 ** -14   # conv_last: fp32 output; on the tensor cores fp32 weights as bf16 hi + lo halves
C_FIRST = 2.0 ** -18  # conv_first: <= 36 fp32 FMAs, one bf16 rounding
REL_LAST = 2e-5       # rel-L2 of conv_last's un-clamped output (bf16 hi alone: 1.6e-3)


def rel_l2(a, b) -> float:
    a = torch.as_tensor(a).double().reshape(-1).cpu()
    b = torch.as_tensor(b).double().reshape(-1).cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def psnr_db(a, b, data_range: float = 1.0) -> float:
    a = torch.as_tensor(a).double().cpu()
    b = torch.as_tensor(b).double().cpu()
    mse = float(((a - b) ** 2).mean())
    return float("inf") if mse == 0 else 10.0 * np.log10(data_range ** 2 / mse)


def _f64(t, device) -> torch.Tensor:
    return torch.as_tensor(t).to(device=device, dtype=torch.float64)


def ulp_bf16(v, mant_bits: int = 7) -> torch.Tensor:
    """Unit in the last place of |v| in a format with `mant_bits` stored mantissa bits (7: bf16, 23: fp32):
    2^(floor(log2|v|) - mant_bits), floored at the smallest normal (2^-126)."""
    e = torch.floor(torch.log2(torch.as_tensor(v).double().abs().clamp_min(2.0 ** -126)))
    return torch.exp2(e - mant_bits)


def assert_bf16_elementwise(got, ref, S, c: float, lip: float = 1.0, what: str = "", mant_bits: int = 7,
                            extra=None) -> float:
    """Per-element check of a kernel's output against a float64 reference of the same operation on the same
    (bf16-exact) operands:  |got - ref| <= ulp_bf16(ref) + lip * c * S  for every element.

    S = sum |w| * |x| + |bias| (the absolute-value convolution, `abs_conv`) bounds what fp32 accumulation in any
    order can lose: c ~ 2^-16 covers the tensor-core layers, 2^-18 the 36 FMAs of conv_first.  `lip` is the
    Lipschitz factor of the epilogue after the accumulation (s0 of a residual layer).  ulp_bf16(ref) takes the final
    rounding to the output format (half an ulp) with a half-ulp margin; `mant_bits=23` makes it fp32's.  `extra`
    (same shape, optional) is an absolute allowance added to c * S, for elements whose operands the kernel may
    legitimately see differently from the reference (see test_gpu_elementwise.py's band seam).

    Tensors are 4-D [B, C, H, W] (any device; the check runs in float64 on ref's device).  On failure the message
    gives the number of violations, the worst element's (b, y, x, c), got, ref, its bound and the largest
    |err| / bound.  Returns that largest ratio, so that a test can print it."""
    ref = torch.as_tensor(ref)
    dev = ref.device
    ref, got, S = _f64(ref, dev), _f64(got, dev), _f64(S, dev)
    if got.shape != ref.shape or S.shape != ref.shape or ref.dim() != 4:
        raise ValueError(f"{what}: shapes got {tuple(got.shape)}, ref {tuple(ref.shape)}, S {tuple(S.shape)}")
    bound = ulp_bf16(ref, mant_bits) + lip * (c * S + (0.0 if extra is None else _f64(extra, dev)))
    ratio = (got - ref).abs() / bound
    ratio = torch.where(torch.isnan(ratio), torch.full_like(ratio, float("inf")), ratio)  # NaN / Inf in got fail
    worst = int(torch.argmax(ratio))
    rmax = float(ratio.reshape(-1)[worst])
    bad = int((ratio > 1.0).sum())
    if bad:
        b, ch, y, x = np.unravel_index(worst, tuple(ref.shape))
        raise AssertionError(
            f"{what}: {bad} of {ref.numel()} elements outside |got - ref| <= ulp_bf16(ref) + {lip:g} * {c:.3g} * S; "
            f"worst at (b, y, x, c) = ({b}, {y}, {x}, {ch}): got {float(got[b, ch, y, x]):.8g}, "
            f"ref {float(ref[b, ch, y, x]):.8g}, bound {float(bound[b, ch, y, x]):.3g}, max |err|/bound = {rmax:.3f}")
    return rmax


def assert_within(got, ref, bound, what: str = "", alt=None) -> float:
    """|got - ref| <= bound for every element (any shape; float64 on ref's device; NaN in got fails).  `alt` =
    (ref2, bound2): an element also passes within bound2 of ref2 (for elements where rounding may take the other
    branch of a clamp).  On failure the message gives the count, the worst index, got, ref and bound.  Returns the
    largest |err| / bound, so that a test can print it."""
    ref = torch.as_tensor(ref)
    dev = ref.device
    ref, got, bound = _f64(ref, dev), _f64(got, dev), _f64(bound, dev).expand_as(ref)
    if got.shape != ref.shape:
        raise ValueError(f"{what}: shapes got {tuple(got.shape)}, ref {tuple(ref.shape)}")
    ratio = torch.where(got == ref, torch.zeros_like(ref), (got - ref).abs() / bound)  # a 0 bound asks for bits
    if alt is not None:
        a0 = _f64(alt[0], dev)
        ratio = torch.minimum(ratio, torch.where(got == a0, torch.zeros_like(ref), (got - a0).abs() / _f64(alt[1], dev)))
    ratio = torch.where(torch.isnan(ratio), torch.full_like(ratio, float("inf")), ratio)
    worst = int(torch.argmax(ratio)) if ratio.numel() else 0
    rmax = float(ratio.reshape(-1)[worst]) if ratio.numel() else 0.0
    bad = int((ratio > 1.0).sum())
    if bad:
        idx = tuple(int(i) for i in np.unravel_index(worst, tuple(ref.shape)))
        raise AssertionError(
            f"{what}: {bad} of {ref.numel()} elements outside |got - ref| <= bound; worst at {idx}: "
            f"got {float(got.reshape(-1)[worst]):.9g}, ref {float(ref.reshape(-1)[worst]):.9g}, "
            f"bound {float(bound.reshape(-1)[worst]):.3g}, max |err|/bound = {rmax:.3f}")
    return rmax


# ---------------------------------------------------------------------------- loss kernels (csrc/loss_kernels.cuh)
# float64 references of the SSIM stages and the rounding bounds the per-element loss tests hold the kernels to
# (tests/test_gpu_loss_elementwise.py); tests/test_loss_elementwise_checker.py shows that fp32 evaluations pass and
# that local faults fail.
U32 = 2.0 ** -24      # unit roundoff of fp32
SSIM_PAD = 9
SSIM_TILE_H, SSIM_TILE_W = 16, 32
STAT_FIELDS = ("minp", "maxp", "mint", "maxt", "nmaxp", "nminp", "dr", "c1", "c2", "use_p", "d_dr", "pad")


def gamma32(k: int) -> float:
    """Relative error bound of k fp32 roundings in a chain (Higham's gamma_k)."""
    return k * U32 / (1 - k * U32)


# A 19-tap correlation in two fp32 passes is 38 FMAs, and an x * x operand adds a rounding; gamma_40 covers both.
MOMENT_GAMMA = gamma32(40)


def stats_record(**kw) -> torch.Tensor:
    """A ScaleStats record (12 floats, fields STAT_FIELDS) with the given fields, others 0."""
    return torch.tensor([float(kw.get(f, 0.0)) for f in STAT_FIELDS], dtype=torch.float32)


def ssim_corr(x, win) -> torch.Tensor:
    """The valid 19 x 19 correlation of [N, H, W] with the outer product of `win`, separably, in x's dtype."""
    w = torch.as_tensor(win, dtype=x.dtype, device=x.device)
    y = F.conv2d(x[:, None], w.view(1, 1, 1, -1))
    return F.conv2d(y, w.view(1, 1, -1, 1))[:, 0]


def ssim_corr_t(m, win) -> torch.Tensor:
    """The transpose of ssim_corr: [N, vh, vw] -> [N, vh + 18, vw + 18], out[x] = sum_v w[x - v] m[v]."""
    w = torch.as_tensor(win, dtype=m.dtype, device=m.device)
    y = F.conv_transpose2d(m[:, None], w.view(1, 1, 1, -1))
    return F.conv_transpose2d(y, w.view(1, 1, -1, 1))[:, 0]


def ssim_moments(p, t, win):
    """(mp, mt, epp, ett, ept) of ssim_stats_kernel over the valid region, in p's dtype."""
    return tuple(ssim_corr(x, win) for x in (p, t, p * p, t * t, p * t))


SSIM_OUTPUTS = ("sim", "cs", "d1", "d2", "ga", "gb", "gc", "vpp_raw")


def ssim_terms(mp, mt, epp, ett, ept, c1, c2, use_sim, kc, rnd=None, keep=None):
    """The per-pixel formulas of ssim_stats_kernel, op for op, in the dtype of the moments: the maps sim and cs, the
    c1 / c2 sensitivities d1 / d2 of the selected map, and the backward maps ga / gb / gc (kc: per-pixel kimg).
    rnd(v) marks each rounded intermediate (identity by default).  keep: the clamp gate of vpp (default
    vpp_raw >= 0)."""
    r = rnd or (lambda v: v)
    vpp_raw = r(epp - r(mp * mp))
    vtt_raw = r(ett - r(mt * mt))
    if keep is None:
        keep = vpp_raw >= 0
    zero = torch.zeros_like(mp)
    # vtt's clamp passes the derivative everywhere: rounding may put a clamped vtt_raw on either side of 0
    vpp, vtt = torch.where(keep, vpp_raw, zero), vtt_raw + (torch.clamp(vtt_raw, min=0.0) - vtt_raw).detach()
    vpt = r(ept - r(mp * mt))
    up = r(2.0 * vpt + c2)
    lo = r(r(vpp + vtt) + c2)
    lum_n = r(r(2.0 * mp * mt) + c1)
    lum_d = r(r(r(mp * mp) + r(mt * mt)) + c1)
    cs, lum = r(up / lo), r(lum_n / lum_d)
    sim = r(lum * cs)
    lo2, ld2 = r(lo * lo), r(lum_d * lum_d)
    dcs_dvpt = r(2.0 / lo)
    dcs_dvpp = torch.where(keep, r(-up / lo2), zero)
    dcs_dc2 = r(r(lo - up) / lo2)
    dlum_dmp = r(r(r(2.0 * mt * lum_d) - r(lum_n * 2.0 * mp)) / ld2)
    dlum_dc1 = r(r(lum_d - lum_n) / ld2)
    if use_sim:
        d_mp, d_vpp, d_vpt = r(dlum_dmp * cs), r(lum * dcs_dvpp), r(lum * dcs_dvpt)
        d1, d2 = r(dlum_dc1 * cs), r(lum * dcs_dc2)
    else:
        d_mp, d_vpp, d_vpt, d1, d2 = zero, dcs_dvpp, dcs_dvpt, zero, dcs_dc2
    ga = r(kc * r(r(d_mp - r(2.0 * mp * d_vpp)) - r(mt * d_vpt)))
    return dict(sim=sim, cs=cs, d1=d1, d2=d2, ga=ga, gb=r(kc * d_vpp), gc=r(kc * d_vpt), vpp_raw=vpp_raw)


def ssim_terms_bounded(p, t, win, c1, c2, use_sim, kc, moments_exact=False, keep=None):
    """float64 ssim_terms of p, t ([N, H, W]) and a first-order bound on what an fp32 evaluation can differ by, per
    output and element: twice (the moment errors, gamma_40 * W (x) |x| or 0 when `moments_exact`, plus one fp32
    rounding of every intermediate, each times |d output / d itself| from float64 autograd), plus 2u |output|.
    kc: [N] kimg.  Returns (refs, bounds), dicts keyed by SSIM_OUTPUTS."""
    p, t = p.double(), t.double()
    with torch.no_grad():
        mom = [m.detach().requires_grad_(True) for m in ssim_moments(p, t, win)]
        err = [None] * 5 if moments_exact else \
            [MOMENT_GAMMA * ssim_corr(x, [abs(float(v)) for v in win]) for x in (p.abs(), t.abs(), p * p, t * t,
                                                                                   (p * t).abs())]
    eps = []

    def rnd(v):
        e = torch.zeros_like(v, requires_grad=True)
        eps.append(e)
        return v * (1.0 + e)

    kcm = torch.as_tensor(kc, dtype=torch.float64, device=p.device).view(-1, 1, 1)
    with torch.enable_grad():
        outs = ssim_terms(*mom, float(c1), float(c2), use_sim, kcm, rnd=rnd, keep=keep)
        refs, bounds = {}, {}
        for name in SSIM_OUTPUTS:
            f = outs[name]
            if not f.requires_grad:  # a constant 0 (d1 / the ssim terms of the cs map)
                refs[name], bounds[name] = f.detach(), torch.zeros_like(f)
                continue
            gs = torch.autograd.grad(f.sum(), mom + eps, retain_graph=True, allow_unused=True)
            b = torch.zeros_like(f)
            for g, e in zip(gs[:5], err):
                if g is not None and e is not None:
                    b = b + g.abs() * e
            for g in gs[5:]:
                if g is not None:
                    b = b + U32 * g.abs()
            refs[name], bounds[name] = f.detach(), (2.0 * b + 2.0 * U32 * f.abs()).detach()
    return refs, bounds


def ssim_maps_bounded(p, t, win, c1, c2, use_sim, kc, moments_exact=False):
    """ssim_terms_bounded with the clamp ambiguity resolved: where |vpp_raw| is within its own bound, an fp32
    evaluation may take either clamp branch, so those elements also get the other branch's (ref, bound) as `alt`.
    Returns {name: (ref, bound, alt or None)}."""
    refs, bounds = ssim_terms_bounded(p, t, win, c1, c2, use_sim, kc, moments_exact)
    amb = (refs["vpp_raw"].abs() <= bounds["vpp_raw"]) & (bounds["vpp_raw"] > 0)  # an exact 0 is not ambiguous
    out = {name: (refs[name], bounds[name], None) for name in SSIM_OUTPUTS}
    if bool(amb.any()):
        r2, b2 = ssim_terms_bounded(p, t, win, c1, c2, use_sim, kc, moments_exact, keep=~(refs["vpp_raw"] >= 0))
        for name in SSIM_OUTPUTS:
            out[name] = (refs[name], bounds[name], (torch.where(amb, r2[name], refs[name]),
                                                    torch.where(amb, b2[name], bounds[name])))
    return out


def ssim_tile_sums(x) -> torch.Tensor:
    """Per-tile sums of a valid-region map [N, vh, vw] in ssim_stats_kernel's tile order: [N, tiles]."""
    n, vh, vw = x.shape
    ty, tx = -(-vh // SSIM_TILE_H), -(-vw // SSIM_TILE_W)
    x = F.pad(x, (0, tx * SSIM_TILE_W - vw, 0, ty * SSIM_TILE_H - vh))
    return x.reshape(n, ty, SSIM_TILE_H, tx, SSIM_TILE_W).sum(dim=(2, 4)).reshape(n, ty * tx)


# each thread adds 2 of a tile's 512 pixels, then a 5-level warp butterfly and 8 warp sums in a row
TILE_SUM_GAMMA = gamma32(2 + 5 + 8)


def ssim_acc_bounded(maps):
    """Reference and bound of ssim_stats_kernel's forward partials acc[N][tiles][4] = per-tile sums of sim, cs, d1,
    d2, from ssim_maps_bounded's output: the sum of the per-element bounds plus gamma_15 * sum |term|."""
    refs, bounds = [], []
    for name in ("sim", "cs", "d1", "d2"):
        ref, bound, alt = maps[name]
        if alt is not None:  # either branch: bound the partial by the larger of the two deviations
            bound = torch.maximum(bound, (alt[0] - ref).abs() + alt[1])
        refs.append(ssim_tile_sums(ref))
        bounds.append(ssim_tile_sums(bound) + TILE_SUM_GAMMA * ssim_tile_sums(ref.abs()))
    return torch.stack(refs, -1), torch.stack(bounds, -1)


def ssim_grad_bounded(ga, gb, gc, p, t, win, st, coarse=None, old=None):
    """float64 ssim_grad_kernel: the transposed correlation of the maps, the data-range term on tied max / min
    pixels (st: the stats record), 0.25 * coarse on the even rows / columns and `old` (accumulate).  Bound:
    gamma_40 * (W' |ga| + 2 |p| W' |gb| + |t| W' |gc|) for the two fp32 passes, plus gamma_8 of every |addend| for
    the roundings of the products and adds that follow.  Returns (ref, bound)."""
    ga, gb, gc, p, t = (x.double() for x in (ga, gb, gc, p, t))
    aw = [abs(float(v)) for v in win]
    g = ssim_corr_t(ga, win) + 2.0 * p * ssim_corr_t(gb, win) + t * ssim_corr_t(gc, win)
    a = ssim_corr_t(ga.abs(), aw) + 2.0 * p.abs() * ssim_corr_t(gb.abs(), aw) + t.abs() * ssim_corr_t(gc.abs(), aw)
    rest = torch.zeros_like(g)
    s = {f: float(v) for f, v in zip(STAT_FIELDS, torch.as_tensor(st).float().cpu().tolist())}
    if s["use_p"] != 0.0 and s["d_dr"] != 0.0:
        dr = (p == s["maxp"]).double() * (float(np.float32(s["d_dr"] / np.float32(s["nmaxp"])))) \
            - (p == s["minp"]).double() * (float(np.float32(s["d_dr"] / np.float32(s["nminp"]))))
        g, rest = g + dr, rest + dr.abs()
    if coarse is not None:
        c = coarse.double()
        up = 0.25 * c.repeat_interleave(2, 1).repeat_interleave(2, 2)
        cg = torch.zeros_like(g)
        cg[:, :up.shape[1], :up.shape[2]] = up
        g, rest = g + cg, rest + cg.abs()
    if old is not None:
        g, rest = g + old.double(), rest + old.double().abs()
    return g, MOMENT_GAMMA * a + gamma32(8) * (a + rest)


# {1, 2} / 32, asymmetric (tap 4 is 1, tap 14 is 2), summing to 33 / 32: the 2-D window sums to more than 1, so
# vpp_raw = S (E[p^2] - S E[p]^2) is negative on constant non-zero patches and exactly 0 on zero patches
DYADIC_TAPS = [a / 32.0 for a in (2, 1, 2, 2, 1, 2, 2, 2, 1, 2, 2, 2, 2, 1, 2, 2, 2, 1, 2)]
DYADIC_C1, DYADIC_C2 = 2.0 ** -10, 2.0 ** -6


def dyadic_stats_fields(n, h, w, seed):
    """Images in {0, 1, 2}: random, with a constant-1 band (columns < 20, preds only: vpp_raw < 0 there while the
    target's variance is positive) and a zero block in both (the last 22 columns of rows < 22: vpp_raw == 0)."""
    g = torch.Generator().manual_seed(seed)
    p = torch.randint(0, 3, (n, h, w), generator=g).float()
    t = torch.randint(0, 3, (n, h, w), generator=g).float()
    p[:, :, :20] = 1.0
    p[:, :22, -22:] = 0.0
    t[:, :22, -22:] = 0.0
    kimg = torch.tensor([0.5, -0.25, 0.75][:n])
    return p, t, kimg


def dyadic_grad_fields(n, h, w, seed):
    """ssim_grad operands: preds in {0, 1, 2} with 4 tied maxima (3) on tile seams and 4 tied minima (-1) on image
    corners, target in {0, 1, 2}, maps in [-2, 2], coarse and the starting gradient in [-4, 4]; the record's
    d_dr / 4 = 0.375 is exact."""
    g = torch.Generator().manual_seed(seed)
    p = torch.randint(0, 3, (n, h, w), generator=g).float()
    t = torch.randint(0, 3, (n, h, w), generator=g).float()
    for (i, y, x) in ((0, 15, 31), (0, 16, 32), (n - 1, min(h - 1, 31), 31), (n - 1, 16, min(w - 1, 63))):
        p[i, y, x] = 3.0
    for (i, y, x) in ((0, 0, 0), (0, h - 1, w - 1), (n - 1, 0, w - 1), (n - 1, h - 1, 0)):
        p[i, y, x] = -1.0
    maps = torch.randint(-2, 3, (3, n, h - 18, w - 18), generator=g).float()
    coarse = torch.randint(-4, 5, (n, h // 2, w // 2), generator=g).float()
    old = torch.randint(-4, 5, (n, h, w), generator=g).float()
    return p, t, maps, coarse, old


def _threads(t: torch.Tensor) -> None:
    if t.device.type == "cpu":
        torch.set_num_threads(os.cpu_count() or 1)


def ref_conv(x, w, b=None) -> torch.Tensor:
    """3x3, padding 1, in float64 on x's device: x [B, Cin, H, W], w [Cout, Cin, 3, 3], b [Cout] or None."""
    x = torch.as_tensor(x)
    _threads(x)
    dev = x.device
    return F.conv2d(_f64(x, dev), _f64(w, dev), None if b is None else _f64(b, dev), padding=1)


def abs_conv(x, w, b=None) -> torch.Tensor:
    """S of `assert_bf16_elementwise`: sum |w| * |x| + |b| over each output's window, float64."""
    x = torch.as_tensor(x)
    return ref_conv(x.abs(), torch.as_tensor(w).abs(), None if b is None else torch.as_tensor(b).abs())


def load_case(golden_dir: str, name: str):
    g = np.load(os.path.join(golden_dir, f"net_{name}.npz"))
    kind_i, nf, nb, seed, counts = (int(v) for v in g["meta"][:5])
    shape = tuple(int(v) for v in g["meta"][5:])
    return g, ("dn", "sr")[kind_i], nf, nb, seed, bool(counts), shape
