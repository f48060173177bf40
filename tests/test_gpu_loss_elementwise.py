"""The loss kernels (csrc/loss_kernels.cuh) element by element, each stage on inputs the test controls or has read
back from the stage before it, so that a bound covers one stage and errors do not compound.  The kernels are called
through _lib with the parameter structs, stream and buffers loss._SsimPipeline and CompositeLoss use; where a stage
reads a ScaleStats record, kimg, maps, coarse or acc, the test passes its own.

Bits are claimed only where they follow from the arithmetic: min / max, tie counts, c1 / c2, the 2x2 pooling, the sums
of small integers, and ssim_grad_kernel on a dyadic window.  Everything else is held to a bound: first-order rounding
bounds from float64 autograd for the SSIM formulas (helpers.ssim_terms_bounded), gamma_k bounds for the sums and
correlations, and the CUDA documentation's ulp figures for logf (1) and powf (4).  On the dyadic window (taps k / 32
from {1, 2} / 32, asymmetric, summing to 33 / 32) and small-integer images, every window moment and vpp_raw, vpt, up,
lo, lum_n and lum_d are exact in fp32, so a dropped tap, a wrong halo, a flipped window or a misplaced tile is an
integer-sized error; the host tests here check that premise.  Every GPU case prints its largest |err| / bound."""
import ctypes
import math

import numpy as np
import pytest
import torch

from helpers import (DYADIC_C1, DYADIC_C2, DYADIC_TAPS, MOMENT_GAMMA, STAT_FIELDS, U32, assert_within,
                     dyadic_grad_fields, dyadic_stats_fields, gamma32, ssim_acc_bounded, ssim_grad_bounded,
                     ssim_maps_bounded, ssim_moments, ssim_terms, stats_record)

K1, K2 = 0.01, 0.05
EXACT = 2 ** 24
LOSS_BLOCKS = 592
EPS = float(np.float32(1e-8))


@pytest.fixture(scope="module")
def dev():
    from xmm_superres_denoise_b200 import _lib

    _lib.check(_lib.load().xmm_check_device())
    return torch.device("cuda:0")


def _report(what, r):
    print(f"{what}: max |err|/bound = {r:.3f}")
    return r


def _call(name, *args):
    from xmm_superres_denoise_b200 import _lib

    _lib.check(getattr(_lib.load(), name)(*args, _lib.stream_ptr()))


def _nan(*shape, dev):
    return torch.full(shape, float("nan"), dtype=torch.float32, device=dev)


def _ptr(x):
    return x.data_ptr() if x is not None else None


# ------------------------------------------------------------------------------------------------ kernel launchers
def _ssim_stats(p, t, st, win, use_sim, kimg=None):
    """xmm_ssim_stats on [N, H, W] images: forward (kimg None) -> acc [N, tiles, 4]; backward -> maps [3, N, vh, vw]."""
    from xmm_superres_denoise_b200 import _lib

    n, h, w = p.shape
    sp = _lib.SsimStatsParams()
    sp.preds, sp.target, sp.nimg, sp.h, sp.w = p.data_ptr(), t.data_ptr(), n, h, w
    sp.stats_dev, sp.window, sp.use_sim = st.data_ptr(), (ctypes.c_float * 19)(*win), int(use_sim)
    if kimg is None:
        out = _nan(n, _lib.load().xmm_ssim_tiles(h, w), 4, dev=p.device)
        sp.acc = out.data_ptr()
    else:
        out = _nan(3, n, h - 18, w - 18, dev=p.device)
        sp.kimg, sp.ga, sp.gb, sp.gc = kimg.data_ptr(), out[0].data_ptr(), out[1].data_ptr(), out[2].data_ptr()
    _call("xmm_ssim_stats", ctypes.byref(sp))
    torch.cuda.synchronize()
    return out


def _ssim_grad(p, t, st, win, maps, coarse=None, old=None):
    """xmm_ssim_grad: grad (old given: accumulate into a copy of it; else overwrite a NaN-filled buffer)."""
    from xmm_superres_denoise_b200 import _lib

    n, h, w = p.shape
    grad = old.clone() if old is not None else _nan(n, h, w, dev=p.device)
    gp = _lib.SsimGradParams()
    gp.preds, gp.target, gp.nimg, gp.h, gp.w = p.data_ptr(), t.data_ptr(), n, h, w
    gp.stats_dev, gp.window = st.data_ptr(), (ctypes.c_float * 19)(*win)
    gp.ga, gp.gb, gp.gc = maps[0].data_ptr(), maps[1].data_ptr(), maps[2].data_ptr()
    gp.coarse, gp.grad, gp.accumulate = _ptr(coarse), grad.data_ptr(), int(old is not None)
    _call("xmm_ssim_grad", ctypes.byref(gp))
    torch.cuda.synchronize()
    return grad


def _loss_reduce(p, t, dev):
    from xmm_superres_denoise_b200 import _lib

    sums, st = _nan(8, dev=dev), torch.zeros(12, device=dev)
    ws = torch.empty(_lib.load().xmm_loss_workspace_floats(), device=dev)
    _call("xmm_loss_reduce", p.data_ptr(), t.data_ptr(), p.numel(), sums.data_ptr(), st.data_ptr(), ws.data_ptr())
    _call("xmm_ssim_prepare", p.data_ptr(), p.numel(), st.data_ptr(), K1, K2)
    torch.cuda.synchronize()
    return sums, st


def _pair(shape, seed, dev, lo=0.0, hi=1.0):
    """Detector-like pair: target with exact zeros, preds = target + noise clamped to [lo, hi] (ties at lo / hi)."""
    g = torch.Generator().manual_seed(seed)
    t = torch.rand(shape, generator=g)
    t[t < 0.3] = 0.0
    p = (t + 0.15 * torch.randn(shape, generator=g)).clamp(lo, hi)
    return p.to(dev), t.to(dev)


# ------------------------------------------------------------------------------------------------ a. reductions
REDUCE_SIZES = [1, 3, 5, 1023, 1024, 1025, 3 * LOSS_BLOCKS * 1024 + 3, 16 * 416 * 416, 16 * 832 * 832]


def _reduce_depth(n: int) -> int:
    """Rounding depth of loss_reduce_kernel's fp32 sums: 4 elements per grid-stride pass (<= 592 blocks x 1024
    elements a pass), a 5-level warp butterfly, 8 warp sums in a row; the finalize adds in double, then rounds once."""
    blocks = min(-(-n // 1024), LOSS_BLOCKS)
    passes = -(-n // (blocks * 1024))
    return 4 * passes + 5 + 8


@pytest.mark.gpu
@pytest.mark.parametrize("n", REDUCE_SIZES)
def test_loss_reduce_and_prepare(dev, n):
    """Sums within gamma_depth * sum|term| (+ per-term rounding) of float64; min / max, use_p, dr, c1, c2 and the tie
    counts bit for bit."""
    p, t = _pair(n, n, dev)
    sums, st = _loss_reduce(p, t, dev)
    s, rec = sums.cpu(), dict(zip(STAT_FIELDS, st.cpu()))
    mm = torch.stack([p.min(), p.max(), t.min(), t.max()]).cpu()
    assert torch.equal(s[3:7], mm) and torch.equal(torch.stack([rec[f] for f in STAT_FIELDS[:4]]), mm)
    rp, rt = (mm[1] - mm[0]), (mm[3] - mm[2])  # fp32 subtraction on the host: the kernel's one rounding
    use_p = 0.0 if float(rt) > float(rp) else 1.0
    dr = rp if use_p else rt
    a, b = torch.tensor(K1, dtype=torch.float32) * dr, torch.tensor(K2, dtype=torch.float32) * dr
    assert float(rec["use_p"]) == use_p and torch.equal(rec["dr"], dr)
    assert torch.equal(rec["c1"], a * a) and torch.equal(rec["c2"], b * b)
    assert float(rec["nmaxp"]) == int((p == p.max()).sum()) and float(rec["nminp"]) == int((p == p.min()).sum())
    assert float(rec["d_dr"]) == 0.0

    gam = gamma32(_reduce_depth(n))
    pd, td = p.double(), t.double()
    d = pd - td
    lg = torch.log(pd + EPS)
    poi = pd - td * lg
    worst = 0.0
    for k, (terms, per_term) in enumerate((
            (d.abs(), U32 * d.abs()),                                              # p - t rounds once
            (poi, 2 * ((3 * U32) * (td * lg).abs() + U32 * td.abs() + U32 * poi.abs())),  # logf 1 ulp, x, t*log, -
            (d * d, 2 * U32 * d * d))):                                            # d rounds, then the FMA
        ref = terms.sum()
        bound = gam * terms.abs().sum() + per_term.sum() + U32 * ref.abs() + 1e-12 * terms.abs().sum()
        worst = max(worst, assert_within(s[k], ref.cpu(), bound.cpu(), what=f"reduce n={n} sum {k}"))
    _report(f"loss_reduce n={n} (depth {_reduce_depth(n)})", worst)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [5, 1025, 3 * LOSS_BLOCKS * 1024 + 3, 16 * 416 * 416])
def test_loss_reduce_exact_on_small_integers(dev, n):
    """|p - t| and (p - t)^2 sums of integers in {0, 1, 2}: every partial sum is an integer below 2^24, so any
    summation order gives the exact sum."""
    g = torch.Generator().manual_seed(n)
    p = torch.randint(0, 3, (n,), generator=g).float()
    t = torch.randint(0, 3, (n,), generator=g).float()
    d = (p - t).double()
    assert float(d.abs().sum()) < EXACT and float((d * d).sum()) < EXACT
    sums, st = _loss_reduce(p.to(dev), t.to(dev), dev)
    assert float(sums[0]) == float(d.abs().sum()) and float(sums[2]) == float((d * d).sum())
    assert float(st[4]) == int((p == 2).sum()) and float(st[5]) == int((p == 0).sum())
    print(f"loss_reduce integers n={n}: |p-t| and (p-t)^2 sums exact")


# ------------------------------------------------------------------------------------------------ b. loss gradient
def _loss_grad_ref(p, t, coef, g, old):
    """float64 g * (a sgn(p-t) + b (1 - t / (p + 1e-8)) + c (p - t)) (+ old), and a bound of 8u of the sum of |terms|
    (p - t, the quotient, 1 - q, three products and two adds, then g) plus the accumulate add."""
    a, b, c = (float(v) for v in coef.cpu())
    pd, td = p.double(), t.double()
    d = pd - td
    q = td / (pd + EPS)
    terms = a * torch.sign(d) + b * (1.0 - q) + c * d
    ref = g * terms
    bound = 8 * U32 * abs(g) * (abs(a) + abs(b) * (1.0 + q.abs()) + (c * d).abs())
    if old is not None:
        ref = ref + old.double()
        bound = bound + 2 * U32 * (old.double().abs() + ref.abs())
    return ref, bound


@pytest.mark.gpu
@pytest.mark.parametrize("accumulate", [0, 1])
@pytest.mark.parametrize("with_gl", [False, True])
def test_loss_grad_per_element(dev, accumulate, with_gl):
    n = 1_000_003  # not a multiple of the 256-thread block
    p, t = _pair(n, 17, dev)
    p[:1000] = t[:1000]                      # p == t: sign 0
    p[1000:2000] = 0.0                       # p = 0, t > 0: t / 1e-8
    t[1000:2000] = torch.linspace(0.01, 1.0, 1000, device=dev)
    coef = torch.tensor([1.5e-3, 2.5e-4, -3.1e-2], device=dev)
    gl = torch.tensor([0.75], device=dev) if with_gl else None
    old = torch.randn(n, generator=torch.Generator(device=dev).manual_seed(3), device=dev) if accumulate else None
    grad = old.clone() if accumulate else _nan(n, dev=dev)
    _call("xmm_loss_grad", p.data_ptr(), t.data_ptr(), n, coef.data_ptr(), _ptr(gl), grad.data_ptr(), accumulate)
    torch.cuda.synchronize()
    ref, bound = _loss_grad_ref(p, t, coef, 0.75 if with_gl else 1.0, old)
    _report(f"loss_grad accumulate={accumulate} gl={'dev' if with_gl else 'null'}",
            assert_within(grad, ref, bound, what="loss_grad"))


@pytest.mark.gpu
def test_composite_l1_poisson_psnr_gradient_per_element(dev):
    """CompositeLoss's gradient for L1 + Poisson + PSNR against float64 autograd of the oracle.  PSNR's coefficient
    comes from the fp32 (p - t)^2 sum, so its term carries that sum's relative bound from test a."""
    from oracle import rrdb_oracle as O
    from xmm_superres_denoise_b200.utils.loss_functions import create_loss

    weights = {"l1": 0.3, "poisson": 0.3, "psnr": 0.4}
    p, t = _pair((2, 1, 416, 416), 21, dev, lo=0.02, hi=0.97)
    pg = p.clone().requires_grad_(True)
    create_loss(None, weights).to(dev)(preds=pg, target=t).backward()
    po = p.double().cpu().requires_grad_(True)
    O.composite_loss(po, t.double().cpu(), weights, None).backward()
    n, b = p.numel(), p.shape[0]
    d = (p.double() - t.double())
    sq = (d * d).sum()
    rel_mse = float((gamma32(_reduce_depth(n)) * sq + 2 * U32 * sq + U32 * sq) / sq) + 4 * U32
    cpsnr = 0.4 * (-20.0 / math.log(10.0)) / n / float(sq / n)
    q = t.double() / (p.double() + EPS)
    bound = 8 * U32 * (0.3 / n + 0.3 / (n * b) * (1.0 + q.abs()) + (cpsnr * d).abs()) + rel_mse * (cpsnr * d).abs()
    r = assert_within(pg.grad, po.grad.to(dev), bound, what="composite l1+poisson+psnr")
    _report(f"CompositeLoss l1+poisson+psnr gradient (psnr coefficient rel bound {rel_mse:.1e})", r)


# ------------------------------------------------------------------------------------------------ c. 2x2 pooling
@pytest.mark.gpu
@pytest.mark.parametrize("b,h,w", [(2, 832, 832), (2, 307, 333)])
def test_avgpool_pyramid_bit_equal(dev, b, h, w):
    """((a00 + a01) + a10) + a11) * 0.25 in fp32, bit for bit, over the five-scale pyramid (307x333 ends at 19x20,
    dropping an odd row or column at three of its four steps)."""
    p, t = _pair((b, h, w), h + w, dev)
    for _ in range(4):
        oh, ow = h // 2, w // 2
        po, to = _nan(b, oh, ow, dev=dev), _nan(b, oh, ow, dev=dev)
        _call("xmm_avgpool2_pair", p.data_ptr(), t.data_ptr(), po.data_ptr(), to.data_ptr(), b, h, w)
        torch.cuda.synchronize()
        for x, o in ((p, po), (t, to)):
            x = x[:, :2 * oh, :2 * ow]
            want = (((x[:, 0::2, 0::2] + x[:, 0::2, 1::2]) + x[:, 1::2, 0::2]) + x[:, 1::2, 1::2]) * 0.25
            assert torch.equal(o, want), f"avgpool {h}x{w} -> {oh}x{ow}"
        p, t, h, w = po, to, oh, ow
    print(f"avgpool pyramid ends at {h}x{w}: bits equal at every scale")


# ------------------------------------------------------------------------------------------------ d. dyadic window
DYADIC_SHAPES = [(2, 70, 100), (3, 35, 51)]


def _dyadic_record(use_p):
    return stats_record(minp=-1.0, maxp=3.0, nmaxp=4.0, nminp=4.0, c1=DYADIC_C1, c2=DYADIC_C2, use_p=use_p,
                        d_dr=1.5, dr=4.0)


def _on_grid(v, k):
    """Every element is a multiple of 2^-k below 2^(24-k) in magnitude: exact in fp32."""
    s = v.double() * 2.0 ** k
    return bool(torch.all(s == torch.round(s))) and float(s.abs().max()) < EXACT


@pytest.mark.parametrize("n,h,w", DYADIC_SHAPES)
def test_dyadic_premise(n, h, w):
    """The premise of the exact tier, checked in float64 on the fields the GPU tests use: the window is asymmetric;
    every window moment, vpp_raw, vpt, up, lo, lum_n and lum_d is on a 2^-20 grid below 2^4 (exact in fp32, and
    so is every partial sum of the 38-FMA correlations, whose |terms| sum below 2^4 on a 2^-10 grid); vpp_raw takes
    negative, zero and positive values; ssim_grad's addends sum below 2^14 on a 2^-10 grid."""
    w19 = torch.tensor(DYADIC_TAPS, dtype=torch.float64)
    assert not torch.equal(w19, w19.flip(0)) and float(w19.sum()) == 33 / 32
    p, t, _ = dyadic_stats_fields(n, h, w, n + h + w)
    mp, mt, epp, ett, ept = ssim_moments(p.double(), t.double(), DYADIC_TAPS)
    f = ssim_terms(mp, mt, epp, ett, ept, DYADIC_C1, DYADIC_C2, True, 1.0)
    vpt = ept - mp * mt
    vpp = f["vpp_raw"].clamp_min(0.0)
    vtt = (ett - mt * mt).clamp_min(0.0)
    for name, v in (("mp", mp), ("mt", mt), ("epp", epp), ("ett", ett), ("ept", ept), ("vpp_raw", f["vpp_raw"]),
                    ("vpt", vpt), ("up", 2 * vpt + DYADIC_C2), ("lo", vpp + vtt + DYADIC_C2),
                    ("lum_n", 2 * mp * mt + DYADIC_C1), ("lum_d", mp * mp + mt * mt + DYADIC_C1),
                    ("mp^2", mp * mp), ("mt^2", mt * mt), ("mp*mt", mp * mt)):
        assert _on_grid(v, 20), name
    vr = f["vpp_raw"]
    assert bool((vr < 0).any()) and bool((vr == 0).any()) and bool((vr > 0).any())
    gp, gt, maps, coarse, old = dyadic_grad_fields(n, h, w, n * h * w)
    assert int((gp == 3).sum()) == 4 and int((gp == -1).sum()) == 4
    _, bound = ssim_grad_bounded(*maps.double(), gp, gt, DYADIC_TAPS, _dyadic_record(1.0), coarse=coarse, old=old)
    addends = bound / (MOMENT_GAMMA + gamma32(8))  # >= sum of |addends| of every output
    assert float(addends.max()) * 2 ** 10 < EXACT


@pytest.mark.gpu
@pytest.mark.parametrize("use_p", [1.0, 0.0])
@pytest.mark.parametrize("n,h,w", DYADIC_SHAPES)
def test_ssim_grad_dyadic_exact(dev, n, h, w, use_p):
    """ssim_grad_kernel on the dyadic window and integer maps / coarse / starting gradient: torch.equal with float64."""
    p, t, maps, coarse, old = dyadic_grad_fields(n, h, w, n * h * w)
    st = _dyadic_record(use_p)
    ref, _ = ssim_grad_bounded(*maps.double(), p, t, DYADIC_TAPS, st, coarse=coarse, old=old)
    got = _ssim_grad(p.to(dev), t.to(dev), st.to(dev), DYADIC_TAPS, maps.to(dev), coarse.to(dev), old.to(dev))
    bad = (got.cpu().double() != ref)
    assert not bool(bad.any()), f"ssim_grad dyadic {n}x{h}x{w}: {int(bad.sum())} elements differ, first at " \
                                f"{tuple(int(i) for i in bad.nonzero()[0])}"
    print(f"ssim_grad dyadic {n}x{h}x{w} use_p={use_p:g}: bits equal")


@pytest.mark.gpu
@pytest.mark.parametrize("use_sim", [1, 0])
@pytest.mark.parametrize("n,h,w", DYADIC_SHAPES)
def test_ssim_stats_dyadic(dev, n, h, w, use_sim):
    """ssim_stats_kernel on exact moments: maps and tile partials within the rounding bounds of the formulas alone."""
    p, t, kimg = dyadic_stats_fields(n, h, w, n + h + w)
    st = stats_record(c1=DYADIC_C1, c2=DYADIC_C2).to(dev)
    pd, td = p.to(dev), t.to(dev)
    maps = _ssim_stats(pd, td, st, DYADIC_TAPS, use_sim, kimg.to(dev))
    acc = _ssim_stats(pd, td, st, DYADIC_TAPS, use_sim)
    want = ssim_maps_bounded(pd, td, DYADIC_TAPS, DYADIC_C1, DYADIC_C2, use_sim, kimg, moments_exact=True)
    assert want["vpp_raw"][2] is None  # exact moments: no clamp ambiguity
    worst = 0.0
    for i, name in enumerate(("ga", "gb", "gc")):
        ref, bound, _ = want[name]
        worst = max(worst, assert_within(maps[i], ref, bound, what=f"dyadic {n}x{h}x{w} {name}"))
    # the clamp branch: gb is exactly 0 where vpp_raw < 0
    assert bool((maps[1][want["vpp_raw"][0] < 0] == 0).all())
    aref, abound = ssim_acc_bounded(want)
    worst = max(worst, assert_within(acc, aref, abound, what=f"dyadic {n}x{h}x{w} acc"))
    _report(f"ssim_stats dyadic {n}x{h}x{w} use_sim={use_sim}", worst)


# ------------------------------------------------------------------------------------------------ e. finalize
BETAS = (0.0448, 0.2856, 0.3001, 0.2363, 0.1333)
# (nscales, batch, channels, gl, weight, tiles per scale, what)
FIN_CASES = [
    (1, 3, 1, None, 1.0, (40,), "ssim, image 1 negative"),
    (1, 2, 2, 0.8, 0.6, (7,), "ssim C=2"),
    (5, 4, 1, 0.8, 0.6, (96, 24, 6, 2, 1), "msssim"),
    (5, 3, 1, None, 1.0, (40, 10, 3, 2, 1), "msssim, means <= 0"),
    (5, 1, 1, 1.25, 1.0, (12, 4, 2, 1, 1), "msssim batch 1"),
    (5, 2, 2, 0.8, 0.6, (12, 4, 2, 1, 1), "msssim C=2"),
    (5, 682, 1, 0.8, 0.6, (5, 3, 2, 1, 1), "msssim 682 images (40 KB)"),
]


def _fin_acc(nscales, nimg, tiles, seed, case):
    """acc[s] [nimg, tiles, 4]: per-tile sums of 512-pixel tiles, map means in [0.3, 0.9], sensitivities ~ N(0, 50).
    "negative": image 1's map negative (passes through a 1-scale SSIM); "<= 0": image 0's mean at scale 2 exactly 0,
    image 2's at scale 1 negative (relu: its product and every dv of that image are 0)."""
    g = torch.Generator().manual_seed(seed)
    accs = []
    for s in range(nscales):
        a = torch.randn(nimg, tiles[s], 4, generator=g) * 50
        a[..., :2] = (0.3 + 0.6 * torch.rand(nimg, tiles[s], 2, generator=g)) * 512
        if "negative" in case:
            a[1, :, 0] *= -1
        if "<= 0" in case:
            if s == 2:
                a[0, :, 1] = 0.0
            if s == 1:
                a[2, :, 1] *= -1
        accs.append(a)
    return accs


@pytest.mark.gpu
@pytest.mark.parametrize("case", FIN_CASES, ids=[c[-1] for c in FIN_CASES])
def test_msssim_finalize(dev, case):
    from xmm_superres_denoise_b200 import _lib

    nscales, batch, channels, gl, weight, tiles, what = case
    nimg = batch * channels
    accs = [a.to(dev) for a in _fin_acc(nscales, nimg, tiles, nimg + nscales, what)]
    nvalid = [512 * tl for tl in tiles]
    st = torch.stack([stats_record(dr=0.9 - 0.1 * s) for s in range(nscales)]).to(dev)
    value, img_val, kimg = _nan(1, dev=dev), _nan(batch, dev=dev), _nan(nscales * nimg, dev=dev)
    gld = torch.tensor([gl], device=dev) if gl is not None else None
    fp = _lib.MsssimFinalizeParams()
    betas = BETAS if nscales > 1 else (1.0,)
    for s in range(nscales):
        fp.acc[s], fp.tiles[s], fp.nvalid[s], fp.betas[s] = accs[s].data_ptr(), tiles[s], nvalid[s], betas[s]
    fp.nscales, fp.batch, fp.channels, fp.k1, fp.k2 = nscales, batch, channels, K1, K2
    fp.stats_dev, fp.value, fp.img_val, fp.kimg = st.data_ptr(), value.data_ptr(), img_val.data_ptr(), kimg.data_ptr()
    fp.gl_dev, fp.weight = _ptr(gld), weight
    _call("xmm_msssim_finalize", ctypes.byref(fp))
    torch.cuda.synchronize()

    acc64 = [a.double().cpu() for a in accs]
    sel = [a[..., 0 if s == nscales - 1 else 1].sum(1) for s, a in enumerate(acc64)]        # [nimg] per scale
    selabs = [a[..., 0 if s == nscales - 1 else 1].abs().sum(1) for s, a in enumerate(acc64)]
    mean = torch.stack([x.view(batch, channels).sum(1) / (nvalid[s] * channels) for s, x in enumerate(sel)])
    # vsum rounds once per image, the mean once more; the double sums are exact to ~2^-50
    dmean = torch.stack([(U32 * x.view(batch, channels).abs().sum(1) + 1e-13 * a.view(batch, channels).sum(1))
                         / (nvalid[s] * channels) for s, (x, a) in enumerate(zip(sel, selabs))]) + U32 * mean.abs()
    if nscales > 1:
        amb = (mean.abs() <= 100 * dmean) & (mean != 0)
        assert not bool(amb.any()), "test data: a scale mean too close to 0 for relu to be decided"
        v = mean.clamp_min(0.0)
        prod = torch.prod(v ** torch.tensor(betas, dtype=torch.float64).view(-1, 1), 0)
        pos = v > 0
        rel = torch.where(pos, torch.tensor(betas, dtype=torch.float64).view(-1, 1) * dmean / v.clamp_min(1e-300)
                          + 9 * U32, torch.zeros_like(v))                                  # powf: 4 ulp <= 8u, * prod
        rel_prod = rel.sum(0) + U32
        dv = torch.where(pos, torch.tensor(betas, dtype=torch.float64).view(-1, 1) * prod / v.clamp_min(1e-300),
                         torch.zeros_like(v))
        rel_k = rel_prod + torch.where(pos, dmean / v.clamp_min(1e-300), torch.zeros_like(v)) + 8 * U32
    else:
        v = mean
        prod = mean[0]
        rel_prod = dmean[0] / mean[0].abs()
        dv = torch.ones_like(v)
        rel_k = torch.full_like(v, 6 * U32)
    gsc = (1.0 if gl is None else float(np.float32(gl))) * float(np.float32(weight)) / batch
    kref = (gsc * dv / (torch.tensor(nvalid, dtype=torch.float64).view(-1, 1) * channels))   # [nscales, batch]
    kref = kref.repeat_interleave(channels, 1).reshape(-1)
    kbound = (kref.abs() * rel_k.repeat_interleave(channels, 1).reshape(-1))
    worst = assert_within(img_val.cpu(), prod, rel_prod * prod.abs(), what=f"finalize {what} img_val")
    worst = max(worst, assert_within(kimg.cpu(), kref, kbound, what=f"finalize {what} kimg"))
    iv = img_val.double().cpu()
    worst = max(worst, assert_within(value.cpu()[0], iv.mean(), U32 * iv.mean().abs() + 1e-13 * iv.abs().mean(),
                                     what=f"finalize {what} value"))
    # d_dr from the kernel's own kimg: p1 / p2 round once per image, the final value once
    k = kimg.double().cpu().view(nscales, nimg)
    stc = st.cpu()
    for s in range(nscales):
        s1, s2 = acc64[s][..., 2].sum(1), acc64[s][..., 3].sum(1)
        dr = float(stc[s, 6])
        f1, f2 = 2 * float(np.float32(K1)) ** 2 * dr, 2 * float(np.float32(K2)) ** 2 * dr
        ref = (k[s] * s1).sum() * f1 + (k[s] * s2).sum() * f2
        bnd = (U32 + 1e-13) * ((k[s] * s1).abs().sum() * abs(f1) + (k[s] * s2).abs().sum() * abs(f2)) + U32 * abs(ref)
        worst = max(worst, assert_within(stc[s, 10], ref, bnd, what=f"finalize {what} d_dr[{s}]"))
        others = [i for i in range(12) if i != 10]
        assert torch.equal(stc[s, others], stats_record(dr=0.9 - 0.1 * s)[others])
    if "<= 0" in what:
        assert float(img_val[0]) == 0.0 and float(img_val[2]) == 0.0
        assert bool(torch.all(kimg.view(nscales, nimg)[:, [0, 2]] == 0))  # 0, not NaN
    if "negative" in what:
        assert float(img_val[1]) < 0
    _report(f"msssim_finalize {what}", worst)


# ------------------------------------------------------------------------------------------------ f. real window
# (b, c, h, w, nscales): the DN / SR training shapes with all five MS-SSIM scales, and the edges of the tiling
PROD_SHAPES = [
    (16, 1, 416, 416, 5),
    (16, 1, 832, 832, 5),
    (1, 1, 19, 19, 1),     # a 1x1 valid region
    (3, 1, 34, 50, 1),     # exactly one 16x32 tile
    (2, 1, 35, 51, 1),     # one more row and column: four tiles
    (2, 1, 307, 333, 5),   # last scale 19x20: a 1x2 valid region
    (2, 2, 70, 90, 1),     # two channels
]


@pytest.mark.gpu
@pytest.mark.parametrize("b,c,h,w,nscales", PROD_SHAPES)
def test_ssim_stages_real_window(dev, b, c, h, w, nscales):
    """Every scale of _SsimPipeline on the 19-tap window, from its own pooled images, stats record and kimg:
    ssim_stats' forward partials (bits equal to the pipeline's own) and backward maps under the first-order bound, and
    ssim_grad on those maps, with the coarser scale's kernel gradient as `coarse`, under its gamma bound."""
    from xmm_superres_denoise_b200 import _lib
    from xmm_superres_denoise_b200.loss import _SsimPipeline, _window

    win = list(_window())
    p, t = _pair((b, c, h, w), b * h + w, dev)
    _, stats0 = _loss_reduce(p, t, dev)
    stats0[4:6] = 0.0  # the pipeline's own xmm_ssim_prepare counts the ties of scale 0
    ws = torch.empty(_lib.load().xmm_loss_workspace_floats(), device=dev)
    pipe = _SsimPipeline(p, t, nscales, stats0, ws)
    pipe._finalize(torch.tensor([0.8], device=dev), 0.6)
    torch.cuda.synchronize()
    nimg = b * c
    coarse = None
    for s in range(nscales - 1, -1, -1):
        hs, wsz = pipe.shapes[s]
        ps, ts = pipe.p[s].reshape(nimg, hs, wsz), pipe.t[s].reshape(nimg, hs, wsz)
        st = pipe.stats[s]
        kimg = pipe.kimg[s * nimg:(s + 1) * nimg]
        rec = dict(zip(STAT_FIELDS, st.cpu().tolist()))
        use_sim = int(s == nscales - 1)
        tag = f"real window {b}x{c}x{h}x{w} scale {s} ({hs}x{wsz})"
        acc = _ssim_stats(ps, ts, st, win, use_sim)
        assert torch.equal(acc.reshape(-1), pipe.acc[s]), tag
        maps = _ssim_stats(ps, ts, st, win, use_sim, kimg)
        want = ssim_maps_bounded(ps, ts, win, rec["c1"], rec["c2"], use_sim, kimg.double())
        worst = 0.0
        for i, name in enumerate(("ga", "gb", "gc")):
            ref, bound, alt = want[name]
            worst = max(worst, assert_within(maps[i], ref, bound, alt=alt, what=f"{tag} {name}"))
        aref, abound = ssim_acc_bounded(want)
        worst = max(worst, assert_within(acc, aref, abound, what=f"{tag} acc"))
        old = torch.randn(nimg, hs, wsz, device=dev, generator=torch.Generator(device=dev).manual_seed(s)) * 1e-6 \
            if s == 0 else None
        grad = _ssim_grad(ps, ts, st, win, maps, coarse, old)
        gref, gbound = ssim_grad_bounded(*maps, ps, ts, win, st, coarse=coarse, old=old)
        worst = max(worst, assert_within(grad, gref, gbound, what=f"{tag} grad"))
        namb = 0 if want["ga"][2] is None else int((want["ga"][2][0] != want["ga"][0]).sum())
        _report(f"{tag} use_sim={use_sim}, {namb} clamp-ambiguous pixels", worst)
        coarse = grad
