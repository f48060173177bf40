"""CPU: the SSIM references and bounds of tests/helpers.py that tests/test_gpu_loss_elementwise.py holds the loss
kernels to.  fp32 evaluations of ssim_stats / ssim_grad (separable fp32 passes, the same formulas in fp32) and
float64 values rounded once to fp32 must pass; each local fault such a tiled stencil can make must fail per element,
although most move the whole-gradient relative L2 by less than test_gpu_loss.py's 3e-3 bar (printed)."""
import pytest
import torch

from helpers import (DYADIC_C1, DYADIC_C2, DYADIC_TAPS, assert_within, dyadic_stats_fields, rel_l2, ssim_acc_bounded,
                     ssim_grad_bounded, ssim_maps_bounded, ssim_moments, ssim_terms, ssim_tile_sums,
                     stats_record)

WHOLE_TENSOR_BAR = 3e-3  # test_gpu_loss.py's relative L2 bar for SSIM / MS-SSIM gradients


@pytest.fixture(scope="module")
def case():
    """A 2 x 416 x 416 pair (test_gpu_loss.py's MS-SSIM shape; valid 398 x 398) on the real 19-tap window, kimg of a
    training step, and a coarse gradient of the fine gradient's size."""
    from xmm_superres_denoise_b200.loss import gaussian_window

    g = torch.Generator().manual_seed(7)
    t = torch.rand(2, 416, 416, generator=g)
    t[t < 0.3] = 0.0
    p = (t + 0.15 * torch.randn(2, 416, 416, generator=g)).clamp(0, 1)
    win = gaussian_window()
    c1, c2 = float(torch.tensor(0.01 ** 2)), float(torch.tensor(0.05 ** 2))
    kc = torch.tensor([3e-6, 2.5e-6])
    coarse = torch.randn(2, 208, 208, generator=g) * 1e-7
    st = stats_record(minp=float(p.min()), maxp=float(p.max()), nmaxp=float((p == p.max()).sum()),
                      nminp=float((p == p.min()).sum()), c1=c1, c2=c2, use_p=1.0, d_dr=2e-3, dr=1.0)
    maps = {use_sim: ssim_maps_bounded(p, t, win, c1, c2, use_sim, kc) for use_sim in (0, 1)}
    return dict(p=p, t=t, win=win, c1=c1, c2=c2, kc=kc, coarse=coarse, st=st, maps=maps)


def _f32_maps(p, t, win, c1, c2, use_sim, kc, keep=None):
    mom = ssim_moments(p.float(), t.float(), torch.tensor(win, dtype=torch.float32))
    return ssim_terms(*mom, c1, c2, use_sim, kc.float().view(-1, 1, 1), keep=keep)


def _f32_grad(maps, p, t, win, st, coarse=None, vwin=None):
    """ssim_grad_kernel in fp32: horizontal pass with `win`, vertical with `vwin` (default win)."""
    w = torch.tensor(win, dtype=torch.float32)
    vw = w if vwin is None else torch.tensor(vwin, dtype=torch.float32)
    s = []
    for m in maps:
        y = torch.nn.functional.conv_transpose2d(m.float()[:, None], w.view(1, 1, 1, -1))
        s.append(torch.nn.functional.conv_transpose2d(y, vw.view(1, 1, -1, 1))[:, 0])
    g = s[0] + 2.0 * p * s[1] + t * s[2]
    f = dict(zip(("minp", "maxp", "nmaxp", "nminp", "d_dr"), (float(st[i]) for i in (0, 1, 4, 5, 10))))
    g = g + (p == f["maxp"]).float() * (f["d_dr"] / f["nmaxp"]) - (p == f["minp"]).float() * (f["d_dr"] / f["nminp"])
    if coarse is not None:
        g[:, :2 * coarse.shape[1], :2 * coarse.shape[2]] += 0.25 * coarse.repeat_interleave(2, 1).repeat_interleave(2, 2)
    return g


def _check_maps(got, want, what):
    worst = 0.0
    for name in ("ga", "gb", "gc"):
        ref, bound, alt = want[name]
        worst = max(worst, assert_within(got[name], ref, bound, alt=alt, what=f"{what} {name}"))
    return worst


def test_fp32_evaluations_pass(case):
    c = case
    for use_sim in (0, 1):
        want = c["maps"][use_sim]
        got = _f32_maps(c["p"], c["t"], c["win"], c["c1"], c["c2"], use_sim, c["kc"])
        r = _check_maps(got, want, f"fp32 use_sim={use_sim}")
        r64 = _check_maps({k: want[k][0].float() for k in ("ga", "gb", "gc")}, want, "f64 rounded")
        aref, abound = ssim_acc_bounded(want)
        gacc = torch.stack([ssim_tile_sums(got[k].double()) for k in ("sim", "cs", "d1", "d2")], -1).float()
        ra = assert_within(gacc, aref, abound, what="fp32 tile sums")
        mk = [want[k][0] for k in ("ga", "gb", "gc")]
        gref, gbound = ssim_grad_bounded(*mk, c["p"], c["t"], c["win"], c["st"], coarse=c["coarse"])
        rg = assert_within(_f32_grad([m.float() for m in mk], c["p"], c["t"], c["win"], c["st"], c["coarse"]), gref,
                           gbound, what="fp32 grad")
        rg64 = assert_within(gref.float(), gref, gbound, what="f64 grad rounded")
        print(f"use_sim={use_sim}: fp32 maps {r:.3f}, f64 rounded {r64:.3f}, tile sums {ra:.3f}, fp32 grad {rg:.3f}, "
              f"f64 grad rounded {rg64:.3f}")


def _rejected(got, ref, bound, what, alt=None):
    with pytest.raises(AssertionError) as e:
        assert_within(got, ref, bound, alt=alt, what=what)
    return float(str(e.value).rsplit("= ", 1)[1])


def _grad_of(c, maps, **kw):
    return ssim_grad_bounded(*maps, c["p"], c["t"], c["win"], c["st"], coarse=c["coarse"], **kw)[0]


def _splice(good, bad, rows, cols):
    out = good.clone()
    out[:, rows, cols] = bad[:, rows, cols]
    return out


TILE1 = (slice(16, 32), slice(32, 64))  # the second tile of the second tile row


def _stats_fault(c, name):
    """Maps (use_sim 1) with one planted fault, and the reference maps."""
    want = c["maps"][1]
    good = {k: want[k][0] for k in ("ga", "gb", "gc")}
    if name == "halo column x=32 read as 0":  # tile 0 (valid x 0..31) reads input columns 0..49
        pz = c["p"].clone()
        pz[:, :, 32] = 0.0
        bad = ssim_maps_bounded(pz, c["t"], c["win"], c["c1"], c["c2"], 1, c["kc"])
        return {k: _splice(good[k], bad[k][0], slice(0, 16), slice(0, 32)) for k in good}, want
    if name == "c1 in place of c2":
        bad = ssim_maps_bounded(c["p"], c["t"], c["win"], c["c1"], c["c1"], 1, c["kc"])
        return {k: _splice(good[k], bad[k][0], *TILE1) for k in good}, want
    if name == "kimg of the neighbouring image":
        bad = {k: v.clone() for k, v in good.items()}
        for k in bad:
            bad[k][1] = good[k][1] * (c["kc"][0] / c["kc"][1])
        return bad, want
    raise KeyError(name)


@pytest.mark.parametrize("name", ["halo column x=32 read as 0", "c1 in place of c2", "kimg of the neighbouring image"])
def test_rejects_ssim_stats_faults(case, name):
    c = case
    bad, want = _stats_fault(c, name)
    worst = 0.0
    for k in ("ga", "gb", "gc"):
        ref, bound, alt = want[k]
        try:
            worst = max(worst, assert_within(bad[k], ref, bound, alt=alt))
        except AssertionError as e:
            worst = max(worst, float(str(e).rsplit("= ", 1)[1]))
    good = [want[k][0] for k in ("ga", "gb", "gc")]
    rl = rel_l2(_grad_of(c, [bad[k] for k in ("ga", "gb", "gc")]), _grad_of(c, good))
    print(f"{name}: max |err|/bound {worst:.3g}, gradient rel-L2 {rl:.1e}")
    assert worst > 1.0
    if name == "c1 in place of c2":  # the other two move a whole image or 18 columns of a tile row: printed only
        assert rl < WHOLE_TENSOR_BAR


@pytest.mark.parametrize("name", ["vertical last tap skipped in one tile", "0.25 missing from the coarse hand-back"])
def test_rejects_ssim_grad_faults(case, name):
    c = case
    want = c["maps"][1]
    mk = [want[k][0] for k in ("ga", "gb", "gc")]
    ref, bound = ssim_grad_bounded(*mk, c["p"], c["t"], c["win"], c["st"], coarse=c["coarse"])
    good = _f32_grad(mk, c["p"], c["t"], c["win"], c["st"], c["coarse"])
    if name.startswith("vertical"):
        vw = list(c["win"])
        vw[0] = 0.0  # the kernel's vertical loop reads w[18 - k]: its last step (k = 18) is w[0]
        bad = _f32_grad(mk, c["p"], c["t"], c["win"], c["st"], c["coarse"], vwin=vw)
    else:
        bad = _f32_grad(mk, c["p"], c["t"], c["win"], c["st"], 4.0 * c["coarse"])
    bad = _splice(good, bad, *TILE1)
    rmax = _rejected(bad, ref, bound, name)
    rl = rel_l2(bad, ref)
    print(f"{name}: max |err|/bound {rmax:.3g}, gradient rel-L2 {rl:.1e}")
    assert rl < WHOLE_TENSOR_BAR


def test_rejects_dyadic_window_faults():
    """On the dyadic window (exact moments, no clamp ambiguity): the window flipped in the gradient (invisible on the
    symmetric Gaussian, which is why the GPU tests use an asymmetric window) and the clamp gate taken from vtt_raw."""
    p, t, kimg = dyadic_stats_fields(2, 70, 100, 1)
    want = ssim_maps_bounded(p, t, DYADIC_TAPS, DYADIC_C1, DYADIC_C2, 1, kimg, moments_exact=True)
    mom = ssim_moments(p.float(), t.float(), torch.tensor(DYADIC_TAPS))
    keep_wrong = (mom[3] - mom[1] * mom[1]) >= 0  # vtt_raw >= 0
    bad = ssim_terms(*mom, DYADIC_C1, DYADIC_C2, 1, kimg.view(-1, 1, 1), keep=keep_wrong)
    rmax = _rejected(bad["gb"], want["gb"][0], want["gb"][1], "clamp on vtt")
    good = [want[k][0] for k in ("ga", "gb", "gc")]
    st = stats_record()
    g_good = ssim_grad_bounded(*good, p, t, DYADIC_TAPS, st)[0]
    g_bad = ssim_grad_bounded(*[bad[k] for k in ("ga", "gb", "gc")], p, t, DYADIC_TAPS, st)[0]
    print(f"clamp gate on vtt_raw: max |err|/bound {rmax:.3g}, gradient rel-L2 {rel_l2(g_bad, g_good):.1e}")
    ref, bound = ssim_grad_bounded(*good, p, t, DYADIC_TAPS, st)
    flipped = _splice(ref, ssim_grad_bounded(*good, p, t, DYADIC_TAPS[::-1], st)[0], *TILE1)
    rmax = _rejected(flipped, ref, bound, "w[18-k] for w[k]")
    print(f"window flipped in one gradient tile: max |err|/bound {rmax:.3g}, gradient rel-L2 {rel_l2(flipped, ref):.1e}")
