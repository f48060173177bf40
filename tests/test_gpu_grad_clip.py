"""GPU (B200): gradient clipping in TrainStep (``gradient_clip_val`` / ``gradient_clip_algorithm``, Lightning's).

* the norm kernel against float64 torch at sizes 1 .. 38 M (F = 64, nb = 23), over many decades, zeros, one inf and
  one NaN: rel error <= 1e-6, the coefficient within 1 ulp of torch's fp32 formula on the reference norm, repeat calls
  bit-identical;
* clipping acts: parameters and both Adam moments over three steps against float64 torch.optim.Adam fed the
  float64-clipped gradient, by norm (max_norm ~ 0.1 x the norm) and by value (a few percent clamped);
* an inactive clip is the plain step, bit for bit;
* world scaling (world forced to 2 with no collective): the norm and the clip apply to g / 2;
* accumulation: one clip per window, at its close, on the window gradient;
* cross-path: the autograd path with clip_grad_norm_ / clip_grad_value_ and torch.optim.Adam;
* determinism with clipping on: run to run, graph replay against eager, memory_efficient on against off;
* the torch-op face against the ctypes calls, bit for bit, and torch's NaN / finite pattern for an inf or NaN gradient.
"""
import pytest
import torch

from helpers import rel_l2

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    from xmm_superres_denoise_b200 import _lib

    _lib.check(_lib.load().xmm_check_device())
    return torch.device("cuda:0")


@pytest.fixture
def det_flag(monkeypatch):
    monkeypatch.delenv("XMM_DETERMINISTIC", raising=False)
    monkeypatch.delenv("XMM_TRAIN_GRAPH", raising=False)
    monkeypatch.delenv("XMM_COMM_MODE", raising=False)
    monkeypatch.setenv("CUBLAS_WORKSPACE_CONFIG", ":4096:8")
    before = torch.are_deterministic_algorithms_enabled()
    yield
    torch.use_deterministic_algorithms(before)


def _model(kind, nf, nb, dev, up=1, memeff=False, seed=31):
    from oracle import rrdb_oracle as O
    from xmm_superres_denoise_b200.models import GeneratorRRDB_DN, GeneratorRRDB_SR

    sd = O.init_state_dict(kind, 1, 1, nf, nb, up, seed=seed)
    m = GeneratorRRDB_DN(1, 1, nf, nb) if kind == "dn" else GeneratorRRDB_SR(1, 1, nf, nb, num_upsample=up)
    m.load_state_dict(sd)
    m.memory_efficient = memeff
    return m.to(dev).train()


def _loss():
    from oracle import rrdb_oracle as O
    from xmm_superres_denoise_b200.utils.loss_functions import create_loss

    return create_loss(O.sc_dict_for("sqrt"), {"l1": 0.5, "poisson": 0.5})


def _batch(b, h, w, s, seed, dev):
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(b, 1, h, w, generator=g).to(dev)
    t = (torch.rand(b, 1, h * s, w * s, generator=g) * 0.5).to(dev)
    return x, t


def _step(m, **kw):
    from xmm_superres_denoise_b200.training import TrainStep

    return TrainStep(m, _loss(), lr=1e-4, **kw)


def _param_count(kind, nf, nb):
    from xmm_superres_denoise_b200.models import GeneratorRRDB_DN, GeneratorRRDB_SR

    with torch.device("meta"):
        m = GeneratorRRDB_DN(1, 1, nf, nb) if kind == "dn" else GeneratorRRDB_SR(1, 1, nf, nb, num_upsample=1)
    return sum(p.numel() for p in m.parameters())


def _coef(out, g, scale, max_norm, dev):
    from xmm_superres_denoise_b200 import training

    ws = training.grad_norm_workspace(g.numel(), dev)
    training.grad_clip_coef(g, scale, max_norm, out, ws)


def _torch_coef(norm64, max_norm, dev):
    """clip_grad_norm_'s coefficient, as torch computes it in fp32, from a given norm."""
    total = torch.tensor(float(norm64), dtype=torch.float32, device=dev)
    return torch.clamp(max_norm / (total + 1e-6), max=1.0)


def _ulps(a, b):
    a, b = a.float().cpu(), b.float().cpu()
    if torch.equal(a, b):
        return 0
    return int((a.view(torch.int32).long() - b.view(torch.int32).long()).abs())


# ------------------------------------------------------------------------------------------------ norm kernel
@pytest.mark.parametrize("size", ["1", "255", "256", "257", "dn", "sr", "f64nb23"])
def test_norm_kernel_against_float64(dev, size):
    n = {"dn": lambda: _param_count("dn", 32, 4), "sr": lambda: _param_count("sr", 32, 4),
         "f64nb23": lambda: _param_count("dn", 64, 23)}.get(size, lambda: int(size))()
    gen = torch.Generator(device=dev).manual_seed(n)
    mag = torch.empty(n, device=dev, dtype=torch.float64).uniform_(-25.0, 15.0, generator=gen)
    sign = torch.randint(0, 2, (n,), device=dev, generator=gen) * 2 - 1
    dec = (sign * torch.pow(10.0, mag)).float()
    out = torch.empty(2, device=dev)
    for case in ("decades", "zeros", "inf", "nan"):
        g = torch.zeros(n, device=dev) if case == "zeros" else dec.clone()
        if case in ("inf", "nan"):
            g[n // 3] = float("inf") if case == "inf" else float("nan")
        ref = float(g.double().pow(2).sum().sqrt())
        for scale in (1.0, 0.5):
            want = ref * scale
            for max_norm in (0.3 * want if want > 0 and want != float("inf") else 0.5, 1e30):
                _coef(out, g, scale, max_norm, dev)
                first = out.clone()
                for _ in range(2):
                    _coef(out, g, scale, max_norm, dev)
                    assert torch.equal(out.view(torch.int32), first.view(torch.int32)), f"{case}: repeat differs"
                got_norm, got_coef = first[0], first[1]
                want_coef = _torch_coef(want, max_norm, dev)
                if case == "nan":
                    assert got_norm.isnan() and got_coef.isnan(), case
                    continue
                if case == "inf":
                    assert got_norm.isinf() and float(got_coef) == 0.0, case
                    continue
                if want == 0.0:
                    assert float(got_norm) == 0.0
                else:
                    assert abs(float(got_norm) - want) <= 1e-6 * want, f"n={n} {case}: {float(got_norm)} vs {want}"
                assert _ulps(got_coef, want_coef) <= 1, f"n={n} {case}: coef {float(got_coef)} vs {float(want_coef)}"
    print(f"n={n}: norm of the decades case {float(dec.double().norm()):.6e}")


# ------------------------------------------------------------------------------------------------ clipping acts
class _RefAdam:
    """float64 torch.optim.Adam from the TrainStep's starting parameters, fed the (clipped) gradients TrainStep saw."""

    def __init__(self, p0):
        self.p = p0.double().clone().requires_grad_(True)
        self.opt = torch.optim.Adam([self.p], lr=1e-4, betas=(0.9, 0.999))

    def step(self, g):
        self.p.grad = g.clone()
        self.opt.step()

    def state(self):
        st = self.opt.state[self.p]
        return self.p.detach(), st["exp_avg"], st["exp_avg_sq"]


def _clip64(g, algorithm, val):
    if algorithm == "value":
        return g.clamp(-val, val)
    norm = g.norm()
    return g * min(val / (float(norm) + 1e-6), 1.0), float(norm)


def _check_against_ref(ts, ref, p0, what, unclipped=None):
    p, m, v = ref.state()
    r_p = rel_l2(ts.flat - p0, p - p0.double())
    r_m = rel_l2(ts.opt.exp_avg, m)
    r_v = rel_l2(ts.opt.exp_avg_sq, v)
    print(f"{what}: parameter step rel-L2 {r_p:.2e}, exp_avg {r_m:.2e}, exp_avg_sq {r_v:.2e}")
    assert r_p < 1e-3 and r_m < 1e-3 and r_v < 1e-3, what
    if unclipped is not None:  # the clip changed what Adam saw: the unclipped reference is far off
        _, mu, vu = unclipped.state()
        far_m, far_v = rel_l2(ts.opt.exp_avg, mu), rel_l2(ts.opt.exp_avg_sq, vu)
        print(f"{what}: against the unclipped reference exp_avg {far_m:.2e}, exp_avg_sq {far_v:.2e}")
        assert far_m > 1e-2 and far_v > 1e-2, what  # ten times the bar


def _first_gradient(dev, x, t):
    ts = _step(_model("dn", 32, 1, dev))
    _, g = ts._fwd_bwd(x, t)
    return g.double().clone()


@pytest.mark.parametrize("algorithm", ["norm", "value"])
def test_clipping_acts_on_adam(dev, det_flag, algorithm):
    torch.use_deterministic_algorithms(False)
    batches = [_batch(2, 96, 80, 1, 60 + j, dev) for j in range(3)]
    g0 = [_first_gradient(dev, x, t) for x, t in batches]  # the batches' gradients differ several-fold in norm
    if algorithm == "norm":
        val = 0.1 * min(float(g.norm()) for g in g0)
    else:
        val = float(torch.quantile(g0[0].abs().float().cpu(), 0.97))
    ts = _step(_model("dn", 32, 1, dev), gradient_clip_val=val, gradient_clip_algorithm=algorithm)
    p0 = ts.flat.clone()
    ref, plain = _RefAdam(p0), _RefAdam(p0)
    for i, (x, t) in enumerate(batches):
        ts(x, t)
        g = ts.engine.last_flat_grad.double()
        if algorithm == "norm":
            gc, norm = _clip64(g, "norm", val)
            print(f"step {i}: norm {norm:.4g}, max_norm {val:.4g}")
            assert norm > 2 * val, f"step {i}: the clip barely acts"
            assert abs(float(ts.grad_norm) - norm) <= 1e-6 * norm, f"step {i}: grad_norm"
            assert ts.grad_norm.dim() == 0 and ts.grad_norm.is_cuda
        else:
            gc = _clip64(g, "value", val)
            frac = float((g.abs() > val).double().mean())
            print(f"step {i}: clip_value clamps {100 * frac:.1f} % of the elements")
            assert 0.005 < frac < 0.2
            assert ts.grad_norm is None
        ref.step(gc)
        plain.step(g)
    _check_against_ref(ts, ref, p0, f"clip by {algorithm}, three steps", unclipped=plain)


@pytest.mark.parametrize("algorithm", ["norm", "value"])
def test_inactive_clip_is_the_plain_step(dev, det_flag, algorithm):
    torch.use_deterministic_algorithms(True)
    runs = []
    for val in (None, 1e30):
        ts = _step(_model("sr", 32, 1, dev), gradient_clip_val=val, gradient_clip_algorithm=algorithm)
        for i in range(3):
            ts(*_batch(2, 96, 80, 2, 70 + i, dev))
        torch.cuda.synchronize()
        runs.append((ts.flat.clone(), ts.opt.exp_avg.clone(), ts.opt.exp_avg_sq.clone()))
        if val is not None and algorithm == "norm":
            assert float(ts.grad_norm) > 0
    for a, b, what in zip(runs[0], runs[1], ("parameters", "exp_avg", "exp_avg_sq")):
        assert torch.equal(a, b), f"{algorithm}: {what} of an inactive clip differ from the plain step"


@pytest.mark.parametrize("algorithm", ["norm", "value"])
def test_world_scaling(dev, det_flag, algorithm):
    """world = 2 without a collective: the gradient Adam sees is g / 2, and so is what gets clipped."""
    torch.use_deterministic_algorithms(False)
    x, t = _batch(2, 96, 80, 1, 61, dev)
    g0 = _first_gradient(dev, x, t) / 2
    val = 0.1 * float(g0.norm()) if algorithm == "norm" else float(torch.quantile(g0.abs().float().cpu(), 0.97))
    ts = _step(_model("dn", 32, 1, dev), gradient_clip_val=val, gradient_clip_algorithm=algorithm)
    ts.world, ts.comm_mode, ts.overlap = 2, "none", False
    p0 = ts.flat.clone()
    ref = _RefAdam(p0)
    ts(x, t)
    g = ts.engine.last_flat_grad.double() / 2
    if algorithm == "norm":
        gc, norm = _clip64(g, "norm", val)
        assert abs(float(ts.grad_norm) - norm) <= 1e-6 * norm, "grad_norm is the norm of g / 2"
    else:
        gc = _clip64(g, "value", val)
    ref.step(gc)
    _check_against_ref(ts, ref, p0, f"world 2, clip by {algorithm}")


def test_accumulation_clips_once_per_window(dev, det_flag):
    torch.use_deterministic_algorithms(False)
    k = 2
    batches = [_batch(2, 96, 80, 1, 62 + j, dev) for j in range(2 * k)]
    g0 = _first_gradient(dev, *batches[0])
    val = 0.1 * float(g0.norm())
    ts = _step(_model("dn", 32, 1, dev), accumulate_grad_batches=k, gradient_clip_val=val)
    p0 = ts.flat.clone()
    ref = _RefAdam(p0)
    for w in range(2):
        before = ts.flat.clone()
        ts(*batches[w * k])
        assert torch.equal(ts.flat, before) and ts.opt.step_count == w, "parameters moved inside a window"
        if w == 0:
            assert ts.grad_norm is None, "clipped before the first window closed"
        ts(*batches[w * k + 1])
        assert ts.opt.step_count == w + 1
        g = ts.engine.last_flat_grad.double()
        gc, norm = _clip64(g, "norm", val)
        assert abs(float(ts.grad_norm) - norm) <= 1e-6 * norm, f"window {w}: the norm of the window gradient"
        ref.step(gc)
    _check_against_ref(ts, ref, p0, "k = 2, clip by norm, two windows")


@pytest.mark.parametrize("algorithm", ["norm", "value"])
def test_matches_autograd_path_with_torch_clipping(dev, det_flag, algorithm):
    """Lightning's own path on the same batch from the same state: loss.backward() on the autograd path,
    torch.nn.utils.clip_grad_norm_ / clip_grad_value_ on the .grad views and torch.optim.Adam, against
    TrainStep(gradient_clip_val=...)."""
    torch.use_deterministic_algorithms(False)
    x, t = _batch(2, 96, 80, 1, 63, dev)
    g0 = _first_gradient(dev, x, t)
    val = 0.1 * float(g0.norm()) if algorithm == "norm" else float(torch.quantile(g0.abs().float().cpu(), 0.97))
    a = _model("dn", 32, 1, dev)
    opt = torch.optim.Adam(a.parameters(), lr=1e-4, betas=(0.9, 0.999))
    ts = _step(_model("dn", 32, 1, dev), gradient_clip_val=val, gradient_clip_algorithm=algorithm)
    p0 = ts.flat.clone()
    _loss()(preds=torch.clamp(a(x), 0, 1), target=t).backward()
    ga = torch.cat([p.grad.reshape(-1) for p in a.parameters()])
    if algorithm == "norm":
        norm_a = float(torch.nn.utils.clip_grad_norm_(a.parameters(), max_norm=val))
    else:
        torch.nn.utils.clip_grad_value_(a.parameters(), val)
    opt.step()
    ts(x, t)
    r_g = rel_l2(ts.engine.last_flat_grad, ga)
    pa = torch.cat([p.detach().reshape(-1) for p in a.parameters()])
    ma = torch.cat([opt.state[p]["exp_avg"].reshape(-1) for p in a.parameters()])
    va = torch.cat([opt.state[p]["exp_avg_sq"].reshape(-1) for p in a.parameters()])
    r_p, r_m, r_v = rel_l2(ts.flat - p0, pa - p0), rel_l2(ts.opt.exp_avg, ma), rel_l2(ts.opt.exp_avg_sq, va)
    print(f"clip by {algorithm}: TrainStep vs autograd + torch clipping + Adam: gradient {r_g:.2e}, parameter step "
          f"{r_p:.2e}, exp_avg {r_m:.2e}, exp_avg_sq {r_v:.2e}"
          + (f", grad_norm {float(ts.grad_norm):.6g} vs {norm_a:.6g}" if algorithm == "norm" else ""))
    if algorithm == "norm":
        assert abs(float(ts.grad_norm) - norm_a) <= 1e-4 * norm_a
    assert r_p < 1e-3 and r_m < 1e-3 and r_v < 1e-3


# ------------------------------------------------------------------------------------------------ determinism
def _run(dev, steps=3, use_graph=False, memeff=False, algorithm="norm"):
    ts = _step(_model("dn", 32, 1, dev, memeff=memeff), use_graph=use_graph, gradient_clip_val=1e-4,
               gradient_clip_algorithm=algorithm)
    norms = []
    for i in range(steps):
        ts(*_batch(2, 96, 80, 1, 80 + i, dev))
        if ts.grad_norm is not None:
            norms.append(ts.grad_norm.clone())
    torch.cuda.synchronize()
    return ts, (norms, ts.flat.clone(), ts.opt.exp_avg.clone(), ts.opt.exp_avg_sq.clone())


def _assert_equal(a, b, what):
    na, pa, ma, va = a
    nb, pb, mb, vb = b
    assert len(na) == len(nb) and all(torch.equal(x, y) for x, y in zip(na, nb)), f"{what}: grad_norm"
    assert torch.equal(pa, pb) and torch.equal(ma, mb) and torch.equal(va, vb), f"{what}: parameters / Adam moments"


@pytest.mark.parametrize("algorithm", ["norm", "value"])
def test_clipped_training_is_bit_reproducible(dev, det_flag, algorithm):
    torch.use_deterministic_algorithms(True)
    _, a = _run(dev, algorithm=algorithm)
    _, b = _run(dev, algorithm=algorithm)
    _assert_equal(a, b, f"clip by {algorithm}: run to run")
    if algorithm == "norm":
        assert len(a[0]) == 3 and all(float(n) > 1e-4 for n in a[0])  # every step was clipped


def test_clipped_graph_replay_matches_eager(dev, det_flag):
    torch.use_deterministic_algorithms(True)
    ts, g = _run(dev, steps=4, use_graph=True)
    assert ts._graph is not None
    _, e = _run(dev, steps=4)
    _assert_equal(g, e, "clip by norm: graph replay vs eager")


def test_clipped_memory_efficient_is_bit_equal(dev, det_flag):
    torch.use_deterministic_algorithms(True)
    _, off = _run(dev)
    _, on = _run(dev, memeff=True)
    _assert_equal(off, on, "clip by norm: memory_efficient on vs off")


# ------------------------------------------------------------------------------------------------ ops face, non-finite
def test_torch_ops_face_is_bit_equal_to_ctypes(dev):
    from xmm_superres_denoise_b200 import torch_ops, training

    ns = torch_ops.load()
    n = 100_003
    gen = torch.Generator(device=dev).manual_seed(5)
    g = torch.randn(n, device=dev, generator=gen) * 1e-3
    p = torch.randn(n, device=dev, generator=gen)
    ws = training.grad_norm_workspace(n, dev)
    out_c, out_t = torch.empty(2, device=dev), torch.empty(2, device=dev)
    training.grad_clip_coef(g, 0.5, 0.01, out_c, ws)
    ns.grad_clip_coef(g, 0.5, 0.01, out_t, ws)
    assert torch.equal(out_c, out_t) and float(out_c[1]) < 1.0
    for kw in ({"clip_coef": out_c[1:]}, {"clip_value": 2e-4}):
        opt = training.FusedAdam(p.clone(), lr=1e-3)
        q, m, v = p.clone(), torch.zeros_like(p), torch.zeros_like(p)
        for step in (1, 2):
            opt.step(g, 0.5, **kw)
            ns.adam_step_clip(q, g, m, v, 1e-3, 0.9, 0.999, 1e-8, step, 0.5, **kw)
        assert torch.equal(opt.params, q) and torch.equal(opt.exp_avg, m) and torch.equal(opt.exp_avg_sq, v), kw
    with pytest.raises(RuntimeError, match="exactly one"):
        ns.adam_step_clip(q, g, m, v, 1e-3, 0.9, 0.999, 1e-8, 3, 1.0)


@pytest.mark.parametrize("algorithm", ["norm", "value"])
@pytest.mark.parametrize("bad", ["inf", "nan"])
def test_non_finite_gradient_follows_torch(dev, algorithm, bad):
    from xmm_superres_denoise_b200 import training

    n = 4099
    gen = torch.Generator(device=dev).manual_seed(9)
    p0 = torch.randn(n, device=dev, generator=gen)
    grads = [torch.randn(n, device=dev, generator=gen) * 1e-2 for _ in range(2)]
    grads[1][n // 2] = float(bad)
    val = 0.05 if algorithm == "norm" else 5e-3
    ref = torch.nn.Parameter(p0.clone())
    opt_t = torch.optim.Adam([ref], lr=1e-3, foreach=False)
    opt = training.FusedAdam(p0.clone(), lr=1e-3)
    out, ws = torch.empty(2, device=dev), training.grad_norm_workspace(n, dev)
    for g in grads:
        ref.grad = g.clone()
        if algorithm == "norm":
            torch.nn.utils.clip_grad_norm_([ref], max_norm=val)
            training.grad_clip_coef(g, 1.0, val, out, ws)
            opt.step(g, 1.0, clip_coef=out[1:])
        else:
            torch.nn.utils.clip_grad_value_([ref], val)
            opt.step(g, 1.0, clip_value=val)
        opt_t.step()
    st = opt_t.state[ref]
    for what, got, want in (("parameters", opt.params, ref.detach()), ("exp_avg", opt.exp_avg, st["exp_avg"]),
                            ("exp_avg_sq", opt.exp_avg_sq, st["exp_avg_sq"])):
        assert torch.equal(got.isnan(), want.isnan()), f"{algorithm} {bad}: NaN pattern of {what}"
        assert torch.equal(got.isfinite(), want.isfinite()), f"{algorithm} {bad}: finite pattern of {what}"
    print(f"{algorithm} {bad}: NaN parameters {int(opt.params.isnan().sum())} of {n}")
