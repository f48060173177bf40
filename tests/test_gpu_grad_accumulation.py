"""GPU (B200): gradient accumulation in TrainStep (``accumulate_grad_batches = k``).

* the window's flat gradient against k calls of ``(loss(model(x_j)) / k).backward()`` on the autograd path (default
  mode), and against the in-order fp32 sum of the k single-micro-batch gradients (deterministic mode: one rounding per
  add);
* one Adam step per window, against torch.optim.Adam in float64 on the accumulated gradient; no parameter changes before
  the window closes;
* k = 1 is the plain step: bit-equal, same launch count;
* bit-reproducible windows (deterministic mode): run to run, CUDA-graph replay against eager, memory_efficient on
  against off, F = 64 and SR-4x;
* the collective schedule on one GPU (world forced to 2, the all-reduce recorded): chunks only in the closing
  micro-batch, covering the buffer once in RRDB order;
* peak memory does not grow with k.
"""
import gc

import pytest
import torch

from helpers import rel_l2

pytestmark = pytest.mark.gpu

U = 2.0 ** -24  # fp32 unit roundoff


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


def _step(m, k=None, **kw):
    from xmm_superres_denoise_b200.training import TrainStep

    if k is None:
        return TrainStep(m, _loss(), lr=1e-4, **kw)
    return TrainStep(m, _loss(), lr=1e-4, accumulate_grad_batches=k, **kw)


def _scale(kind, up):
    return 1 if kind == "dn" else 2 ** up


# ------------------------------------------------------------------------------------------------ window gradient
@pytest.mark.parametrize("kind,nb", [("dn", 2), ("sr", 1)])
def test_window_gradient_matches_autograd_path(dev, det_flag, kind, nb):
    torch.use_deterministic_algorithms(False)
    k, s = 3, _scale(kind, 1)
    batches = [_batch(2, 96, 80, s, 40 + j, dev) for j in range(k)]
    ts = _step(_model(kind, 32, nb, dev), k)
    for x, t in batches:
        ts(x, t)
    got = ts.engine.last_flat_grad.clone()
    ref = _model(kind, 32, nb, dev)
    loss = _loss()
    for x, t in batches:
        (loss(preds=torch.clamp(ref(x), 0, 1), target=t) / k).backward()
    want = torch.cat([p.grad.reshape(-1) for p in ref.parameters()])
    r = rel_l2(got, want)
    print(f"{kind} nb={nb}: window gradient rel-L2 vs autograd accumulation = {r:.2e}")
    assert r <= 1e-6


@pytest.mark.parametrize("kind,nb", [("dn", 2), ("sr", 1)])
def test_deterministic_window_is_the_sum_of_its_micro_batches(dev, det_flag, kind, nb):
    """The first micro-batch writes g_1 bit for bit; every later one adds its g_j with one rounding.  The finalize and
    weight-gradient reductions fuse their scale (conv5's 0.2 / 0.04) into that add, dst + scale * s, as one FMA: it
    adds the unrounded product, which differs from the stored g_j = round(scale * s) by up to u |g_j|.  So
    |acc - sum_j g_j| <= u sum_{j >= 2} (sum_{i <= j} |g_i| + |g_j|)  (<= k u sum_j |g_j|; (k - 1) u sum_j |g_j| where
    the scale is 1)."""
    torch.use_deterministic_algorithms(True)
    k, s = 3, _scale(kind, 1)
    batches = [_batch(2, 96, 80, s, 50 + j, dev) for j in range(k)]
    ref = _step(_model(kind, 32, nb, dev), 1)
    ref._seed.fill_(1.0 / k)
    singles = [ref._fwd_bwd(x, t)[1].double() for x, t in batches]
    ts = _step(_model(kind, 32, nb, dev), k)
    ts(*batches[0])
    assert torch.equal(ts.engine.last_flat_grad.double(), singles[0])  # the first micro-batch writes, as k = 1 does
    for x, t in batches[1:]:
        ts(x, t)
    got = ts.engine.last_flat_grad.double()
    want = sum(singles)
    err = (got - want).abs()
    running = singles[0].abs()
    bound = torch.zeros_like(running)
    for g in singles[1:]:
        running = running + g.abs()
        bound += U * (running + g.abs())
    bound = bound * (1 + 2.0 ** -20) + 2.0 ** -140  # (second-order terms, subnormals)
    plain = (k - 1) * U * running + 2.0 ** -140
    ratio = float((err / bound).max())
    print(f"{kind} nb={nb}: max |acc - sum g_j| / bound = {ratio:.3f} (/ ((k - 1) u sum |g_j|) = "
          f"{float((err / plain).max()):.3f})")
    assert ratio <= 1.0


# ------------------------------------------------------------------------------------------------ optimizer step
def test_one_adam_step_per_window(dev, det_flag):
    torch.use_deterministic_algorithms(False)
    k = 3
    ts = _step(_model("dn", 32, 1, dev), k)
    p0 = ts.flat.clone()
    for j in range(k):
        assert ts.pending == j
        ts(*_batch(2, 96, 80, 1, 60 + j, dev))
        if j < k - 1:
            assert torch.equal(ts.flat, p0) and ts.opt.step_count == 0, f"parameters moved after micro-batch {j}"
    assert ts.pending == 0 and ts.opt.step_count == 1
    g = ts.engine.last_flat_grad.double()
    p = p0.double().clone().requires_grad_(True)
    opt = torch.optim.Adam([p], lr=1e-4, betas=(0.9, 0.999))
    p.grad = g.clone()
    opt.step()
    st = opt.state[p]
    r_p = rel_l2(ts.flat - p0, p.detach() - p0.double())
    r_m = rel_l2(ts.opt.exp_avg, st["exp_avg"])
    r_v = rel_l2(ts.opt.exp_avg_sq, st["exp_avg_sq"])
    print(f"one window: parameter step rel-L2 {r_p:.2e}, exp_avg {r_m:.2e}, exp_avg_sq {r_v:.2e}")
    assert r_p < 1e-3 and r_m < 1e-3 and r_v < 1e-3


def test_k1_is_the_plain_step(dev, det_flag):
    from xmm_superres_denoise_b200 import ops

    torch.use_deterministic_algorithms(True)
    runs = []
    for k in (None, 1):
        ts = _step(_model("sr", 32, 1, dev), k)
        assert ts._grad is None
        torch.cuda.synchronize()
        ops.LAUNCHES = 0
        losses, grads = [], []
        for i in range(3):
            losses.append(ts(*_batch(2, 96, 80, 2, 70 + i, dev)).clone())
            grads.append(ts.engine.last_flat_grad.clone())
        torch.cuda.synchronize()
        runs.append((ops.LAUNCHES, losses, grads, ts.flat.clone(), ts.opt.exp_avg.clone(), ts.opt.exp_avg_sq.clone()))
    a, b = runs
    assert a[0] == b[0], f"launch counts {a[0]} vs {b[0]}"
    for i in range(3):
        assert torch.equal(a[1][i], b[1][i]) and torch.equal(a[2][i], b[2][i]), i
    assert torch.equal(a[3], b[3]) and torch.equal(a[4], b[4]) and torch.equal(a[5], b[5])


# ------------------------------------------------------------------------------------------------ reproducibility
def _windows(kind, nf, nb, up, dev, k=2, windows=2, use_graph=False, memeff=False):
    ts = _step(_model(kind, nf, nb, dev, up, memeff), k, use_graph=use_graph)
    losses, grads = [], []
    for i in range(k * windows):
        losses.append(ts(*_batch(2, 96, 80, _scale(kind, up), 80 + i, dev)).clone())
        grads.append(ts.engine.last_flat_grad.clone())
    torch.cuda.synchronize()
    return ts, (losses, grads, ts.flat.clone(), ts.opt.exp_avg.clone(), ts.opt.exp_avg_sq.clone())


def _assert_equal(a, b, what):
    la, ga, pa, ma, va = a
    lb, gb, pb, mb, vb = b
    for i in range(len(la)):
        assert torch.equal(la[i], lb[i]), f"{what}: loss of micro-batch {i}"
        assert torch.equal(ga[i], gb[i]), f"{what}: flat gradient after micro-batch {i}"
    assert torch.equal(pa, pb) and torch.equal(ma, mb) and torch.equal(va, vb), f"{what}: parameters / Adam moments"


CASES = [("dn", 32, 1, 1), ("sr", 32, 1, 1), ("dn", 64, 1, 1), ("sr", 32, 1, 2)]


@pytest.mark.parametrize("kind,nf,nb,up", CASES)
def test_windows_are_bit_reproducible(dev, det_flag, kind, nf, nb, up):
    torch.use_deterministic_algorithms(True)
    _, a = _windows(kind, nf, nb, up, dev)
    _, b = _windows(kind, nf, nb, up, dev)
    _assert_equal(a, b, f"{kind} F={nf} up={up}")
    assert not torch.equal(a[1][0], a[1][1])  # the second micro-batch added something


def test_graph_replay_of_windows_matches_eager(dev, det_flag):
    torch.use_deterministic_algorithms(True)
    ts, g = _windows("dn", 32, 1, 1, dev, windows=3, use_graph=True)
    assert ts._graph is not None and len(ts._graph) == 2  # a window's first micro-batch and the later one
    _, e = _windows("dn", 32, 1, 1, dev, windows=3)
    _assert_equal(g, e, "graph replay vs eager, k = 2")


@pytest.mark.parametrize("kind,nf,up", [("dn", 32, 1), ("sr", 32, 2), ("dn", 64, 1)])
def test_memory_efficient_windows_are_bit_equal(dev, det_flag, kind, nf, up):
    torch.use_deterministic_algorithms(True)
    _, off = _windows(kind, nf, 1, up, dev)
    _, on = _windows(kind, nf, 1, up, dev, memeff=True)
    _assert_equal(off, on, f"{kind} F={nf} up={up}: memory_efficient on vs off, k = 2")


# ------------------------------------------------------------------------------------------------ collectives
@pytest.mark.parametrize("comm", ["overlap", "serial"])
def test_collective_schedule(dev, det_flag, comm):
    torch.use_deterministic_algorithms(False)
    k, nb = 3, 3
    ts = _step(_model("dn", 32, nb, dev), k, use_graph=False)
    ts.world, ts.comm_mode, ts.overlap = 2, comm, comm == "overlap"
    calls = []
    ts._allreduce_range = lambda flat, lo, hi: calls.append((ts.pending, lo, hi))
    total = ts.flat.numel()
    if comm == "overlap":  # RRDB nb-1 with the tail layers, then RRDB nb-2 .. 0, then conv_first
        los = [ts._chunks[i][0] for i in range(nb - 1, -1, -1)]
        want = list(zip(los + [0], [total] + los))
    else:
        want = [(0, total)]
    for window in range(2):
        calls.clear()
        for j in range(k):
            ts(*_batch(2, 96, 80, 1, 90 + j, dev))
        assert {c[0] for c in calls} == {k - 1}, "a collective outside the closing micro-batch"
        assert [c[1:] for c in calls] == want, window
    assert ts.opt.step_count == 2


# ------------------------------------------------------------------------------------------------ memory
def test_peak_memory_does_not_grow_with_k(dev, det_flag):
    torch.use_deterministic_algorithms(False)
    peaks = {}
    for k in (1, 4):
        gc.collect()
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats(dev)
        base = torch.cuda.memory_allocated(dev)
        ts = _step(_model("dn", 32, 4, dev), k)
        for j in range(k):
            ts(*_batch(4, 416, 416, 1, 5 + j, dev))
        torch.cuda.synchronize()
        peaks[k] = torch.cuda.max_memory_allocated(dev) - base
        del ts
    grad_bytes = 4 * sum(p.numel() for p in _model("dn", 32, 4, dev).parameters())
    print(f"DN F=32 nb=4 batch 4 416^2: peak k=1 {peaks[1] / 2**20:.1f} MiB, k=4 {peaks[4] / 2**20:.1f} MiB "
          f"(gradient buffer {grad_bytes / 2**20:.1f} MiB)")
    assert abs(peaks[4] - peaks[1]) <= 4 * 2**20
