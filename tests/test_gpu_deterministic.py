"""GPU (B200): the deterministic training mode (determinism.py, XMM_DETERMINISTIC / torch.use_deterministic_algorithms).

* per reduction site: the deterministic form gives the same bits over repeats while a side stream changes CTA timing,
  and stays within a float64 bound derived from its summation depth;
* the finalize kernel itself: a workspace with one slot dropped or duplicated fails that bound;
* whole training steps (TrainStep, the autograd path, the CUDA-graph replay): bit-identical losses, gradients,
  parameters and Adam moments from the same state;
* against the default (atomic) path: only the summation order differs; off means off.

Float64 bounds.  A float32 sum of values a_1..a_m whose evaluation tree has depth D (every value passes through at
most D additions) is within gamma(D) * sum |a_i| of the exact sum, gamma(D) = D u / (1 - D u), u = 2^-24.  Each site
is a three-level tree: per-thread (or per-lane) running sums over L values, a fixed in-CTA combination of depth I,
then xmm_det_finalize over the K slots in slot order -- D = L + I + K, plus one rounding for a final scale.
"""
import math

import pytest
import torch

from helpers import C_TC, GRAD_REL, abs_conv, ref_conv, rel_l2

pytestmark = pytest.mark.gpu

U = 2.0 ** -24


def gamma(d: int) -> float:
    return d * U / (1 - d * U)


@pytest.fixture(scope="module")
def dev():
    from xmm_superres_denoise_b200 import _lib

    _lib.check(_lib.load().xmm_check_device())
    return torch.device("cuda:0")


@pytest.fixture
def det_flag(monkeypatch):
    monkeypatch.delenv("XMM_DETERMINISTIC", raising=False)
    monkeypatch.setenv("CUBLAS_WORKSPACE_CONFIG", ":4096:8")
    before = torch.are_deterministic_algorithms_enabled()
    yield
    torch.use_deterministic_algorithms(before)


class SideLoad:
    """Elementwise work on a side stream, enqueued just before a measured launch (so that the two overlap): repeat k
    runs k passes, so the launch's CTAs start on differently busy SMs every repeat."""

    def __init__(self, dev):
        self.s = torch.cuda.Stream(dev)
        self.buf = torch.rand(64 << 20, device=dev)

    def __call__(self, k: int) -> None:
        self.s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(self.s):
            for _ in range(k):
                self.buf.mul_(0.999).add_(1e-3)


def _finalize_one(dev, ws, count, stride, dst, n, scale, accumulate=1, col0=0):
    """xmm_det_finalize on one job, called directly."""
    from xmm_superres_denoise_b200 import _lib, ops

    job = _lib.DetJob(ws.data_ptr() + 4 * col0, count, stride, 0, n, scale, accumulate)
    table = torch.frombuffer(bytearray(bytes(job)), dtype=torch.uint8).to(dev)
    ops.det_finalize(table, 1, n, dst)


# ---------------------------------------------------------------------------------------------------- per site
B, H, W, CIN = 2, 416, 416, 96  # a dense block's data gradient of x_2 at the F = 32 training shape
FAMILIES = {"tap_view": dict(tap_mode=1), "column_scatter": dict(tap_mode=7), "column_scatter_g2": dict(tap_mode=8),
            "row_hop": dict(tap_mode=9)}


def _conv_case(dev):
    from xmm_superres_denoise_b200.engine import WeightArena, _Blob, _Segment

    g = torch.Generator().manual_seed(3)
    # positive operands: the column sums do not cancel, so the float64 bound is tight enough to see one slot
    x = torch.rand(B, H, W, 160, generator=g).to(torch.bfloat16).to(dev)
    wgt = (torch.rand(32, CIN, 3, 3, generator=g) * 0.02).to(dev)
    mask = (torch.rand(B, H, W, 32, generator=g) + 0.01).to(torch.bfloat16).to(dev)
    arena = WeightArena()
    arena.add(_Blob("c", 32, 32, CIN // 32, [_Segment(wgt, CIN, 0, 0, 0, 0, CIN, 1.0)], None))
    arena.add(_Blob("c.row", 32, 32, CIN // 32, [_Segment(wgt, CIN, 0, 0, 0, 0, CIN, 1.0)], None, tap_order=1))
    arena.ensure(dev)
    return x, wgt, mask, arena


def _conv(x, mask, arena, fam, out, **kw):
    from xmm_superres_denoise_b200 import ops

    extra = dict(FAMILIES[fam])
    if fam == "row_hop":
        extra["wblob_row"] = arena.ptr("c.row")
    ops.conv3x3(x, 32, CIN, arena.ptr("c"), 32, 32, out, 0, mask=mask, mask_coff=0, mask_slope=0.2, **extra, **kw)


def _conv_bound(dev, x, wgt, count):
    """float64 column sums 0.2 * sum_p y[p][n] and their bound.  Each value v the kernel adds is the fp32 epilogue value
    (before the bf16 store): |v - y| <= C_TC * S per element (helpers.assert_bf16_elementwise's accumulation term).
    Depth: a lane adds one pixel per 128-pixel tile / row step it owns; the static schedules give a CTA at most twice
    its even share plus two (pre-tile, ragged tail), L <= 2 ceil(P / (128 G)) + 2; then 5 shuffle levels; then the
    K = 8 G warp slots."""
    xin = x[..., 32:32 + CIN].permute(0, 3, 1, 2)
    wq = wgt.to(torch.bfloat16)
    y = ref_conv(xin, wq)
    s = abs_conv(xin, wq)
    grid = count // 8
    depth = 2 * math.ceil(B * H * W / (128 * grid)) + 2 + 5 + count
    want = 0.2 * y.sum(dim=(0, 2, 3))
    acc = C_TC * s.sum(dim=(0, 2, 3))
    bound = 0.2 * (acc + gamma(depth) * (y.abs().sum(dim=(0, 2, 3)) + acc)) + U * want.abs()
    return want, bound


@pytest.mark.parametrize("fam", list(FAMILIES))
def test_fused_bias_sums_are_deterministic(dev, fam):
    from xmm_superres_denoise_b200 import _lib, determinism, ops

    x, wgt, mask, arena = _conv_case(dev)
    load = SideLoad(dev)
    out = torch.empty(B, H, W, 32, dtype=torch.bfloat16, device=dev)
    plan = determinism.DetPlan(dev)
    dst = torch.zeros(32, device=dev)
    det, atomic = [], []
    for rep in range(5):
        dst.zero_()
        plan.begin(dst)
        kw = plan.conv_kwargs(B, H, W, dst, 0.2)
        load(rep)
        _conv(x, mask, arena, fam, out, **kw)
        plan.flush()
        torch.cuda.synchronize()
        det.append(dst.clone())
        cs = torch.zeros(32, device=dev)
        load(rep)
        _conv(x, mask, arena, fam, out, colsum=cs, colsum_scale=0.2)
        torch.cuda.synchronize()
        atomic.append(cs)
    for r in det[1:]:
        assert torch.equal(r, det[0])
    ndiff = sum(int((a != atomic[0]).sum()) for a in atomic[1:])
    print(f"{fam}: default (atomic) path, elements differing from repeat 0 over 4 repeats: {ndiff} of 128")
    count = ops.det_slots(_lib.DET_CONV3X3, B, H, W, 32)
    want, bound = _conv_bound(dev, x, wgt, count)
    err = (det[0].double() - want).abs()
    print(f"{fam}: max |err| / bound = {float((err / bound).max()):.3f}")
    assert bool((err <= bound).all())


@pytest.mark.parametrize("fault", ["zeroed", "duplicated"])
def test_finalize_fails_the_bound_with_a_slot_dropped_or_duplicated(dev, fault):
    from xmm_superres_denoise_b200 import _lib, ops

    x, wgt, mask, arena = _conv_case(dev)
    count = ops.det_slots(_lib.DET_CONV3X3, B, H, W, 32)
    ws = torch.zeros(count * 32, device=dev)
    dst = torch.zeros(32, device=dev)
    out = torch.empty(B, H, W, 32, dtype=torch.bfloat16, device=dev)
    _conv(x, mask, arena, "column_scatter", out, colsum=dst, colsum_scale=0.2, colsum_ws=ws)
    torch.cuda.synchronize()
    slots = ws.view(count, 32)
    k = int(slots.sum(dim=1).argmax())
    if fault == "zeroed":
        slots[k].zero_()
    else:
        other = (k + 1) % count
        slots[other] += slots[k]
    _finalize_one(dev, ws, count, 32, dst, 32, 0.2, accumulate=0)
    torch.cuda.synchronize()
    assert float(ws.abs().max()) == 0.0  # the finalize leaves its slots zero
    want, bound = _conv_bound(dev, x, wgt, count)
    ratio = float(((dst.double() - want).abs() / bound).max())
    print(f"slot {fault}: max |err| / bound = {ratio:.2f}")
    assert ratio > 1.0


def test_colsum_multi_five_segments_is_deterministic(dev):
    from xmm_superres_denoise_b200 import _lib, determinism, ops

    g = torch.Generator().manual_seed(4)
    G = torch.randn(B, H, W, 160, generator=g).to(torch.bfloat16).to(dev)
    scales = [1.0, 1.0, 1.0, 1.0, 0.2]
    load = SideLoad(dev)
    plan = determinism.DetPlan(dev)
    dst = torch.zeros(160, device=dev)
    det, atomic = [], []
    for rep in range(5):
        dst.zero_()
        plan.begin(dst)
        load(rep)
        plan.colsum([G], [(32 * k, 32, dst[32 * k:32 * (k + 1)], scales[k], True) for k in range(5)])
        plan.flush()
        torch.cuda.synchronize()
        det.append(dst.clone())
        ref = torch.zeros(160, device=dev)
        load(rep)
        ops.colsum_multi(G, [(32 * k, 32, ref[32 * k:32 * (k + 1)], scales[k], False) for k in range(5)])
        torch.cuda.synchronize()
        atomic.append(ref)
    for r in det[1:]:
        assert torch.equal(r, det[0])
    print(f"colsum_multi: default path, elements differing over 4 repeats: "
          f"{sum(int((a != atomic[0]).sum()) for a in atomic[1:])} of 640")
    # depth: a thread adds ceil(P / (G ppb)) pixels, the CTA then adds its ppb pixel lanes in order, then K = G slots
    count = ops.det_slots(_lib.DET_COLSUM, B, H, W, 160)
    ppb = 256 // 20
    depth = math.ceil(B * H * W / (count * ppb)) + ppb + count
    sc = torch.tensor([scales[c // 32] for c in range(160)], dtype=torch.float64, device=dev)
    Gd = G.double()
    want = sc * Gd.sum(dim=(0, 1, 2))
    bound = sc * gamma(depth + 1) * Gd.abs().sum(dim=(0, 1, 2)) + U * want.abs()
    assert bool(((det[0].double() - want).abs() <= bound).all())


def _shift(s, dy, dx):
    """s[y - dy][x - dx] with zero outside ([B, ns, H, W] float64)."""
    p = torch.nn.functional.pad(s, (1, 1, 1, 1))
    h, w = s.shape[-2:]
    return p[..., 1 - dy:1 - dy + h, 1 - dx:1 - dx + w]


@pytest.mark.parametrize("form", ["conv_last", "conv_first"])
def test_edge_wgrad_is_deterministic(dev, form):
    from xmm_superres_denoise_b200 import _lib, determinism, ops

    g = torch.Generator().manual_seed(5)
    f = 32
    s = torch.randn(B, 1, H, W, generator=g).to(dev)
    v = torch.randn(B, H, W, f, generator=g).to(torch.bfloat16).to(dev)
    kw, v2 = {}, None
    if form == "conv_last":
        gate = (torch.rand(B, 1, H, W, generator=g) * 1.4 - 0.2).to(dev)
        kw = dict(gate=gate)
        se = s * ((gate >= 0) & (gate <= 1))
    else:
        v2 = torch.randn(B, H, W, f, generator=g).to(torch.bfloat16).to(dev)
        kw = dict(v2=v2, v2_coff=0)
        se = s
    load = SideLoad(dev)
    plan = determinism.DetPlan(dev)
    dst = torch.zeros(f * 9 + 1, device=dev)
    det, atomic = [], []
    for rep in range(5):
        dst.zero_()
        plan.begin(dst)
        load(rep)
        plan.edge_wgrad(s, v, 0, f, dst[:f * 9].view(1, f, 9), ssum=dst[f * 9:] if form == "conv_last" else None, **kw)
        plan.flush()
        torch.cuda.synchronize()
        det.append(dst.clone())
        r = torch.zeros(1, f, 9, device=dev)
        ss = torch.zeros(1, device=dev)
        load(rep)
        ops.edge_wgrad(s, v, 0, f, r, ssum=ss if form == "conv_last" else None, **kw)
        torch.cuda.synchronize()
        atomic.append(torch.cat([r.reshape(-1), ss]))
    for r in det[1:]:
        assert torch.equal(r, det[0])
    print(f"edge_wgrad {form}: default path, elements differing over 4 repeats: "
          f"{sum(int((a != atomic[0]).sum()) for a in atomic[1:])} of {atomic[0].numel() * 4}")
    # reference: R[c][t] = sum_q s[q - off(t)] V[q][c], V = v (+ v2, one fp32 rounding), S = sum_q s[q]
    sd = se.double()
    V = v.double() + (v2.double() if v2 is not None else 0.0)
    Va = v.double().abs() + (v2.double().abs() if v2 is not None else 0.0)
    want = torch.empty(f, 9, dtype=torch.float64, device=dev)
    mag = torch.empty(f, 9, dtype=torch.float64, device=dev)
    for t in range(9):
        sh = _shift(sd, t // 3 - 1, t % 3 - 1)[:, 0, :, :, None]
        want[:, t] = (sh * V).sum(dim=(0, 1, 2))
        mag[:, t] = (sh.abs() * Va).sum(dim=(0, 1, 2))
    # depth: a thread's FMAs over its pixels (rows * W / PPI, rows <= 8, PPI = 256 / (f / 8) pixels per pass),
    # 3 shuffle levels, the 8 warps in order, then the K CTA slots; + 1 for the v + v2 rounding
    count = ops.det_slots(_lib.DET_EDGE_WGRAD, B, H, W, f)
    depth = math.ceil(8 * W / (256 // (f // 8))) + 3 + 8 + count + 1
    got = det[0][:f * 9].view(f, 9).double()
    assert bool(((got - want).abs() <= gamma(depth) * mag + U * want.abs()).all())
    if form == "conv_last":
        # S: a thread's share of the staged rows ((8 + 2) * (W + 2) / 256), 5 shuffle levels, 8 warps, K slots
        depth_s = math.ceil(10 * (W + 2) / 256) + 5 + 8 + count
        ws_ = sd.sum()
        assert abs(float(det[0][f * 9]) - float(ws_)) <= gamma(depth_s) * float(sd.abs().sum()) + U * abs(float(ws_))


# ---------------------------------------------------------------------------------------------------- training
def _model(kind, nf, nb, seed, dev, up=1):
    from oracle import rrdb_oracle as O
    from xmm_superres_denoise_b200.models import GeneratorRRDB_DN, GeneratorRRDB_SR

    sd = O.init_state_dict(kind, 1, 1, nf, nb, up, seed=seed)
    m = GeneratorRRDB_DN(1, 1, nf, nb) if kind == "dn" else GeneratorRRDB_SR(1, 1, nf, nb, num_upsample=up)
    m.load_state_dict(sd)
    return m.to(dev).train()


def _batch(b, h, w, s, seed, dev):
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(b, 1, h, w, generator=g).to(dev)
    t = (torch.rand(b, 1, h * s, w * s, generator=g) * 0.5).to(dev)
    return x, t


def _train_run(kind, nf, nb, up, b, h, w, dev, steps=3, use_graph=False):
    from oracle import rrdb_oracle as O
    from xmm_superres_denoise_b200.training import TrainStep
    from xmm_superres_denoise_b200.utils.loss_functions import create_loss

    m = _model(kind, nf, nb, 31, dev, up)
    step = TrainStep(m, create_loss(O.sc_dict_for("sqrt"), {"l1": 0.5, "poisson": 0.5}), lr=1e-4,
                     use_graph=use_graph)
    s = 1 if kind == "dn" else 2 ** up
    losses, grads = [], []
    for i in range(steps):
        x, t = _batch(b, h, w, s, 100 + i, dev)
        losses.append(step(x, t).detach().clone())
        grads.append(step.engine.last_flat_grad.clone())
    torch.cuda.synchronize()
    return losses, grads, step.flat.clone(), step.opt.exp_avg.clone(), step.opt.exp_avg_sq.clone()


def _assert_runs_equal(a, b, what):
    la, ga, pa, ma, va = a
    lb, gb, pb, mb, vb = b
    for i in range(len(la)):
        assert torch.equal(la[i], lb[i]), f"{what}: loss of step {i}"
        assert torch.equal(ga[i], gb[i]), f"{what}: flat gradient of step {i}"
    assert torch.equal(pa, pb) and torch.equal(ma, mb) and torch.equal(va, vb), f"{what}: parameters / Adam moments"


TRAIN_CASES = [("dn", 32, 1, 1, 2, 416, 416), ("sr", 32, 1, 1, 2, 416, 416), ("dn", 64, 1, 1, 2, 416, 416),
               ("sr", 64, 1, 1, 2, 416, 416), ("sr", 32, 1, 2, 2, 416, 416), ("dn", 32, 1, 1, 2, 200, 136),
               ("dn", 32, 4, 1, 16, 416, 416)]  # (last: the bench's DN training shape)


@pytest.mark.parametrize("kind,nf,nb,up,b,h,w", TRAIN_CASES)
def test_trainstep_is_bit_reproducible(dev, det_flag, kind, nf, nb, up, b, h, w):
    torch.use_deterministic_algorithms(True)
    a = _train_run(kind, nf, nb, up, b, h, w, dev)
    c = _train_run(kind, nf, nb, up, b, h, w, dev)
    _assert_runs_equal(a, c, f"{kind} F={nf} nb={nb} up={up} {b}x{h}x{w}")


@pytest.mark.parametrize("kind", ["dn", "sr"])
def test_autograd_path_is_bit_reproducible(dev, det_flag, kind):
    from oracle import rrdb_oracle as O
    from xmm_superres_denoise_b200.utils.loss_functions import create_loss

    torch.use_deterministic_algorithms(True)
    loss = create_loss(O.sc_dict_for("sqrt"), {"l1": 0.5, "poisson": 0.5})
    x, t = _batch(2, 416, 416, 1 if kind == "dn" else 2, 7, dev)
    runs = []
    for _ in range(2):
        m = _model(kind, 32, 1, 31, dev)
        loss(preds=torch.clamp(m(x), 0, 1), target=t).backward()
        runs.append([p.grad.clone() for p in m.parameters()])
    for n, (ga, gb) in enumerate(zip(*runs)):
        assert torch.equal(ga, gb), n


def test_cuda_graph_replay_is_bit_reproducible(dev, det_flag):
    torch.use_deterministic_algorithms(True)
    a = _train_run("dn", 32, 1, 1, 2, 416, 416, dev, steps=4, use_graph=True)
    c = _train_run("dn", 32, 1, 1, 2, 416, 416, dev, steps=4, use_graph=True)
    _assert_runs_equal(a, c, "XMM_TRAIN_GRAPH")
    e = _train_run("dn", 32, 1, 1, 2, 416, 416, dev, steps=4)
    _assert_runs_equal(a, e, "graph replay vs eager")


def _grads(kind, nf, dev, x, t, det: bool):
    from oracle import rrdb_oracle as O
    from xmm_superres_denoise_b200.utils.loss_functions import create_loss

    torch.use_deterministic_algorithms(det)
    m = _model(kind, nf, 1, 31, dev)
    create_loss(O.sc_dict_for("sqrt"), {"l1": 0.5, "poisson": 0.5})(preds=torch.clamp(m(x), 0, 1), target=t).backward()
    return {n: p.grad.clone() for n, p in m.named_parameters()}


@pytest.mark.parametrize("kind,nf", [("dn", 32), ("sr", 32), ("dn", 64)])
def test_deterministic_gradients_match_the_default_path(dev, det_flag, kind, nf):
    x, t = _batch(2, 416, 416, 1 if kind == "dn" else 2, 9, dev)
    gd = _grads(kind, nf, dev, x, t, True)
    g0 = _grads(kind, nf, dev, x, t, False)
    worst = max((rel_l2(gd[n], g0[n]), n) for n in gd)
    print(f"{kind} F={nf}: worst per-tensor rel-L2 deterministic vs default = {worst[0]:.2e} ({worst[1]})")
    assert worst[0] <= 1e-5


def test_deterministic_gradient_vector_vs_oracle(dev, det_flag):
    """The bar of test_gpu_training's full-gradient check, with the mode on."""
    import os

    import numpy as np

    from oracle import rrdb_oracle as O
    from oracle.make_golden import LR_MAX
    from oracle.synthetic import count_batch

    kind, nf, nb = "dn", 32, 4
    sd = O.init_state_dict(kind, 1, 1, nf, nb, 1, seed=21)
    lr, hr, t_lr, t_hr = count_batch(2, seed=5, kind=kind)
    x = O.normalize_image(torch.from_numpy(lr[:, :, 160:256, 168:248].astype(np.float32) / t_lr), LR_MAX, "sqrt")
    sdg = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    torch.set_num_threads(os.cpu_count() or 1)
    want_out = O.model_forward(x, sdg, kind, 1)
    target = (want_out.detach() * 0.7 + 0.05).clamp(0, 1)
    ((want_out - target).abs().mean() + ((want_out - target) ** 2).mean()).backward()
    torch.use_deterministic_algorithms(True)
    from xmm_superres_denoise_b200.models import GeneratorRRDB_DN

    m = GeneratorRRDB_DN(1, 1, nf, nb)
    m.load_state_dict(sd)
    m = m.to(dev).train()
    out = torch.clamp(m(x.to(dev)), 0, 1)
    tt = target.to(dev)
    ((out - tt).abs().mean() + ((out - tt) ** 2).mean()).backward()
    got = torch.cat([p.grad.reshape(-1) for _, p in m.named_parameters()]).cpu()
    want = torch.cat([sdg[n].grad.reshape(-1) for n, _ in m.named_parameters()])
    r = rel_l2(got, want)
    print(f"deterministic full gradient rel-L2 vs oracle = {r:.3e}")
    assert r < GRAD_REL


def test_off_means_off(dev, det_flag):
    """Mode off: no plan, no workspace, no finalize launch, and the default path's launch count."""
    from xmm_superres_denoise_b200 import ops

    torch.use_deterministic_algorithms(False)
    counts = {}
    for det in (False, True):
        torch.use_deterministic_algorithms(det)
        m = _model("sr", 32, 2, 31, dev)
        step_eng = m._get_engine(train=True)
        x, t = _batch(2, 96, 80, 2, 3, dev)
        out, bufs = step_eng.forward_train(x)
        ops.LAUNCHES = 0
        step_eng.backward(bufs, step_eng.generation, x, torch.ones_like(out) * 1e-3, need_x_grad=False)
        torch.cuda.synchronize()
        counts[det] = ops.LAUNCHES
        if not det:
            assert "det" not in bufs and step_eng._det is None
        else:
            assert "det" in bufs
    # deterministic: one finalize per RRDB + one for the edge layers, nothing else added
    assert counts[True] == counts[False] + 2 + 1, counts
