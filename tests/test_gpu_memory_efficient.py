"""GPU: memory-efficient training (the generator's ``memory_efficient``; engine_train.TrainEngine keeps one F-channel
input per dense block and recomputes x1..x4 before the block's backward).

* the chain flag XMM_CHAIN_SKIP_LAST: x1..x4 bit-equal to what the full chain stores, the last layer's output never
  written, on the fused path (single CTAs and CTA pairs: conv1..conv3, then the conv4-only form), layer by layer (odd
  image height), and at F = 64 (the engine's split layers);
* xmm_copy_channels_bf16 against a torch slice copy;
* training steps with the flag on against off from the same state: bit-equal losses, gradients, parameters and Adam
  moments in the deterministic mode (TrainStep, the autograd path, the CUDA-graph replay), rel-L2 1e-6 with the default
  atomic reductions, and a bit-equal forward output;
* the peak memory of a step with the flag against one without.
"""
import gc

import pytest
import torch

from helpers import rel_l2
from test_gpu_rdb_pair import F32, _block
from xmm_superres_denoise_b200 import ops

pytestmark = pytest.mark.gpu

SENTINEL = -7.0


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


# ---------------------------------------------------------------------------------------------------- chain flag
def _chain(arena, x0, xr, mode):
    """One dense block (RDB3 form: residuals r1, r2) through conv3x3_chain; returns (feature buffer, output)."""
    f = F32
    b, h, w, _ = x0.shape
    buf = torch.full((b, h, w, 5 * f), SENTINEL, dtype=torch.bfloat16, device=x0.device)
    buf[..., :f] = x0
    out = torch.full((b, h, w, f), SENTINEL, dtype=torch.bfloat16, device=x0.device)
    layers = [((buf, 0, k * f, arena.ptr(f"c{k}"), 32, f, buf, k * f), dict(lrelu=0.2, wblob_row=arena.ptr(f"c{k}.row")))
              for k in range(1, 5)]
    layers.append(((buf, 0, 5 * f, arena.ptr("c5"), 32, f, out, 0),
                   dict(wblob_row=arena.ptr("c5.row"), s0=0.04, r1=buf, r1_coff=0, s1=0.2, r2=xr, r2_coff=0, s2=1.0)))
    ops.conv3x3_chain(layers, mode)
    torch.cuda.synchronize()
    return buf, out, ops.LAST_CHAIN_LAUNCHES


@pytest.mark.parametrize("b,h,w,form", [(1, 416, 416, ops.CHAIN_RDB_SINGLE), (1, 416, 416, ops.CHAIN_RDB_PAIR),
                                        (16, 416, 416, ops.CHAIN_RDB_SINGLE), (16, 416, 416, ops.CHAIN_RDB_PAIR),
                                        (3, 40, 131, ops.CHAIN_RDB_PAIR), (2, 8, 70, ops.CHAIN_RDB_SINGLE)])
def test_skip_last_fused_matches_the_full_chain(dev, b, h, w, form):
    arena = _block(dev, 3 * b + h + w)
    g = torch.Generator().manual_seed(b * h + w)
    x0 = torch.randn(b, h, w, F32, generator=g).to(torch.bfloat16).to(dev)
    xr = torch.randn(b, h, w, F32, generator=g).to(torch.bfloat16).to(dev)
    full, _, _ = _chain(arena, x0, xr, ops.CHAIN_AUTO | form)
    part, out, launches = _chain(arena, x0, xr, ops.CHAIN_AUTO | form | ops.CHAIN_SKIP_LAST)
    assert launches == 2
    for k in range(1, 5):
        sl = slice(k * F32, (k + 1) * F32)
        assert torch.equal(part[..., sl], full[..., sl]), f"x{k}"
        assert not torch.all(part[..., sl] == SENTINEL), f"x{k} stored"
    assert torch.all(out == SENTINEL), "the last layer's output was written"


@pytest.mark.parametrize("b,h,w,mode", [(2, 39, 64, ops.CHAIN_AUTO), (1, 40, 131, ops.CHAIN_LAYER_BY_LAYER)])
def test_skip_last_layer_by_layer(dev, b, h, w, mode):
    arena = _block(dev, 17)
    g = torch.Generator().manual_seed(17)
    x0 = torch.randn(b, h, w, F32, generator=g).to(torch.bfloat16).to(dev)
    xr = torch.randn(b, h, w, F32, generator=g).to(torch.bfloat16).to(dev)
    full, _, n_full = _chain(arena, x0, xr, mode)
    part, out, n_part = _chain(arena, x0, xr, mode | ops.CHAIN_SKIP_LAST)
    assert (n_full, n_part) == (5, 4)
    assert torch.equal(part, full), "x1..x4"
    assert torch.all(out == SENTINEL)


def test_skip_last_excludes_skip_dead_stores(dev):
    arena = _block(dev, 5)
    x0 = torch.zeros(1, 8, 16, F32, dtype=torch.bfloat16, device=dev)
    with pytest.raises(RuntimeError, match="exclude each other"):
        _chain(arena, x0, x0, ops.CHAIN_FUSED | ops.CHAIN_SKIP_LAST | ops.CHAIN_SKIP_DEAD_STORES)


def test_skip_last_at_64_filters_recomputes_the_forward_maps(dev):
    """F = 64: the engine's split layers; conv1..conv4 are the forward's own launches."""
    m = _model("dn", 64, 1, 31, dev)
    eng = m._get_engine(train=True)
    eng.arena.ensure(dev)
    f = 64
    g = torch.Generator().manual_seed(2)
    x0 = torch.randn(2, 96, 80, f, generator=g).to(torch.bfloat16).to(dev)
    bufs = [torch.full((2, 96, 80, 5 * f), SENTINEL, dtype=torch.bfloat16, device=dev) for _ in range(2)]
    outs = [torch.full((2, 96, 80, f), SENTINEL, dtype=torch.bfloat16, device=dev) for _ in range(2)]
    for buf in bufs:
        buf[..., :f] = x0
    eng._rdb_forward("f.0.1", bufs[0], outs[0], s0=0.2, s1=1.0, r2=None, s2=0.0)
    first4, last = eng._rdb_layers("f.0.1", bufs[1], outs[1], s0=0.2, s1=1.0, r2=None, s2=0.0)
    assert len(first4) + len(last) > 5  # split layers: no chain
    eng._run(first4)
    torch.cuda.synchronize()
    assert torch.equal(bufs[1], bufs[0])
    assert torch.all(outs[1] == SENTINEL) and not torch.all(outs[0] == SENTINEL)


@pytest.mark.parametrize("src_c,src_off,dst_c,dst_off,n", [(32, 0, 160, 0, 32), (160, 0, 32, 0, 32), (320, 64, 64, 0, 64),
                                                            (160, 8, 160, 120, 40)])
def test_copy_channels(dev, src_c, src_off, dst_c, dst_off, n):
    g = torch.Generator().manual_seed(src_c + dst_off)
    src = torch.randn(3, 37, 29, src_c, generator=g).to(torch.bfloat16).to(dev)
    dst = torch.randn(3, 37, 29, dst_c, generator=g).to(torch.bfloat16).to(dev)
    want = dst.clone()
    want[..., dst_off:dst_off + n] = src[..., src_off:src_off + n]
    ops.copy_channels(src, src_off, dst, dst_off, n)
    torch.cuda.synchronize()
    assert torch.equal(dst, want)
    with pytest.raises(RuntimeError, match="multiples of 8"):
        ops.copy_channels(src, 4, dst, 0, 8)


# ---------------------------------------------------------------------------------------------------- training
def _model(kind, nf, nb, seed, dev, up=1, memeff=False):
    from oracle import rrdb_oracle as O
    from xmm_superres_denoise_b200.models import GeneratorRRDB_DN, GeneratorRRDB_SR

    sd = O.init_state_dict(kind, 1, 1, nf, nb, up, seed=seed)
    m = GeneratorRRDB_DN(1, 1, nf, nb) if kind == "dn" else GeneratorRRDB_SR(1, 1, nf, nb, num_upsample=up)
    m.load_state_dict(sd)
    m.memory_efficient = memeff
    return m.to(dev).train()


def _batch(b, h, w, s, seed, dev):
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(b, 1, h, w, generator=g).to(dev)
    t = (torch.rand(b, 1, h * s, w * s, generator=g) * 0.5).to(dev)
    return x, t


def _loss():
    from oracle import rrdb_oracle as O
    from xmm_superres_denoise_b200.utils.loss_functions import create_loss

    return create_loss(O.sc_dict_for("sqrt"), {"l1": 0.5, "poisson": 0.5})


def _train_run(kind, nf, nb, up, b, h, w, dev, memeff, steps=3, use_graph=False):
    from xmm_superres_denoise_b200.training import TrainStep

    m = _model(kind, nf, nb, 31, dev, up, memeff)
    step = TrainStep(m, _loss(), lr=1e-4, use_graph=use_graph)
    s = 1 if kind == "dn" else 2 ** up
    losses, grads = [], []
    for i in range(steps):
        x, t = _batch(b, h, w, s, 100 + i, dev)
        losses.append(step(x, t).detach().clone())
        grads.append(step.engine.last_flat_grad.clone())
    torch.cuda.synchronize()
    assert ("ckpt" in next(iter(step.engine._bufs.values()))) == memeff
    return losses, grads, step.flat.clone(), step.opt.exp_avg.clone(), step.opt.exp_avg_sq.clone()


def _assert_runs_equal(a, b, what):
    la, ga, pa, ma, va = a
    lb, gb, pb, mb, vb = b
    for i in range(len(la)):
        assert torch.equal(la[i], lb[i]), f"{what}: loss of step {i}"
        assert torch.equal(ga[i], gb[i]), f"{what}: flat gradient of step {i}"
    assert torch.equal(pa, pb) and torch.equal(ma, mb) and torch.equal(va, vb), f"{what}: parameters / Adam moments"


TRAIN_CASES = [("dn", 32, 2, 1, 2, 416, 416), ("sr", 32, 1, 1, 2, 416, 416), ("sr", 32, 1, 2, 2, 208, 208),
               ("dn", 64, 1, 1, 2, 416, 416)]


@pytest.mark.parametrize("kind,nf,nb,up,b,h,w", TRAIN_CASES)
def test_trainstep_memory_efficient_is_bit_equal(dev, det_flag, kind, nf, nb, up, b, h, w):
    torch.use_deterministic_algorithms(True)
    off = _train_run(kind, nf, nb, up, b, h, w, dev, False)
    on = _train_run(kind, nf, nb, up, b, h, w, dev, True)
    _assert_runs_equal(off, on, f"{kind} F={nf} nb={nb} up={up}: memory_efficient on vs off")


def test_autograd_path_memory_efficient_is_bit_equal(dev, det_flag):
    torch.use_deterministic_algorithms(True)
    x, t = _batch(2, 416, 416, 2, 7, dev)
    runs = []
    for memeff in (False, True):
        m = _model("sr", 32, 1, 31, dev, memeff=memeff)
        _loss()(preds=torch.clamp(m(x), 0, 1), target=t).backward()
        runs.append([p.grad.clone() for p in m.parameters()])
    for n, (ga, gb) in enumerate(zip(*runs)):
        assert torch.equal(ga, gb), n


def test_cuda_graph_replay_memory_efficient(dev, det_flag):
    torch.use_deterministic_algorithms(True)
    graph_on = _train_run("dn", 32, 1, 1, 2, 416, 416, dev, True, steps=4, use_graph=True)
    eager_off = _train_run("dn", 32, 1, 1, 2, 416, 416, dev, False, steps=4)
    _assert_runs_equal(graph_on, eager_off, "graph replay (memory_efficient) vs eager (off)")


@pytest.mark.parametrize("kind,nf", [("dn", 32), ("sr", 32)])
def test_default_mode_gradients_agree(dev, det_flag, kind, nf):
    torch.use_deterministic_algorithms(False)
    x, t = _batch(2, 416, 416, 1 if kind == "dn" else 2, 9, dev)
    outs, grads = [], []
    for memeff in (False, True):
        m = _model(kind, nf, 2, 31, dev, memeff=memeff)
        eng = m._get_engine(train=True)
        out, bufs = eng.forward_train(x)
        outs.append(out.clone())
        gout = torch.full_like(out, 1e-3)
        eng.backward(bufs, eng.generation, x, gout, need_x_grad=False)
        grads.append(eng.last_flat_grad.clone())
    assert torch.equal(outs[0], outs[1]), "forward output"
    r = rel_l2(grads[1], grads[0])
    print(f"{kind} F={nf}: flat gradient rel-L2 memory_efficient vs off (atomic reductions) = {r:.2e}")
    assert r <= 1e-6


def test_memory_efficient_halves_the_peak(dev):
    from xmm_superres_denoise_b200.training import TrainStep

    peaks = {}
    for memeff in (False, True):
        gc.collect()
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats(dev)
        base = torch.cuda.memory_allocated(dev)
        m = _model("dn", 32, 4, 31, dev, memeff=memeff)
        step = TrainStep(m, _loss(), lr=1e-4)
        x, t = _batch(4, 416, 416, 1, 5, dev)
        step(x, t)
        torch.cuda.synchronize()
        peaks[memeff] = torch.cuda.max_memory_allocated(dev) - base
        del m, step, x, t
    ratio = peaks[True] / peaks[False]
    print(f"DN F=32 nb=4 batch 4 416^2: peak {peaks[False] / 2**20:.0f} MiB -> {peaks[True] / 2**20:.0f} MiB "
          f"({ratio:.3f})")
    assert ratio <= 0.5
