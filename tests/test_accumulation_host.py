"""CPU: the host side of gradient accumulation -- train.py's [trainer] accumulate_grad_batches and
--accumulate-grad-batches, TrainStep's argument check, the caller-owned gradient buffer of TrainEngine.backward, and the
accumulate flag of every weight-gradient destination.  No GPU: buffers live on the CPU or the meta device and the
launches are recorded."""
import os
import subprocess
import sys

import pytest
import torch

import __graft_entry__ as entry


@pytest.fixture
def train_mod():
    sys.path.insert(0, entry.ROOT)
    import train

    return train


def test_train_py_key_and_flag(tmp_path, train_mod):
    train = train_mod
    cfg = train.load_run_config(None)
    assert cfg["trainer"]["accumulate_grad_batches"] == 1
    assert train.accumulate_grad_batches(cfg, None) == 1
    assert train.parser().parse_args(["fit"]).accumulate_grad_batches is None
    run = tmp_path / "run.toml"
    run.write_text("[trainer]\naccumulate_grad_batches = 4\n")
    cfg = train.load_run_config(str(run))
    assert cfg["trainer"]["accumulate_grad_batches"] == 4 and cfg["trainer"]["deterministic"] is False
    assert train.accumulate_grad_batches(cfg, None) == 4
    a = train.parser().parse_args(["fit", str(run), "--accumulate-grad-batches", "2"])
    assert a.accumulate_grad_batches == 2
    assert train.accumulate_grad_batches(cfg, a.accumulate_grad_batches) == 2  # the flag wins over the run file
    for bad in (0, -3, 1.5, True):
        with pytest.raises(ValueError, match="accumulate_grad_batches"):
            train.accumulate_grad_batches(train.load_run_config(None), bad)
    run.write_text("[trainer]\naccumulate_grad_batches = 0\n")
    with pytest.raises(ValueError, match="accumulate_grad_batches"):
        train.accumulate_grad_batches(train.load_run_config(str(run)), None)
    out = subprocess.run([sys.executable, os.path.join(entry.ROOT, "train.py"), "--help"], capture_output=True,
                         text=True, check=True).stdout
    assert "--accumulate-grad-batches" in out


def test_trainstep_rejects_a_window_below_one():
    from xmm_superres_denoise_b200.training import TrainStep

    for bad in (0, -1, 2.0, True):
        with pytest.raises(ValueError, match="accumulate_grad_batches"):
            TrainStep(torch.nn.Linear(2, 2), None, accumulate_grad_batches=bad)


def _gen(kind, nf, nb=1, device="cpu"):
    from xmm_superres_denoise_b200.models import GeneratorRRDB_DN, GeneratorRRDB_SR

    torch.manual_seed(3)
    g = GeneratorRRDB_DN(1, 1, nf, nb) if kind == "dn" else GeneratorRRDB_SR(1, 1, nf, nb, num_upsample=1)
    return g.to(device)


def test_caller_buffer_is_zeroed_or_kept():
    """A window's first backward starts from zero; a later one keeps the gradients and zeroes only the deterministic
    scratch floats after them (destinations that are copied into a gradient)."""
    from xmm_superres_denoise_b200.engine_train import TrainEngine

    g = _gen("sr", 32)
    eng = TrainEngine(g, "sr")
    total = sum(p.numel() for p in g.parameters())
    extra = eng._det_scratch_floats()
    buf = eng.grad_buffer(torch.device("cpu"))
    assert buf.numel() == total + extra and not buf.any()
    for det_extra in (0, extra):
        buf.fill_(5.0)
        views = eng._grad_views(torch.device("cpu"), det_extra, buf, accumulate=True)
        assert torch.all(buf[:total] == 5.0) and not buf[total:total + det_extra].any()
        assert eng.last_flat_grad.data_ptr() == buf.data_ptr() and eng.last_flat_grad.numel() == total
        assert [v.shape for v in views] == [p.shape for p in g.parameters()]
        assert views[0].data_ptr() == buf.data_ptr()
        eng._grad_views(torch.device("cpu"), det_extra, buf, accumulate=False)
        assert not buf[:total + det_extra].any()
    with pytest.raises(RuntimeError, match="caller-owned"):
        eng._grad_views(torch.device("cpu"), 0, None, accumulate=True)
    with pytest.raises(RuntimeError, match="grad_buffer"):
        eng._grad_views(torch.device("cpu"), 0, torch.zeros(total), accumulate=True)


@pytest.mark.parametrize("kind,nf", [("dn", 32), ("sr", 32), ("dn", 64)])
def test_every_weight_gradient_destination_follows_the_flag(monkeypatch, kind, nf):
    """The dense blocks' and the single convs' weight-gradient destinations overwrite on a window's first micro-batch
    and add on the later ones (meta buffers, launches recorded)."""
    from xmm_superres_denoise_b200 import ops
    from xmm_superres_denoise_b200.engine_train import TrainEngine

    g = _gen(kind, nf)
    eng = TrainEngine(g, kind)
    meta = torch.device("meta")
    bufs = eng._train_buffers(1, 16, 16, meta, False)
    dsts = []
    monkeypatch.setattr(ops, "conv3x3_wgrad", lambda x, dy, roles, d: dsts.extend(d))
    monkeypatch.setattr(ops, "colsum", lambda *a, **k: None)
    monkeypatch.setattr(ops, "colsum_multi", lambda *a, **k: None)
    for acc in (0, 1):
        dsts.clear()
        grads = eng._grad_views(meta)
        eng._acc = acc
        try:
            for r in range(3):
                eng._rdb_wgrad(0, r, bufs, grads)
            eng._single_conv_wgrad(g.trunk_conv, bufs["trunk"], bufs["d_trunk"], grads)
            if kind == "sr":
                eng._single_conv_wgrad(g.upsampling[0], bufs["trunk"], bufs["d_up0"], grads, perm=1)
                eng._single_conv_wgrad(g.HRconv, bufs["up0"], bufs["d_hr"], grads)
        finally:
            eng._acc = 0
        assert dsts and {d[9] for d in dsts} == {acc}
