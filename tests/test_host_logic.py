"""CPU: host-side mirror of the reference interface (names, state_dict, error behaviour)."""
import os

import numpy as np
import pytest
import torch

from oracle import ref_loader
from oracle import rrdb_oracle as O
from oracle.make_golden import init_fingerprint
from xmm_superres_denoise_b200.models import GeneratorRRDB_DN, GeneratorRRDB_SR
from xmm_superres_denoise_b200.models.modules import RRDB, ResidualDenseBlock_5C, make_layer
from xmm_superres_denoise_b200.transforms import ImageUpsample, Normalize


@pytest.mark.parametrize("kind", ["dn", "sr"])
def test_state_dict_keys_shapes_and_param_count(kind):
    m = GeneratorRRDB_DN(1, 1, 32, 4) if kind == "dn" else GeneratorRRDB_SR(1, 1, 32, 4, num_upsample=1)
    sd = m.state_dict()
    want = O.init_state_dict(kind, 1, 1, 32, 4, 1)
    assert sorted(sd.keys()) == sorted(want.keys())
    assert all(tuple(sd[k].shape) == tuple(want[k].shape) for k in sd)
    assert sum(p.numel() for p in m.parameters()) == (1670657 if kind == "dn" else 1716897)  # SURVEY a6
    assert len(sd) == (126 if kind == "dn" else 130)
    m.load_state_dict(want)  # strict


def test_default_num_upsample_and_attributes():
    m = GeneratorRRDB_SR(1, 1, 32, 1)
    assert m.num_upsample == 2 and "upsampling.3.weight" in m.state_dict()
    assert (m.in_channels, m.out_channels, m.num_filters, m.num_res_blocks, m.memory_efficient) == (1, 1, 32, 1, False)
    assert isinstance(m.rrdb[0], RRDB) and isinstance(m.rrdb[0].RDB2, ResidualDenseBlock_5C)
    assert len(make_layer(lambda: RRDB(32, 32), 3)) == 3


@pytest.mark.parametrize("kind", ["dn", "sr"])
def test_same_seed_gives_the_reference_initialisation(golden_dir, kind):
    """The reference's initialisation is torch's default one, drawn in its module construction order.  The stored
    fingerprint of it (tests/golden/init_seed123.npz: keys, sizes, exact sampled values, sums) was recorded from these
    classes, which the comparison below holds bit-equal to the reference's own classes where its source is present."""
    cls = GeneratorRRDB_DN if kind == "dn" else GeneratorRRDB_SR
    got = init_fingerprint(cls, kind)
    g = np.load(os.path.join(golden_dir, "init_seed123.npz"))
    assert list(got["keys"]) == list(g[f"{kind}.keys"])
    np.testing.assert_array_equal(got["numel"], g[f"{kind}.numel"])
    np.testing.assert_array_equal(got["sample"], g[f"{kind}.sample"])
    np.testing.assert_allclose(got["moments"], g[f"{kind}.moments"], rtol=1e-9, atol=1e-12)
    if not ref_loader.available():
        return
    ref = ref_loader.load_reference()
    torch.manual_seed(123)
    a = ref.GeneratorRRDB_DN(1, 1, 32, 2) if kind == "dn" else ref.GeneratorRRDB_SR(1, 1, 32, 2, num_upsample=1)
    torch.manual_seed(123)
    b = GeneratorRRDB_DN(1, 1, 32, 2) if kind == "dn" else GeneratorRRDB_SR(1, 1, 32, 2, num_upsample=1)
    sa, sb = a.state_dict(), b.state_dict()
    assert list(sa.keys()) == list(sb.keys())
    assert all(torch.equal(sa[k], sb[k]) for k in sa)


def test_no_cpu_fallback():
    m = GeneratorRRDB_DN(1, 1, 32, 1).eval()
    with torch.no_grad(), pytest.raises(RuntimeError, match="no CPU path"):
        m(torch.rand(1, 1, 16, 16))
    with pytest.raises(RuntimeError):
        Normalize(1.0, 1.0, "sqrt").normalize_lr_image(torch.rand(4, 4))
    with pytest.raises(RuntimeError):
        ImageUpsample(2)(torch.rand(1, 1, 4, 4))
    with pytest.raises(NotImplementedError):
        GeneratorRRDB_DN(1, 1, 48, 1).eval()._get_engine()


def test_normalize_interface():
    n = Normalize(lr_max=0.0022336, hr_max=0.0005584, stretch_mode="asinh")
    assert n.stretch_mode == "asinh" and n.lr_max.ndim == 0 and abs(float(n.hr_max) - 0.0005584) < 1e-9
    assert n.normalize_hr_image(None) is None
    x = torch.linspace(0, 1, 9)
    assert torch.allclose(n.denorm(n.norm(x)), x, atol=1e-6)
    with pytest.raises(ValueError, match="is not implemented"):
        Normalize(1.0, 1.0, "cbrt")
    with pytest.raises(ValueError):
        ImageUpsample(1.5)


def test_model_wrapper_mirrors_reference_interface():
    """models.Model: constructor / method names of the reference's LightningModule (models/model.py:13-247)."""
    import types

    from xmm_superres_denoise_b200.models import Model

    cfg = types.SimpleNamespace(name="esr_gen", memory_efficient=False, batch_size=4,
                                model=types.SimpleNamespace(in_channels=1, out_channels=1, filters=32, residual_blocks=1),
                                optimizer=types.SimpleNamespace(learning_rate=1e-4, betas=(0.9, 0.999)))
    m = Model(cfg, (416, 416), (832, 832), loss=None, metrics=None, extended_metrics=None, in_metrics=None,
              in_extended_metrics=None)
    assert m.model is None
    m.configure_model()
    assert type(m.model).__name__ == "GeneratorRRDB_SR" and m.model.num_upsample == 1
    opt = m.configure_optimizers()
    assert opt.defaults["lr"] == 1e-4 and tuple(opt.defaults["betas"]) == (0.9, 0.999)
    for name in ("forward", "training_step", "validation_step", "test_step", "on_validation_start",
                 "on_validation_epoch_end", "on_test_epoch_end", "_on_step", "_on_epoch_end"):
        assert callable(getattr(m, name))
    cfg.name = "swinfir"
    m2 = Model(cfg, (416, 416), (416, 416), loss=None)
    import pytest

    with pytest.raises(NotImplementedError):
        m2.configure_model()
    bad = Model(types.SimpleNamespace(**{**cfg.__dict__, "name": "esr_gen"}), (416, 416), (1248, 1248), loss=None)
    with pytest.raises(ValueError):
        bad.configure_model()


def test_train_py_reads_the_reference_config_files(tmp_path, monkeypatch):
    """train.py (reference: xmm_superres_denoise/train.py:27-55,66-67): the model table of res/configs/models.toml named
    by [model].name, the [loss] percentages + [scaling.<mode>] of res/configs/loss_functions.toml when use_scaling is
    set, and dataset.<side>.clamp_max as the normalisation maxima."""
    import importlib.util
    import os

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("xmm_train_entry", os.path.join(root, "train.py"))
    train = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(train)
    cfgdir = tmp_path / "res" / "configs"
    cfgdir.mkdir(parents=True)
    (cfgdir / "models.toml").write_text(
        '[esr_gen]\nin_channels = 1\nout_channels = 1\nfilters = 64\nresidual_blocks = 8\nlearning_rate = 2e-4\nbetas = [0.5, 0.9]\n')
    (cfgdir / "loss_functions.toml").write_text(
        '[loss]\nuse_scaling = true\nl1 = 0.25\npoisson = 0.0\npsnr = 0.0\nssim = 0.0\nms_ssim = 0.75\n'
        '[scaling.sqrt]\nl1 = { scaling = 9.5, correction = -0.5 }\nms_ssim = { scaling = -3.0, correction = 2.6 }\n'
        '[scaling.linear]\nl1 = { scaling = 27.0, correction = -0.57 }\n')
    run = tmp_path / "run.toml"
    run.write_text('[model]\nname = "esr_gen"\nbatch_size = 4\n[dataset]\nscaling = "sqrt"\n'
                   '[dataset.lr]\nclamp_max = 0.002\nres = 416\nexps = [20]\n[dataset.hr]\nclamp_max = 0.0005\nres = 832\nexp = 50\n')
    monkeypatch.chdir(tmp_path)
    cfg = train.load_run_config(str(run))
    assert cfg["model"]["model"]["filters"] == 64 and cfg["model"]["model"]["residual_blocks"] == 8
    assert cfg["model"]["optimizer"] == {"learning_rate": 2e-4, "betas": [0.5, 0.9]}
    assert cfg["dataset"]["lr"]["max"] == 0.002 and cfg["dataset"]["hr"]["max"] == 0.0005
    assert cfg["loss"]["ms_ssim"] == 0.75 and cfg["sc_dict"]["l1"] == {"scaling": 9.5, "correction": -0.5}
    # without the files: the run file's own tables, unscaled
    monkeypatch.chdir(tmp_path / "res")
    cfg = train.load_run_config(str(run))
    assert cfg["sc_dict"] is None and cfg["model"]["model"]["filters"] == 32
