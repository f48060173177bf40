"""CPU: the host side of gradient clipping -- train.py's [trainer] gradient_clip_val / gradient_clip_algorithm and their
flags, the shared argument check, TrainStep's rejection of bad settings, and None / 0 meaning no clipping."""
import math
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


def test_settings_check():
    from xmm_superres_denoise_b200.training import gradient_clip_settings

    assert gradient_clip_settings() == (None, "norm")
    assert gradient_clip_settings(None, "value") == (None, "value")
    assert gradient_clip_settings(0, "norm") == (None, "norm")  # Lightning: 0 is off
    assert gradient_clip_settings(0.0, "value") == (None, "value")
    assert gradient_clip_settings(0.5) == (0.5, "norm")
    assert gradient_clip_settings(2, None) == (2.0, "norm")  # Lightning's None algorithm is "norm"
    assert gradient_clip_settings(math.inf, "value") == (math.inf, "value")
    for bad in (-1e-3, -2, math.nan, True, "1.0"):
        with pytest.raises(ValueError, match="gradient_clip_val"):
            gradient_clip_settings(bad)
    for bad in ("l2", "Norm", "", 2):
        with pytest.raises(ValueError, match="gradient_clip_algorithm"):
            gradient_clip_settings(1.0, bad)
    with pytest.raises(ValueError, match="gradient_clip_algorithm"):
        gradient_clip_settings(None, "inf")  # an unknown algorithm is an error even with clipping off


def test_train_py_keys_and_flags(tmp_path, train_mod):
    train = train_mod
    cfg = train.load_run_config(None)
    assert cfg["trainer"]["gradient_clip_val"] is None and cfg["trainer"]["gradient_clip_algorithm"] == "norm"
    assert train.gradient_clip(cfg, None, None) == (None, "norm")
    a = train.parser().parse_args(["fit"])
    assert a.gradient_clip_val is None and a.gradient_clip_algorithm is None
    run = tmp_path / "run.toml"
    run.write_text('[trainer]\ngradient_clip_val = 0.5\ngradient_clip_algorithm = "value"\n')
    cfg = train.load_run_config(str(run))
    assert cfg["trainer"]["accumulate_grad_batches"] == 1  # the other [trainer] defaults stay
    assert train.gradient_clip(cfg, None, None) == (0.5, "value")
    a = train.parser().parse_args(["fit", str(run), "--gradient-clip-val", "2.5"])
    assert train.gradient_clip(cfg, a.gradient_clip_val, a.gradient_clip_algorithm) == (2.5, "value")
    a = train.parser().parse_args(["fit", str(run), "--gradient-clip-algorithm", "norm"])
    assert train.gradient_clip(cfg, a.gradient_clip_val, a.gradient_clip_algorithm) == (0.5, "norm")
    a = train.parser().parse_args(["fit", str(run), "--gradient-clip-val", "0"])
    assert train.gradient_clip(cfg, a.gradient_clip_val, a.gradient_clip_algorithm) == (None, "value")  # flag turns it off
    run.write_text("[trainer]\ngradient_clip_val = 1\n")
    assert train.gradient_clip(train.load_run_config(str(run)), None, None) == (1.0, "norm")
    run.write_text("[trainer]\ngradient_clip_val = -1.0\n")
    with pytest.raises(ValueError, match="gradient_clip_val"):
        train.gradient_clip(train.load_run_config(str(run)), None, None)
    run.write_text('[trainer]\ngradient_clip_val = 1.0\ngradient_clip_algorithm = "l2"\n')
    with pytest.raises(ValueError, match="gradient_clip_algorithm"):
        train.gradient_clip(train.load_run_config(str(run)), None, None)
    with pytest.raises(ValueError, match="gradient_clip_val"):
        train.gradient_clip(train.load_run_config(None), -0.1, None)
    out = subprocess.run([sys.executable, os.path.join(entry.ROOT, "train.py"), "--help"], capture_output=True,
                         text=True, check=True).stdout
    assert "--gradient-clip-val" in out and "--gradient-clip-algorithm" in out


def test_trainstep_rejects_bad_settings():
    """The check runs before TrainStep touches the model or the GPU."""
    from xmm_superres_denoise_b200.training import TrainStep

    for val, algorithm, what in ((-1.0, "norm", "gradient_clip_val"), (math.nan, "value", "gradient_clip_val"),
                                 (1.0, "l2", "gradient_clip_algorithm")):
        with pytest.raises(ValueError, match=what):
            TrainStep(torch.nn.Linear(2, 2), None, gradient_clip_val=val, gradient_clip_algorithm=algorithm)


def test_fused_adam_clip_arguments_are_checked(monkeypatch):
    """FusedAdam.step rejects both clips at once and a non-positive clip_value before any launch (the CUDA-tensor check
    is stubbed so that CPU tensors get that far)."""
    from xmm_superres_denoise_b200 import training

    monkeypatch.setattr(training._lib, "require_cuda_tensor", lambda t, dtype, name: None)
    opt = training.FusedAdam(torch.zeros(4))
    with pytest.raises(ValueError, match="not both"):
        opt.step(torch.zeros(4), 1.0, clip_coef=torch.ones(1), clip_value=1.0)
    for bad in (0.0, -1.0, math.nan):
        with pytest.raises(ValueError, match="clip_value"):
            opt.step(torch.zeros(4), 1.0, clip_value=bad)
    assert opt.step_count == 0
