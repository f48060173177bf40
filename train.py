#!/usr/bin/env python
"""Training entry point (reference: xmm_superres_denoise/train.py:19-165 ``python train.py fit run.toml``).

The reference builds DatasetCfg / ModelCfg / LossCfg / TrainerCfg from a TOML run file plus ``res/configs/models.toml``
and ``res/configs/loss_functions.toml`` and hands a LightningModule to ``lightning.Trainer``.  Lightning, astropy and
the pydantic schemas are outside the accelerated path (SURVEY.md section 2: out of scope) and not installed here, so
this script is the plain-torch loop of ``xmm_superres_denoise_b200.training.TrainStep`` -- engine-direct
forward/backward, NCCL all-reduce overlapped with backward, fused Adam -- on seeded Poisson count images of the
reference shape (``--synthetic``; FITS directories need the reference's XmmDataModule).  There is no ``test``
routine and no Lightning branch.  What it keeps of the reference's configuration, under the reference's key names:

* the run file's [model] name / memory_efficient / batch_size, [dataset] scaling, lr / hr ``res``, ``exps`` / ``exp`` and
  ``clamp_max`` (train.py:66-67: the normalisation maxima; ``max`` is accepted as an alias), [trainer] epochs;
* ``res/configs/models.toml`` (train.py:35-36) when present in the working directory: the table named by
  [model].name supplies in/out channels, filters, residual_blocks, learning_rate and betas;
* [trainer] deterministic (Lightning's ``Trainer(deterministic=...)``; ``--deterministic`` sets it too):
  ``torch.use_deterministic_algorithms(True)`` and a seeded torch generator, so two runs of the same configuration on
  the same GPU give the same weights bit for bit (the gradient all-reduce of multi-GPU runs is outside that promise);
* ``res/configs/loss_functions.toml`` (train.py:45-53) when present: the [loss] percentages and, with
  ``use_scaling = true``, the [scaling.<dataset scaling>] table as ``sc_dict`` of ``create_loss``.  Without the file the
  [loss] table of the run file is used, unscaled (the scaling constants live in that file only).

    python train.py fit run.toml [--synthetic] [--steps N] [--deterministic]
    python -m torch.distributed.run --nproc-per-node 8 train.py fit run.toml --synthetic
"""
from __future__ import annotations

import argparse
import os
import sys
import time
import types

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import numpy as np  # noqa: E402
import torch  # noqa: E402

DEFAULTS = {
    "model": {"name": "rrdb_denoise", "memory_efficient": False, "batch_size": 16,
              "model": {"in_channels": 1, "out_channels": 1, "filters": 32, "residual_blocks": 4},
              "optimizer": {"learning_rate": 1e-4, "betas": [0.9, 0.999]}},
    "loss": {"l1": 0.5, "poisson": 0.5, "psnr": 0.0, "ssim": 0.0, "ms_ssim": 0.0, "use_scaling": True},
    "dataset": {"scaling": "sqrt", "lr": {"max": 0.0022336, "res": 416, "exps": [20]},
                "hr": {"max": 0.0022336, "res": 416, "exp": 50}},
    "trainer": {"epochs": 1, "deterministic": False},
}

DETERMINISTIC_SEED = 0


def _merge(base: dict, over: dict) -> dict:
    out = dict(base)
    for k, v in over.items():
        out[k] = _merge(base[k], v) if isinstance(v, dict) and isinstance(base.get(k), dict) else v
    return out


def _ns(d):
    return types.SimpleNamespace(**{k: _ns(v) if isinstance(v, dict) else v for k, v in d.items()})


def load_run_config(path):
    import tomllib

    cfg = dict(DEFAULTS)
    if path:
        with open(path, "rb") as f:
            cfg = _merge(DEFAULTS, tomllib.load(f))
    for side in ("lr", "hr"):  # train.py:66-67 reads dataset.<side>.clamp_max
        if "clamp_max" in cfg["dataset"][side]:
            cfg["dataset"][side]["max"] = cfg["dataset"][side]["clamp_max"]
    models_toml = os.path.join("res", "configs", "models.toml")  # train.py:35-42
    if os.path.exists(models_toml):
        with open(models_toml, "rb") as f:
            table = tomllib.load(f).get(cfg["model"]["name"])
        if table is not None:
            table = dict(table)
            cfg["model"]["optimizer"] = {"learning_rate": table.pop("learning_rate"), "betas": table.pop("betas")}
            cfg["model"]["model"] = _merge(cfg["model"]["model"], table)
    cfg["sc_dict"] = None
    loss_toml = os.path.join("res", "configs", "loss_functions.toml")  # train.py:45-53
    if os.path.exists(loss_toml):
        with open(loss_toml, "rb") as f:
            lc = tomllib.load(f)
        cfg["loss"] = dict(lc["loss"])
        if cfg["loss"].get("use_scaling"):
            cfg["sc_dict"] = lc["scaling"][cfg["dataset"]["scaling"]]
    return cfg


def configure_determinism(cfg: dict, flag: bool) -> bool:
    """--deterministic or [trainer] deterministic = true: deterministic algorithms (the engine's reductions then run in
    a fixed order, determinism.enabled) and a seeded torch generator (the initial weights).  Returns the mode."""
    det = bool(flag) or bool(cfg["trainer"].get("deterministic", False))
    if det:
        os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")  # what torch asks of cuBLAS under the flag
        torch.use_deterministic_algorithms(True)
        torch.manual_seed(DETERMINISTIC_SEED)
    return det


def synthetic_batch(kind: str, batch: int, seed: int, cfg: dict, device):
    """Seeded Poisson count images of the reference shape (SURVEY.md 8d), normalised on the GPU."""
    from xmm_superres_denoise_b200 import ops

    rng = np.random.default_rng(seed)
    lam = 0.11 + 3.0 * rng.random((batch, 1, 1)) * np.exp(-((np.arange(411)[None, :, None] - 205) ** 2 +
                                                               (np.arange(403)[None, None, :] - 201) ** 2) / 8000.0)
    d = cfg["dataset"]
    lr = torch.from_numpy(rng.poisson(lam).astype(np.int32)).to(device)
    up = 2 if kind == "sr" else 1
    lam_hr = np.repeat(np.repeat(lam, up, 1), up, 2) * (d["hr"]["exp"] / d["lr"]["exps"][0]) / up ** 2
    hr = torch.from_numpy(rng.poisson(lam_hr).astype(np.int32)).to(device)
    x = ops.prepare_counts([lr], d["lr"]["res"], d["lr"]["max"], d["scaling"], exposure=d["lr"]["exps"][0] * 1000.0)
    y = ops.prepare_counts([hr], d["hr"]["res"], d["hr"]["max"], d["scaling"], exposure=d["hr"]["exp"] * 1000.0)
    return x, y


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("routine", choices=["fit"])
    ap.add_argument("config", nargs="?", default=None, help="run TOML (reference layout); defaults are the DeNoise setup")
    ap.add_argument("--synthetic", action="store_true")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--deterministic", action="store_true",
                    help="bit-reproducible training on one GPU ([trainer] deterministic = true does the same)")
    a = ap.parse_args()
    cfg = load_run_config(a.config)
    configure_determinism(cfg, a.deterministic)

    import torch.distributed as dist

    from xmm_superres_denoise_b200.models import Model
    from xmm_superres_denoise_b200.training import TrainStep
    from xmm_superres_denoise_b200.utils.loss_functions import create_loss

    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("NCCL_MAX_CTAS", "4")  # a 6.7 MB all-reduce needs no more; see TrainStep.sm_reserve
        dist.init_process_group("nccl")
    if not a.synthetic:
        raise SystemExit("FITS datasets are read by the reference's XmmDataModule (astropy); run with --synthetic here, "
                         "or feed raw count planes through xmm_superres_denoise_b200.data.CountsFeed")
    mcfg = _ns(cfg["model"])
    d = cfg["dataset"]
    kind = "sr" if d["hr"]["res"] > d["lr"]["res"] else "dn"
    mcfg.name = "esr_gen" if kind == "sr" else "rrdb_denoise"
    loss = create_loss(cfg["sc_dict"], {k: float(v) for k, v in cfg["loss"].items() if k != "use_scaling"}).to(dev)
    model = Model(mcfg, (d["lr"]["res"],) * 2, (d["hr"]["res"],) * 2, loss)
    model.configure_model()
    model = model.to(dev).train()
    step = TrainStep(model.model, loss, lr=mcfg.optimizer.learning_rate, betas=tuple(mcfg.optimizer.betas))
    t0 = time.time()
    for it in range(a.steps):
        x, y = synthetic_batch(kind, mcfg.batch_size, 1234 + rank + world * it, cfg, dev)
        val = step(x, y)
        if rank == 0 and (it % 5 == 0 or it == a.steps - 1):
            print(f"step {it:4d}  train/loss {float(val):.5f}  ({(it + 1) * mcfg.batch_size * world / (time.time() - t0):.1f} img/s)")
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
