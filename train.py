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
* [trainer] accumulate_grad_batches (Lightning's ``Trainer`` argument; ``--accumulate-grad-batches`` overrides it;
  default 1): k micro-batches of ``batch_size`` per optimizer step, their gradients added in place, one all-reduce and
  one Adam step per window (``TrainStep``).  ``--steps`` counts optimizer steps, each consuming k seeded micro-batches;
  the printed img/s counts every image and the printed loss is the mean over the window.  As under Lightning, the loss
  terms are defined per micro-batch (the Poisson term's division by the batch size, MS-SSIM's data range), so this is
  not one batch of k * batch_size;
* [trainer] gradient_clip_val and gradient_clip_algorithm (Lightning's ``Trainer`` arguments;
  ``--gradient-clip-val`` / ``--gradient-clip-algorithm`` override them; default: no clipping, algorithm "norm"): the
  averaged gradient of every optimizer step is clipped by its global L2 norm (``clip_grad_norm_``) or by value
  (``clip_grad_value_``) before Adam; 0 turns clipping off.  With "norm" the printed lines add the pre-clip norm;
* ``res/configs/loss_functions.toml`` (train.py:45-53) when present: the [loss] percentages and, with
  ``use_scaling = true``, the [scaling.<dataset scaling>] table as ``sc_dict`` of ``create_loss``.  Without the file the
  [loss] table of the run file is used, unscaled (the scaling constants live in that file only).

    python train.py fit run.toml [--synthetic] [--steps N] [--deterministic] [--accumulate-grad-batches K]
                                 [--gradient-clip-val V] [--gradient-clip-algorithm {norm,value}]
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
    "trainer": {"epochs": 1, "deterministic": False, "accumulate_grad_batches": 1, "gradient_clip_val": None,
                "gradient_clip_algorithm": "norm"},
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


def accumulate_grad_batches(cfg: dict, flag) -> int:
    """--accumulate-grad-batches (when given) or [trainer] accumulate_grad_batches: micro-batches per optimizer step."""
    k = flag if flag is not None else cfg["trainer"].get("accumulate_grad_batches", 1)
    if isinstance(k, bool) or not isinstance(k, int) or k < 1:
        raise ValueError(f"accumulate_grad_batches = {k!r}: expected an integer >= 1")
    return k


def gradient_clip(cfg: dict, val_flag, algorithm_flag):
    """--gradient-clip-val / --gradient-clip-algorithm (when given) or [trainer] gradient_clip_val /
    gradient_clip_algorithm, checked as TrainStep checks them: (max value or None when off, algorithm)."""
    from xmm_superres_denoise_b200.training import gradient_clip_settings

    t = cfg["trainer"]
    val = val_flag if val_flag is not None else t.get("gradient_clip_val")
    algorithm = algorithm_flag if algorithm_flag is not None else t.get("gradient_clip_algorithm", "norm")
    return gradient_clip_settings(val, algorithm)


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


def parser() -> argparse.ArgumentParser:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("routine", choices=["fit"])
    ap.add_argument("config", nargs="?", default=None, help="run TOML (reference layout); defaults are the DeNoise setup")
    ap.add_argument("--synthetic", action="store_true")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--deterministic", action="store_true",
                    help="bit-reproducible training on one GPU ([trainer] deterministic = true does the same)")
    ap.add_argument("--accumulate-grad-batches", type=int, default=None, metavar="K",
                    help="micro-batches per optimizer step (default: [trainer] accumulate_grad_batches, else 1)")
    ap.add_argument("--gradient-clip-val", type=float, default=None, metavar="V",
                    help="clip each optimizer step's averaged gradient at V (0: off; default: [trainer] "
                         "gradient_clip_val, else off)")
    ap.add_argument("--gradient-clip-algorithm", default=None, metavar="{norm,value}",
                    help="clip by global L2 norm (default) or by value (default: [trainer] gradient_clip_algorithm)")
    return ap


def main() -> None:
    a = parser().parse_args()
    cfg = load_run_config(a.config)
    k = accumulate_grad_batches(cfg, a.accumulate_grad_batches)
    clip_val, clip_algorithm = gradient_clip(cfg, a.gradient_clip_val, a.gradient_clip_algorithm)
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
    step = TrainStep(model.model, loss, lr=mcfg.optimizer.learning_rate, betas=tuple(mcfg.optimizer.betas),
                     accumulate_grad_batches=k, gradient_clip_val=clip_val, gradient_clip_algorithm=clip_algorithm)
    t0 = time.time()
    for it in range(a.steps):  # optimizer steps; micro-batch m = it * k + j has seed 1234 + rank + world * m
        vals = []
        for j in range(k):
            x, y = synthetic_batch(kind, mcfg.batch_size, 1234 + rank + world * (it * k + j), cfg, dev)
            vals.append(step(x, y))
        if rank == 0 and (it % 5 == 0 or it == a.steps - 1):
            val = vals[0] if k == 1 else torch.stack(vals).mean()
            rate = (it + 1) * k * mcfg.batch_size * world / (time.time() - t0)
            norm = "" if step.grad_norm is None else f"  grad_norm {float(step.grad_norm):.5g}"
            print(f"step {it:4d}  train/loss {float(val):.5f}{norm}  ({rate:.1f} img/s)")
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
