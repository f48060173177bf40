"""Generate tests/golden/*.npz by RUNNING THE REFERENCE (imported from /root/reference by file
path; see oracle/ref_loader.py) -- TEST INFRASTRUCTURE.  Run in the authoring container:

    python -m oracle.make_golden

The reference ships no tests or golden vectors (SURVEY.md section 4), so these fixtures are
"outputs of the reference itself run here".  Weights and inputs are closed-form
(``rrdb_oracle.init_state_dict`` / ``splitmix_uniform``), so the fixtures hold only the
reference's outputs plus one example count image (config 1 of BASELINE.json).
"""
from __future__ import annotations

import os

import numpy as np
import torch

from . import rrdb_oracle as O
from .fits_min import read_primary
from .ref_loader import REF_ROOT, load_reference
from .synthetic import pad_to

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
EXAMPLE = "data/example_data/real/20ks/0852030101_image_split_500_2000_20ks_3_1.fits"
LR_MAX = 0.0022336


def det_input(shape, seed: int) -> torch.Tensor:
    n = int(np.prod(shape))
    return torch.from_numpy(O.splitmix_uniform(n, seed).astype("float32")).reshape(shape)


def counts_like_input(shape, seed: int) -> torch.Tensor:
    """Discrete sqrt-stretched count values min(1, sqrt(k/44.672)) -- what real inputs look like."""
    u = O.splitmix_uniform(int(np.prod(shape)), seed)
    k = np.floor(-np.log(1 - u) * 1.2)  # geometric-ish counts, mean ~1
    return torch.from_numpy(np.minimum(1.0, np.sqrt(k / 44.672)).astype("float32")).reshape(shape)


def probe_like(shape, seed: int) -> torch.Tensor:
    """Positive, non-constant cotangent for the backward fixtures.  A zero-mean probe makes every
    gradient a near-cancelling sum, whose relative error then measures clamp-boundary flips of a
    reduced-precision forward rather than the backward arithmetic; real loss gradients are coherent."""
    return det_input(shape, seed) * 0.5 + 0.25


def grad_summary(g: torch.Tensor) -> np.ndarray:
    g = g.detach().double().reshape(-1)
    return np.array([g.sum().item(), g.norm().item(), g.abs().max().item()])


def net_case(ref, kind: str, nf: int, nb: int, seed: int, shape, counts: bool):
    cls = ref.GeneratorRRDB_DN if kind == "dn" else ref.GeneratorRRDB_SR
    kwargs = dict(in_channels=1, out_channels=1, num_filters=nf, num_res_blocks=nb)
    if kind == "sr":
        kwargs["num_upsample"] = 1
    model = cls(**kwargs)
    sd = O.init_state_dict(kind, 1, 1, nf, nb, 1, seed=seed)
    missing = model.load_state_dict(sd, strict=True)
    assert not missing.missing_keys and not missing.unexpected_keys
    x = (counts_like_input if counts else det_input)(shape, seed + 17)
    x.requires_grad_(True)
    out = torch.clamp(model(x), 0.0, 1.0)  # Model.forward, models/model.py:48-49
    probe = probe_like(tuple(out.shape), seed + 29)
    (out * probe).sum().backward()
    res = {"out": out.detach().numpy(), "grad_x": x.grad.numpy()}
    for name, p in model.named_parameters():
        res[f"gsum.{name}"] = grad_summary(p.grad)
    for name in ("conv_first.weight", "conv_last.weight", "rrdb.0.RDB2.conv3.weight", "trunk_conv.bias"):
        res[f"grad.{name}"] = dict(model.named_parameters())[name].grad.numpy()
    return res


INIT_SEED, INIT_NF, INIT_NB = 123, 32, 2
INIT_SAMPLES = 64  # values kept per tensor: the full state_dict (3.4 MB per generator) is too large to store


def init_fingerprint(cls, kind: str) -> dict:
    """What ``torch.manual_seed(123); cls(1, 1, 32, 2[, num_upsample=1]).state_dict()`` holds: keys in order, element
    counts, INIT_SAMPLES evenly spaced values of every tensor (exact fp32) and its float64 sum and sum of squares."""
    torch.manual_seed(INIT_SEED)
    model = cls(1, 1, INIT_NF, INIT_NB) if kind == "dn" else cls(1, 1, INIT_NF, INIT_NB, num_upsample=1)
    flat = [v.detach().reshape(-1) for v in model.state_dict().values()]
    picks = [np.linspace(0, v.numel() - 1, min(v.numel(), INIT_SAMPLES)).round().astype(np.int64) for v in flat]
    return {"keys": np.array(list(model.state_dict().keys())),
            "numel": np.array([v.numel() for v in flat]),
            "sample": np.concatenate([v.numpy()[i] for v, i in zip(flat, picks)]),
            "moments": np.array([[v.double().sum().item(), v.double().square().sum().item()] for v in flat])}


def write_init_golden(gen_dn, gen_sr, source: str) -> None:
    """tests/golden/init_seed123.npz: the default initialisation of both generators under one seed."""
    res = {"source": np.array(source)}
    for kind, cls in (("dn", gen_dn), ("sr", gen_sr)):
        res.update({f"{kind}.{k}": v for k, v in init_fingerprint(cls, kind).items()})
    np.savez_compressed(os.path.join(OUT, "init_seed123.npz"), **res)


def main() -> None:
    os.makedirs(OUT, exist_ok=True)
    torch.manual_seed(0)
    torch.set_num_threads(8)
    ref = load_reference()

    # (A) network forward (seeds chosen so that most outputs fall strictly inside the clamp range) + backward, reference classes, closed-form weights/inputs
    cases = {
        "dn_f32_nb1_rand": ("dn", 32, 1, 25, (2, 1, 32, 32), False),
        "sr_f32_nb1_rand": ("sr", 32, 1, 15, (2, 1, 32, 32), False),
        "dn_f32_nb2_counts": ("dn", 32, 2, 10, (1, 1, 48, 40), True),
        "sr_f32_nb2_counts": ("sr", 32, 2, 29, (1, 1, 48, 40), True),
        "dn_f8_nb1_rand": ("dn", 8, 1, 19, (2, 1, 24, 24), False),
        "sr_f8_nb1_rand": ("sr", 8, 1, 21, (2, 1, 24, 24), False),
    }
    for name, (kind, nf, nb, seed, shape, counts) in cases.items():
        res = net_case(ref, kind, nf, nb, seed, shape, counts)
        res["meta"] = np.array([{"dn": 0, "sr": 1}[kind], nf, nb, seed, int(counts)] + list(shape))
        np.savez_compressed(os.path.join(OUT, f"net_{name}.npz"), **res)
        print(name, res["out"].shape, float(res["out"].mean()))

    # (B) BASELINE.json config 1: DeNoise, one real example image, F=32 nb=4, fp32 CPU reference
    counts, hdr = read_primary(os.path.join(REF_ROOT, EXAMPLE))
    exposure = float(hdr["EXPOSURE"])
    assert counts.shape == (411, 403) and counts.max() < 256
    padded = pad_to(counts.astype(np.float32), 416)
    norm = ref.Normalize(lr_max=LR_MAX, hr_max=LR_MAX, stretch_mode="sqrt")
    lr = norm.normalize_lr_image(torch.from_numpy(padded / exposure)[None])  # (1,416,416) rate units (SURVEY I4)
    model = ref.GeneratorRRDB_DN(1, 1, 32, 4)
    model.load_state_dict(O.init_state_dict("dn", 1, 1, 32, 4, seed=21))
    with torch.no_grad():
        out = torch.clamp(model(lr[None]), 0.0, 1.0)[0, 0].numpy()
    blocks = out.reshape(26, 16, 26, 16).mean(axis=(1, 3))
    stats = np.array([out.mean(), out.std(), np.sqrt((out.astype(np.float64) ** 2).sum()), out.min(), out.max(),
                      (out == 1.0).mean(), (out == 0.0).mean()], dtype=np.float64)
    np.savez_compressed(os.path.join(OUT, "config1_dn_example.npz"), counts=counts.astype(np.uint8),
                        exposure=np.array(exposure), lr_crop=lr[0, 176:240, 176:240].numpy(),
                        out_crop=out[176:240, 176:240], out_blocks=blocks.astype(np.float32), out_stats=stats,
                        seed=np.array(21))
    print("config1", stats)

    # (C) Normalize, all stretch modes + the max_val<=0 branch + denorm callables
    vals = np.concatenate([np.array([-1e-3, 0.0, 1e-9, 5e-5, 1e-4, 1.1168e-3, 2.2336e-3, 2.3e-3, 1.0], dtype=np.float32),
                           (O.splitmix_uniform(247, 5) * 3e-3).astype(np.float32)])
    res = {"vals": vals}
    for mode in ("linear", "sqrt", "asinh", "log"):
        n = ref.Normalize(lr_max=LR_MAX, hr_max=0.0005584, stretch_mode=mode)
        res[f"lr.{mode}"] = n.normalize_lr_image(torch.from_numpy(vals.copy())).numpy()
        res[f"hr.{mode}"] = n.normalize_hr_image(torch.from_numpy(vals.copy())).numpy()
        res[f"dynmax.{mode}"] = n.normalize_image(torch.from_numpy(np.abs(vals)), torch.tensor(0.0)).numpy()
        unit = torch.linspace(0, 1, 33)
        res[f"denormfn.{mode}"] = n.denorm(unit.clone()).numpy()
        res[f"denorm.{mode}"] = n.denormalize_image(unit.clone().reshape(1, 1, 3, 11), torch.tensor([LR_MAX])).numpy()
    np.savez_compressed(os.path.join(OUT, "normalize.npz"), **res)

    # (D) ImageUpsample
    img = det_input((2, 1, 5, 7), 77)
    np.savez_compressed(os.path.join(OUT, "imageupsample.npz"), x=img.numpy(),
                        up2=ref.ImageUpsample(2)(img).numpy(), up3_single=ref.ImageUpsample(3)(img[0]).numpy())

    # (E) default initialisation under a fixed seed
    write_init_golden(ref.GeneratorRRDB_DN, ref.GeneratorRRDB_SR, "reference classes")
    print("golden fixtures written to", OUT)


if __name__ == "__main__":
    main()
