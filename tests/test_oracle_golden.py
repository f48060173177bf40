"""CPU: pin the oracle restatement to what the reference itself computed (tests/golden, generated
by oracle/make_golden.py from the live reference), and -- when /root/reference is mounted -- to
the live reference classes on fresh inputs."""
import os

import numpy as np
import pytest
import torch

from oracle import ref_loader
from oracle import rrdb_oracle as O
from oracle.make_golden import LR_MAX, counts_like_input, det_input, probe_like
from oracle.synthetic import pad_to

from helpers import load_case, rel_l2

NET_CASES = ["dn_f32_nb1_rand", "sr_f32_nb1_rand", "dn_f32_nb2_counts", "sr_f32_nb2_counts", "dn_f8_nb1_rand",
             "sr_f8_nb1_rand"]


@pytest.mark.parametrize("name", NET_CASES)
def test_network_forward_backward_matches_reference_golden(golden_dir, name):
    g, kind, nf, nb, seed, counts, shape = load_case(golden_dir, name)
    sd = {k: v.clone().requires_grad_(True) for k, v in O.init_state_dict(kind, 1, 1, nf, nb, 1, seed=seed).items()}
    x = (counts_like_input if counts else det_input)(shape, seed + 17).requires_grad_(True)
    out = O.model_forward(x, sd, kind, 1)
    assert out.shape == g["out"].shape
    np.testing.assert_allclose(out.detach().numpy(), g["out"], rtol=0, atol=2e-6)
    probe = probe_like(tuple(out.shape), seed + 29)
    (out * probe).sum().backward()
    assert rel_l2(x.grad, g["grad_x"]) < 1e-5
    for key in g.files:
        if key.startswith("grad."):
            assert rel_l2(sd[key[5:]].grad, g[key]) < 1e-5, key
        if key.startswith("gsum."):
            gr = sd[key[5:]].grad.double()
            assert abs(float(gr.norm()) - g[key][1]) <= 1e-5 * max(g[key][1], 1e-12), key


def test_config1_example_image_matches_reference_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "config1_dn_example.npz"))
    counts = g["counts"].astype(np.float32)
    lr = O.normalize_image(torch.from_numpy(pad_to(counts, 416) / float(g["exposure"])), LR_MAX, "sqrt")
    np.testing.assert_allclose(lr[176:240, 176:240].numpy(), g["lr_crop"], rtol=0, atol=1e-7)
    sd = O.init_state_dict("dn", 1, 1, 32, 4, seed=int(g["seed"]))
    torch.set_num_threads(os.cpu_count() or 1)
    with torch.no_grad():
        out = O.model_forward(lr[None, None], sd, "dn")[0, 0].numpy()
    np.testing.assert_allclose(out[176:240, 176:240], g["out_crop"], rtol=0, atol=5e-6)
    np.testing.assert_allclose(out.reshape(26, 16, 26, 16).mean(axis=(1, 3)), g["out_blocks"], rtol=0, atol=5e-6)
    assert abs(out.mean() - g["out_stats"][0]) < 1e-6


def test_normalize_matches_reference_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "normalize.npz"))
    vals = torch.from_numpy(g["vals"])
    for mode in ("linear", "sqrt", "asinh", "log"):
        np.testing.assert_allclose(O.normalize_image(vals, LR_MAX, mode).numpy(), g[f"lr.{mode}"], rtol=0, atol=1e-7)
        np.testing.assert_allclose(O.normalize_image(vals, 0.0005584, mode).numpy(), g[f"hr.{mode}"], rtol=0, atol=1e-7)
        np.testing.assert_allclose(O.normalize_image(vals.abs(), 0.0, mode).numpy(), g[f"dynmax.{mode}"], rtol=0,
                                   atol=1e-7)
        unit = torch.linspace(0, 1, 33)
        np.testing.assert_allclose(O.unstretch(unit, mode).numpy(), g[f"denormfn.{mode}"], rtol=1e-6, atol=1e-9)
        np.testing.assert_allclose(O.denormalize_image(unit.reshape(1, 1, 3, 11), torch.tensor([LR_MAX]), mode).numpy(),
                                   g[f"denorm.{mode}"], rtol=1e-6, atol=1e-10)
    with pytest.raises(ValueError):
        O.stretch(vals, "cbrt")


def test_image_upsample_matches_reference_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "imageupsample.npz"))
    x = torch.from_numpy(g["x"])
    np.testing.assert_array_equal(O.image_upsample(x, 2).numpy(), g["up2"])
    np.testing.assert_array_equal(O.image_upsample(x[0], 3).numpy(), g["up3_single"])
    assert abs(float(O.image_upsample(x, 2).sum()) - float(x.sum())) < 1e-4  # brightness preserved


def test_combine_mask_pad_geometry():
    # data/tools.py:103-126: 411x403 -> 416x416 with 2 rows before / 3 after, 6 cols before / 7 after
    img = torch.ones(1, 411, 403)
    out = O.combine_mask_pad(img, None, None, None, 416)
    assert out.shape == (1, 416, 416)
    assert out[0, :2].sum() == 0 and out[0, 413:].sum() == 0 and out[0, 2:413, 6:409].min() == 1
    assert out[0, :, :6].sum() == 0 and out[0, :, 409:].sum() == 0
    m = torch.zeros(411, 403)
    m[100:200] = 1
    out = O.combine_mask_pad(img, img * 2, img * 3, m, 416)
    assert float(out.sum()) == 6 * 100 * 403


@pytest.mark.skipif(not ref_loader.available(),
                    reason="needs the reference's source tree (XMM_REFERENCE_ROOT, or its copy in oracle/_ref)")
@pytest.mark.parametrize("kind", ["dn", "sr"])
def test_oracle_matches_live_reference(kind):
    ref = ref_loader.load_reference()
    torch.manual_seed(5)
    model = (ref.GeneratorRRDB_DN(1, 1, 16, 2) if kind == "dn" else ref.GeneratorRRDB_SR(1, 1, 16, 2, num_upsample=1))
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    x = torch.rand(2, 1, 20, 28)
    with torch.no_grad():
        want = torch.clamp(model(x), 0, 1)
        got = O.model_forward(x, sd, kind, 1)
    assert torch.allclose(got, want, atol=2e-6)
    # the oracle's closed-form init has the reference's keys and shapes
    mine = O.init_state_dict(kind, 1, 1, 16, 2, 1, seed=1)
    assert sorted(mine.keys()) == sorted(sd.keys())
    assert {k: tuple(v.shape) for k, v in mine.items()} == {k: tuple(v.shape) for k, v in sd.items()}
