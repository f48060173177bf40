"""Shared helpers for the parity tests (tolerances are the ones BASELINE.json's north_star states)."""
from __future__ import annotations

import os

import numpy as np
import torch
import torch.nn.functional as F

# bf16 compute: per-pixel relative L2 <= 1e-2; loss / gradient relative error <= 1e-2
REL_L2_BF16 = 1e-2
GRAD_REL = 1e-2
PSNR_DELTA_DB = 0.05

# per-element bounds (assert_bf16_elementwise): c of |got - ref| <= ulp(ref) + lip * c * S, fixed by
# tests/test_elementwise_checker.py (correct rounding passes, every local fault there fails)
C_TC = 2.0 ** -16     # tensor-core 3x3 layers: bf16 operands, fp32 accumulation, bf16 output
C_LAST = 2.0 ** -14   # conv_last: fp32 output; on the tensor cores fp32 weights as bf16 hi + lo halves
C_FIRST = 2.0 ** -18  # conv_first: <= 36 fp32 FMAs, one bf16 rounding
REL_LAST = 2e-5       # rel-L2 of conv_last's un-clamped output (bf16 hi alone: 1.6e-3)


def rel_l2(a, b) -> float:
    a = torch.as_tensor(a).double().reshape(-1).cpu()
    b = torch.as_tensor(b).double().reshape(-1).cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def psnr_db(a, b, data_range: float = 1.0) -> float:
    a = torch.as_tensor(a).double().cpu()
    b = torch.as_tensor(b).double().cpu()
    mse = float(((a - b) ** 2).mean())
    return float("inf") if mse == 0 else 10.0 * np.log10(data_range ** 2 / mse)


def _f64(t, device) -> torch.Tensor:
    return torch.as_tensor(t).to(device=device, dtype=torch.float64)


def ulp_bf16(v, mant_bits: int = 7) -> torch.Tensor:
    """Unit in the last place of |v| in a format with `mant_bits` stored mantissa bits (7: bf16, 23: fp32):
    2^(floor(log2|v|) - mant_bits), floored at the smallest normal (2^-126)."""
    e = torch.floor(torch.log2(torch.as_tensor(v).double().abs().clamp_min(2.0 ** -126)))
    return torch.exp2(e - mant_bits)


def assert_bf16_elementwise(got, ref, S, c: float, lip: float = 1.0, what: str = "", mant_bits: int = 7,
                            extra=None) -> float:
    """Per-element check of a kernel's output against a float64 reference of the same operation on the same
    (bf16-exact) operands:  |got - ref| <= ulp_bf16(ref) + lip * c * S  for every element.

    S = sum |w| * |x| + |bias| (the absolute-value convolution, `abs_conv`) bounds what fp32 accumulation in any
    order can lose: c ~ 2^-16 covers the tensor-core layers, 2^-18 the 36 FMAs of conv_first.  `lip` is the
    Lipschitz factor of the epilogue after the accumulation (s0 of a residual layer).  ulp_bf16(ref) takes the final
    rounding to the output format (half an ulp) with a half-ulp margin; `mant_bits=23` makes it fp32's.  `extra`
    (same shape, optional) is an absolute allowance added to c * S, for elements whose operands the kernel may
    legitimately see differently from the reference (see test_gpu_elementwise.py's band seam).

    Tensors are 4-D [B, C, H, W] (any device; the check runs in float64 on ref's device).  On failure the message
    gives the number of violations, the worst element's (b, y, x, c), got, ref, its bound and the largest
    |err| / bound.  Returns that largest ratio, so that a test can print it."""
    ref = torch.as_tensor(ref)
    dev = ref.device
    ref, got, S = _f64(ref, dev), _f64(got, dev), _f64(S, dev)
    if got.shape != ref.shape or S.shape != ref.shape or ref.dim() != 4:
        raise ValueError(f"{what}: shapes got {tuple(got.shape)}, ref {tuple(ref.shape)}, S {tuple(S.shape)}")
    bound = ulp_bf16(ref, mant_bits) + lip * (c * S + (0.0 if extra is None else _f64(extra, dev)))
    ratio = (got - ref).abs() / bound
    ratio = torch.where(torch.isnan(ratio), torch.full_like(ratio, float("inf")), ratio)  # NaN / Inf in got fail
    worst = int(torch.argmax(ratio))
    rmax = float(ratio.reshape(-1)[worst])
    bad = int((ratio > 1.0).sum())
    if bad:
        b, ch, y, x = np.unravel_index(worst, tuple(ref.shape))
        raise AssertionError(
            f"{what}: {bad} of {ref.numel()} elements outside |got - ref| <= ulp_bf16(ref) + {lip:g} * {c:.3g} * S; "
            f"worst at (b, y, x, c) = ({b}, {y}, {x}, {ch}): got {float(got[b, ch, y, x]):.8g}, "
            f"ref {float(ref[b, ch, y, x]):.8g}, bound {float(bound[b, ch, y, x]):.3g}, max |err|/bound = {rmax:.3f}")
    return rmax


def _threads(t: torch.Tensor) -> None:
    if t.device.type == "cpu":
        torch.set_num_threads(os.cpu_count() or 1)


def ref_conv(x, w, b=None) -> torch.Tensor:
    """3x3, padding 1, in float64 on x's device: x [B, Cin, H, W], w [Cout, Cin, 3, 3], b [Cout] or None."""
    x = torch.as_tensor(x)
    _threads(x)
    dev = x.device
    return F.conv2d(_f64(x, dev), _f64(w, dev), None if b is None else _f64(b, dev), padding=1)


def abs_conv(x, w, b=None) -> torch.Tensor:
    """S of `assert_bf16_elementwise`: sum |w| * |x| + |b| over each output's window, float64."""
    x = torch.as_tensor(x)
    return ref_conv(x.abs(), torch.as_tensor(w).abs(), None if b is None else torch.as_tensor(b).abs())


def load_case(golden_dir: str, name: str):
    g = np.load(os.path.join(golden_dir, f"net_{name}.npz"))
    kind_i, nf, nb, seed, counts = (int(v) for v in g["meta"][:5])
    shape = tuple(int(v) for v in g["meta"][5:])
    return g, ("dn", "sr")[kind_i], nf, nb, seed, bool(counts), shape
