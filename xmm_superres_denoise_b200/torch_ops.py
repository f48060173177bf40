"""``torch.ops.xmm_b200.*`` -- the torch custom-op face of the C ABI (SURVEY.md section 8b).

``csrc/torch_ops.cpp`` registers ``TORCH_LIBRARY(xmm_b200, m)`` shims (CUDA dispatch key only: a CPU tensor raises
``NotImplementedError`` from the dispatcher -- there is no fallback) over the ``extern "C"`` launchers of
``libxmm_b200.so``.  ``load()`` loads ``libxmm_b200_torch.so`` once; afterwards

    torch.ops.xmm_b200.conv3x3_fwd(inp, in_coff, cin, wblob, kc, cout, out, out_coff, lrelu=0.2, wblob_row=...)
    torch.ops.xmm_b200.conv3x3_dgrad / normalize / denormalize / image_upsample / adam_step / abi_version
    torch.ops.xmm_b200.grad_clip_coef / adam_step_clip  (gradient clipping, training.FusedAdam)

are ordinary dispatcher ops (mutating their ``out`` argument, returning nothing).  The engine itself keeps calling
the launchers through ctypes (``_lib.py``): both faces end in the same C entry point, and the engine's calls are
either GPU-bound (large batches) or replayed from a CUDA graph (small batches), so the per-call host cost does not
show in throughput; ``ops.conv3x3`` routes through the registered op when ``XMM_TORCH_OPS=1``.
"""
from __future__ import annotations

import os

import torch

from . import _lib

TORCH_LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "libxmm_b200_torch.so")
_loaded = False


def load():
    """Register the ops (idempotent); returns ``torch.ops.xmm_b200``."""
    global _loaded
    if not _loaded:
        _lib.load()  # libxmm_b200.so first: clearer error when nothing is built
        if not os.path.exists(TORCH_LIB_PATH):
            raise RuntimeError(f"{TORCH_LIB_PATH} is not built. Run `python -c 'import __graft_entry__ as g; g.build()'`.")
        torch.ops.load_library(TORCH_LIB_PATH)
        if torch.ops.xmm_b200.abi_version() != _lib.load().xmm_version():
            raise RuntimeError("libxmm_b200_torch.so and libxmm_b200.so disagree on the ABI version: rebuild both")
        _loaded = True
    return torch.ops.xmm_b200
