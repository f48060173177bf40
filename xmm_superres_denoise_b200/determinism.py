"""Deterministic training mode: bit-identical gradients from run to run.

Three reductions of the backward pass add partial sums with float atomics in an order that depends on CTA timing:
the bias gradients fused into the F = 32 data-gradient launches, the column-sum bias gradients, and the edge-layer
weight gradients (conv_last, conv_first).  In deterministic mode each of them stores its partial sums to its own
slots of a workspace instead, and one ``det_finalize`` launch per RRDB (just before that RRDB's gradient chunk is
handed to the all-reduce hook) and one for the edge layers add them in a fixed order.

The mode is off by default.  ``enabled()`` resolves it on every backward call: ``XMM_DETERMINISTIC=1`` / ``0`` when
set, otherwise ``torch.are_deterministic_algorithms_enabled()`` -- so ``torch.use_deterministic_algorithms(True)``
(what Lightning's ``Trainer(deterministic=True)`` calls) switches it on.
"""
from __future__ import annotations

import os
from typing import Callable, List, Optional, Tuple

import torch

from . import _lib, ops


def enabled() -> bool:
    env = os.environ.get("XMM_DETERMINISTIC")
    if env is not None and env.strip() != "":
        if env.strip() not in ("0", "1"):
            raise ValueError(f"XMM_DETERMINISTIC={env!r}: expected 0 or 1")
        return env.strip() == "1"
    return torch.are_deterministic_algorithms_enabled()


Job = Tuple[int, int, int, int, int, float, int]  # (slots pointer, count, stride, dst offset, n, scale, accumulate)


class DetPlan:
    """Slot ranges and finalize jobs of one training shape.

    The backward pass asks for its slot ranges in a fixed order; the first deterministic backward of a shape allocates
    them (zeroed: the finalize leaves every slot it reads zero again), later ones get the same ranges back.  Jobs name
    their destination as an offset into the backward's gradient buffer, so the device job table of every finalize is
    built once and reused although that buffer is new on every call.  ``flush()`` closes a group: one finalize launch
    for the jobs added since the previous flush, then the host-side steps registered with ``after()``.
    """

    def __init__(self, device: torch.device, slot_count: Callable[..., int] = ops.det_slots) -> None:
        self.device = device
        self.slot_count = slot_count
        self.regions: List[torch.Tensor] = []
        self.tables: List[Tuple[Tuple[Job, ...], Optional[torch.Tensor], int]] = []
        self._base: Optional[torch.Tensor] = None
        self._ri = self._fi = 0
        self._jobs: List[Job] = []
        self._post: List[Callable[[], None]] = []

    # ------------------------------------------------------------------ bookkeeping
    def begin(self, base: torch.Tensor) -> None:
        """Start a backward pass whose destinations all lie in ``base`` (fp32, contiguous)."""
        self._base = base
        self._ri = self._fi = 0
        self._jobs, self._post = [], []

    def slots(self, count: int, row: int) -> torch.Tensor:
        if self._ri == len(self.regions):
            self.regions.append(torch.zeros(count * row, dtype=torch.float32, device=self.device))
        r = self.regions[self._ri]
        if r.numel() != count * row:
            raise RuntimeError("deterministic plan: this backward asks for another slot layout than the one recorded "
                               "for its shape")
        self._ri += 1
        return r

    def job(self, slots: torch.Tensor, count: int, stride: int, dst: torch.Tensor, n: int, scale: float = 1.0,
            accumulate: bool = True) -> None:
        base = self._base
        if not dst.is_contiguous() or dst.dtype != torch.float32 or dst.numel() < n:
            raise RuntimeError("deterministic plan: a destination must be n contiguous fp32 elements")
        off = (dst.data_ptr() - base.data_ptr()) // 4
        if off < 0 or off + n > base.numel() or dst.data_ptr() != base.data_ptr() + 4 * off:
            raise RuntimeError("deterministic plan: destination outside the gradient buffer")
        for j in self._jobs:  # jobs of one finalize run concurrently: no shared destinations
            if j[3] < off + n and off < j[3] + j[4]:
                raise RuntimeError("deterministic plan: two jobs of one finalize write the same gradient")
        self._jobs.append((slots.data_ptr(), int(count), int(stride), int(off), int(n), float(scale), int(accumulate)))

    def after(self, fn: Callable[[], None]) -> None:
        """Run ``fn`` right after the next flush (a copy out of a finalized scratch destination)."""
        self._post.append(fn)

    def flush(self) -> None:
        jobs = tuple(self._jobs)
        if jobs:
            if self._fi == len(self.tables):
                self.tables.append(((), None, 0))
            if self.tables[self._fi][0] != jobs:
                arr = (_lib.DetJob * len(jobs))(*[_lib.DetJob(*j) for j in jobs])
                table = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8).to(self.device)
                self.tables[self._fi] = (jobs, table, max(j[4] for j in jobs))
            _, table, max_n = self.tables[self._fi]
            ops.det_finalize(table, len(jobs), max_n, self._base)
            self._fi += 1
        for fn in self._post:
            fn()
        self._jobs, self._post = [], []

    # ------------------------------------------------------------------ the three sites
    def conv_kwargs(self, b: int, h: int, w: int, dst: torch.Tensor, scale: float) -> dict:
        """conv3x3 keywords of a fused bias gradient (cout = 32) in deterministic form, and its job."""
        count = self.slot_count(_lib.DET_CONV3X3, b, h, w, 32)
        ws = self.slots(count, 32)
        self.job(ws, count, 32, dst, 32, scale)
        return dict(colsum=dst, colsum_scale=scale, colsum_ws=ws)

    def colsum(self, inputs, segments) -> None:
        """Column sums of the same channel windows of every buffer in ``inputs`` (one shape), added into the segments'
        destinations: segments [(c0, n, dst, scale, accumulate)].  All inputs share one job per segment, so a gradient
        with several integrands (conv_first's bias) is still one finalize job."""
        b, h, w = inputs[0].shape[:3]
        row = sum(seg[1] for seg in segments)
        count = self.slot_count(_lib.DET_COLSUM, b, h, w, row)
        ws = self.slots(len(inputs) * count, row)
        for k, inp in enumerate(inputs):
            ops.colsum_multi_det(inp, [(c0, n, scale) for c0, n, _, scale, _ in segments],
                                 ws[k * count * row:(k + 1) * count * row])
        col = 0
        for c0, n, dst, scale, accumulate in segments:
            self.job(ws[col:], len(inputs) * count, row, dst, n, scale, accumulate)
            col += n

    def edge_wgrad(self, s: torch.Tensor, v: torch.Tensor, v_coff: int, channels: int, r: torch.Tensor,
                   ssum: Optional[torch.Tensor] = None, **kw) -> None:
        b, ns, h, w = s.shape
        nr = ns * channels * 9
        row = nr + ns
        count = self.slot_count(_lib.DET_EDGE_WGRAD, b, h, w, channels)
        ws = self.slots(count, row)
        ops.edge_wgrad(s, v, v_coff, channels, r, ssum=ssum, ws=ws, **kw)
        self.job(ws, count, row, r, nr)
        if ssum is not None:
            self.job(ws[nr:], count, row, ssum, ns)
