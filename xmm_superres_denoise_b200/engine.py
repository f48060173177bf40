"""Execution engine behind ``GeneratorRRDB_DN`` / ``GeneratorRRDB_SR``.

Owns what the reference leaves to autograd and cuDNN:

* the packed bf16 weight images of every 3x3 layer (rebuilt by ONE kernel launch whenever a
  parameter changes -- after ``optimizer.step()`` or ``load_state_dict``),
* the NHWC bf16 activation buffers: one ``5*F``-channel buffer per dense block, so that
  ``torch.cat`` (rrdb_blocks.py:49-52) is a channel offset,
* the launch sequence of the forward pass (and, in ``engine_train.py``, the backward pass).
"""
from __future__ import annotations

import gc

import ctypes
import os
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Tuple

import torch
from torch import nn

from . import _lib, ops
from ._lib import PackJob

_ALIGN = 1024


def _round_up(x: int, a: int) -> int:
    return (x + a - 1) // a * a


@dataclass
class _Segment:
    param: torch.Tensor
    src_cin: int
    o_off: int
    i_off: int
    transpose: int
    k_off: int
    k_count: int
    scale: float
    n_off: int = 0
    n_count: int = -1  # -1: all rows of the blob
    part: int = 0      # 1: low-order half bf16(w - bf16(w)) of a split-precision layer


@dataclass
class _Blob:
    """One packed layer: `nt` GEMM columns (output channels), K = nchunks*kc input channels."""
    name: str
    nt: int
    kc: int
    nchunks: int
    segments: List[_Segment]
    bias: Optional[torch.Tensor] = None
    perm: int = 0
    bias_n: int = -1  # rows that take a bias (-1: all)
    offset: int = 0  # byte offset inside the blob arena
    tap_order: int = 0  # 1: the row-hop kernel's block order dx*3 + (2 - dy) (xmm_pack_job.tap_order)

    @property
    def nbytes(self) -> int:
        return self.nchunks * 9 * self.nt * self.kc * 2 + self.nt * 4


class WeightArena:
    """All packed layers of one model in one device buffer + the device-side job table."""

    def __init__(self) -> None:
        self.blobs: Dict[str, _Blob] = {}
        self._order: List[_Blob] = []
        self._arena: Optional[torch.Tensor] = None
        self._jobs_dev: Optional[torch.Tensor] = None
        self._key: Optional[tuple] = None
        self._versions: Optional[tuple] = None

    def add(self, blob: _Blob) -> None:
        if blob.name in self.blobs:
            raise KeyError(blob.name)
        self.blobs[blob.name] = blob
        self._order.append(blob)

    def invalidate(self) -> None:
        """Force a re-pack on the next ensure() (for writers that bypass tensor version counters)."""
        self._versions = None

    def ptr(self, name: str) -> int:
        assert self._arena is not None
        return self._arena.data_ptr() + self.blobs[name].offset

    def _params(self) -> List[torch.Tensor]:
        ps = []
        for b in self._order:
            ps.extend(s.param for s in b.segments)
            if b.bias is not None:
                ps.append(b.bias)
        return ps

    def ensure(self, device: torch.device) -> None:
        """(Re)build the job table if parameter storage moved; re-pack if any parameter changed."""
        params = self._params()
        key = (str(device),) + tuple(p.data_ptr() for p in params)
        if key != self._key:
            off = 0
            for b in self._order:
                b.offset = off
                off = _round_up(off + b.nbytes, _ALIGN)
            self._arena = torch.empty(off, dtype=torch.uint8, device=device)
            jobs = (PackJob * len(self._order))()
            for j, b in zip(jobs, self._order):
                j.dst = self._arena.data_ptr() + b.offset
                j.bias = b.bias.data_ptr() if b.bias is not None else None
                j.nt, j.kc, j.nchunks, j.nseg, j.perm, j.n_valid = b.nt, b.kc, b.nchunks, len(b.segments), b.perm, b.nt
                j.bias_n = b.nt if b.bias_n < 0 else b.bias_n
                j.tap_order = b.tap_order
                if len(b.segments) > 5:
                    raise RuntimeError(f"{b.name}: a packed layer takes at most 5 source segments")
                for s_c, s in zip(j.seg, b.segments):
                    if s.param.dtype != torch.float32 or not s.param.is_contiguous() or s.param.device != device:
                        raise RuntimeError(f"{b.name}: parameters must be contiguous fp32 tensors on {device}")
                    s_c.src, s_c.src_cin, s_c.o_off, s_c.i_off = s.param.data_ptr(), s.src_cin, s.o_off, s.i_off
                    s_c.transpose, s_c.k_off, s_c.k_count, s_c.scale = s.transpose, s.k_off, s.k_count, s.scale
                    s_c.n_off, s_c.n_count = s.n_off, (b.nt if s.n_count < 0 else s.n_count)
                    s_c.part = s.part
            raw = bytes(jobs)
            self._jobs_dev = torch.frombuffer(bytearray(raw), dtype=torch.uint8).to(device)
            self._key = key
            self._versions = None
        versions = tuple(p._version for p in params)
        if versions != self._versions:
            ops.pack_weights(self._jobs_dev.data_ptr(), len(self._order))
            self._versions = versions


def _fwd_blob(name: str, conv: nn.Conv2d, kc: int, perm: int = 0) -> _Blob:
    cout, cin = conv.weight.shape[0], conv.weight.shape[1]
    return _Blob(name, cout, kc, cin // kc,
                 [_Segment(conv.weight, cin, 0, 0, 0, 0, cin, 1.0)], conv.bias, perm)


class _LayerPlans:
    """Mixin: packed forward layers of an engine (``self.arena``, ``self.plans``, ``self.kc``)."""

    def _add_forward_layer(self, name: str, conv: nn.Conv2d, perm: int = 0) -> None:
        """Packed weights of one forward conv.  The kernels keep a layer's weights resident in shared memory; a
        layer that does not fit (F=64: 9*cin*cout*2 bytes reaches 368 KB) is split along its OUTPUT channels into
        parts of 32 (128 for the pixel-shuffle conv) packed with 32-channel K chunks, and runs as one launch per
        part into adjacent output windows."""
        cout, cin = conv.weight.shape[0], conv.weight.shape[1]
        if 9 * cin * cout * 2 <= _WEIGHT_BUDGET:
            self.arena.add(_fwd_blob(name, conv, self.kc, perm))
            self.plans[name] = [(name, self.kc, cout, 0, self._row_twin(_fwd_blob(name, conv, self.kc, perm)))]
            return
        part = 128 if perm else 32
        if cout % part or 9 * cin * part * 2 > 190 * 1024:
            raise NotImplementedError(f"{name}: a {cin}->{cout} conv does not fit the resident-weight kernels")
        plan = []
        for n0 in range(0, cout, part):
            pname = f"{name}.n{n0}"

            def mk(pname=pname, n0=n0):
                return _Blob(pname, part, 32, cin // 32, [_Segment(conv.weight, cin, n0, 0, 0, 0, cin, 1.0)],
                             conv.bias, perm)

            self.arena.add(mk())
            plan.append((pname, 32, part, n0, self._row_twin(mk())))
        self.plans[name] = plan

    def _row_twin(self, blob: _Blob) -> Optional[str]:
        """The same layer packed a second time in the row-hop kernel's block order (``xmm_conv3x3_params.wblob_row``)
        where that kernel can take it: cout == kc in (32, 64), no pixel-shuffle permutation.  Whether a launch
        really uses it is decided per call by the library (image height, shared memory)."""
        if blob.perm or blob.nt != blob.kc or blob.nt not in (32, 64):
            return None
        blob.name += ".row"
        blob.tap_order = 1
        self.arena.add(blob)
        return blob.name

    def _add_planned(self, name: str, rows: int, k_total: int, make_blob) -> None:
        """A packed layer described by ``make_blob(blob_name, n0, nt, kc) -> _Blob`` (rows [n0, n0+nt) of the layer's
        `rows` GEMM columns, K = k_total channels): one blob if its weights fit next to the pipeline stages, else
        parts of 32 rows with 32-channel K chunks (data-gradient layers of the 64-filter generators)."""
        if 9 * k_total * rows * 2 <= _WEIGHT_BUDGET:
            self.arena.add(make_blob(name, 0, rows, self.kc))
            self.plans[name] = [(name, self.kc, rows, 0, self._row_twin(make_blob(name, 0, rows, self.kc)))]
            return
        if rows % 32 or 9 * k_total * 32 * 2 > 190 * 1024:
            raise NotImplementedError(f"{name}: a {k_total}->{rows} layer does not fit the resident-weight kernels")
        plan = []
        for n0 in range(0, rows, 32):
            pname = f"{name}.n{n0}"
            self.arena.add(make_blob(pname, n0, 32, 32))
            plan.append((pname, 32, 32, n0, self._row_twin(make_blob(pname, n0, 32, 32))))
        self.plans[name] = plan

    def _conv(self, name: str, inp: torch.Tensor, in_coff: int, cin: int, out: torch.Tensor, out_coff: int, **kw):
        """The launches of one planned layer as (args, kwargs) for ops.conv3x3 / ops.conv3x3_chain."""
        calls = []
        shuffle = kw.get("pixel_shuffle", 0) == 1
        plan = self.plans[name]
        rows = sum(p[2] for p in plan)
        for blob, kc, nt, n0, row_blob in plan:
            k2 = dict(kw)
            if row_blob is not None and k2.get("pixel_shuffle", 0) == 0:
                k2["wblob_row"] = self.arena.ptr(row_blob)
            for key in ("r1_coff", "r2_coff", "mask_coff"):
                if key in k2 and k2.get(key[:-5]) is not None:
                    k2[key] = k2[key] + n0
            if k2.get("colsum") is not None:  # fused bias gradient: this part's window of the bias gradient
                if k2.get("colsum_ws") is not None and len(plan) > 1:
                    raise RuntimeError(f"{name}: the deterministic fused bias gradient needs an unsplit layer")
                k2["colsum"] = k2["colsum"][n0:n0 + nt]
            if k2.get("pixel_shuffle", 0) == 2 and len(plan) > 1:
                k2["shuffle_stride"] = rows  # the four (y&1, x&1) blocks are a full layer apart
            calls.append(((inp, in_coff, cin, self.arena.ptr(blob), kc, nt, out, out_coff + (n0 // 4 if shuffle else n0)),
                          k2))
        return calls

    def _run(self, calls) -> None:
        for a, kw in calls:
            ops.conv3x3(*a, **kw)



# Shared memory a conv CTA can spend on resident weights and still keep >= 2 activation stages (227 KB opt-in).
_WEIGHT_BUDGET = 150 * 1024


class RRDBEngine(_LayerPlans):
    """Forward pass of the RRDB generators on the tensor-core kernels (inference half)."""

    def __init__(self, gen: nn.Module, kind: str) -> None:
        self.kind = kind
        self.nf = gen.num_filters
        self.nb = gen.num_res_blocks
        if self.nf not in (32, 64):
            raise NotImplementedError(
                f"num_filters={self.nf}: the sm_100a kernels are built for 32 or 64 filters (no fallback path)")
        self.kc = 32 if self.nf == 32 else 64
        self.num_upsample = getattr(gen, "num_upsample", 0)
        self._gen_ref = [gen]  # no nn.Module registration (avoid a reference cycle in the module tree)
        self.arena = WeightArena()
        self.plans: Dict[str, List[Tuple[str, int, int, int, Optional[str]]]] = {}
        g = gen
        for i, rrdb in enumerate(g.rrdb):
            for r, rdb in enumerate((rrdb.RDB1, rrdb.RDB2, rrdb.RDB3)):
                for k in range(1, 6):
                    self._add_forward_layer(f"f.{i}.{r}.{k}", getattr(rdb, f"conv{k}"))
        self._add_forward_layer("f.trunk", g.trunk_conv)
        if kind == "sr":
            for s in range(self.num_upsample):
                self._add_forward_layer(f"f.up{s}", g.upsampling[3 * s], perm=1)
            self._add_forward_layer("f.hr", g.HRconv)
        # conv_last (F -> out_channels) on the tensor cores with fp32-accurate weights: a 32-row layer whose rows
        # [0, cout) hold bf16(w) and rows [16, 16 + cout) the low-order halves bf16(w - bf16(w)); the image epilogue
        # of the conv kernel adds the two partial sums, the bias and the DN residual and clamps (fp32 NCHW out)
        cl = g.conv_last
        co = cl.weight.shape[0]
        if co <= 4 and self.nf % 32 == 0:
            self.arena.add(_Blob("f.last", 32, 32, self.nf // 32,
                                 [_Segment(cl.weight, self.nf, 0, 0, 0, 0, self.nf, 1.0, 0, co, 0),
                                  _Segment(cl.weight, self.nf, 0, 0, 0, 0, self.nf, 1.0, 16, co, 1)],
                                 cl.bias, 0, bias_n=co))
            self._last_blob = "f.last"
        else:
            self._last_blob = None
        self._bufs: Dict[tuple, Dict[str, torch.Tensor]] = {}
        # how a dense block's five dependent convs are launched (ops.CHAIN_*): by default the library decides --
        # the fused dense-block kernels (conv1-3 + conv4-5, conv3x3_rdb.cuh) where the layers qualify (F = 32, even
        # image height), else layer by layer; XMM_CHAIN_MODE=2 forces layer by layer, 1 the pipelined single launch
        self.chain_mode = int(os.environ.get("XMM_CHAIN_MODE", ops.CHAIN_AUTO))
        self._keep_all = True  # set per forward: training keeps every block's x1..x4 for the backward pass
        # CUDA-graph replay of small-batch inference (XMM_CUDA_GRAPH=0 disables)
        self.use_graph = os.environ.get("XMM_CUDA_GRAPH", "1") != "0"
        self.graph_max_batch = 8
        self._graphs: Dict[tuple, tuple] = {}

    @property
    def gen(self) -> nn.Module:
        return self._gen_ref[0]

    def _last_ptr(self):
        return self.arena.ptr(self._last_blob) if self._last_blob is not None else None

    # ------------------------------------------------------------------ buffers
    def _inference_buffers(self, b: int, h: int, w: int, device: torch.device) -> Dict[str, torch.Tensor]:
        key = ("inf", b, h, w, str(device))
        bufs = self._bufs.get(key)
        if bufs is None:
            self._bufs.clear()  # one live shape at a time: these are multi-GB at batch 64
            self._graphs.clear()  # captured launch sequences point into the dropped buffers
            f = self.nf
            bufs = {f"rdb{r}": torch.empty(b, h, w, 5 * f, dtype=torch.bfloat16, device=device) for r in range(3)}
            bufs["fea"] = torch.empty(b, h, w, f, dtype=torch.bfloat16, device=device)
            bufs["trunk"] = torch.empty(b, h, w, f, dtype=torch.bfloat16, device=device)
            hh, ww = h, w
            for s in range(self.num_upsample if self.kind == "sr" else 0):
                hh, ww = 2 * hh, 2 * ww
                bufs[f"up{s}"] = torch.empty(b, hh, ww, f, dtype=torch.bfloat16, device=device)
            if self.kind == "sr":
                bufs["hr"] = torch.empty(b, hh, ww, f, dtype=torch.bfloat16, device=device)
            self._bufs[key] = bufs
        return bufs

    # ------------------------------------------------------------------ dense blocks
    def _rdb_forward(self, name: str, buf: torch.Tensor, out: torch.Tensor, *, s0: float, s1: float,
                     r2: Optional[torch.Tensor], s2: float) -> None:
        """One ResidualDenseBlock_5C (rrdb_blocks.py:37-54): x in buf[..., :F]; result -> out[..., :F]."""
        f = self.nf
        layers = []
        for k in range(1, 5):
            layers += self._conv(f"{name}.{k}", buf, 0, k * f, buf, k * f, lrelu=0.2)
        layers += self._conv(f"{name}.5", buf, 0, 5 * f, out, 0, s0=s0, r1=buf, r1_coff=0, s1=s1, r2=r2, r2_coff=0, s2=s2)
        if len(layers) == 5:
            # inference keeps nothing of a block but its output: x4 need not be written (training reads x1..x4 back)
            ops.conv3x3_chain(layers, self.chain_mode | (0 if self._keep_all else ops.CHAIN_SKIP_DEAD_STORES))
        else:  # split layers (F=64): plain launches
            self._run(layers)

    def _trunk_forward(self, x: torch.Tensor, rdb_bufs: List[torch.Tensor], fea: torch.Tensor,
                       trunk_out: torch.Tensor) -> None:
        """_GeneratorRRDB.forward (generator_rrdb.py:66-69).  rdb_bufs: 3 buffers (ping-pong, inference)
        or 3*nb + 1 buffers (training: every dense block keeps its activations)."""
        g, f = self.gen, self.nf
        ring = len(rdb_bufs)
        keep_all = ring > 3
        self._keep_all = keep_all
        first = rdb_bufs[0]
        if keep_all:
            ops.conv_first(x, g.conv_first.weight, g.conv_first.bias, first, 0)
            fea = first  # RDB 0's input window is never overwritten in training
        else:
            ops.conv_first(x, g.conv_first.weight, g.conv_first.bias, first, 0, out2=fea, out2_coff=0)
        idx = 0
        for i in range(self.nb):
            x_rrdb = rdb_bufs[idx % ring]
            for r in range(3):
                cur = rdb_bufs[idx % ring]
                nxt = rdb_bufs[(idx + 1) % ring]
                if r < 2:
                    # x5 * 0.2 + x
                    self._rdb_forward(f"f.{i}.{r}", cur, nxt, s0=0.2, s1=1.0, r2=None, s2=0.0)
                else:
                    # (x5 * 0.2 + x_rdb3) * 0.2 + x_rrdb   (rrdb_blocks.py:54,70)
                    self._rdb_forward(f"f.{i}.{r}", cur, nxt, s0=0.04, s1=0.2, r2=x_rrdb, s2=1.0)
                idx += 1
        last = rdb_bufs[idx % ring]
        self._run(self._conv("f.trunk", last, 0, f, trunk_out, 0, s0=1.0, r1=fea, r1_coff=0, s1=1.0))

    # ------------------------------------------------------------------ public
    def _check_input(self, x: torch.Tensor) -> None:
        g = self.gen
        if x.dim() != 4 or x.shape[1] != g.in_channels:
            raise RuntimeError(f"expected input (B,{g.in_channels},H,W), got {tuple(x.shape)}")
        if not x.is_cuda:
            raise RuntimeError("xmm_superres_denoise_b200 runs on CUDA (sm_100a) only; there is no CPU path")
        if g.in_channels > 4 or g.out_channels > 4:
            raise NotImplementedError("in_channels / out_channels above 4 are not built")
        for p in g.parameters():
            if p.device != x.device or p.dtype != torch.float32:
                raise RuntimeError("model parameters must be fp32 and on the input's device")

    @torch.no_grad()
    def forward_inference(self, x: torch.Tensor) -> torch.Tensor:
        """Inference forward.  Small batches (<= ``graph_max_batch`` images) are launch-bound -- ~80-150 kernel
        launches of ~10 us each through Python -- so their launch sequence is captured once per input shape into a
        CUDA graph and replayed (weights are re-packed outside the graph; a moved parameter storage re-captures)."""
        self._check_input(x)
        x = x.contiguous().float()
        self.arena.ensure(x.device)
        if not (self.use_graph and x.shape[0] <= self.graph_max_batch) or torch.cuda.is_current_stream_capturing():
            return self._forward_inference_eager(x)
        key = (tuple(x.shape), str(x.device), self.arena._key)
        entry = self._graphs.get(key)
        if entry is None:
            if len(self._graphs) >= 4:
                self._graphs.clear()
            static_in = x.clone()
            side = torch.cuda.Stream(device=x.device)
            side.wait_stream(torch.cuda.current_stream(x.device))
            with torch.cuda.stream(side):  # first-call setup (function attributes, TMA descriptors) outside the capture
                self._forward_inference_eager(static_in)
            torch.cuda.current_stream(x.device).wait_stream(side)
            gc.collect()  # a collected engine / graph releasing device memory in mid-capture would invalidate the capture
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                static_out = self._forward_inference_eager(static_in)
            entry = (graph, static_in, static_out)
            self._graphs[key] = entry
        graph, static_in, static_out = entry
        static_in.copy_(x)
        graph.replay()
        return static_out.clone()

    def _forward_inference_eager(self, x: torch.Tensor) -> torch.Tensor:
        g = self.gen
        b, _, h, w = x.shape
        bufs = self._inference_buffers(b, h, w, x.device)
        self._trunk_forward(x, [bufs["rdb0"], bufs["rdb1"], bufs["rdb2"]], bufs["fea"], bufs["trunk"])
        if self.kind == "dn":
            if g.in_channels != g.out_channels:
                raise RuntimeError("GeneratorRRDB_DN adds its input to its output: in_channels must equal out_channels")
            out = torch.empty(b, g.out_channels, h, w, dtype=torch.float32, device=x.device)
            ops.conv_last(bufs["trunk"], 0, g.conv_last.weight, g.conv_last.bias, out, residual=x, clamp=True,
                          wblob_ptr=self._last_ptr())
            return out
        cur = bufs["trunk"]
        for s in range(self.num_upsample):
            self._run(self._conv(f"f.up{s}", cur, 0, self.nf, bufs[f"up{s}"], 0, lrelu=0.01, pixel_shuffle=1))
            cur = bufs[f"up{s}"]
        self._run(self._conv("f.hr", cur, 0, self.nf, bufs["hr"], 0, lrelu=0.2))
        hh, ww = cur.shape[1], cur.shape[2]
        out = torch.empty(b, g.out_channels, hh, ww, dtype=torch.float32, device=x.device)
        ops.conv_last(bufs["hr"], 0, g.conv_last.weight, g.conv_last.bias, out, clamp=True, wblob_ptr=self._last_ptr())
        return out


# ---------------------------------------------------------------------- standalone blocks
class _BlockRunner(_LayerPlans):
    """RRDB / ResidualDenseBlock_5C called on their own (reference exports them from
    models/modules/__init__.py:1).  Inference only."""

    def __init__(self, rdbs) -> None:
        nf, gc = rdbs[0].nf, rdbs[0].gc
        if nf != gc or nf not in (32, 64):
            raise NotImplementedError(f"standalone dense block with nf={nf}, gc={gc}: only nf == gc in (32, 64) is built")
        self.nf, self.kc = nf, (32 if nf == 32 else 64)
        self.arena = WeightArena()
        self.plans = {}
        for r, rdb in enumerate(rdbs):
            for k in range(1, 6):
                self._add_forward_layer(f"{r}.{k}", getattr(rdb, f"conv{k}"))
        self.n = len(rdbs)

    def run(self, x: torch.Tensor, rrdb: bool) -> torch.Tensor:
        if not x.is_cuda:
            raise RuntimeError("xmm_superres_denoise_b200 runs on CUDA (sm_100a) only; there is no CPU path")
        f, kc = self.nf, self.kc
        b, c, h, w = x.shape
        if c != f:
            raise RuntimeError(f"expected {f} channels, got {c}")
        self.arena.ensure(x.device)
        bufs = [torch.empty(b, h, w, 5 * f, dtype=torch.bfloat16, device=x.device) for _ in range(self.n + 1)]
        bufs[0][..., :f] = x.permute(0, 2, 3, 1)
        for r in range(self.n):
            last = rrdb and r == self.n - 1
            cur, nxt = bufs[r], bufs[r + 1]
            for k in range(1, 5):
                self._run(self._conv(f"{r}.{k}", cur, 0, k * f, cur, k * f, lrelu=0.2))
            self._run(self._conv(f"{r}.5", cur, 0, 5 * f, nxt, 0, s0=0.04 if last else 0.2, r1=cur, r1_coff=0,
                                 s1=0.2 if last else 1.0, r2=bufs[0] if last else None, r2_coff=0,
                                 s2=1.0 if last else 0.0))
        return bufs[self.n][..., :f].permute(0, 3, 1, 2).float().contiguous()


def standalone_block_forward(rdbs, x: torch.Tensor, rrdb: bool) -> torch.Tensor:
    if torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for m in rdbs for p in m.parameters())):
        raise NotImplementedError(
            "autograd through a standalone RRDB / ResidualDenseBlock_5C is not built; use GeneratorRRDB_SR/DN "
            "(whole-generator backward) or wrap the call in torch.no_grad()")
    runner = rdbs[0].__dict__.get("_xmm_runner")
    if runner is None or runner.n != len(rdbs):
        runner = _BlockRunner(rdbs)
        rdbs[0].__dict__["_xmm_runner"] = runner
    with torch.no_grad():
        return runner.run(x, rrdb)
