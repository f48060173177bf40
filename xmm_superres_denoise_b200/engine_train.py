"""Training half of the engine: forward with saved activations + the hand-scheduled backward.

What autograd + cuDNN do for the reference (conv bwd-data, conv bwd-filter, LeakyReLU / clamp /
pixel-shuffle / residual backward, rrdb_blocks.py:37-70, generator_rrdb.py:66-137) is here an
explicit launch sequence over the same two tensor-core kernels:

* data gradients reuse ``conv3x3`` (the gradient of a correlation is a correlation with the
  flipped, transposed filter).  For a dense block the gradient of x_j is ONE convolution over
  the already-complete gradient slots dY_{j+1..5} -- they are adjacent channels of the block's
  gradient buffer, mirroring how the forward reads x_0..x_{k-1} -- with LeakyReLU' taken from
  the stored activation (in-place LeakyReLU keeps only the output; slope > 0 makes sign(out)
  exact) fused in the epilogue, and the block / RRDB skip connections as scaled residual terms;
* weight gradients use ``conv3x3_wgrad`` once per dense block (all five layers at once).

Buffers per dense block: activations A = [x0|x1|x2|x3|x4] (kept from the forward), gradients
G = [dY1|dY2|dY3|dY4|g] where g = dL/d(block output) (conv5's 0.2 is folded into the packed
weights).  Three G buffers rotate: RDB3 -> ring[2], RDB2 -> ring[1], RDB1 -> ring[0].
"""
from __future__ import annotations

from typing import Dict, List, Optional

import torch

from . import determinism, ops
from .engine import RRDBEngine, _Blob, _Segment


def _dgrad_blob(name: str, convs, j: int, f: int, kc: int, conv5_scale: float, n0: int = 0, nt: int = -1) -> _Blob:
    """Gradient of x_j of a dense block (its channels [n0, n0+nt)): K runs over dY_{j+1}..dY_5 (F channels each)."""
    nt = f if nt < 0 else nt
    segs = []
    for k in range(j + 1, 6):
        w = convs[k - 1].weight
        segs.append(_Segment(w, w.shape[1], 0, j * f + n0, 1, (k - j - 1) * f, f, conv5_scale if k == 5 else 1.0))
    return _Blob(name, nt, kc, (5 - j) * f // kc, segs, None)


def _transpose_blob(name: str, conv, kc: int, perm: int = 0, n0: int = 0, nt: int = -1) -> _Blob:
    """Data gradient of a plain conv: rows = its input channels ([n0, n0+nt)), K = its output channels."""
    cout, cin = conv.weight.shape[0], conv.weight.shape[1]
    nt = cin if nt < 0 else nt
    return _Blob(name, nt, kc, cout // kc, [_Segment(conv.weight, cin, 0, n0, 1, 0, cout, 1.0)], None, perm)


class TrainEngine(RRDBEngine):
    def __init__(self, gen, kind: str) -> None:
        super().__init__(gen, kind)
        f = self.nf
        # bias gradients ride on the data-gradient launches that produce their integrands (Cout = 32 kernels);
        # the 64-filter generators take one colsum pass per dense block instead
        self.fuse_bias = f == 32
        for i, rrdb in enumerate(gen.rrdb):
            for r, rdb in enumerate((rrdb.RDB1, rrdb.RDB2, rrdb.RDB3)):
                convs = [getattr(rdb, f"conv{k}") for k in range(1, 6)]
                for j in range(5):
                    self._add_planned(f"d.{i}.{r}.{j}", f, (5 - j) * f,
                                      lambda nm, n0, nt, kc, convs=convs, j=j, r=r: _dgrad_blob(
                                          nm, convs, j, f, kc, 0.04 if r == 2 else 0.2, n0, nt))
        self._add_planned("d.trunk", f, f, lambda nm, n0, nt, kc: _transpose_blob(nm, gen.trunk_conv, kc, 0, n0, nt))
        if kind == "sr":
            for s in range(self.num_upsample):
                self._add_planned(f"d.up{s}", f, 4 * f, lambda nm, n0, nt, kc, s=s: _transpose_blob(
                    nm, gen.upsampling[3 * s], kc, 1, n0, nt))
            self._add_planned("d.hr", f, f, lambda nm, n0, nt, kc: _transpose_blob(nm, gen.HRconv, kc, 0, n0, nt))
        self.generation = 0
        self._params = list(gen.parameters())
        self._pindex = {id(p): n for n, p in enumerate(self._params)}
        self._det: Optional[determinism.DetPlan] = None  # the running backward's plan in deterministic mode

    # ------------------------------------------------------------------ buffers
    def _train_buffers(self, b: int, h: int, w: int, device: torch.device) -> Dict[str, object]:
        key = ("train", b, h, w, str(device))
        bufs = self._bufs.get(key)
        if bufs is None:
            self._bufs.clear()
            self._graphs.clear()
            f = self.nf
            bf = dict(dtype=torch.bfloat16, device=device)
            nrdb = 3 * self.nb
            act = [torch.empty(b, h, w, 5 * f, **bf) for _ in range(nrdb)]
            act.append(torch.empty(b, h, w, f, **bf))  # output of the last RRDB
            bufs = {"act": act, "trunk": torch.empty(b, h, w, f, **bf),
                    "ring": [torch.empty(b, h, w, 5 * f, **bf) for _ in range(3)],
                    "d_trunk": torch.empty(b, h, w, f, **bf), "d_fea": torch.empty(b, h, w, f, **bf)}
            hh, ww = h, w
            if self.kind == "sr":
                for s in range(self.num_upsample):
                    hh, ww = 2 * hh, 2 * ww
                    bufs[f"up{s}"] = torch.empty(b, hh, ww, f, **bf)
                    bufs[f"d_up{s}"] = torch.empty(b, hh // 2, ww // 2, 4 * f, **bf)  # un-shuffled gradient
                bufs["hr"] = torch.empty(b, hh, ww, f, **bf)
                bufs["d_hr"] = torch.empty(b, hh, ww, f, **bf)
            bufs["pre"] = torch.empty(b, self.gen.out_channels, hh, ww, dtype=torch.float32, device=device)
            self._bufs[key] = bufs
        return bufs

    # ------------------------------------------------------------------ forward
    def forward_train(self, x: torch.Tensor):
        self._check_input(x)
        g = self.gen
        x = x.contiguous().float()
        b, _, h, w = x.shape
        self.arena.ensure(x.device)
        bufs = self._train_buffers(b, h, w, x.device)
        self.generation += 1
        self._trunk_forward(x, bufs["act"], bufs["act"][0], bufs["trunk"])
        if self.kind == "dn":
            if g.in_channels != g.out_channels:
                raise RuntimeError("GeneratorRRDB_DN adds its input to its output: in_channels must equal out_channels")
            out = torch.empty(b, g.out_channels, h, w, dtype=torch.float32, device=x.device)
            ops.conv_last(bufs["trunk"], 0, g.conv_last.weight, g.conv_last.bias, out, residual=x, pre=bufs["pre"],
                          wblob_ptr=self._last_ptr())
            return out, bufs
        cur = bufs["trunk"]
        for s in range(self.num_upsample):
            self._run(self._conv(f"f.up{s}", cur, 0, self.nf, bufs[f"up{s}"], 0, lrelu=0.01, pixel_shuffle=1))
            cur = bufs[f"up{s}"]
        self._run(self._conv("f.hr", cur, 0, self.nf, bufs["hr"], 0, lrelu=0.2))
        out = torch.empty(b, g.out_channels, cur.shape[1], cur.shape[2], dtype=torch.float32, device=x.device)
        ops.conv_last(bufs["hr"], 0, g.conv_last.weight, g.conv_last.bias, out, pre=bufs["pre"], wblob_ptr=self._last_ptr())
        return out, bufs

    # ------------------------------------------------------------------ backward
    def _grad_views(self, device: torch.device, extra: int = 0) -> List[torch.Tensor]:
        """Fresh flat fp32 gradient buffer (autograd may adopt the returned tensors as .grad).  extra: zeroed scratch
        floats after the gradients (deterministic mode: destinations that are copied into a gradient afterwards)."""
        total = sum(p.numel() for p in self._params)
        flat = torch.zeros(total + extra, dtype=torch.float32, device=device)
        views, off = [], 0
        for p in self._params:
            views.append(flat[off:off + p.numel()].view(p.shape))
            off += p.numel()
        self.last_flat_grad = flat[:total] if extra else flat
        self._flat_ext, self._ext_off = flat, total
        return views

    def _scratch(self, n: int) -> torch.Tensor:
        t = self._flat_ext[self._ext_off:self._ext_off + n]
        self._ext_off += n
        return t

    def _det_scratch_floats(self) -> int:
        return self.gen.in_channels * self.nf * 9 + (4 * self.nf * self.num_upsample if self.kind == "sr" else 0)

    def _colsum(self, inp: torch.Tensor, segments) -> None:
        """Bias gradients from one buffer: segments [(c0, n, dst, scale, accumulate)]."""
        if self._det is not None:
            self._det.colsum([inp], segments)
        elif len(segments) == 1:
            ops.colsum(inp, *segments[0])
        else:
            ops.colsum_multi(inp, segments)

    def _edge_wgrad(self, *a, **kw) -> None:
        if self._det is not None:
            self._det.edge_wgrad(*a, **kw)
        else:
            ops.edge_wgrad(*a, **kw)

    def _gv(self, grads, p: torch.Tensor) -> torch.Tensor:
        return grads[self._pindex[id(p)]]

    def _single_conv_wgrad(self, conv, x: torch.Tensor, dy: torch.Tensor, grads, perm: int = 0) -> None:
        f = self.nf
        n = conv.weight.shape[0]
        dw = self._gv(grads, conv.weight)
        # F -> F / F -> 4F: stacked roles (M = up to 128 dY channels, N = 3 dx taps x 32 X channels; 3 MMAs per 16
        # pixels instead of 9 narrow ones with most of the M rows aliased), one per (32 X channels, 128 dY channels)
        roles, dsts = [], []
        for x0 in range(0, f, 32):
            for y0 in range(0, n, 128):
                m = min(128, n - y0)
                roles.append((0, 3, x0, 1 if m <= 64 else 2, y0, 96, 1))
                dsts.append((dw, m, f, x0, x0 + 32, len(roles) - 1, 0, 0, 1.0, 0, perm, y0, n))
        ops.conv3x3_wgrad(x, dy, roles, dsts)
        if conv.bias is not None:
            db = self._gv(grads, conv.bias)
            if perm:
                if self._det is None:
                    tmp = torch.empty(n, dtype=torch.float32, device=dy.device)
                    ops.colsum(dy, 0, n, tmp)
                    db.copy_(tmp.view(4, n // 4).t().reshape(n))  # packed g*F+c -> channel 4c+g
                else:
                    tmp = self._scratch(n)
                    self._det.colsum([dy], [(0, n, tmp, 1.0, False)])
                    self._det.after(lambda: db.copy_(tmp.view(4, n // 4).t().reshape(n)))
            else:
                self._colsum(dy, [(0, n, db, 1.0, True)])  # db is a view of the zero-initialised flat buffer

    def _rdb_backward(self, i: int, r: int, bufs, grads, d_fea: torch.Tensor) -> None:
        f, kc, a = self.nf, self.kc, self.arena
        act, ring = bufs["act"], bufs["ring"]
        A, G = act[3 * i + r], ring[r]
        rdb = self._rdb(i, r)
        layers = []
        for j in range(4, 0, -1):  # dY_j = LeakyReLU'(x_j) * sum_k dgrad_k(dY_k); its column sums are conv_j's bias grad
            layers += self._conv(f"d.{i}.{r}.{j}", G, j * f, (5 - j) * f, G, (j - 1) * f, mask=A, mask_coff=j * f,
                                 mask_slope=0.2, **self._bias_sum(grads, getattr(rdb, f"conv{j}"), 1.0))
        # gradient of the block input: + skip connection(s).  The result is the output gradient g of the NEXT block to be
        # processed, i.e. the integrand of that block's conv5 bias gradient (scaled by its folded residual factor).
        if r == 2:    # out_rrdb = 0.2 * out_rdb3 + x_rrdb ; G[4] holds E_i = dL/d(out_rrdb)
            layers += self._conv(f"d.{i}.{r}.0", G, 0, 5 * f, ring[1], 4 * f, r1=G, r1_coff=4 * f, s1=0.2,
                                 **self._bias_sum(grads, self._rdb(i, 1).conv5, 0.2))
        elif r == 1:
            layers += self._conv(f"d.{i}.{r}.0", G, 0, 5 * f, ring[0], 4 * f, r1=G, r1_coff=4 * f, s1=1.0,
                                 **self._bias_sum(grads, self._rdb(i, 0).conv5, 0.2))
        else:         # RDB1: + g_1 + E_i (RRDB skip); result is E_{i-1}, or dL/d(fea) through the trunk for i == 0
            out, ocoff = (ring[2], 4 * f) if i > 0 else (d_fea, 0)
            extra = self._bias_sum(grads, self._rdb(i - 1, 2).conv5, 0.04) if i > 0 else {}
            layers += self._conv(f"d.{i}.{r}.0", G, 0, 5 * f, out, ocoff, r1=G, r1_coff=4 * f, s1=1.0, r2=ring[2],
                                 r2_coff=4 * f, s2=1.0, **extra)
        if len(layers) == 5:
            ops.conv3x3_chain(layers, self.chain_mode)
        else:  # split layers (F = 64): plain launches
            self._run(layers)

    def _rdb(self, i: int, r: int):
        rrdb = self.gen.rrdb[i]
        return (rrdb.RDB1, rrdb.RDB2, rrdb.RDB3)[r]

    def _bias_sum(self, grads, conv, scale: float) -> dict:
        """conv3x3 keywords that make the producing layer accumulate `conv`'s bias gradient (views of the
        zero-initialised flat gradient buffer)."""
        if conv.bias is None or not self.fuse_bias:
            return {}
        if self._det is not None:
            return self._det.conv_kwargs(*self._det_bhw, self._gv(grads, conv.bias), scale)
        return dict(colsum=self._gv(grads, conv.bias), colsum_scale=scale)

    def _rdb_wgrad(self, i: int, r: int, bufs, grads) -> None:
        f = self.nf
        rrdb = self.gen.rrdb[i]
        rdb = (rrdb.RDB1, rrdb.RDB2, rrdb.RDB3)[r]
        A, G = bufs["act"][3 * i + r], bufs["ring"][r]
        s5 = 0.04 if r == 2 else 0.2
        convs = [getattr(rdb, f"conv{k}") for k in range(1, 6)]
        dws = [self._gv(grads, c.weight) for c in convs]
        if not self.fuse_bias:  # the five bias gradients: one pass over the block's gradient buffer
            segs = [((k - 1) * f, f, self._gv(grads, c.bias), s5 if k == 5 else 1.0, True)
                    for k, c in enumerate(convs, 1) if c.bias is not None]
            if segs:
                self._colsum(G, segs)
        if f == 64:
            self._rdb_wgrad_64(A, G, dws, s5)
            return
        # x0..x3 against all five dY slots, one role per filter row; x4 x dY5 as a stacked role (three dx taps per
        # MMA, operands swapped: lanes = channels of the [dY4|dY5] box)
        roles = [(3 * d, 3, 0, 2, 0, 5 * f) for d in range(3)] + [(0, 3, 4 * f, 1, 3 * f, 3 * f, 1)]
        dsts = []
        for k in range(1, 6):
            sc = s5 if k == 5 else 1.0
            for d in range(3):
                dsts.append((dws[k - 1], f, k * f, 0, min(k * f, 4 * f), d, 0, (k - 1) * f, sc, 0, 0))
            if k == 5:
                dsts.append((dws[k - 1], f, 5 * f, 4 * f, 5 * f, 3, f, 0, sc, 0, 0))
        # (bias gradients: accumulated by the conv launches that produced G's slots -- _rdb_backward / backward)
        ops.conv3x3_wgrad(A, G, roles, dsts)

    @staticmethod
    def _rdb_wgrad_64(A: torch.Tensor, G: torch.Tensor, dws, s5: float) -> None:
        """64 filters: X and dY are 320 channels, the needed (x_i, dY_k) blocks (i < k) are 64 x 64.  An M tile is two
        X slots (128 channels), a role keeps taps * N <= 512 accumulator columns -> five launches:
        [x0|x1] x [dY1|dY2], [x0|x1] x [dY3|dY4], [x2|x3] x [dY3|dY4] (one role per filter row, N = 128),
        [x0|x1] and [x2|x3] x dY5 (N = 64, 5 + 4 taps per role), x4 x dY5 (stacked roles, 32 X channels each)."""
        f = 64
        dw1, dw2, dw3, dw4, dw5 = dws

        def rows(x_c0: int, y_c0: int):
            return [(3 * d, 3, x_c0, 2, y_c0, 2 * f) for d in range(3)]

        ops.conv3x3_wgrad(A, G, rows(0, 0),
                          [(dw1, f, f, 0, f, d, 0, 0, 1.0, 0, 0) for d in range(3)] +
                          [(dw2, f, 2 * f, 0, 2 * f, d, 0, f, 1.0, 0, 0) for d in range(3)])
        ops.conv3x3_wgrad(A, G, rows(0, 2 * f),
                          [(dw3, f, 3 * f, 0, 2 * f, d, 0, 0, 1.0, 0, 0) for d in range(3)] +
                          [(dw4, f, 4 * f, 0, 2 * f, d, 0, f, 1.0, 0, 0) for d in range(3)])
        ops.conv3x3_wgrad(A, G, rows(2 * f, 2 * f),
                          [(dw3, f, 3 * f, 2 * f, 3 * f, d, 0, 0, 1.0, 0, 0) for d in range(3)] +
                          [(dw4, f, 4 * f, 2 * f, 4 * f, d, 0, f, 1.0, 0, 0) for d in range(3)])
        roles = [(0, 5, 0, 2, 4 * f, f), (5, 4, 0, 2, 4 * f, f), (0, 5, 2 * f, 2, 4 * f, f), (5, 4, 2 * f, 2, 4 * f, f)]
        ops.conv3x3_wgrad(A, G, roles,
                          [(dw5, f, 5 * f, 0, 2 * f, q, 0, 0, s5, 0, 0) for q in (0, 1)] +
                          [(dw5, f, 5 * f, 2 * f, 4 * f, q, 0, 0, s5, 0, 0) for q in (2, 3)])
        ops.conv3x3_wgrad(A, G, [(0, 3, 4 * f, 1, 4 * f, 96, 1), (0, 3, 4 * f + 32, 1, 4 * f, 96, 1)],
                          [(dw5, f, 5 * f, 4 * f, 4 * f + 32, 0, 0, 0, s5, 0, 0),
                           (dw5, f, 5 * f, 4 * f + 32, 5 * f, 1, 0, 0, s5, 0, 0)])

    def backward(self, bufs, generation: int, x: torch.Tensor, gout: torch.Tensor, need_x_grad: bool,
                 rrdb_done_hook=None):
        if generation != self.generation:
            raise RuntimeError("backward through a GeneratorRRDB forward whose saved activations were overwritten by a "
                               "later forward (run backward before the next training-mode forward)")
        if not determinism.enabled():
            self._det = None
            return self._backward(bufs, x, gout, need_x_grad, rrdb_done_hook)
        # deterministic mode: the plan (slot ranges, finalize job tables) lives with this shape's training buffers
        plan = bufs.get("det")
        if plan is None:
            plan = bufs["det"] = determinism.DetPlan(x.device)
        self._det = plan
        try:
            return self._backward(bufs, x, gout, need_x_grad, rrdb_done_hook)
        except BaseException:
            bufs.pop("det", None)  # slots written without their finalize: start the next deterministic call afresh
            raise
        finally:
            self._det = None

    def _backward(self, bufs, x: torch.Tensor, gout: torch.Tensor, need_x_grad: bool, rrdb_done_hook):
        g, f, kc, a = self.gen, self.nf, self.kc, self.arena
        det = self._det
        gout = gout.contiguous().float()
        x = x.contiguous().float()
        grads = self._grad_views(x.device, self._det_scratch_floats() if det is not None else 0)
        if det is not None:
            det.begin(self._flat_ext)
            self._det_bhw = tuple(bufs["trunk"].shape[:3])
        pre = bufs["pre"]
        # flipped / transposed conv_last filter: data gradient of an F->1 conv is a 1->F stencil (288 floats)
        wt_last = g.conv_last.weight.detach().flip(2, 3).permute(1, 0, 2, 3).contiguous()
        dw_last = self._gv(grads, g.conv_last.weight)
        db_last = self._gv(grads, g.conv_last.bias) if g.conv_last.bias is not None else None
        if self.kind == "dn":
            feat_in = bufs["trunk"]
            ops.conv_first(gout, wt_last, None, bufs["d_trunk"], 0, gate=pre)
            self._edge_wgrad(gout, feat_in, 0, f, dw_last.view(g.out_channels, f, 9), ssum=db_last, gate=pre)
        else:
            hr = bufs["hr"]
            ops.conv_first(gout, wt_last, None, bufs["d_hr"], 0, gate=pre, mask=hr, mask_coff=0, mask_slope=0.2)
            self._edge_wgrad(gout, hr, 0, f, dw_last.view(g.out_channels, f, 9), ssum=db_last, gate=pre)
            ups = [bufs["trunk"]] + [bufs[f"up{s}"] for s in range(self.num_upsample)]
            self._single_conv_wgrad(g.HRconv, ups[-1], bufs["d_hr"], grads)
            dy = bufs["d_hr"]
            blob = "d.hr"
            nin = f
            for s in range(self.num_upsample - 1, -1, -1):
                # gradient w.r.t. the shuffled, LeakyReLU(0.01)-activated upsample output, stored un-shuffled
                self._run(self._conv(blob, dy, 0, nin, bufs[f"d_up{s}"], 0, mask=ups[s + 1], mask_coff=0,
                                     mask_slope=0.01, pixel_shuffle=2))
                dy, blob, nin = bufs[f"d_up{s}"], f"d.up{s}", 4 * f
                self._single_conv_wgrad(g.upsampling[3 * s], ups[s], dy, grads, perm=1)
            self._run(self._conv(blob, dy, 0, nin, bufs["d_trunk"], 0))
        d_trunk = bufs["d_trunk"]  # dL/d(fea + trunk_conv(...)): feeds trunk_conv and the `fea` skip
        last_act = bufs["act"][3 * self.nb]
        self._single_conv_wgrad(g.trunk_conv, last_act, d_trunk, grads)
        ring = bufs["ring"]
        d_fea = bufs["d_fea"]
        if self.nb > 0:
            self._run(self._conv("d.trunk", d_trunk, 0, f, ring[2], 4 * f,  # E_{nb-1} = g of the last RDB3
                                 **self._bias_sum(grads, self._rdb(self.nb - 1, 2).conv5, 0.04)))
            for i in range(self.nb - 1, -1, -1):
                for r in (2, 1, 0):
                    self._rdb_backward(i, r, bufs, grads, d_fea)
                    self._rdb_wgrad(i, r, bufs, grads)
                if det is not None:  # this RRDB's (and, first time round, the tail layers') reductions, in order
                    det.flush()
                if rrdb_done_hook is not None:  # every gradient of RRDB i (and of all later layers) is enqueued
                    rrdb_done_hook(i, self.last_flat_grad)
        else:
            self._run(self._conv("d.trunk", d_trunk, 0, f, d_fea, 0))
        # conv_first: dL/d(fea) = d_fea (through the RRDBs) + d_trunk (skip)
        cin = g.in_channels
        dwf = self._gv(grads, g.conv_first.weight)
        if det is None:
            r_first = torch.zeros(cin, f, 9, dtype=torch.float32, device=x.device)
            ops.edge_wgrad(x, d_fea, 0, f, r_first, v2=d_trunk, v2_coff=0)
            dwf.copy_(r_first.flip(2).permute(1, 0, 2).reshape(f, cin, 3, 3))
            if g.conv_first.bias is not None:
                dbf = self._gv(grads, g.conv_first.bias)
                ops.colsum(d_fea, 0, f, dbf)
                ops.colsum(d_trunk, 0, f, dbf, accumulate=True)
        else:
            r_first = self._scratch(cin * f * 9).view(cin, f, 9)
            det.edge_wgrad(x, d_fea, 0, f, r_first, v2=d_trunk, v2_coff=0)
            det.after(lambda: dwf.copy_(r_first.flip(2).permute(1, 0, 2).reshape(f, cin, 3, 3)))
            if g.conv_first.bias is not None:  # both integrands in one job: d_fea's slots, then d_trunk's
                det.colsum([d_fea, d_trunk], [(0, f, self._gv(grads, g.conv_first.bias), 1.0, False)])
            det.flush()
        gx = None
        if need_x_grad:
            # dL/dx = conv_first^T(dL/dfea) (+ the DN residual path); an F->cin stencil = conv_last kernel
            wt_first = g.conv_first.weight.detach().flip(2, 3).permute(1, 0, 2, 3).contiguous()
            gx1 = torch.empty_like(x)
            base = None
            if self.kind == "dn":
                base = torch.where((pre >= 0) & (pre <= 1), gout, torch.zeros_like(gout))
            ops.conv_last(d_fea, 0, wt_first, None, gx1, residual=base, clamp=False)
            gx = torch.empty_like(x)
            ops.conv_last(d_trunk, 0, wt_first, None, gx, residual=gx1, clamp=False)
        return gx, grads
