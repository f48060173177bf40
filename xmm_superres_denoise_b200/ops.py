"""Thin Python wrappers over the C ABI: one function per kernel family.

Tensors are torch CUDA tensors used purely as device-memory handles; activations are NHWC
bf16 ``[B, H, W, C]`` and a convolution reads / writes a *channel window* of them.
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional

import torch

from . import _lib
from ._lib import (Conv3x3Params, ConvFirstParams, ConvLastParams, EdgeWgradParams, NormalizeParams, WgradDst,
                   WgradParams, WgradRole)


LAST_CHAIN_LAUNCHES = 0
LAUNCHES = 0  # kernels launched through this module since the caller last reset it (bench.py's gpu_launches)


def _count(n: int = 1) -> None:
    global LAUNCHES
    LAUNCHES += n


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _nhwc(t: torch.Tensor, name: str) -> None:
    _lib.require_cuda_tensor(t, torch.bfloat16, name)
    if t.dim() != 4:
        raise RuntimeError(f"{name}: expected [B,H,W,C], got {tuple(t.shape)}")


def _conv3x3_params(p: Conv3x3Params, inp: torch.Tensor, in_coff: int, cin: int, wblob_ptr: int, kc: int, cout: int,
                    out: torch.Tensor, out_coff: int, *, lrelu: float = 1.0, s0: float = 1.0,
                    r1: Optional[torch.Tensor] = None, r1_coff: int = 0, s1: float = 0.0,
                    r2: Optional[torch.Tensor] = None, r2_coff: int = 0, s2: float = 0.0,
                    mask: Optional[torch.Tensor] = None, mask_coff: int = 0, mask_slope: float = 1.0,
                    pixel_shuffle: int = 0, tap_mode: int = 0, colsum: Optional[torch.Tensor] = None,
                    colsum_scale: float = 1.0, shuffle_stride: int = 0, wblob_row: Optional[int] = None,
                    colsum_ws: Optional[torch.Tensor] = None) -> None:
    _nhwc(inp, "conv3x3 input")
    _nhwc(out, "conv3x3 output")
    b, h, w, ctot = inp.shape
    p.in_, p.in_ctot, p.in_coff, p.cin = inp.data_ptr(), ctot, in_coff, cin
    p.wblob, p.kc, p.cout = wblob_ptr, kc, cout
    p.wblob_row = wblob_row
    p.batch, p.height, p.width = b, h, w
    p.lrelu_slope = lrelu
    if mask is not None:
        _nhwc(mask, "conv3x3 mask")
        p.mask, p.mask_ctot, p.mask_coff = mask.data_ptr(), mask.shape[3], mask_coff
    p.mask_slope = mask_slope
    p.s0 = s0
    if r1 is not None:
        _nhwc(r1, "conv3x3 r1")
        p.r1, p.r1_ctot, p.r1_coff = r1.data_ptr(), r1.shape[3], r1_coff
    p.s1 = s1
    if r2 is not None:
        _nhwc(r2, "conv3x3 r2")
        p.r2, p.r2_ctot, p.r2_coff = r2.data_ptr(), r2.shape[3], r2_coff
    p.s2 = s2
    pixel_shuffle = int(pixel_shuffle)
    exp = {0: (b, h, w), 1: (b, 2 * h, 2 * w), 2: (b, h // 2, w // 2)}[pixel_shuffle]
    if tuple(out.shape[:3]) != exp:
        raise RuntimeError(f"conv3x3 output: expected spatial shape {exp}, got {tuple(out.shape[:3])}")
    p.out, p.out_ctot, p.out_coff = out.data_ptr(), out.shape[3], out_coff
    p.pixel_shuffle = pixel_shuffle
    p.shuffle_stride = shuffle_stride
    p.tap_mode = tap_mode
    if colsum is not None:
        _lib.require_cuda_tensor(colsum, torch.float32, "conv3x3 colsum")
        if colsum.numel() != cout:
            raise RuntimeError("conv3x3 colsum: one float per output channel")
        p.colsum, p.colsum_scale = colsum.data_ptr(), colsum_scale
        if colsum_ws is not None:
            _lib.require_cuda_tensor(colsum_ws, torch.float32, "conv3x3 colsum_ws")
            p.colsum_ws, p.colsum_ws_slots = colsum_ws.data_ptr(), colsum_ws.numel() // 32


def conv3x3(inp: torch.Tensor, in_coff: int, cin: int, wblob_ptr: int, kc: int, cout: int,
            out: torch.Tensor, out_coff: int, **kw) -> None:
    """out[..., out_coff:out_coff+cout] = epilogue(conv3x3(inp[..., in_coff:in_coff+cin])).

    Keywords: lrelu, s0, r1/r1_coff/s1, r2/r2_coff/s2, mask/mask_coff/mask_slope, pixel_shuffle, tap_mode,
    colsum/colsum_scale (fused bias gradient: colsum += scale * column sums of the written values), colsum_ws (its
    deterministic form: unscaled per-warp sums to slots of 32 floats, for det_finalize; colsum is then not written),
    wblob_row (the layer's row-hop weight image: lets the library pick conv3x3_row.cuh where the shape qualifies).
    See ``xmm_conv3x3_params`` in include/xmm_b200.h for the epilogue definition."""
    if _TORCH_OPS and not (kw.keys() - _TORCH_FWD_KEYS):
        # the registered dispatcher op (csrc/torch_ops.cpp) instead of ctypes: same launcher, same arguments
        from . import torch_ops

        torch_ops.load().conv3x3_fwd(inp, in_coff, cin, wblob_ptr, kc, cout, out, out_coff, kw.get("lrelu", 1.0),
                                     kw.get("s0", 1.0), kw.get("r1"), kw.get("r1_coff", 0), kw.get("s1", 0.0),
                                     kw.get("r2"), kw.get("r2_coff", 0), kw.get("s2", 0.0), kw.get("wblob_row") or 0,
                                     kw.get("tap_mode", 0))
        _count()
        return
    p = Conv3x3Params()
    _conv3x3_params(p, inp, in_coff, cin, wblob_ptr, kc, cout, out, out_coff, **kw)
    _lib.check(_lib.load().xmm_conv3x3_bf16(ctypes.byref(p), _lib.stream_ptr()))
    _count()


_TORCH_OPS = os.environ.get("XMM_TORCH_OPS", "0") == "1"
_TORCH_FWD_KEYS = {"lrelu", "s0", "r1", "r1_coff", "s1", "r2", "r2_coff", "s2", "wblob_row", "tap_mode"}


CHAIN_AUTO, CHAIN_PIPELINED, CHAIN_LAYER_BY_LAYER, CHAIN_FUSED = 0, 1, 2, 3
CHAIN_SKIP_DEAD_STORES = 0x100  # flag: outputs of layers 1..n-1 are not read after the call (inference)
CHAIN_RDB_PAIR, CHAIN_RDB_SINGLE = 0x200, 0x400  # flags: both kernels of the fused block as CTA pairs / single CTAs
CHAIN_SKIP_LAST = 0x800  # flag: layers 1..n-1 only, the last layer's output is not written (recompute for a backward)
_chain_ws: dict = {}
_chain_ws_retired: list = []  # outgrown workspaces stay allocated: a captured CUDA graph may still hold their address


def conv3x3_chain(layers, mode: int = CHAIN_AUTO) -> None:
    """Dependent 3x3 convolutions (one dense block: forward convs or backward data gradients) through
    ``xmm_conv3x3_chain_bf16``.  ``layers``: list of (args, kwargs) exactly as for :func:`conv3x3`; the result equals
    calling conv3x3 on them in order (up to fp32 summation order).  mode: CHAIN_AUTO (the fused dense-block kernels
    where the layers qualify, else layer by layer) / CHAIN_PIPELINED (one launch, layers pipelined over SM groups) /
    CHAIN_LAYER_BY_LAYER / CHAIN_FUSED (error if the layers are not a dense block), optionally
    ``| CHAIN_SKIP_DEAD_STORES`` or ``| CHAIN_SKIP_LAST``, and ``| CHAIN_RDB_PAIR`` or ``| CHAIN_RDB_SINGLE``."""
    n = len(layers)
    arr = (Conv3x3Params * n)()
    for p, (a, kw) in zip(arr, layers):
        _conv3x3_params(p, *a, **kw)
    lib = _lib.load()
    dev = layers[0][0][0].device
    need = int(lib.xmm_conv3x3_chain_workspace_bytes(n, arr[0].batch, arr[0].height))
    ws = _chain_ws.get(dev)
    if ws is None or ws.numel() < need:
        if ws is not None:
            _chain_ws_retired.append(ws)
        ws = torch.empty(max(need, 1 << 16), dtype=torch.uint8, device=dev)
        _chain_ws[dev] = ws
    _lib.check(lib.xmm_conv3x3_chain_bf16(arr, n, int(mode), ws.data_ptr(), ws.numel(), _lib.stream_ptr()))
    global LAST_CHAIN_LAUNCHES
    LAST_CHAIN_LAUNCHES = int(lib.xmm_last_chain_launches())  # 2 fused, 1 pipelined, n layer by layer
    _count(LAST_CHAIN_LAUNCHES)


def copy_channels(src: torch.Tensor, src_coff: int, dst: torch.Tensor, dst_coff: int, channels: int) -> None:
    """dst[..., dst_coff:dst_coff+channels] = src[..., src_coff:src_coff+channels] for two NHWC bf16 buffers of the same
    spatial shape (a dense block's input into and out of its 5F-channel buffer); 16-byte accesses."""
    _nhwc(src, "copy_channels source")
    _nhwc(dst, "copy_channels destination")
    if tuple(src.shape[:3]) != tuple(dst.shape[:3]):
        raise RuntimeError(f"copy_channels: spatial shapes {tuple(src.shape[:3])} and {tuple(dst.shape[:3])} differ")
    b, h, w, _ = src.shape
    _lib.check(_lib.load().xmm_copy_channels_bf16(src.data_ptr(), src.shape[3], src_coff, dst.data_ptr(), dst.shape[3],
                                                  dst_coff, channels, b * h * w, _lib.stream_ptr()))
    _count()


def conv_first(x: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor], out: torch.Tensor,
               out_coff: int, out2: Optional[torch.Tensor] = None, out2_coff: int = 0, *,
               gate: Optional[torch.Tensor] = None, mask: Optional[torch.Tensor] = None, mask_coff: int = 0,
               mask_slope: float = 1.0) -> None:
    """fp32 NCHW image -> bf16 NHWC features (generator_rrdb.py:31-37,67)."""
    _lib.require_cuda_tensor(x, torch.float32, "conv_first input")
    _lib.require_cuda_tensor(weight, torch.float32, "conv_first weight")
    _nhwc(out, "conv_first output")
    b, cin, h, w = x.shape
    p = ConvFirstParams()
    p.in_, p.weight, p.bias = x.data_ptr(), weight.data_ptr(), _ptr(bias)
    p.batch, p.cin, p.height, p.width, p.filters = b, cin, h, w, weight.shape[0]
    p.out, p.out_ctot, p.out_coff = out.data_ptr(), out.shape[3], out_coff
    if out2 is not None:
        _nhwc(out2, "conv_first output2")
        p.out2, p.out2_ctot, p.out2_coff = out2.data_ptr(), out2.shape[3], out2_coff
    if gate is not None:
        _lib.require_cuda_tensor(gate, torch.float32, "conv_first gate")
        if gate.shape != x.shape:
            raise RuntimeError("conv_first gate: shape must equal the input shape")
        p.gate = gate.data_ptr()
    if mask is not None:
        _nhwc(mask, "conv_first mask")
        p.mask, p.mask_ctot, p.mask_coff = mask.data_ptr(), mask.shape[3], mask_coff
    p.mask_slope = mask_slope
    _lib.check(_lib.load().xmm_conv_first(ctypes.byref(p), _lib.stream_ptr()))
    _count()


def conv_last(inp: torch.Tensor, in_coff: int, weight: torch.Tensor, bias: Optional[torch.Tensor],
              out: torch.Tensor, residual: Optional[torch.Tensor] = None, pre: Optional[torch.Tensor] = None,
              clamp: bool = True, wblob_ptr: Optional[int] = None) -> None:
    """bf16 NHWC features -> fp32 NCHW image (+ residual, clamp) (generator_rrdb.py:48-54,107-108,132-135).
    wblob_ptr: packed split-precision layer -> tensor-core path (see xmm_conv_last_params.wblob)."""
    _nhwc(inp, "conv_last input")
    _lib.require_cuda_tensor(weight, torch.float32, "conv_last weight")
    _lib.require_cuda_tensor(out, torch.float32, "conv_last output")
    b, h, w, ctot = inp.shape
    p = ConvLastParams()
    p.in_, p.in_ctot, p.in_coff = inp.data_ptr(), ctot, in_coff
    p.weight, p.bias = weight.data_ptr(), _ptr(bias)
    if residual is not None:
        _lib.require_cuda_tensor(residual, torch.float32, "conv_last residual")
        if residual.shape != out.shape:
            raise RuntimeError("conv_last residual: shape must equal the output shape")
        p.residual = residual.data_ptr()
    if pre is not None:
        _lib.require_cuda_tensor(pre, torch.float32, "conv_last pre")
        p.pre = pre.data_ptr()
    p.out = out.data_ptr()
    p.batch, p.cout, p.height, p.width, p.filters = b, weight.shape[0], h, w, weight.shape[1]
    p.clamp = 1 if clamp else 0
    p.wblob = wblob_ptr
    _lib.check(_lib.load().xmm_conv_last(ctypes.byref(p), _lib.stream_ptr()))
    _count()


def normalize(inp: torch.Tensor, max_val: float, stretch_mode: str, *, out: Optional[torch.Tensor] = None,
              mask: Optional[torch.Tensor] = None, pre_scale: float = 1.0) -> torch.Tensor:
    """Fused clamp / divide / stretch / clamp (+ detector mask, + counts->rate scale)."""
    if stretch_mode not in _lib.STRETCH_MODES:
        raise ValueError(f"Stretching function {stretch_mode} is not implemented")
    if not inp.is_cuda or not inp.is_contiguous() or inp.dtype not in (torch.float32, torch.int32):
        raise RuntimeError("normalize: expected a contiguous CUDA fp32 or int32 tensor")
    if out is None:
        out = torch.empty(inp.shape, dtype=torch.float32, device=inp.device)
    _lib.require_cuda_tensor(out, torch.float32, "normalize output")
    p = NormalizeParams()
    p.in_, p.in_is_int32 = inp.data_ptr(), int(inp.dtype == torch.int32)
    if mask is not None:
        _lib.require_cuda_tensor(mask, torch.uint8, "normalize mask")
        p.mask, p.mask_n = mask.data_ptr(), mask.numel()
    p.out, p.n = out.data_ptr(), inp.numel()
    p.pre_scale, p.max_val, p.stretch_mode = pre_scale, float(max_val), _lib.STRETCH_MODES[stretch_mode]
    scratch = None
    if not max_val > 0:
        scratch = torch.zeros(1, dtype=torch.float32, device=inp.device)
        p.scratch = scratch.data_ptr()
    _lib.check(_lib.load().xmm_normalize(ctypes.byref(p), _lib.stream_ptr()))
    _count(1 if max_val > 0 else 2)
    return out


def denormalize(inp: torch.Tensor, max_vals: torch.Tensor, stretch_mode: str) -> torch.Tensor:
    if stretch_mode not in _lib.STRETCH_MODES:
        raise ValueError(f"Stretching function {stretch_mode} is not implemented")
    _lib.require_cuda_tensor(inp, torch.float32, "denormalize input")
    mv = max_vals.to(device=inp.device, dtype=torch.float32).reshape(-1).contiguous()
    out = torch.empty_like(inp)
    per_image = inp.numel() // inp.shape[0] if inp.dim() > 0 and inp.shape[0] > 0 else inp.numel()
    _lib.check(_lib.load().xmm_denormalize(inp.data_ptr(), out.data_ptr(), inp.numel(), per_image, mv.data_ptr(),
                                           mv.numel(), _lib.STRETCH_MODES[stretch_mode], _lib.stream_ptr()))
    _count()
    return out


def restretch(x: torch.Tensor, from_mode: str, to_mode: str) -> torch.Tensor:
    """norm_to(denorm_from(x)) in one pass (metrics/xmm_metric_collection.py:135-143)."""
    for m in (from_mode, to_mode):
        if m not in _lib.STRETCH_MODES:
            raise ValueError(f"Stretching function {m} is not implemented")
    _lib.require_cuda_tensor(x, torch.float32, "restretch input")
    out = torch.empty_like(x)
    _lib.check(_lib.load().xmm_restretch(x.data_ptr(), out.data_ptr(), x.numel(), _lib.STRETCH_MODES[from_mode],
                                         _lib.STRETCH_MODES[to_mode], _lib.stream_ptr()))
    _count()
    return out


def prepare_counts(planes, res, max_val: float, stretch_mode: str, *, det_mask: Optional[torch.Tensor] = None,
                   exposure=1.0, upsample: int = 1, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Raw count planes -> normalised network input, one kernel (data/dataset.py:24-49,258-270).

    planes: 1..3 tensors [B,h,w] or [B,1,h,w] (image, AGN, background), all int32 or all fp32, on the GPU;
    res: int or (res_h, res_w); exposure: seconds, a float or a [B] tensor; returns [B,1,res_h,res_w] fp32."""
    if stretch_mode not in _lib.STRETCH_MODES:
        raise ValueError(f"Stretching function {stretch_mode} is not implemented")
    planes = [p for p in planes if p is not None]
    if not 1 <= len(planes) <= 3:
        raise RuntimeError("prepare_counts: 1..3 source planes")
    first = planes[0]
    if first.dim() == 4:
        if first.shape[1] != 1:
            raise RuntimeError("prepare_counts: single-channel count images only")
        planes = [p.reshape(p.shape[0], p.shape[2], p.shape[3]) for p in planes]
        first = planes[0]
    b, h, w = first.shape
    for p in planes:
        if not p.is_cuda or not p.is_contiguous() or p.dtype != first.dtype or p.shape != first.shape:
            raise RuntimeError("prepare_counts: planes must be contiguous CUDA tensors of one dtype and shape")
    if first.dtype not in (torch.int32, torch.float32):
        raise RuntimeError("prepare_counts: planes must be int32 or fp32")
    res_h, res_w = (res, res) if isinstance(res, int) else res
    if out is None:
        out = torch.empty(b, 1, res_h, res_w, dtype=torch.float32, device=first.device)
    _lib.require_cuda_tensor(out, torch.float32, "prepare_counts output")
    p = _lib.PrepareCountsParams()
    for k, t in enumerate(planes):
        p.src[k] = t.data_ptr()
    p.nsrc, p.src_is_int32 = len(planes), int(first.dtype == torch.int32)
    if det_mask is not None:
        _lib.require_cuda_tensor(det_mask, torch.uint8, "prepare_counts det_mask")
        if det_mask.numel() != h * w:
            raise RuntimeError("prepare_counts: det_mask must have the shape of one source image")
        p.mask = det_mask.data_ptr()
    p.batch, p.h, p.w, p.up, p.res_h, p.res_w = b, h, w, int(upsample), res_h, res_w
    keep = None
    if isinstance(exposure, torch.Tensor):
        keep = (1.0 / exposure.to(device=first.device, dtype=torch.float32)).reshape(-1).contiguous()
        if keep.numel() != b:
            raise RuntimeError("prepare_counts: one exposure per image")
        p.pre_scale, p.pre_scale_dev = 1.0, keep.data_ptr()
    else:
        p.pre_scale = 1.0 / float(exposure)
    p.max_val, p.stretch_mode, p.out = float(max_val), _lib.STRETCH_MODES[stretch_mode], out.data_ptr()
    _lib.check(_lib.load().xmm_prepare_counts(ctypes.byref(p), _lib.stream_ptr()))
    _count()
    return out


def image_upsample(x: torch.Tensor, scale: int) -> torch.Tensor:
    """Nearest upsample by an integer factor, divided by factor**2 (imageupsample.py:10-26)."""
    _lib.require_cuda_tensor(x, torch.float32, "image_upsample input")
    h, w = x.shape[-2:]
    n_img = x.numel() // (h * w) if h * w else 0
    out = torch.empty(*x.shape[:-2], h * scale, w * scale, dtype=torch.float32, device=x.device)
    _lib.check(_lib.load().xmm_image_upsample(x.data_ptr(), out.data_ptr(), n_img, h, w, scale, _lib.stream_ptr()))
    _count()
    return out


def pack_weights(jobs_dev_ptr: int, njobs: int) -> None:
    """Repack every layer listed in the device-side job table (one launch)."""
    _lib.check(_lib.load().xmm_pack_weights(jobs_dev_ptr, njobs, _lib.stream_ptr()))
    _count()


_WS = {}


def wgrad_workspace(device: torch.device) -> torch.Tensor:
    ws = _WS.get(str(device))
    if ws is None:
        ws = torch.empty(_lib.load().xmm_wgrad_workspace_bytes() // 4, dtype=torch.float32, device=device)
        _WS[str(device)] = ws
    return ws


def conv3x3_wgrad(x: torch.Tensor, dy: torch.Tensor, roles, dsts) -> None:
    """Tensor-core weight gradient.  roles: [(tap_begin, tap_count, x_c0, x_boxes, y_c0, n[, mode])];
    dsts: [(dw, o_count, i_total, i_begin, i_end, role, lane0, col0, scale, accumulate, perm[, o_begin, o_total])]."""
    _nhwc(x, "wgrad x")
    _nhwc(dy, "wgrad dy")
    if x.shape[:3] != dy.shape[:3]:
        raise RuntimeError("wgrad: x and dy must have the same batch / spatial shape")
    p = WgradParams()
    p.x, p.x_ctot, p.dy, p.dy_ctot = x.data_ptr(), x.shape[3], dy.data_ptr(), dy.shape[3]
    p.batch, p.height, p.width = x.shape[0], x.shape[1], x.shape[2]
    p.nroles = len(roles)
    for dst, r in zip(p.roles, roles):
        dst.tap_begin, dst.tap_count, dst.x_c0, dst.x_boxes, dst.y_c0, dst.n = r[:6]
        dst.mode = r[6] if len(r) > 6 else 0
    p.ndst = len(dsts)
    for dst, d in zip(p.dst, dsts):
        dw = d[0]
        _lib.require_cuda_tensor(dw, torch.float32, "wgrad dw")
        (dst.o_count, dst.i_total, dst.i_begin, dst.i_end, dst.role, dst.lane0, dst.col0, dst.scale, dst.accumulate,
         dst.perm) = d[1:11]
        dst.o_begin, dst.o_total = (d[11], d[12]) if len(d) > 11 else (0, 0)
        dst.dw = dw.data_ptr()
    p.workspace = wgrad_workspace(x.device).data_ptr()
    _lib.check(_lib.load().xmm_conv3x3_wgrad(ctypes.byref(p), _lib.stream_ptr()))
    _count(2)


def colsum(inp: torch.Tensor, c0: int, n: int, out: torch.Tensor, scale: float = 1.0, accumulate: bool = False) -> None:
    """out[i] (+)= scale * sum over pixels of inp[..., c0 + i]  (bias gradient)."""
    _nhwc(inp, "colsum input")
    _lib.require_cuda_tensor(out, torch.float32, "colsum output")
    npix = inp.shape[0] * inp.shape[1] * inp.shape[2]
    _lib.check(_lib.load().xmm_colsum_bf16(inp.data_ptr(), inp.shape[3], c0, n, npix, out.data_ptr(), scale,
                                           int(accumulate), _lib.stream_ptr()))
    _count()


def colsum_multi(inp: torch.Tensor, segments) -> None:
    """Several bias gradients in one pass over ``inp``.  segments: [(c0, n, out, scale, accumulate)]."""
    _nhwc(inp, "colsum input")
    arr = (_lib.ColsumSegment * len(segments))()
    for a, (c0, n, out, scale, accumulate) in zip(arr, segments):
        _lib.require_cuda_tensor(out, torch.float32, "colsum output")
        a.c0, a.n, a.out, a.scale, a.accumulate = c0, n, out.data_ptr(), scale, int(accumulate)
    npix = inp.shape[0] * inp.shape[1] * inp.shape[2]
    _lib.check(_lib.load().xmm_colsum_multi_bf16(inp.data_ptr(), inp.shape[3], npix, arr, len(segments),
                                                 _lib.stream_ptr()))
    _count()


def edge_wgrad(s: torch.Tensor, v: torch.Tensor, v_coff: int, channels: int, r: torch.Tensor,
               ssum: Optional[torch.Tensor] = None, gate: Optional[torch.Tensor] = None,
               v2: Optional[torch.Tensor] = None, v2_coff: int = 0, ws: Optional[torch.Tensor] = None) -> None:
    """r[o][c][tap] += sum_p s[o][p] * (v + v2)[p + off(tap)][c];  ssum[o] += sum_p s[o][p].
    ws: deterministic form -- per-CTA sums to slots of ns * channels * 9 + ns floats (r / ssum are not written)."""
    _lib.require_cuda_tensor(s, torch.float32, "edge_wgrad s")
    _nhwc(v, "edge_wgrad v")
    _lib.require_cuda_tensor(r, torch.float32, "edge_wgrad r")
    p = EdgeWgradParams()
    p.s, p.gate = s.data_ptr(), _ptr(gate)
    p.v, p.v_ctot, p.v_coff = v.data_ptr(), v.shape[3], v_coff
    if v2 is not None:
        _nhwc(v2, "edge_wgrad v2")
        p.v2, p.v2_ctot, p.v2_coff = v2.data_ptr(), v2.shape[3], v2_coff
    p.r, p.ssum = r.data_ptr(), _ptr(ssum)
    p.batch, p.ns, p.height, p.width, p.channels = s.shape[0], s.shape[1], s.shape[2], s.shape[3], channels
    if ws is not None:
        _lib.require_cuda_tensor(ws, torch.float32, "edge_wgrad ws")
        p.ws, p.ws_slots = ws.data_ptr(), ws.numel() // (s.shape[1] * channels * 9 + s.shape[1])
    _lib.check(_lib.load().xmm_edge_wgrad(ctypes.byref(p), _lib.stream_ptr()))
    _count()


def colsum_multi_det(inp: torch.Tensor, segments, ws: torch.Tensor) -> None:
    """Deterministic form of :func:`colsum_multi`: segments [(c0, n, scale)]; each CTA stores the unscaled sums of the
    segments' channels (concatenated) to its own slot of ``ws`` (sum(n) floats per slot, zero on entry)."""
    _nhwc(inp, "colsum input")
    _lib.require_cuda_tensor(ws, torch.float32, "colsum ws")
    arr = (_lib.ColsumSegment * len(segments))()
    for a, (c0, n, scale) in zip(arr, segments):
        a.c0, a.n, a.scale = c0, n, scale
    npix = inp.shape[0] * inp.shape[1] * inp.shape[2]
    row = sum(n for _, n, _ in segments)
    _lib.check(_lib.load().xmm_colsum_multi_det_bf16(inp.data_ptr(), inp.shape[3], npix, arr, len(segments),
                                                     ws.data_ptr(), ws.numel() // row, _lib.stream_ptr()))
    _count()


def det_slots(site: int, batch: int, height: int, width: int, channels: int) -> int:
    """Slots one call of a deterministic reduction site writes at most (_lib.DET_*; xmm_det_slots)."""
    n = int(_lib.load().xmm_det_slots(site, batch, height, width, channels))
    if n == 0:
        raise RuntimeError(f"xmm_det_slots: no slot layout for site {site} at {batch}x{height}x{width}x{channels} "
                           f"({_lib.load().xmm_last_error().decode()})")
    return n


def det_finalize(jobs_dev: torch.Tensor, njobs: int, max_n: int, dst_base: torch.Tensor) -> None:
    """One launch for a device table of :class:`_lib.DetJob`: dst_base[dst + i] (+)= scale * sum of the slots, in
    slot order; the slots read are left zero."""
    _lib.require_cuda_tensor(dst_base, torch.float32, "det_finalize dst_base")
    _lib.check(_lib.load().xmm_det_finalize(jobs_dev.data_ptr(), njobs, max_n, dst_base.data_ptr(), _lib.stream_ptr()))
    _count()
