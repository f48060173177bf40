"""ctypes binding of ``libxmm_b200.so`` (the C ABI declared in ``include/xmm_b200.h``).

The product path has no CPU or PyTorch-eager fallback: if the shared library is missing, or
the device is not an sm_100a GPU, every entry point raises.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_float, c_int, c_size_t, c_void_p

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libxmm_b200.so")


class PackSegment(Structure):
    _fields_ = [("src", c_void_p), ("src_cin", c_int), ("o_off", c_int), ("i_off", c_int), ("transpose", c_int),
                ("k_off", c_int), ("k_count", c_int), ("scale", c_float), ("n_off", c_int), ("n_count", c_int),
                ("part", c_int)]


class PackJob(Structure):
    _fields_ = [("dst", c_void_p), ("bias", c_void_p), ("nt", c_int), ("kc", c_int), ("nchunks", c_int),
                ("nseg", c_int), ("perm", c_int), ("n_valid", c_int), ("bias_n", c_int), ("seg", PackSegment * 5),
                ("tap_order", c_int)]


class Conv3x3Params(Structure):
    _fields_ = [("in_", c_void_p), ("in_ctot", c_int), ("in_coff", c_int), ("cin", c_int),
                ("wblob", c_void_p), ("kc", c_int), ("cout", c_int),
                ("batch", c_int), ("height", c_int), ("width", c_int),
                ("lrelu_slope", c_float),
                ("mask", c_void_p), ("mask_ctot", c_int), ("mask_coff", c_int), ("mask_slope", c_float),
                ("s0", c_float),
                ("r1", c_void_p), ("r1_ctot", c_int), ("r1_coff", c_int), ("s1", c_float),
                ("r2", c_void_p), ("r2_ctot", c_int), ("r2_coff", c_int), ("s2", c_float),
                ("out", c_void_p), ("out_ctot", c_int), ("out_coff", c_int),
                ("pixel_shuffle", c_int), ("tap_mode", c_int), ("colsum", c_void_p), ("colsum_scale", c_float),
                ("shuffle_stride", c_int), ("wblob_row", c_void_p), ("colsum_ws", c_void_p), ("colsum_ws_slots", c_size_t)]


class NormalizeParams(Structure):
    _fields_ = [("in_", c_void_p), ("in_is_int32", c_int), ("mask", c_void_p), ("mask_n", c_size_t),
                ("out", c_void_p), ("n", c_size_t), ("pre_scale", c_float), ("max_val", c_float),
                ("stretch_mode", c_int), ("scratch", c_void_p)]


class ConvFirstParams(Structure):
    _fields_ = [("in_", c_void_p), ("weight", c_void_p), ("bias", c_void_p),
                ("batch", c_int), ("cin", c_int), ("height", c_int), ("width", c_int), ("filters", c_int),
                ("out", c_void_p), ("out_ctot", c_int), ("out_coff", c_int),
                ("out2", c_void_p), ("out2_ctot", c_int), ("out2_coff", c_int),
                ("gate", c_void_p), ("mask", c_void_p), ("mask_ctot", c_int), ("mask_coff", c_int),
                ("mask_slope", c_float)]


class ConvLastParams(Structure):
    _fields_ = [("in_", c_void_p), ("in_ctot", c_int), ("in_coff", c_int),
                ("weight", c_void_p), ("bias", c_void_p), ("residual", c_void_p),
                ("out", c_void_p), ("pre", c_void_p),
                ("batch", c_int), ("cout", c_int), ("height", c_int), ("width", c_int), ("filters", c_int),
                ("clamp", c_int), ("wblob", c_void_p)]


class WgradRole(Structure):
    _fields_ = [("tap_begin", c_int), ("tap_count", c_int), ("x_c0", c_int), ("x_boxes", c_int), ("y_c0", c_int),
                ("n", c_int), ("mode", c_int)]


class WgradDst(Structure):
    _fields_ = [("dw", c_void_p), ("o_count", c_int), ("i_total", c_int), ("i_begin", c_int), ("i_end", c_int),
                ("role", c_int), ("lane0", c_int), ("col0", c_int), ("scale", c_float), ("accumulate", c_int),
                ("perm", c_int), ("o_begin", c_int), ("o_total", c_int)]


class WgradParams(Structure):
    _fields_ = [("x", c_void_p), ("x_ctot", c_int), ("dy", c_void_p), ("dy_ctot", c_int),
                ("batch", c_int), ("height", c_int), ("width", c_int),
                ("nroles", c_int), ("roles", WgradRole * 4), ("ndst", c_int), ("dst", WgradDst * 16),
                ("workspace", c_void_p)]


class EdgeWgradParams(Structure):
    _fields_ = [("s", c_void_p), ("gate", c_void_p), ("v", c_void_p), ("v_ctot", c_int), ("v_coff", c_int),
                ("v2", c_void_p), ("v2_ctot", c_int), ("v2_coff", c_int), ("r", c_void_p), ("ssum", c_void_p),
                ("batch", c_int), ("ns", c_int), ("height", c_int), ("width", c_int), ("channels", c_int),
                ("ws", c_void_p), ("ws_slots", c_size_t)]


class ScaleStats(Structure):
    _fields_ = [(n, c_float) for n in ("minp", "maxp", "mint", "maxt", "nmaxp", "nminp", "dr", "c1", "c2", "use_p",
                                       "d_dr", "pad")]


class SsimStatsParams(Structure):
    _fields_ = [("preds", c_void_p), ("target", c_void_p), ("nimg", c_int), ("h", c_int), ("w", c_int),
                ("stats_dev", c_void_p), ("window", c_float * 19), ("use_sim", c_int), ("acc", c_void_p),
                ("kimg", c_void_p), ("ga", c_void_p), ("gb", c_void_p), ("gc", c_void_p)]


class SsimGradParams(Structure):
    _fields_ = [("preds", c_void_p), ("target", c_void_p), ("nimg", c_int), ("h", c_int), ("w", c_int),
                ("stats_dev", c_void_p), ("window", c_float * 19), ("ga", c_void_p), ("gb", c_void_p),
                ("gc", c_void_p), ("coarse", c_void_p), ("grad", c_void_p), ("accumulate", c_int)]


class MsssimFinalizeParams(Structure):
    _fields_ = [("acc", c_void_p * 5), ("tiles", c_int * 5), ("nvalid", c_int * 5), ("nscales", c_int),
                ("batch", c_int), ("channels", c_int), ("betas", c_float * 5), ("k1", c_float), ("k2", c_float),
                ("stats_dev", c_void_p), ("value", c_void_p), ("img_val", c_void_p), ("kimg", c_void_p),
                ("gl_dev", c_void_p), ("weight", c_float)]


class PrepareCountsParams(Structure):
    _fields_ = [("src", c_void_p * 3), ("nsrc", c_int), ("src_is_int32", c_int), ("mask", c_void_p),
                ("batch", c_int), ("h", c_int), ("w", c_int), ("up", c_int), ("res_h", c_int), ("res_w", c_int),
                ("pre_scale", c_float), ("pre_scale_dev", c_void_p), ("max_val", c_float), ("stretch_mode", c_int),
                ("out", c_void_p)]


class ColsumSegment(Structure):
    _fields_ = [("c0", c_int), ("n", c_int), ("out", c_void_p), ("scale", c_float), ("accumulate", c_int)]


class DetJob(Structure):
    _fields_ = [("slots", c_void_p), ("count", c_int), ("stride", c_int), ("dst", c_size_t), ("n", c_int),
                ("scale", c_float), ("accumulate", c_int)]


DET_CONV3X3, DET_COLSUM, DET_EDGE_WGRAD = 0, 1, 2


EXTRA_STRUCTS = {"xmm_colsum_segment": ColsumSegment, "xmm_prepare_counts_params": PrepareCountsParams, "xmm_scale_stats": ScaleStats, "xmm_ssim_stats_params": SsimStatsParams,
                 "xmm_ssim_grad_params": SsimGradParams, "xmm_msssim_finalize_params": MsssimFinalizeParams,
                 "xmm_wgrad_role": WgradRole, "xmm_wgrad_dst": WgradDst, "xmm_wgrad_params": WgradParams,
                 "xmm_edge_wgrad_params": EdgeWgradParams, "xmm_det_job": DetJob}

# name -> (restype, argtypes); the non-GPU test-suite checks every name in include/xmm_b200.h is here
# and exported by the shared object.
SIGNATURES = {
    "xmm_last_error": (c_char_p, []),
    "xmm_version": (c_int, []),
    "xmm_check_device": (c_int, []),
    "xmm_set_sm_reserve": (c_int, [c_int]),
    "xmm_pack_blob_bytes": (c_size_t, [c_int, c_int, c_int]),
    "xmm_pack_weights": (c_int, [c_void_p, c_int, c_void_p]),
    "xmm_conv3x3_bf16": (c_int, [POINTER(Conv3x3Params), c_void_p]),
    "xmm_conv3x3_chain_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "xmm_last_chain_launches": (c_int, []),
    "xmm_conv3x3_chain_bf16": (c_int, [POINTER(Conv3x3Params), c_int, c_int, c_void_p, c_size_t, c_void_p]),
    "xmm_normalize": (c_int, [POINTER(NormalizeParams), c_void_p]),
    "xmm_denormalize": (c_int, [c_void_p, c_void_p, c_size_t, c_size_t, c_void_p, c_int, c_int, c_void_p]),
    "xmm_restretch": (c_int, [c_void_p, c_void_p, c_size_t, c_int, c_int, c_void_p]),
    "xmm_prepare_counts": (c_int, [POINTER(PrepareCountsParams), c_void_p]),
    "xmm_image_upsample": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "xmm_conv_first": (c_int, [POINTER(ConvFirstParams), c_void_p]),
    "xmm_conv_last": (c_int, [POINTER(ConvLastParams), c_void_p]),
    "xmm_wgrad_workspace_bytes": (c_size_t, []),
    "xmm_conv3x3_wgrad": (c_int, [POINTER(WgradParams), c_void_p]),
    "xmm_colsum_bf16": (c_int, [c_void_p, c_int, c_int, c_int, c_size_t, c_void_p, c_float, c_int, c_void_p]),
    "xmm_colsum_multi_bf16": (c_int, [c_void_p, c_int, c_size_t, POINTER(ColsumSegment), c_int, c_void_p]),
    "xmm_colsum_multi_det_bf16": (c_int, [c_void_p, c_int, c_size_t, POINTER(ColsumSegment), c_int, c_void_p, c_size_t,
                                          c_void_p]),
    "xmm_edge_wgrad": (c_int, [POINTER(EdgeWgradParams), c_void_p]),
    "xmm_det_slots": (c_size_t, [c_int, c_int, c_int, c_int, c_int]),
    "xmm_det_finalize": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "xmm_loss_workspace_floats": (c_size_t, []),
    "xmm_loss_reduce": (c_int, [c_void_p, c_void_p, c_size_t, c_void_p, c_void_p, c_void_p, c_void_p]),
    "xmm_loss_grad": (c_int, [c_void_p, c_void_p, c_size_t, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "xmm_avgpool2_pair": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "xmm_ssim_prepare": (c_int, [c_void_p, c_size_t, c_void_p, c_float, c_float, c_void_p]),
    "xmm_ssim_tiles": (c_int, [c_int, c_int]),
    "xmm_ssim_stats": (c_int, [POINTER(SsimStatsParams), c_void_p]),
    "xmm_ssim_grad": (c_int, [POINTER(SsimGradParams), c_void_p]),
    "xmm_msssim_finalize": (c_int, [POINTER(MsssimFinalizeParams), c_void_p]),
    "xmm_adam_step": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_float, c_float, c_float, c_float,
                              c_int, c_float, c_void_p]),
}

_lib = None


def load() -> ctypes.CDLL:
    """Load the shared library (no device required)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is not built. Run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). xmm_superres_denoise_b200 has no CPU / eager fallback.")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        msg = load().xmm_last_error()
        raise RuntimeError(f"libxmm_b200 error {rc}: {msg.decode() if msg else '?'}")


def stream_ptr() -> int:
    """cudaStream_t of torch's current stream (launches join torch's stream order)."""
    return torch.cuda.current_stream().cuda_stream


def require_cuda_tensor(t: torch.Tensor, dtype: torch.dtype, name: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(f"{name}: expected a CUDA tensor (xmm_superres_denoise_b200 has no CPU path)")
    if t.dtype != dtype:
        raise RuntimeError(f"{name}: expected dtype {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise RuntimeError(f"{name}: expected a contiguous tensor")
    # The library launches on the CURRENT device and on its current stream (stream_ptr): a tensor of another GPU
    # would be an illegal address -- or, with peer access on, a silent run on the wrong GPU.
    if t.device.index != torch.cuda.current_device():
        raise RuntimeError(f"{name}: tensor lives on {t.device} but the current device is cuda:"
                           f"{torch.cuda.current_device()}; call torch.cuda.set_device / use torch.cuda.device(...)")


STRETCH_MODES = {"linear": 0, "sqrt": 1, "asinh": 2, "log": 3}
