"""ctypes binding of libmcb200.so (the C-ABI declared in include/mcb200.h).

There is no fallback: if the shared library is missing or a call fails this module raises.  Build the library
with ``python -c "import __graft_entry__ as g; g.build()"`` (or ``make -C modelcompression_b200/csrc``).
"""
import ctypes
import os
from ctypes import (POINTER, c_char_p, c_double, c_float, c_int, c_int64, c_size_t, c_uint8, c_void_p)

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmcb200.so")

MC_MAX_SEGMENTS = 64
MC_EPI_PNHWC, MC_EPI_REORG2, MC_EPI_NCHW_F32, MC_EPI_DECODE = 0, 1, 2, 4


class McError(RuntimeError):
    """A libmcb200 entry point returned a non-zero status."""


class mc_decode_params(ctypes.Structure):
    _fields_ = [
        ("d_boxes", c_void_p), ("d_cls", c_void_p), ("d_head", c_void_p),
        ("A", c_int), ("nc", c_int), ("conf_thresh", c_float), ("only_objectness", c_int),
        ("anchors", c_float * 32),
    ]


class mc_conv_desc(ctypes.Structure):
    _fields_ = [
        ("d_in", c_void_p), ("d_wpack", c_void_p), ("d_scale", c_void_p), ("d_shift", c_void_p), ("d_out", c_void_p),
        ("B", c_int), ("H", c_int), ("W", c_int),
        ("Cin", c_int), ("Cin_ld", c_int),
        ("N", c_int), ("Npad", c_int),
        ("ksize", c_int), ("leaky", c_int), ("epi_mode", c_int),
        ("ldc", c_int), ("ch_off", c_int),
        ("block_n", c_int), ("stages", c_int), ("block_k", c_int), ("in_cols", c_int),
        ("decode", POINTER(mc_decode_params)),
        ("d_ws", c_void_p), ("ws_bytes", c_size_t),
        ("d_stat_sum", c_void_p), ("d_stat_sumsq", c_void_p),
    ]


# name -> (restype, argtypes); every symbol include/mcb200.h declares
_SIGNATURES = {
    "mc_version": (c_int, []),
    "mc_last_error_string": (c_char_p, []),
    "mc_device_ok": (c_int, []),
    "mc_kth_abs_select": (c_int, [POINTER(c_void_p), POINTER(c_int64), c_int, c_int64, c_float, c_void_p,
                                  c_void_p, c_size_t, c_void_p]),
    "mc_workspace_bytes_kth_abs_select": (c_size_t, [c_int64]),
    "mc_weight_prune_masks": (c_int, [POINTER(c_void_p), POINTER(c_void_p), POINTER(c_int64), c_int, c_int64, c_float,
                                      c_void_p, c_void_p, c_size_t, c_void_p]),
    "mc_debug_select_used_fast": (c_int, [c_void_p, c_void_p]),
    "mc_debug_select_tstamps": (c_int, [c_void_p, c_void_p, c_void_p]),
    "mc_mask_apply_gt": (c_int, [POINTER(c_void_p), POINTER(c_void_p), POINTER(c_int64), c_int, c_void_p, c_int,
                                 c_void_p]),
    "mc_apply_masks": (c_int, [POINTER(c_void_p), POINTER(c_void_p), POINTER(c_int64), c_int, c_void_p]),
    "mc_count_zeros": (c_int, [POINTER(c_void_p), POINTER(c_int64), c_int, c_void_p, c_void_p]),
    "mc_masked_residual": (c_int, [POINTER(c_void_p), POINTER(c_void_p), POINTER(c_int64), c_int, c_void_p,
                                   c_void_p]),
    "mc_filter_values": (c_int, [POINTER(c_void_p), POINTER(c_int), POINTER(c_int), POINTER(c_int), POINTER(c_int),
                                 c_int, c_void_p, c_void_p]),
    "mc_filter_prune": (c_int, [POINTER(c_void_p), POINTER(c_int), POINTER(c_int), POINTER(c_int), POINTER(c_int), c_int,
                                c_int64, c_double, c_void_p, c_void_p, POINTER(c_void_p), c_void_p, c_void_p, c_size_t,
                                c_void_p]),
    "mc_workspace_bytes_filter_prune": (c_size_t, []),
    "mc_filter_prune_greedy": (c_int, [POINTER(c_void_p), POINTER(c_int), POINTER(c_int), POINTER(c_int),
                                       POINTER(c_int), c_int, c_int64, c_int64, c_double, c_int, c_void_p, c_void_p,
                                       POINTER(c_void_p), c_void_p, c_size_t, c_void_p]),
    "mc_workspace_bytes_filter_prune_greedy": (c_size_t, [c_int]),
    "mc_decode_region": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, POINTER(c_float), c_float, c_int,
                                 c_void_p, c_void_p, c_void_p, c_void_p]),
    "mc_nms_batched": (c_int, [c_void_p, c_void_p, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p]),
    "mc_nms_detect": (c_int, [c_void_p, c_void_p, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p, c_int, c_float,
                              c_void_p, c_void_p, c_void_p]),
    "mc_compact_detections": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_int,
                                      c_void_p, c_void_p, c_void_p]),
    "mc_bbox_ious": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p]),
    "mc_reorg_nchw": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "mc_conv_fwd": (c_int, [POINTER(mc_conv_desc), c_void_p]),
    "mc_conv_chain_fwd": (c_int, [POINTER(mc_conv_desc), c_int, c_void_p]),
    "mc_workspace_bytes_conv_chain": (c_size_t, [POINTER(mc_conv_desc), c_int]),
    "mc_workspace_bytes_conv_fwd": (c_size_t, [POINTER(mc_conv_desc)]),
    "mc_conv_last_plan": (c_int, [POINTER(c_int)]),
    "mc_conv_direct_supported": (c_int, [c_int, c_int, c_int]),
    "mc_conv_direct_fwd": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                   c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "mc_conv_thin_geometry": (c_int, [c_int, c_int, c_int, c_int, c_int, POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    "mc_conv_thin_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int,
                                 c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "mc_conv_im2col_supported": (c_int, [c_int, c_int, c_int, c_int]),
    "mc_conv_im2col_geometry": (c_int, [c_int, c_int, c_int, c_int, POINTER(c_int), POINTER(c_int), POINTER(c_int),
                                        POINTER(c_int)]),
    "mc_conv_im2col_fwd": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                   c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "mc_debug_im2col_timeout": (c_int, []),
    "mc_debug_conv_trace": (c_int, [c_void_p]),
    "mc_conv_window_supported": (c_int, [c_int, c_int, c_int, c_int]),
    "mc_conv_window_geometry": (c_int, [c_int, c_int, c_int, c_int, POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    "mc_conv_window_fwd": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                   c_int, c_int, c_int, c_int, c_void_p]),
    "mc_pack_conv_weights": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_int,
                                     c_void_p, c_int, c_int, c_void_p]),
    "mc_maxpool2x2": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "mc_unpack_pnhwc": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "mc_pack_pnhwc": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "mc_col_stats": (c_int, [c_void_p, c_int64, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "mc_bn_finalize": (c_int, [c_void_p, c_void_p, c_int, c_double, c_void_p, c_void_p, c_float, c_float, c_void_p,
                               c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "mc_bn_apply": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p, c_int,
                            c_int, c_int, c_void_p]),
    "mc_bn_backward": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p,
                               c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "mc_maxpool2x2_backward": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int,
                                       c_int, c_void_p]),
    "mc_workspace_bytes_region_loss": (c_size_t, [c_int]),
    "mc_region_loss": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, POINTER(c_double), c_float, c_float,
                               c_float, c_float, c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "mc_voc_table": (c_int, [c_void_p, c_int64, c_void_p, c_float, c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "mc_workspace_bytes_voc_match": (c_size_t, [c_int64, c_int64]),
    "mc_voc_match": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_int64, c_double, c_void_p,
                             c_void_p, c_void_p, c_size_t, c_void_p]),
    "mc_bn_pool_supported": (c_int, [c_int]),
    "mc_bn_apply_pool": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p, c_int,
                                 c_void_p]),
    "mc_bn_pool_backward": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p,
                                    c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int,
                                    c_void_p]),
    "mc_pack_conv_weights_dgrad": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_int, c_void_p]),
    "mc_conv_wgrad": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p,
                              c_void_p, c_int, c_void_p, c_size_t, c_void_p]),
    "mc_workspace_bytes_conv_wgrad": (c_size_t, [c_int, c_int, c_int, c_int, c_int, c_int]),
    "mc_conv_wgrad_plan": (c_int, [c_int, c_int, c_int, c_int, c_int, c_int, POINTER(c_int)]),
    "mc_conv_wgrad_first": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p,
                                    c_void_p, c_size_t, c_void_p]),
    "mc_workspace_bytes_conv_wgrad_first": (c_size_t, [c_int, c_int, c_int, c_int, c_int]),
    "mc_sgd_momentum_step": (c_int, [POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p), POINTER(c_int64), c_int,
                                     c_float, c_float, c_float, c_int, c_void_p]),
}

EXPORTED_SYMBOLS = tuple(sorted(_SIGNATURES))

_lib = None


def load():
    """Load libmcb200.so (once) and set the ctypes prototypes.  Raises if the library is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "modelcompression_b200: %s is not built. There is no CPU/PyTorch fallback for this path; build it with "
            "`python -c 'import __graft_entry__ as g; g.build()'` or `make -C modelcompression_b200/csrc`." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so is stale
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what=""):
    if rc != 0:
        msg = load().mc_last_error_string()
        raise McError("%s failed (%d): %s" % (what or "libmcb200 call", rc, msg.decode() if msg else "?"))


def stream_ptr():
    import torch
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr_array(tensors):
    """ctypes array of device pointers for a list of torch tensors (None -> NULL)."""
    arr = (c_void_p * len(tensors))()
    for i, t in enumerate(tensors):
        arr[i] = None if t is None else t.data_ptr()
    return arr


def int64_array(vals):
    return (c_int64 * len(vals))(*[int(v) for v in vals])


def int_array(vals):
    return (c_int * len(vals))(*[int(v) for v in vals])


def require_cuda(t, what):
    if not t.is_cuda:
        raise RuntimeError(
            "%s: tensor is on %s. modelcompression_b200 runs this path on a B200 (sm_100a) only; there is no CPU "
            "fallback (move the model/tensors to CUDA)." % (what, t.device))
