"""Thin ctypes loader for ``liblsfa_b200.so`` (the C ABI of ``include/lsfa_ops.h``).

Holds no state beyond the loaded handle.  There is NO fallback: if the library is
missing or fails to load, every operator of this package raises ``LsfaLibraryError``.
ctypes releases the GIL around each call, so N host threads can drive N devices
(the threading model of the reference's tester.py:301-309).
"""
from __future__ import annotations

import ctypes as C
import os

from . import _build

# --- enums (mirror include/lsfa_ops.h) ---------------------------------------------------
ABI_VERSION = 1
OK, E_BADARG, E_SHAPE, E_ALIGN, E_CUDA, E_UNSUPPORTED = 0, -1, -2, -3, -4, -5
REQ_NULL, REQ_WRITE, REQ_INPLACE, REQ_ADD = 0, 1, 2, 3
POOL_CENTRE2X2, POOL_AVG16 = 0, 1
FLOW_PREPOOLED, FLOW_RAW_I32, FLOW_RAW_F32, FLOW_GRID, FLOW_COVIAR_I32 = 0, 1, 2, 3, 4
W_NONE, W_ADD, W_MEAN, W_LOGITS, W_COSINE = 0, 1, 2, 3, 4
LAYOUT_NCHW_F32, LAYOUT_NHWC_F32, LAYOUT_NHWC_BF16 = 0, 1, 2

_ERR_NAMES = {E_BADARG: "LSFA_E_BADARG", E_SHAPE: "LSFA_E_SHAPE", E_ALIGN: "LSFA_E_ALIGN",
              E_CUDA: "LSFA_E_CUDA", E_UNSUPPORTED: "LSFA_E_UNSUPPORTED"}


class LsfaLibraryError(RuntimeError):
    """The CUDA library is missing / unloadable.  Never swallowed, never worked around."""


class LsfaError(RuntimeError):
    """A C-ABI call returned a negative status (message from lsfa_last_error())."""

    def __init__(self, code, message):
        super().__init__("%s (%d): %s" % (_ERR_NAMES.get(code, "LSFA_E_?"), code, message))
        self.code = code


class LsfaAggArgs(C.Structure):
    _fields_ = [
        ("struct_bytes", C.c_int32), ("layout", C.c_int32),
        ("N", C.c_int32), ("C", C.c_int32), ("H", C.c_int32), ("W", C.c_int32),
        ("key_h", C.c_int32), ("key_w", C.c_int32), ("num_keys", C.c_int32),
        ("key", C.c_void_p), ("key_index", C.c_void_p),
        ("flow_kind", C.c_int32), ("flow", C.c_void_p),
        ("mv_h", C.c_int32), ("mv_w", C.c_int32), ("im_scale", C.c_double),
        ("pool_mode", C.c_int32),
        ("scale_map", C.c_void_p), ("res", C.c_void_p), ("rnet_w", C.c_void_p),
        ("rnet_b", C.c_void_p),
        ("cur", C.c_void_p), ("weight_mode", C.c_int32), ("logits", C.c_void_p),
        ("emb_warp", C.c_void_p), ("emb_cur", C.c_void_p), ("E", C.c_int32),
        ("bypass", C.c_void_p),
        ("out", C.c_void_p), ("req", C.c_int32),
        ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t),
        ("mv_src_h", C.c_int32), ("mv_src_w", C.c_int32), ("mv_negate", C.c_int32), ("mv_hflip", C.c_int32),
        ("force_generic", C.c_int32),
    ]


class LsfaAggGrads(C.Structure):
    _fields_ = [
        ("struct_bytes", C.c_int32), ("out_grad", C.c_void_p),
        ("grad_key", C.c_void_p), ("req_key", C.c_int32),
        ("grad_flow", C.c_void_p), ("req_flow", C.c_int32),
        ("grad_scale", C.c_void_p), ("req_scale", C.c_int32),
        ("grad_cur", C.c_void_p), ("req_cur", C.c_int32),
        ("grad_logits", C.c_void_p), ("req_logits", C.c_int32),
        ("grad_res", C.c_void_p), ("req_res", C.c_int32),
        ("grad_rnet_w", C.c_void_p), ("grad_rnet_b", C.c_void_p), ("req_rnet", C.c_int32),
        ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t),
        ("grad_emb_warp", C.c_void_p), ("grad_emb_cur", C.c_void_p), ("req_emb", C.c_int32),
    ]


class LsfaHostAggArgs(C.Structure):
    _fields_ = [
        ("struct_bytes", C.c_int32),
        ("N", C.c_int32), ("C", C.c_int32), ("H", C.c_int32), ("W", C.c_int32),
        ("mv_h", C.c_int32), ("mv_w", C.c_int32), ("im_scale", C.c_double),
        ("weight_mode", C.c_int32), ("num_new_keys", C.c_int32),
        ("key", C.c_void_p), ("key_slot", C.c_void_p), ("key_index", C.c_void_p),
        ("scale_map", C.c_void_p), ("cur", C.c_void_p), ("mv", C.c_void_p), ("logits", C.c_void_p),
        ("out", C.c_void_p),
        ("key_table", C.c_void_p), ("num_slots", C.c_int32),
        ("chunk", C.c_int32), ("depth", C.c_int32),
        ("staging", C.c_void_p), ("staging_bytes", C.c_size_t),
        ("stream_in", C.c_void_p), ("stream_run", C.c_void_p), ("stream_out", C.c_void_p),
    ]


_I, _D, _P, _SZ = C.c_int, C.c_double, C.c_void_p, C.c_size_t

# name -> (restype, argtypes); also the list the symbol-export test checks
PROTOTYPES = {
    "lsfa_version": (_I, []),
    "lsfa_last_error": (C.c_char_p, []),
    "lsfa_mv_pool_i32": (_I, [_P, _P, _I, _I, _I, _D, _I, _P]),
    "lsfa_mv_pool_f32": (_I, [_P, _P, _I, _I, _I, _D, _I, _P]),
    "lsfa_res_pool_i32": (_I, [_P, _P, _I, _I, _I, _P, _D, _I, _P]),
    "lsfa_res_pool_f32": (_I, [_P, _P, _I, _I, _I, _P, _D, _I, _P]),
    "lsfa_res_coviar_pool_i32": (_I, [_P, _P, _I, _I, _I, _I, _I, _D, _I, _P, _D, _I, _P]),
    "lsfa_mv_centre_rows_h2d": (_I, [_P, _P, _I, _I, _I, _P, _P]),
    "lsfa_host_aggregate_staging_bytes": (_SZ, [C.POINTER(LsfaHostAggArgs)]),
    "lsfa_host_aggregate_f32_nchw": (_I, [C.POINTER(LsfaHostAggArgs)]),
    "lsfa_host_aggregate_bytes": (_I, [C.POINTER(LsfaHostAggArgs), C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
    "lsfa_mv_prepare_i32": (_I, [_P, _P, _I, _I, _I, _I, _I, _D, _I, _I, _P]),
    "lsfa_grid_generator_warp_f32": (_I, [_P, _P, _I, _I, _I, _P]),
    "lsfa_bilinear_sampler_f32": (_I, [_P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P]),
    "lsfa_sampler_coords_f32": (_I, [_P, _I, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "lsfa_warp_scale_aggregate": (_I, [C.POINTER(LsfaAggArgs), _P]),
    "lsfa_warp_scale_aggregate_f32_nchw": (_I, [C.POINTER(LsfaAggArgs), _P]),
    "lsfa_warp_scale_aggregate_bf16_nhwc": (_I, [C.POINTER(LsfaAggArgs), _P]),
    "lsfa_warp_scale_aggregate_workspace_bytes": (_SZ, [C.POINTER(LsfaAggArgs)]),
    "lsfa_warp_scale_aggregate_num_launches": (_I, [C.POINTER(LsfaAggArgs)]),
    "lsfa_cosine_logits": (_I, [_P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "lsfa_cosine_logits_workspace_bytes": (_SZ, [_I, _I, _I, _I, _I]),
    "lsfa_cosine_logits_ws": (_I, [_P, _P, _P, _I, _I, _I, _I, _I, _P, _SZ, _P]),
    "lsfa_cosine_logits_backward_workspace_bytes": (_SZ, [_I, _I, _I, _I]),
    "lsfa_cosine_logits_backward_f32_nchw": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P, _SZ, _I, _P]),
    "lsfa_unfused_chain_f32_nchw": (_I, [_P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "lsfa_unfused_chain_num_launches": (_I, []),
    "lsfa_blend_logits_f32": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "lsfa_choose_feat_f32": (_I, [_P, _P, _P, _P, _I, C.c_longlong, _P]),
    "lsfa_mv_accumulate_workspace_bytes": (_SZ, [_I, _I, _I]),
    "lsfa_mv_accumulate_i32": (_I, [_P, _P, _I, _I, _I, _I, _I, _P, _P, _SZ, _P]),
    "lsfa_mv_accumulate_trace_workspace_bytes": (_SZ, [_I, _I, _I, _I]),
    "lsfa_mv_accumulate_algo_i32": (_I, [_P, _P, _I, _I, _I, _I, _I, _P, _P, _SZ, _I, _P]),
    "lsfa_coviar_residual_u8": (_I, [_P, _P, _P, _P, _I, _I, _I, _P]),
    "lsfa_bilinear_sampler_backward_workspace_bytes": (_SZ, [_I, _I, _I, _I, _I, _I]),
    "lsfa_bilinear_sampler_backward_f32": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _P, _SZ, _I, _P]),
    "lsfa_bilinear_sampler_backward_num_launches": (_I, [_I, _I, _I, _I, _I, _I, _I, _I, _SZ, _I]),
    "lsfa_grid_generator_warp_backward_f32": (_I, [_P, _P, _I, _I, _I, _I, _P]),
    "lsfa_warp_backward_f32": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P, _SZ, _I, _P]),
    "lsfa_pack_conv_weight_bf16": (_I, [_P, _P, _I, _I, _I, _P]),
    "lsfa_conv_bf16_nhwc": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P]),
    "lsfa_embed_cosine_logits_workspace_bytes": (_SZ, [_I, _I, _I, _I, _I, _I]),
    "lsfa_embed_cosine_logits_bf16_nhwc": (_I, [_P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P, _SZ, _P]),
    "lsfa_nq_logits_bf16_nhwc": (_I, [_P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "lsfa_warp_scale_aggregate_backward_workspace_bytes": (_SZ, [C.POINTER(LsfaAggArgs), C.POINTER(LsfaAggGrads)]),
    "lsfa_warp_scale_aggregate_backward_f32_nchw": (_I, [C.POINTER(LsfaAggArgs), C.POINTER(LsfaAggGrads), _P]),
    "lsfa_nchw_to_nhwc": (_I, [_P, _P, _I, _I, _I, _I, _I, _P]),
    "lsfa_nhwc_to_nchw": (_I, [_P, _P, _I, _I, _I, _I, _I, _P]),
    "lsfa_graph_begin": (_I, [_P]),
    "lsfa_graph_end": (_I, [_P, C.POINTER(C.c_void_p)]),
    "lsfa_graph_launch": (_I, [_P, _P]),
    "lsfa_graph_destroy": (_I, [_P]),
}

_lib = None


def library_path() -> str:
    return os.environ.get("LSFA_B200_LIB", _build.LIB_PATH)


def load():
    """dlopen the library once and bind prototypes.  Raises LsfaLibraryError if absent."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.exists(path):
        raise LsfaLibraryError(
            "%s not found: build it with `python -m lsfa_b200._build` (needs nvcc, sm_100a). "
            "lsfa_b200 has no CPU or PyTorch fallback." % path)
    try:
        lib = C.CDLL(path)
    except OSError as e:  # pragma: no cover - environment specific
        raise LsfaLibraryError("cannot load %s: %s" % (path, e)) from e
    for name, (res, args) in PROTOTYPES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:
            raise LsfaLibraryError("%s does not export %s" % (path, name)) from e
        fn.restype = res
        fn.argtypes = args
    ver = lib.lsfa_version()
    if ver != ABI_VERSION:
        raise LsfaLibraryError("ABI mismatch: library %d, python binding %d" % (ver, ABI_VERSION))
    if C.sizeof(LsfaAggArgs) <= 0:  # pragma: no cover
        raise LsfaLibraryError("bad LsfaAggArgs layout")
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != OK:
        msg = load().lsfa_last_error()
        raise LsfaError(rc, msg.decode("utf-8", "replace") if msg else "")


def new_args(**kw) -> LsfaAggArgs:
    a = LsfaAggArgs()
    a.struct_bytes = C.sizeof(LsfaAggArgs)
    for k, v in kw.items():
        setattr(a, k, v)
    return a
