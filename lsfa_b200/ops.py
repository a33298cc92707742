"""Host-side mirror of the reference's operator surface for the non-key-frame path.

Names, argument meaning and error behaviour follow the reference symbols so the parity
tests read like the reference graph (SYM = dff_rfcn/symbols/resnet_v1_101_flownet_rfcn.py):

    GridGenerator(data, transform_type='warp')      mx.sym.GridGenerator   SYM:571
    BilinearSampler(data, grid)                     mx.sym.BilinearSampler SYM:572
    transform_mv_res / mv_pool / res_pool           lib/utils/image.py:202-228
    Nq_aggregate / Fgfa_aggregate                   SYM:94-109 / 132-148 (tails)
    ChooseFeat, tile_as                             operator_py/choose_feat.py, tile_as.py
    warp_scale_aggregate(...)                       the fused operator (SURVEY.md 8a)

PyTorch is used only for device memory and streams: every function takes CUDA tensors,
enqueues hand-written sm_100a kernels through the C ABI (``include/lsfa_ops.h``) on the
current torch stream and returns without synchronising.  There is no CPU path and no
PyTorch-op fallback; a missing library raises ``LsfaLibraryError``.
"""
from __future__ import annotations

import math
from typing import Optional, Sequence

import torch

from . import _cabi as A

__all__ = [
    "GridGenerator", "BilinearSampler", "BilinearSampler_backward", "GridGenerator_backward", "warp_backward",
    "mv_prepare", "mv_pool", "res_pool", "transform_mv_res",
    "sampler_coords", "warp_scale_aggregate", "cur_frame_path", "Nq_aggregate", "Fgfa_aggregate",
    "mean_aggregate", "blend_logits", "ChooseFeat", "tile_as", "cosine_logits", "cosine_logits_backward", "unfused_chain", "mv_accumulate", "coviar_residual", "to_nhwc",
    "to_nchw", "num_launches",
]

_POOL = {"centre2x2": A.POOL_CENTRE2X2, "center2x2": A.POOL_CENTRE2X2, "avg16": A.POOL_AVG16,
         A.POOL_CENTRE2X2: A.POOL_CENTRE2X2, A.POOL_AVG16: A.POOL_AVG16}
_REQ = {"null": A.REQ_NULL, "write": A.REQ_WRITE, "inplace": A.REQ_INPLACE, "add": A.REQ_ADD,
        A.REQ_NULL: A.REQ_NULL, A.REQ_WRITE: A.REQ_WRITE, A.REQ_INPLACE: A.REQ_INPLACE,
        A.REQ_ADD: A.REQ_ADD}
_WMODE = {"none": A.W_NONE, "add": A.W_ADD, "mean": A.W_MEAN, "logits": A.W_LOGITS,
          "cosine": A.W_COSINE}
_LAYOUT = {"nchw": A.LAYOUT_NCHW_F32, "nchw_f32": A.LAYOUT_NCHW_F32, "nhwc_f32": A.LAYOUT_NHWC_F32,
           "nhwc_bf16": A.LAYOUT_NHWC_BF16}


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _dev(t: torch.Tensor, name: str, dtype=None) -> torch.Tensor:
    if not isinstance(t, torch.Tensor):
        raise TypeError("%s must be a torch.Tensor, got %r" % (name, type(t)))
    if not t.is_cuda:
        raise ValueError("%s must live on a CUDA device (lsfa_b200 has no CPU path)" % name)
    if t.device.index != torch.cuda.current_device():
        # the C library launches on the calling thread's CURRENT device and this wrapper enqueues on that device's
        # current stream: a tensor of another device would be read through the wrong context (illegal address / silent
        # peer access).  One host thread per GPU sets its device once (tester.py:301-309).
        raise ValueError("%s lives on cuda:%d but the current device is cuda:%d: call torch.cuda.set_device(...) (or use "
                         "`with torch.cuda.device(...)`) in the thread that drives this GPU"
                         % (name, t.device.index, torch.cuda.current_device()))
    if dtype is not None and t.dtype != dtype:
        raise TypeError("%s must be %s, got %s" % (name, dtype, t.dtype))
    if not t.is_contiguous():
        raise ValueError("%s must be contiguous" % name)
    return t


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _feat_dtype(layout: int):
    return torch.bfloat16 if layout == A.LAYOUT_NHWC_BF16 else torch.float32


def _ceil16(v: int) -> int:
    return (v + 15) // 16


# ------------------------------------------------------------------------------------------
# a7 / a8: the two MXNet operators
# ------------------------------------------------------------------------------------------
def GridGenerator(data: torch.Tensor, transform_type: str = "warp", out=None) -> torch.Tensor:
    """mx.sym.GridGenerator(data=flow, transform_type='warp') - (N,2,H,W) f32 -> (N,2,H,W)."""
    if transform_type != "warp":
        raise NotImplementedError("only transform_type='warp' is on the LSFA path (SYM:306,320,468,571,678)")
    _dev(data, "data", torch.float32)
    if data.dim() != 4 or data.shape[1] != 2:
        raise ValueError("GridGenerator(warp): data must be (N,2,H,W), got %s" % (tuple(data.shape),))
    grid = torch.empty_like(data) if out is None else _dev(out, "out", torch.float32)
    N, _, H, W = data.shape
    A.check(A.load().lsfa_grid_generator_warp_f32(data.data_ptr(), grid.data_ptr(), N, H, W, _stream()))
    return grid


def BilinearSampler(data: torch.Tensor, grid: torch.Tensor, out=None, req="write") -> torch.Tensor:
    """mx.sym.BilinearSampler(data, grid): data (N,C,Hi,Wi), grid (N,2,Ho,Wo) in [-1,1]."""
    _dev(data, "data", torch.float32)
    _dev(grid, "grid", torch.float32)
    if data.dim() != 4 or grid.dim() != 4 or grid.shape[1] != 2 or grid.shape[0] != data.shape[0]:
        raise ValueError("BilinearSampler: data (N,C,Hi,Wi) and grid (N,2,Ho,Wo) expected, got %s %s"
                         % (tuple(data.shape), tuple(grid.shape)))
    N, Cc, Hi, Wi = data.shape
    Ho, Wo = grid.shape[2], grid.shape[3]
    if out is None:
        if _REQ[req] == A.REQ_ADD:
            raise ValueError("req='add' needs an existing out tensor")
        out = torch.empty((N, Cc, Ho, Wo), dtype=torch.float32, device=data.device)
    _dev(out, "out", torch.float32)
    if tuple(out.shape) != (N, Cc, Ho, Wo):
        raise ValueError("out has shape %s, expected %s" % (tuple(out.shape), (N, Cc, Ho, Wo)))
    A.check(A.load().lsfa_bilinear_sampler_f32(data.data_ptr(), grid.data_ptr(), out.data_ptr(), N, Cc,
                                               Hi, Wi, Ho, Wo, _REQ[req], _stream()))
    return out


_KERNEL = {"auto": 0, "scatter": 1, "gather": 2, 0: 0, 1: 1, 2: 2}


def _sampler_backward(fn_name, data, coords, out_grad, grad_data, grad_coords, req_data, req_coords, workspace, kernel):
    _dev(data, "data", torch.float32)
    _dev(coords, "grid/flow", torch.float32)
    _dev(out_grad, "out_grad", torch.float32)
    if data.dim() != 4 or coords.dim() != 4 or coords.shape[1] != 2 or coords.shape[0] != data.shape[0]:
        raise ValueError("backward: data (N,C,Hi,Wi) and grid/flow (N,2,Ho,Wo) expected, got %s %s"
                         % (tuple(data.shape), tuple(coords.shape)))
    N, Cc, Hi, Wi = data.shape
    Ho, Wo = coords.shape[2], coords.shape[3]
    if tuple(out_grad.shape) != (N, Cc, Ho, Wo):
        raise ValueError("out_grad has shape %s, expected %s" % (tuple(out_grad.shape), (N, Cc, Ho, Wo)))
    rd, rc = _REQ[req_data], _REQ[req_coords]
    if rd != A.REQ_NULL:
        if grad_data is None:
            if rd == A.REQ_ADD:
                raise ValueError("req_data='add' needs an existing grad_data")
            grad_data = torch.empty_like(data)
        _dev(grad_data, "grad_data", torch.float32)
        if grad_data.shape != data.shape:
            raise ValueError("grad_data must have data's shape")
    if rc != A.REQ_NULL:
        if grad_coords is None:
            if rc == A.REQ_ADD:
                raise ValueError("req_grid='add' needs an existing grad_grid")
            grad_coords = torch.empty_like(coords)
        _dev(grad_coords, "grad_grid", torch.float32)
        if grad_coords.shape != coords.shape:
            raise ValueError("grad_grid must have the grid's shape")
    lib = A.load()
    k = _KERNEL[kernel]
    if workspace is None and k != 1:
        need = lib.lsfa_bilinear_sampler_backward_workspace_bytes(N, Cc, Hi, Wi, Ho, Wo)
        workspace = torch.empty(need, dtype=torch.uint8, device=data.device)
    ws_ptr, ws_bytes = (None, 0) if workspace is None or workspace is False else (
        workspace.data_ptr(), workspace.numel() * workspace.element_size())
    gd = _ptr(grad_data) if rd != A.REQ_NULL else None
    gc = _ptr(grad_coords) if rc != A.REQ_NULL else None
    if fn_name == "sampler":
        A.check(lib.lsfa_bilinear_sampler_backward_f32(data.data_ptr(), coords.data_ptr(), out_grad.data_ptr(), gd, gc,
                                                       N, Cc, Hi, Wi, Ho, Wo, rd, rc, ws_ptr, ws_bytes, k, _stream()))
    else:
        if (Hi, Wi) != (Ho, Wo):
            raise ValueError("warp_backward: key and flow must share H,W")
        A.check(lib.lsfa_warp_backward_f32(data.data_ptr(), coords.data_ptr(), out_grad.data_ptr(), gd, gc, N, Cc, Ho, Wo,
                                           rd, rc, ws_ptr, ws_bytes, k, _stream()))
    return (grad_data if rd != A.REQ_NULL else None), (grad_coords if rc != A.REQ_NULL else None)


def BilinearSampler_backward(data, grid, out_grad, grad_data=None, grad_grid=None, req_data="write", req_grid="write",
                             workspace=None, kernel="auto"):
    """Backward of mx.sym.BilinearSampler (MXNet BilinearSamplerBackward): returns (grad_data, grad_grid);
    a 'null' req skips that gradient (SYM:320-321 needs grad_data only: the motion vector is data)."""
    return _sampler_backward("sampler", data, grid, out_grad, grad_data, grad_grid, req_data, req_grid, workspace, kernel)


def GridGenerator_backward(grad_grid, grad_flow=None, req="write"):
    """Backward of mx.sym.GridGenerator(transform_type='warp'): grad_flow = grad_grid / [(W-1)/2, (H-1)/2]."""
    _dev(grad_grid, "grad_grid", torch.float32)
    if grad_grid.dim() != 4 or grad_grid.shape[1] != 2:
        raise ValueError("grad_grid must be (N,2,H,W)")
    rq = _REQ[req]
    if grad_flow is None:
        if rq == A.REQ_ADD:
            raise ValueError("req='add' needs an existing grad_flow")
        grad_flow = torch.empty_like(grad_grid)
    _dev(grad_flow, "grad_flow", torch.float32)
    N, _, H, W = grad_grid.shape
    A.check(A.load().lsfa_grid_generator_warp_backward_f32(grad_grid.data_ptr(), grad_flow.data_ptr(), N, H, W, rq, _stream()))
    return grad_flow


def warp_backward(key, flow, out_grad, grad_key=None, grad_flow=None, req_key="write", req_flow="write",
                  workspace=None, kernel="auto"):
    """Backward of BilinearSampler(key, GridGenerator(flow,'warp')) in one pass (SYM:306-307, 320-321):
    returns (grad_key, grad_flow)."""
    return _sampler_backward("warp", key, flow, out_grad, grad_key, grad_flow, req_key, req_flow, workspace, kernel)


def sampler_coords(flow_or_grid: torch.Tensor, key_hw=None, is_grid=False):
    """Index math of a7+a8 alone: returns x0,y0 (int32) and wx,wy (f32), each (N,H,W)."""
    _dev(flow_or_grid, "flow_or_grid", torch.float32)
    N, two, H, W = flow_or_grid.shape
    Hi, Wi = key_hw if key_hw is not None else (H, W)
    dev = flow_or_grid.device
    x0 = torch.empty((N, H, W), dtype=torch.int32, device=dev)
    y0 = torch.empty_like(x0)
    wx = torch.empty((N, H, W), dtype=torch.float32, device=dev)
    wy = torch.empty_like(wx)
    A.check(A.load().lsfa_sampler_coords_f32(flow_or_grid.data_ptr(), int(bool(is_grid)), x0.data_ptr(),
                                             y0.data_ptr(), wx.data_ptr(), wy.data_ptr(), N, H, W, Hi,
                                             Wi, _stream()))
    return x0, y0, wx, wy


# ------------------------------------------------------------------------------------------
# a1-a6: MV / residual preparation (lib/utils/image.py)
# ------------------------------------------------------------------------------------------
def cv_round(v: float) -> int:
    """cvRound (round-half-to-even), used by cv2.resize for dsize."""
    return int(round(v))  # Python's round() is banker's rounding


def mv_prepare(mv_coviar: torch.Tensor, im_scale: float = 1.0, negate: bool = True,
               flipped: bool = False) -> torch.Tensor:
    """image.py:53-60 + :204: (N,h,w,2) int32 from coviar -> sign (+flip) -> cv2-style bilinear
    resize by im_scale -> (N,h',w',2) float32."""
    _dev(mv_coviar, "mv_coviar", torch.int32)
    if mv_coviar.dim() != 4 or mv_coviar.shape[3] != 2:
        raise ValueError("mv_coviar must be (N,h,w,2)")
    N, h, w, _ = mv_coviar.shape
    oh, ow = (h, w) if im_scale == 1.0 else (cv_round(h * im_scale), cv_round(w * im_scale))
    out = torch.empty((N, oh, ow, 2), dtype=torch.float32, device=mv_coviar.device)
    A.check(A.load().lsfa_mv_prepare_i32(mv_coviar.data_ptr(), out.data_ptr(), N, h, w, oh, ow,
                                         float(im_scale), int(negate), int(flipped), _stream()))
    return out


def mv_pool(mv: torch.Tensor, im_scale: float = 1.0, mode="centre2x2", out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """image.py:207-215,220-228 for the MV: (N,h,w,2) int32|f32 -> flow (N,2,ceil(h/16),ceil(w/16)) (``out``: a
    caller-owned destination, e.g. inside a recorded graph)."""
    _dev(mv, "mv")
    if mv.dim() != 4 or mv.shape[3] != 2:
        raise ValueError("mv must be (N,h,w,2), got %s" % (tuple(mv.shape),))
    N, h, w, _ = mv.shape
    shape = (N, 2, _ceil16(h), _ceil16(w))
    if out is None:
        flow = torch.empty(shape, dtype=torch.float32, device=mv.device)
    else:
        _dev(out, "out", torch.float32)
        if tuple(out.shape) != shape or not out.is_contiguous():
            raise ValueError("out must be a contiguous %s float32 tensor, got %s" % (shape, tuple(out.shape)))
        flow = out
    lib = A.load()
    if mv.dtype == torch.int32:
        fn = lib.lsfa_mv_pool_i32
    elif mv.dtype == torch.float32:
        fn = lib.lsfa_mv_pool_f32
    else:
        raise TypeError("mv must be int32 or float32, got %s" % mv.dtype)
    A.check(fn(mv.data_ptr(), flow.data_ptr(), N, h, w, float(im_scale), _POOL[mode], _stream()))
    return flow


def res_pool(res: torch.Tensor, pixel_means: Sequence[float] = (0.0, 0.0, 0.0),
             pixel_scale: float = 1.0, mode="centre2x2") -> torch.Tensor:
    """image.py:207-222 for the residual (incl. the aliasing of :217-218): (N,h,w,3) -> (N,3,H,W)."""
    import ctypes
    _dev(res, "res")
    if res.dim() != 4 or res.shape[3] != 3:
        raise ValueError("res must be (N,h,w,3), got %s" % (tuple(res.shape),))
    N, h, w, _ = res.shape
    out = torch.empty((N, 3, _ceil16(h), _ceil16(w)), dtype=torch.float32, device=res.device)
    means = (ctypes.c_double * 3)(*[float(m) for m in pixel_means])
    lib = A.load()
    if res.dtype == torch.int32:
        fn = lib.lsfa_res_pool_i32
    elif res.dtype == torch.float32:
        fn = lib.lsfa_res_pool_f32
    else:
        raise TypeError("res must be int32 or float32, got %s" % res.dtype)
    A.check(fn(res.data_ptr(), out.data_ptr(), N, h, w, ctypes.cast(means, ctypes.c_void_p),
               float(pixel_scale), _POOL[mode], _stream()))
    return out


def res_coviar_pool(res_coviar: torch.Tensor, im_scale: float = 1.0, flipped: bool = False,
                    pixel_means: Sequence[float] = (0.0, 0.0, 0.0), pixel_scale: float = 1.0,
                    mode="centre2x2") -> torch.Tensor:
    """The residual half of get_image + transform_mv_res (image.py:52,59,205,207-222) in one launch:
    (N,h,w,3) int32 exactly as ``coviar_py2.load(..., 2, True)`` returns it -> (N,3,H,W) float32."""
    import ctypes
    _dev(res_coviar, "res_coviar", torch.int32)
    if res_coviar.dim() != 4 or res_coviar.shape[3] != 3:
        raise ValueError("res_coviar must be (N,h,w,3), got %s" % (tuple(res_coviar.shape),))
    N, h, w, _ = res_coviar.shape
    oh, ow = (h, w) if im_scale == 1.0 else (cv_round(h * im_scale), cv_round(w * im_scale))
    out = torch.empty((N, 3, _ceil16(oh), _ceil16(ow)), dtype=torch.float32, device=res_coviar.device)
    means = (ctypes.c_double * 3)(*[float(m) for m in pixel_means])
    A.check(A.load().lsfa_res_coviar_pool_i32(res_coviar.data_ptr(), out.data_ptr(), N, h, w, oh, ow, float(im_scale),
                                              int(flipped), ctypes.cast(means, ctypes.c_void_p), float(pixel_scale),
                                              _POOL[mode], _stream()))
    return out


def transform_mv_res(motion_vector: torch.Tensor, res_diff: torch.Tensor, im_scale: float,
                     pixel_means=(0.0, 0.0, 0.0), pixel_scale: float = 1.0):
    """Device version of lib/utils/image.py:202-228 for inputs already at network scale
    (``im_scale`` only rescales the MV values, stage 1 done by ``mv_prepare``):
    (N,h,w,2),(N,h,w,3) -> (N,2,H,W),(N,3,H,W) float32."""
    return mv_pool(motion_vector, im_scale), res_pool(res_diff, pixel_means, pixel_scale)


# ------------------------------------------------------------------------------------------
# the fused operator
# ------------------------------------------------------------------------------------------
def _feature_dims(t: torch.Tensor, layout: int):
    if t.dim() != 4:
        raise ValueError("feature tensors must be 4-D, got %s" % (tuple(t.shape),))
    if layout == A.LAYOUT_NCHW_F32:
        n, c, h, w = t.shape
    else:
        n, h, w, c = t.shape
    return n, c, h, w


def _build_args(key, flow, *, cur=None, scale_map=None, res=None, rnet_w=None, rnet_b=None,
                weight_mode="none", logits=None, emb_warp=None, emb_cur=None, bypass=None,
                key_index=None, flow_kind="flow", im_scale=1.0, pool_mode="centre2x2", negate=True, flipped=False,
                layout="nchw", out=None, req="write", workspace=None, force_generic=False):
    lay = _LAYOUT[layout] if isinstance(layout, str) else layout
    fdt = _feat_dtype(lay)
    _dev(key, "key", fdt)
    nk, Cc, Hk, Wk = _feature_dims(key, lay)
    keep = [key]

    if flow_kind in ("flow", "grid"):
        _dev(flow, "flow", torch.float32)
        if flow.dim() != 4 or flow.shape[1] != 2:
            raise ValueError("flow/grid must be (N,2,H,W), got %s" % (tuple(flow.shape),))
        N, _, H, W = flow.shape
        fk = A.FLOW_PREPOOLED if flow_kind == "flow" else A.FLOW_GRID
        mv_h = mv_w = 0
    elif flow_kind == "raw":
        _dev(flow, "flow (raw mv)")
        if flow.dim() != 4 or flow.shape[3] != 2:
            raise ValueError("raw mv must be (N,h,w,2), got %s" % (tuple(flow.shape),))
        N, mv_h, mv_w, _ = flow.shape
        H, W = _ceil16(mv_h), _ceil16(mv_w)
        if flow.dtype == torch.int32:
            fk = A.FLOW_RAW_I32
        elif flow.dtype == torch.float32:
            fk = A.FLOW_RAW_F32
        else:
            raise TypeError("raw mv must be int32 or float32")
    elif flow_kind == "coviar":
        # the MV exactly as coviar_py2.load(..., 1, True) returns it (image.py:53): sign, flip and the
        # im_scale resize of image.py:54-60,204 happen in the kernel
        _dev(flow, "flow (coviar mv)", torch.int32)
        if flow.dim() != 4 or flow.shape[3] != 2:
            raise ValueError("coviar mv must be (N,h,w,2) int32, got %s" % (tuple(flow.shape),))
        N, src_h, src_w, _ = flow.shape
        mv_h, mv_w = (src_h, src_w) if im_scale == 1.0 else (cv_round(src_h * im_scale), cv_round(src_w * im_scale))
        H, W = _ceil16(mv_h), _ceil16(mv_w)
        fk = A.FLOW_COVIAR_I32
    else:
        raise ValueError("flow_kind must be 'flow', 'grid', 'raw' or 'coviar'")
    keep.append(flow)

    if key_index is not None:
        _dev(key_index, "key_index", torch.int32)
        if key_index.numel() != N:
            raise ValueError("key_index must have N=%d entries" % N)
        keep.append(key_index)
    elif nk != N:
        raise ValueError("key has %d frames but flow has %d (pass key_index to share key features)" % (nk, N))

    out_shape = (N, Cc, H, W) if lay == A.LAYOUT_NCHW_F32 else (N, H, W, Cc)
    wm = _WMODE[weight_mode] if isinstance(weight_mode, str) else weight_mode
    rq = _REQ[req]
    if out is None:
        if rq == A.REQ_ADD:
            raise ValueError("req='add' needs an existing out tensor")
        out = torch.empty(out_shape, dtype=fdt, device=key.device)
    _dev(out, "out", fdt)
    if tuple(out.shape) != out_shape:
        raise ValueError("out has shape %s, expected %s" % (tuple(out.shape), out_shape))

    def same(t, name):
        if t is None:
            return None
        _dev(t, name, fdt)
        if tuple(t.shape) != out_shape:
            raise ValueError("%s has shape %s, expected %s" % (name, tuple(t.shape), out_shape))
        keep.append(t)
        return t

    same(scale_map, "scale_map")
    same(cur, "cur")
    if res is not None:
        _dev(res, "res", torch.float32)
        if tuple(res.shape) != (N, 3, H, W):
            raise ValueError("res must be (N,3,H,W)=%s, got %s" % ((N, 3, H, W), tuple(res.shape)))
        if rnet_w is None or rnet_b is None:
            raise ValueError("res needs rnet_w (C,3[,1,1]) and rnet_b (C,)")
        _dev(rnet_w, "rnet_w", torch.float32)
        _dev(rnet_b, "rnet_b", torch.float32)
        if rnet_w.numel() != Cc * 3 or rnet_b.numel() != Cc:
            raise ValueError("rnet_w must have C*3 and rnet_b C elements")
        keep += [res, rnet_w, rnet_b]
    if logits is not None:
        _dev(logits, "logits", torch.float32)
        if tuple(logits.shape) != (N, 2, H, W):
            raise ValueError("logits must be (N,2,H,W)=%s, got %s" % ((N, 2, H, W), tuple(logits.shape)))
        keep.append(logits)
    E = 0
    if emb_warp is not None or emb_cur is not None:
        if emb_warp is None or emb_cur is None:
            raise ValueError("emb_warp and emb_cur go together")
        _dev(emb_warp, "emb_warp", fdt)
        _dev(emb_cur, "emb_cur", fdt)
        if emb_warp.shape != emb_cur.shape:
            raise ValueError("emb_warp / emb_cur shapes differ")
        en, E, eh, ew = _feature_dims(emb_warp, lay)
        if (en, eh, ew) != (N, H, W):
            raise ValueError("embeddings must cover (N,H,W)=%s" % ((N, H, W),))
        keep += [emb_warp, emb_cur]
    if bypass is not None:
        _dev(bypass, "bypass", torch.uint8)
        if bypass.numel() != N:
            raise ValueError("bypass must have N entries")
        keep.append(bypass)

    args = A.new_args(
        layout=lay, N=N, C=Cc, H=H, W=W, key_h=Hk, key_w=Wk, num_keys=nk,
        key=_ptr(key), key_index=_ptr(key_index), flow_kind=fk, flow=_ptr(flow), mv_h=mv_h,
        mv_w=mv_w, im_scale=float(im_scale), pool_mode=_POOL[pool_mode],
        scale_map=_ptr(scale_map), res=_ptr(res), rnet_w=_ptr(rnet_w), rnet_b=_ptr(rnet_b),
        cur=_ptr(cur), weight_mode=wm, logits=_ptr(logits), emb_warp=_ptr(emb_warp),
        emb_cur=_ptr(emb_cur), E=E, bypass=_ptr(bypass), out=_ptr(out), req=rq,
        force_generic=int(force_generic))
    if fk == A.FLOW_COVIAR_I32:
        args.mv_src_h, args.mv_src_w = src_h, src_w
        args.mv_negate, args.mv_hflip = int(bool(negate)), int(bool(flipped))
    lib = A.load()
    need = lib.lsfa_warp_scale_aggregate_workspace_bytes(args)
    if workspace is False and wm != A.W_COSINE:
        need = 0                      # caller opts out of the scheduling scratch: static work split
    if need:
        if workspace is None or workspace is False:
            workspace = torch.empty(need, dtype=torch.uint8, device=key.device)
        _dev(workspace, "workspace")
        if workspace.numel() * workspace.element_size() < need:
            raise ValueError("workspace too small: need %d bytes" % need)
        args.workspace = workspace.data_ptr()
        args.workspace_bytes = workspace.numel() * workspace.element_size()
        keep.append(workspace)
    return args, out, keep


def warp_scale_aggregate(key, flow, **kw) -> torch.Tensor:
    """out = blend(BilinearSampler(key, GridGenerator_warp(flow)) [*scale_map] [+rnet(res)], cur).

    Keyword arguments: cur, scale_map, res, rnet_w, rnet_b, weight_mode ('none'|'add'|'mean'|
    'logits'|'cosine'), logits (N,2,H,W), emb_warp, emb_cur, bypass (N,) uint8, key_index (N,)
    int32, flow_kind ('flow'|'grid'|'raw'|'coviar'), im_scale, pool_mode, negate, flipped, layout ('nchw'|'nhwc_f32'|
    'nhwc_bf16'), out, req, workspace, force_generic (kernel choice - NCHW: 0 auto, 1 generic gather, 2 plane-resident
    LDG/STG, 3 all-TMA, 4 2-CTA cluster form; channels-last: 0 auto, 1 LDG/STG tile kernel, 3 all-TMA gather by bulk copy,
    5 window-resident all-TMA on tensor maps).
    ``workspace``: None = allocated here when the chosen path can use one, False = none (static work split).
    """
    args, out, _keep = _build_args(key, flow, **kw)
    A.check(A.load().lsfa_warp_scale_aggregate(args, _stream()))
    return out


class PreparedAggregate:
    """Arguments validated once, launched many times (the batch harness / bench loop):
    what a bound MXNet executor is to a symbol.  ``run()`` is one C-ABI call."""

    def __init__(self, key, flow, **kw):
        self.args, self.out, self._keep = _build_args(key, flow, **kw)
        self._lib = A.load()
        self.launches = self._lib.lsfa_warp_scale_aggregate_num_launches(self.args)

    def run(self, stream: Optional[int] = None) -> torch.Tensor:
        A.check(self._lib.lsfa_warp_scale_aggregate(self.args, _stream() if stream is None else stream))
        return self.out


class RecordedGraph:
    """A sequence of this package's calls recorded into ONE CUDA graph through the C ABI (``lsfa_graph_begin`` /
    ``lsfa_graph_end`` / ``lsfa_graph_launch``): the reference issues the operators of a frame one by one
    (core/tester.py:138-145); replaying them costs one launch.

        g = RecordedGraph(stream)
        with g:                       # every ops.* / PreparedAggregate.run(stream) call on `stream` is recorded
            p.run(stream)
        g.launch()                    # same buffers, new contents

    The recorded calls' tensors must stay alive and in place for the lifetime of the graph."""

    def __init__(self, stream: int):
        if not stream:
            raise ValueError("recording needs an explicit, non-default stream handle")
        self._lib = A.load()
        self.stream = stream
        self._h = None

    def __enter__(self):
        A.check(self._lib.lsfa_graph_begin(self.stream))
        return self

    def __exit__(self, et, ev, tb):
        import ctypes
        h = ctypes.c_void_p()
        rc = self._lib.lsfa_graph_end(self.stream, ctypes.byref(h))
        if et is None:
            A.check(rc)
            self._h = h
        return False

    def launch(self, stream: Optional[int] = None):
        if self._h is None:
            raise RuntimeError("nothing recorded")
        A.check(self._lib.lsfa_graph_launch(self._h, self.stream if stream is None else stream))

    def close(self):
        if self._h is not None:
            self._lib.lsfa_graph_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def warp_scale_aggregate_backward(out_grad, key, flow, *, want=("key", "flow", "scale", "cur", "logits", "res", "rnet", "emb_warp",
                                                              "emb_cur"), **kw):
    """Backward of ``warp_scale_aggregate`` (NCHW float32; SYM:306-338 needs it for training): returns a dict of the
    gradients that exist for these inputs among ``want`` - 'key', 'flow' (prepooled flow or grid only: raw motion vectors
    are data), 'scale', 'cur', 'logits' (logits mode), 'res', 'rnet_w' + 'rnet_b', 'emb_warp' + 'emb_cur' (cosine mode).
    ``kw`` = the forward's keyword arguments."""
    import ctypes
    kw = dict(kw)
    kw.pop("out", None)
    kw.pop("req", None)
    kw["workspace"] = False
    _dev(out_grad, "out_grad", torch.float32)
    args, _out, keep = _build_args(key, flow, **kw)
    if tuple(out_grad.shape) != tuple(_out.shape):
        raise ValueError("out_grad has shape %s, expected %s" % (tuple(out_grad.shape), tuple(_out.shape)))
    g = A.LsfaAggGrads()
    g.struct_bytes = ctypes.sizeof(A.LsfaAggGrads)
    g.out_grad = out_grad.data_ptr()
    res = {}
    fk = kw.get("flow_kind", "flow")
    mode = kw.get("weight_mode", "none")

    def mk(name, like, cond):
        if name in want and cond:
            res[name] = torch.empty_like(like)
            return res[name].data_ptr(), A.REQ_WRITE
        return None, A.REQ_NULL
    g.grad_key, g.req_key = mk("key", key, kw.get("key_index") is None)
    g.grad_flow, g.req_flow = mk("flow", flow, fk in ("flow", "grid"))
    g.grad_scale, g.req_scale = mk("scale", kw.get("scale_map"), kw.get("scale_map") is not None)
    g.grad_cur, g.req_cur = mk("cur", kw.get("cur"), kw.get("cur") is not None and mode != "none")
    g.grad_logits, g.req_logits = mk("logits", kw.get("logits"), mode == "logits")
    g.grad_res, g.req_res = mk("res", kw.get("res"), kw.get("res") is not None)
    g.grad_emb_warp, rw = mk("emb_warp", kw.get("emb_warp"), mode == "cosine")
    g.grad_emb_cur, rc = mk("emb_cur", kw.get("emb_cur"), mode == "cosine")
    g.req_emb = max(rw, rc)
    if "rnet" in want and kw.get("res") is not None:
        res["rnet_w"] = torch.empty_like(kw["rnet_w"])
        res["rnet_b"] = torch.empty_like(kw["rnet_b"])
        g.grad_rnet_w, g.grad_rnet_b, g.req_rnet = res["rnet_w"].data_ptr(), res["rnet_b"].data_ptr(), A.REQ_WRITE
    lib = A.load()
    need = lib.lsfa_warp_scale_aggregate_backward_workspace_bytes(args, g)
    if need == 0:
        A.check(lib.lsfa_warp_scale_aggregate_backward_f32_nchw(args, g, _stream()))     # raises with the library's message
    ws = torch.empty(need + 256, dtype=torch.uint8, device=key.device)
    off = (-ws.data_ptr()) % 256
    g.workspace, g.workspace_bytes = ws.data_ptr() + off, need
    A.check(lib.lsfa_warp_scale_aggregate_backward_f32_nchw(args, g, _stream()))
    del keep
    return res


def num_launches(**kw) -> int:
    args, _, _ = _build_args(**kw)
    return A.load().lsfa_warp_scale_aggregate_num_launches(args)


# ------------------------------------------------------------------------------------------
# reference graph pieces expressed through the fused operator
# ------------------------------------------------------------------------------------------
def cur_frame_path(feat_key, motion_vector, res_diff, rnet_w, rnet_b, small_net_feat, **kw):
    """get_cur_test_symbol as shipped (SYM:570-586, yaml:49-60):
    warp(feat_key, motion_vector) + rnet_conv0(res_diff) + fuse_reduce_add(small net)."""
    return warp_scale_aggregate(feat_key, motion_vector, cur=small_net_feat, res=res_diff,
                                rnet_w=rnet_w, rnet_b=rnet_b, weight_mode="add", **kw)


def Nq_aggregate(feat_key_old, flow, scale_map, conv_feat, nq_logits, is_first_frame=None, **kw):
    """Key-frame long-term aggregation with Nq weights (SYM:468-472,104-108,477)."""
    return warp_scale_aggregate(feat_key_old, flow, cur=conv_feat, scale_map=scale_map,
                                weight_mode="logits", logits=nq_logits, bypass=is_first_frame, **kw)


def Fgfa_aggregate(feat_key_old, flow, scale_map, conv_feat, emb_warp, emb_cur,
                   is_first_frame=None, **kw):
    """Same with cosine-embedding weights (SYM:473-474,132-148)."""
    return warp_scale_aggregate(feat_key_old, flow, cur=conv_feat, scale_map=scale_map,
                                weight_mode="cosine", emb_warp=emb_warp, emb_cur=emb_cur,
                                bypass=is_first_frame, **kw)


def mean_aggregate(feat_key_old, flow, scale_map, conv_feat, **kw):
    """0.5 * (warp*scale + conv_feat) (SYM:315,476)."""
    return warp_scale_aggregate(feat_key_old, flow, cur=conv_feat, scale_map=scale_map,
                                weight_mode="mean", **kw)


def ChooseFeat(conv_feat, conv_feat_prop, eq_flag):
    """operator_py/choose_feat.py:23-31 without the host sync: the flag stays on the device and
    the select is the fused kernel's bypass path (identity warp is NOT used: prop is copied)."""
    _dev(conv_feat, "conv_feat", torch.float32)
    _dev(conv_feat_prop, "conv_feat_prop", torch.float32)
    _dev(eq_flag, "eq_flag", torch.uint8)
    if conv_feat.shape != conv_feat_prop.shape or eq_flag.numel() != conv_feat.shape[0]:
        raise ValueError("ChooseFeat: shapes %s %s flag %s" % (tuple(conv_feat.shape),
                         tuple(conv_feat_prop.shape), tuple(eq_flag.shape)))
    out = torch.empty_like(conv_feat)
    n = conv_feat.shape[0]
    A.check(A.load().lsfa_choose_feat_f32(conv_feat.data_ptr(), conv_feat_prop.data_ptr(),
                                          eq_flag.data_ptr(), out.data_ptr(), n,
                                          conv_feat.numel() // n, _stream()))
    return out


def blend_logits(src0, cur, logits, bypass=None, out=None) -> torch.Tensor:
    """Nq / Fgfa tail on two materialised features (SYM:104-108,141-147): softmax(logits) blend, NCHW f32."""
    _dev(src0, "src0", torch.float32)
    _dev(cur, "cur", torch.float32)
    _dev(logits, "logits", torch.float32)
    N, Cc, H, W = src0.shape
    if cur.shape != src0.shape or tuple(logits.shape) != (N, 2, H, W):
        raise ValueError("blend_logits: src0/cur (N,C,H,W) and logits (N,2,H,W) expected")
    if bypass is not None:
        _dev(bypass, "bypass", torch.uint8)
    out = torch.empty_like(src0) if out is None else _dev(out, "out", torch.float32)
    A.check(A.load().lsfa_blend_logits_f32(src0.data_ptr(), cur.data_ptr(), logits.data_ptr(), _ptr(bypass),
                                           out.data_ptr(), N, Cc, H, W, _stream()))
    return out


def tile_as(n: int, device) -> torch.Tensor:
    """operator_py/tile_as.py:16-19 without materialising the copies: the (n,) key_index that makes
    every frame of the batch sample key feature 0."""
    return torch.zeros(n, dtype=torch.int32, device=device)


def cosine_logits(emb_warp, emb_cur, layout="nchw", workspace=None) -> torch.Tensor:
    """compute_weight x2 of Fgfa_net (SYM:111-116,137-139) -> (N,2,H,W) f32.  NCHW embeddings go through the all-TMA
    pre-pass (scratch allocated here unless given; ``workspace=False`` pins the LDG kernel)."""
    lay = _LAYOUT[layout]
    fdt = _feat_dtype(lay)
    _dev(emb_warp, "emb_warp", fdt)
    _dev(emb_cur, "emb_cur", fdt)
    N, E, H, W = _feature_dims(emb_warp, lay)
    logits = torch.empty((N, 2, H, W), dtype=torch.float32, device=emb_warp.device)
    lib = A.load()
    if workspace is None:
        need = lib.lsfa_cosine_logits_workspace_bytes(N, E, H, W, lay)
        workspace = torch.empty(need, dtype=torch.uint8, device=emb_warp.device) if need else False
    if workspace is False:
        A.check(lib.lsfa_cosine_logits(emb_warp.data_ptr(), emb_cur.data_ptr(), logits.data_ptr(), N, E, H, W, lay, _stream()))
    else:
        A.check(lib.lsfa_cosine_logits_ws(emb_warp.data_ptr(), emb_cur.data_ptr(), logits.data_ptr(), N, E, H, W, lay,
                                          workspace.data_ptr(), workspace.numel() * workspace.element_size(), _stream()))
    return logits


_COS_KERNEL = {"auto": 0, "plain": 1, "tma": 2, 0: 0, 1: 1, 2: 2}


def cosine_logits_backward(emb_warp, emb_cur, grad_logits, grad_emb_warp=None, grad_emb_cur=None, req_warp="write",
                           req_cur="write", workspace=None, kernel="auto"):
    """Backward of ``cosine_logits`` (NCHW float32): from d/d(logits) (N,2,H,W) to (grad_emb_warp, grad_emb_cur), each
    (N,E,H,W) or None where its req is 'null'.  The logits are recomputed as ``cosine_logits`` computes them with its
    default workspace.  ``kernel``: 'auto', 'plain' (LDG/STG) or 'tma' (all-TMA; raises where it cannot serve the
    shape); both give the same bits.  The gradients must not overlap the inputs."""
    _dev(emb_warp, "emb_warp", torch.float32)
    _dev(emb_cur, "emb_cur", torch.float32)
    _dev(grad_logits, "grad_logits", torch.float32)
    if emb_warp.dim() != 4 or emb_cur.shape != emb_warp.shape:
        raise ValueError("emb_warp and emb_cur must be (N,E,H,W) of one shape, got %s %s" % (tuple(emb_warp.shape), tuple(emb_cur.shape)))
    N, E, H, W = emb_warp.shape
    if tuple(grad_logits.shape) != (N, 2, H, W):
        raise ValueError("grad_logits must be (N,2,H,W)=%s, got %s" % ((N, 2, H, W), tuple(grad_logits.shape)))
    grads = []
    for g, rq, nme in ((grad_emb_warp, _REQ[req_warp], "grad_emb_warp"), (grad_emb_cur, _REQ[req_cur], "grad_emb_cur")):
        if rq != A.REQ_NULL:
            if g is None:
                if rq == A.REQ_ADD:
                    raise ValueError("req 'add' needs an existing %s" % nme)
                g = torch.empty_like(emb_warp)
            _dev(g, nme, torch.float32)
            if g.shape != emb_warp.shape:
                raise ValueError("%s must have the embeddings' shape" % nme)
        grads.append(g if rq != A.REQ_NULL else None)
    lib = A.load()
    if workspace is None:
        workspace = torch.empty(lib.lsfa_cosine_logits_backward_workspace_bytes(N, E, H, W), dtype=torch.uint8, device=emb_warp.device)
    _dev(workspace, "workspace")
    A.check(lib.lsfa_cosine_logits_backward_f32_nchw(emb_warp.data_ptr(), emb_cur.data_ptr(), grad_logits.data_ptr(), _ptr(grads[0]),
                                                     _ptr(grads[1]), N, E, H, W, _REQ[req_warp], _REQ[req_cur], workspace.data_ptr(),
                                                     workspace.numel() * workspace.element_size(), _COS_KERNEL[kernel], _stream()))
    return grads[0], grads[1]


def unfused_chain(key, flow, scale_map, cur, logits, tmp=None) -> torch.Tensor:
    """The reference graph operator by operator (ablation baseline, 9 kernels)."""
    for t, nme in ((key, "key"), (flow, "flow"), (scale_map, "scale_map"), (cur, "cur"), (logits, "logits")):
        _dev(t, nme, torch.float32)
    N, Cc, H, W = key.shape
    out = torch.empty_like(key)
    if tmp is None:
        tmp = torch.empty(5 * key.numel(), dtype=torch.float32, device=key.device)
    A.check(A.load().lsfa_unfused_chain_f32_nchw(key.data_ptr(), flow.data_ptr(), scale_map.data_ptr(),
                                                 cur.data_ptr(), logits.data_ptr(), out.data_ptr(),
                                                 tmp.data_ptr(), N, Cc, H, W, _stream()))
    return out


_MVACC_ALGO = {"auto": 0, "field": 1, "trace": 2}


def mv_accumulate(mvs: torch.Tensor, counts: torch.Tensor, height: int, width: int, workspace=None, algo="auto") -> torch.Tensor:
    """coviar's accumulated MV field (coviar_data_loader.c:71-139, accumulate=1) for N GOPs at once.
    mvs (N,T,M,6) int32 {w,h,src_x,src_y,dst_x,dst_y} per P-frame in list order, counts (N,T) int32
    -> (N,height,width,2) int32, the array coviar_py2.load(video, gop, pos=T, 1, True) returns."""
    _dev(mvs, "mvs", torch.int32)
    _dev(counts, "counts", torch.int32)
    if mvs.dim() != 4 or mvs.shape[3] != 6 or tuple(counts.shape) != tuple(mvs.shape[:2]):
        raise ValueError("mvs must be (N,T,M,6) and counts (N,T)")
    N, T, M, _ = mvs.shape
    lib = A.load()
    need = lib.lsfa_mv_accumulate_workspace_bytes(N, height, width)
    if workspace is None:
        workspace = torch.empty(need, dtype=torch.uint8, device=mvs.device)
    out = torch.empty((N, height, width, 2), dtype=torch.int32, device=mvs.device)
    A.check(lib.lsfa_mv_accumulate_algo_i32(mvs.data_ptr(), counts.data_ptr(), N, T, M, height, width, out.data_ptr(),
                                            workspace.data_ptr(), workspace.numel() * workspace.element_size(),
                                            _MVACC_ALGO[algo], _stream()))
    return out


def coviar_residual(iframe: torch.Tensor, cur: torch.Tensor, mv: torch.Tensor) -> torch.Tensor:
    """coviar_data_loader.c:141-175: res = cur - iframe[(x,y) - mv]; frames (N,h,w,3) uint8, mv (N,h,w,2) int32."""
    _dev(iframe, "iframe", torch.uint8)
    _dev(cur, "cur", torch.uint8)
    _dev(mv, "mv", torch.int32)
    N, h, w, _ = cur.shape
    res = torch.empty((N, h, w, 3), dtype=torch.int32, device=cur.device)
    A.check(A.load().lsfa_coviar_residual_u8(iframe.data_ptr(), cur.data_ptr(), mv.data_ptr(), res.data_ptr(), N, h, w,
                                             _stream()))
    return res


def to_nhwc(x: torch.Tensor, dtype=torch.float32, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """(N,C,H,W) f32 -> (N,H,W,C) f32|bf16 with our transpose kernel (``out``: a contiguous (N,H,W,C) destination,
    e.g. a slice along N of a larger buffer)."""
    _dev(x, "x", torch.float32)
    N, Cc, H, W = x.shape
    lay = A.LAYOUT_NHWC_BF16 if dtype == torch.bfloat16 else A.LAYOUT_NHWC_F32
    if out is None:
        out = torch.empty((N, H, W, Cc), dtype=dtype, device=x.device)
    else:
        _dev(out, "out", dtype)
        if tuple(out.shape) != (N, H, W, Cc):
            raise ValueError("out must be (N,H,W,C)=%s, got %s" % ((N, H, W, Cc), tuple(out.shape)))
    A.check(A.load().lsfa_nchw_to_nhwc(x.data_ptr(), out.data_ptr(), N, Cc, H, W, lay, _stream()))
    return out


def to_nchw(x: torch.Tensor) -> torch.Tensor:
    """(N,H,W,C) f32|bf16 -> (N,C,H,W) f32."""
    _dev(x, "x")
    N, H, W, Cc = x.shape
    lay = A.LAYOUT_NHWC_BF16 if x.dtype == torch.bfloat16 else A.LAYOUT_NHWC_F32
    out = torch.empty((N, Cc, H, W), dtype=torch.float32, device=x.device)
    A.check(A.load().lsfa_nhwc_to_nchw(x.data_ptr(), out.data_ptr(), N, Cc, H, W, lay, _stream()))
    return out


# ------------------------------------------------------------------------------------------
# SURVEY 8f rank 2: the embedding / quality networks on tensor cores (csrc/conv_gemm_tc.cu)
# ------------------------------------------------------------------------------------------
def pack_conv_weight(w: torch.Tensor) -> torch.Tensor:
    """MXNet's (Cout,Cin,k,k) float32 convolution weight -> (Cout, k*k*Cin) bf16 (K index = tap*Cin + cin), once per
    parameter set."""
    _dev(w, "w", torch.float32)
    if w.dim() != 4 or w.shape[2] != w.shape[3] or w.shape[2] not in (1, 3):
        raise ValueError("conv weight must be (Cout,Cin,k,k) with k in {1,3}, got %s" % (tuple(w.shape),))
    Cout, Cin, k, _ = w.shape
    out = torch.empty((Cout, k * k * Cin), dtype=torch.bfloat16, device=w.device)
    A.check(A.load().lsfa_pack_conv_weight_bf16(w.data_ptr(), out.data_ptr(), Cout, Cin, k, _stream()))
    return out


def _ksize(w_packed: torch.Tensor, Cin: int) -> int:
    taps, rem = divmod(w_packed.shape[1], Cin)
    if rem or taps not in (1, 9):
        raise ValueError("packed weight (Cout, %d) does not match Cin=%d for a 1x1 or 3x3 kernel" % (w_packed.shape[1], Cin))
    return 1 if taps == 1 else 3


def conv_bf16_nhwc(x: torch.Tensor, w_packed: torch.Tensor, bias: torch.Tensor, relu: bool = False, out=None) -> torch.Tensor:
    """mx.sym.Convolution (stride 1, 'same' padding, with bias) [+ ReLU] on tensor cores: x (NB,H,W,Cin) bf16 channels-last,
    w_packed from pack_conv_weight, bias (Cout,) f32 -> (NB,H,W,Cout) bf16.  Cin % 64 == 0, Cout % 256 == 0."""
    _dev(x, "x", torch.bfloat16)
    _dev(w_packed, "w_packed", torch.bfloat16)
    _dev(bias, "bias", torch.float32)
    NB, H, W, Cin = x.shape
    Cout = w_packed.shape[0]
    k = _ksize(w_packed, Cin)
    if out is None:
        out = torch.empty((NB, H, W, Cout), dtype=torch.bfloat16, device=x.device)
    _dev(out, "out", torch.bfloat16)
    A.check(A.load().lsfa_conv_bf16_nhwc(x.data_ptr(), w_packed.data_ptr(), bias.data_ptr(), out.data_ptr(), NB, H, W, Cin, Cout,
                                         k, int(bool(relu)), _stream()))
    return out


def embed_cosine_logits(x: torch.Tensor, packed_params, workspace=None) -> torch.Tensor:
    """get_embednet + compute_weight of Fgfa_net (SYM:111-139) in three tensor-core launches + a tiny finalise:
    x = Concat_0(conv_feat, warp_feat) (2N,H,W,C) bf16 channels-last; packed_params = (w1p, b1, w2p, b2, w3p, b3) with the
    weights from pack_conv_weight -> logits (N,2,H,W) f32 ([n,0] warp vs cur, [n,1] cur vs cur).  The 2048-channel
    embeddings are reduced in em_conv3's epilogue and never written."""
    _dev(x, "x", torch.bfloat16)
    w1, b1, w2, b2, w3, b3 = packed_params
    for t, nme in ((w1, "w1"), (w2, "w2"), (w3, "w3")):
        _dev(t, nme, torch.bfloat16)
    for t, nme in ((b1, "b1"), (b2, "b2"), (b3, "b3")):
        _dev(t, nme, torch.float32)
    NB, H, W, Cc = x.shape
    if NB % 2:
        raise ValueError("x must hold Concat_0(conv_feat, warp_feat): an even number of images")
    N = NB // 2
    C1, C2, E = w1.shape[0], w2.shape[0], w3.shape[0]
    if w1.shape[1] != Cc or w2.shape[1] != 9 * C1 or w3.shape[1] != C2:
        raise ValueError("embedding weights do not chain: %s %s %s for C=%d" % (tuple(w1.shape), tuple(w2.shape), tuple(w3.shape), Cc))
    lib = A.load()
    need = lib.lsfa_embed_cosine_logits_workspace_bytes(N, H, W, C1, C2, E)
    if workspace is None:
        workspace = torch.empty(need + 256, dtype=torch.uint8, device=x.device)
    off = (-workspace.data_ptr()) % 256
    logits = torch.empty((N, 2, H, W), dtype=torch.float32, device=x.device)
    A.check(lib.lsfa_embed_cosine_logits_bf16_nhwc(x.data_ptr(), w1.data_ptr(), b1.data_ptr(), w2.data_ptr(), b2.data_ptr(),
                                                   w3.data_ptr(), b3.data_ptr(), logits.data_ptr(), N, H, W, Cc, C1, C2, E,
                                                   workspace.data_ptr() + off, workspace.numel() - off, _stream()))
    return logits


def nq_logits(x: torch.Tensor, packed_params) -> torch.Tensor:
    """The convolutions of Nq_net (SYM:95-101) in one tensor-core launch: x = Concat_0(warp_feat, conv_feat) (2N,H,W,C) bf16
    channels-last; packed_params = (w1p, b1, w2, b2, w3, b3): w1p = pack_conv_weight(Nq_conv1), the rest float32 as MXNet holds
    them ((16,256,1,1), (16,), (1,16,1,1), (1,)) -> logits (N,2,H,W) f32 ([n,0] warp, [n,1] current)."""
    _dev(x, "x", torch.bfloat16)
    w1, b1, w2, b2, w3, b3 = packed_params
    _dev(w1, "w1", torch.bfloat16)
    for t, nme in ((b1, "b1"), (w2, "w2"), (b2, "b2"), (w3, "w3"), (b3, "b3")):
        _dev(t, nme, torch.float32)
    NB, H, W, Cc = x.shape
    if NB % 2:
        raise ValueError("x must hold Concat_0(warp_feat, conv_feat): an even number of images")
    if w1.shape[0] != 256 or w1.shape[1] != 9 * Cc or w2.numel() != 16 * 256 or b2.numel() != 16 or w3.numel() != 16 or b3.numel() != 1:
        raise ValueError("Nq_net parameters must be 3x3 C->256, 1x1 256->16, 1x1 16->1 (SYM:97-101)")
    N = NB // 2
    logits = torch.empty((N, 2, H, W), dtype=torch.float32, device=x.device)
    A.check(A.load().lsfa_nq_logits_bf16_nhwc(x.data_ptr(), w1.data_ptr(), b1.data_ptr(), w2.data_ptr(), b2.data_ptr(),
                                              w3.data_ptr(), b3.data_ptr(), logits.data_ptr(), N, H, W, Cc, _stream()))
    return logits
