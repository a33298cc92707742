"""PyTorch custom-op harness (``torch.library``) over the C ABI.

The role ``mx.operator.CustomOpProp`` plays in the reference (list_arguments / infer_shape /
create_operator, operator_py/choose_feat.py:45-68): each op has a real implementation that
enqueues our CUDA kernels and a ``register_fake`` that is the ``infer_shape``.  Registered under
the ``lsfa::`` namespace:

    lsfa::grid_generator_warp(flow) -> grid
    lsfa::bilinear_sampler(data, grid) -> out
    lsfa::mv_pool(mv, im_scale, mode) -> flow
    lsfa::warp_scale_aggregate(key, flow, cur?, scale_map?, logits?, bypass?, weight_mode, flow_kind,
                               im_scale, layout) -> out
    lsfa::cosine_logits(emb_warp, emb_cur) -> logits      (NCHW float32; Fgfa trains as
                               warp_scale_aggregate(..., logits=cosine_logits(ew, ec), weight_mode=3))

This is harness only - shapes, dtypes and dispatch; the arithmetic is in liblsfa_b200.so.
"""
from __future__ import annotations

from typing import Optional

import torch

from . import ops

_MODES = ("none", "add", "mean", "logits", "cosine")
_FLOWS = ("flow", "grid", "raw")
_LAYOUTS = ("nchw", "nhwc_f32", "nhwc_bf16")


@torch.library.custom_op("lsfa::grid_generator_warp", mutates_args=())
def grid_generator_warp(flow: torch.Tensor) -> torch.Tensor:
    return ops.GridGenerator(flow, transform_type="warp")


@grid_generator_warp.register_fake
def _(flow):
    torch._check(flow.dim() == 4 and flow.shape[1] == 2, lambda: "flow must be (N,2,H,W)")
    return torch.empty_like(flow)


@torch.library.custom_op("lsfa::bilinear_sampler", mutates_args=())
def bilinear_sampler(data: torch.Tensor, grid: torch.Tensor) -> torch.Tensor:
    return ops.BilinearSampler(data, grid)


@bilinear_sampler.register_fake
def _(data, grid):
    torch._check(data.dim() == 4 and grid.dim() == 4 and grid.shape[1] == 2 and grid.shape[0] == data.shape[0],
                 lambda: "data (N,C,Hi,Wi), grid (N,2,Ho,Wo)")
    return data.new_empty((data.shape[0], data.shape[1], grid.shape[2], grid.shape[3]))


@torch.library.custom_op("lsfa::bilinear_sampler_backward", mutates_args=())
def bilinear_sampler_backward(data: torch.Tensor, grid: torch.Tensor, out_grad: torch.Tensor) -> tuple[torch.Tensor, torch.Tensor]:
    gd, gg = ops.BilinearSampler_backward(data, grid, out_grad.contiguous())
    return gd, gg


@bilinear_sampler_backward.register_fake
def _(data, grid, out_grad):
    return torch.empty_like(data), torch.empty_like(grid)


@torch.library.custom_op("lsfa::grid_generator_warp_backward", mutates_args=())
def grid_generator_warp_backward(grad_grid: torch.Tensor) -> torch.Tensor:
    return ops.GridGenerator_backward(grad_grid.contiguous())


@grid_generator_warp_backward.register_fake
def _(grad_grid):
    return torch.empty_like(grad_grid)


# declare_backward_dependency / backward of the two MXNet operators (operator_py/*.py:declare_backward_dependency
# is where a CustomOpProp says what its backward needs): the sampler's backward needs data and grid, the grid
# generator's only the incoming gradient
def _bs_setup(ctx, inputs, output):
    ctx.save_for_backward(*inputs)


def _bs_backward(ctx, grad_out):
    data, grid = ctx.saved_tensors
    gd, gg = bilinear_sampler_backward(data, grid, grad_out)
    return gd, gg


bilinear_sampler.register_autograd(_bs_backward, setup_context=_bs_setup)
grid_generator_warp.register_autograd(lambda ctx, g: grid_generator_warp_backward(g))


@torch.library.custom_op("lsfa::mv_pool", mutates_args=())
def mv_pool(mv: torch.Tensor, im_scale: float, mode: int) -> torch.Tensor:
    return ops.mv_pool(mv, im_scale, mode)


@mv_pool.register_fake
def _(mv, im_scale, mode):
    torch._check(mv.dim() == 4 and mv.shape[3] == 2, lambda: "mv must be (N,h,w,2)")
    return mv.new_empty((mv.shape[0], 2, (mv.shape[1] + 15) // 16, (mv.shape[2] + 15) // 16), dtype=torch.float32)


@torch.library.custom_op("lsfa::warp_scale_aggregate", mutates_args=())
def warp_scale_aggregate(key: torch.Tensor, flow: torch.Tensor, cur: Optional[torch.Tensor],
                         scale_map: Optional[torch.Tensor], logits: Optional[torch.Tensor],
                         bypass: Optional[torch.Tensor], weight_mode: int, flow_kind: int,
                         im_scale: float, layout: int) -> torch.Tensor:
    return ops.warp_scale_aggregate(key, flow, cur=cur, scale_map=scale_map, logits=logits, bypass=bypass,
                                    weight_mode=_MODES[weight_mode], flow_kind=_FLOWS[flow_kind],
                                    im_scale=im_scale, layout=_LAYOUTS[layout])


@warp_scale_aggregate.register_fake
def _(key, flow, cur, scale_map, logits, bypass, weight_mode, flow_kind, im_scale, layout):
    torch._check(key.dim() == 4 and flow.dim() == 4, lambda: "key and flow must be 4-D")
    if flow_kind == 2:
        n, h, w = flow.shape[0], (flow.shape[1] + 15) // 16, (flow.shape[2] + 15) // 16
    else:
        n, h, w = flow.shape[0], flow.shape[2], flow.shape[3]
    if layout == 0:
        return key.new_empty((n, key.shape[1], h, w))
    return key.new_empty((n, h, w, key.shape[3]))


# backward of the fused operator (csrc/aggregate_backward.cu): NCHW float32, modes none/add/mean/logits; raw motion vectors
# are data (no gradient), a prepooled flow / grid gets one
@torch.library.custom_op("lsfa::warp_scale_aggregate_backward", mutates_args=())
def warp_scale_aggregate_backward(out_grad: torch.Tensor, key: torch.Tensor, flow: torch.Tensor, cur: Optional[torch.Tensor],
                                  scale_map: Optional[torch.Tensor], logits: Optional[torch.Tensor],
                                  bypass: Optional[torch.Tensor], weight_mode: int, flow_kind: int,
                                  im_scale: float) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    g = ops.warp_scale_aggregate_backward(out_grad.contiguous(), key, flow, cur=cur, scale_map=scale_map, logits=logits, bypass=bypass,
                                          weight_mode=_MODES[weight_mode], flow_kind=_FLOWS[flow_kind], im_scale=im_scale)
    z = lambda t: torch.zeros_like(t) if t is not None else out_grad.new_zeros(1)  # noqa: E731
    flow_like = flow if flow.dtype == torch.float32 else None
    return (g["key"], g.get("flow", z(flow_like)), g.get("cur", z(cur)), g.get("scale", z(scale_map)), g.get("logits", z(logits)))


@warp_scale_aggregate_backward.register_fake
def _(out_grad, key, flow, cur, scale_map, logits, bypass, weight_mode, flow_kind, im_scale):
    e = lambda t: torch.empty_like(t) if t is not None else out_grad.new_empty(1)  # noqa: E731
    return torch.empty_like(key), e(flow if flow.dtype == torch.float32 else None), e(cur), e(scale_map), e(logits)


def _wsa_setup(ctx, inputs, output):
    key, flow, cur, scale_map, logits, bypass, weight_mode, flow_kind, im_scale, layout = inputs
    if layout != 0 or weight_mode == 4:
        ctx.unsupported = "the backward is built for NCHW float32 and the modes none/add/mean/logits"
        return
    ctx.unsupported = None
    ctx.meta = (weight_mode, flow_kind, im_scale)
    ctx.has = (cur is not None, scale_map is not None, logits is not None, bypass is not None)
    ctx.save_for_backward(*[t for t in (key, flow, cur, scale_map, logits, bypass) if t is not None])


def _wsa_backward(ctx, grad_out):
    if ctx.unsupported:
        raise RuntimeError("lsfa::warp_scale_aggregate: " + ctx.unsupported)
    saved = list(ctx.saved_tensors)
    key, flow = saved[0], saved[1]
    rest = saved[2:]
    opt = []
    for present in ctx.has:
        opt.append(rest.pop(0) if present else None)
    cur, scale_map, logits, bypass = opt
    weight_mode, flow_kind, im_scale = ctx.meta
    gk, gf, gc, gs, gl = warp_scale_aggregate_backward(grad_out, key, flow, cur, scale_map, logits, bypass, weight_mode, flow_kind, im_scale)
    return (gk, gf if (flow_kind in (0, 1) and flow.dtype == torch.float32) else None, gc if cur is not None else None,
            gs if scale_map is not None else None, gl if (logits is not None and weight_mode == 3) else None, None, None, None, None, None)


warp_scale_aggregate.register_autograd(_wsa_backward, setup_context=_wsa_setup)


# Fgfa_net's weights (SYM:111-116,137-139): the same kernels the fused COSINE mode runs, so that mode trains as
# warp_scale_aggregate(..., logits=cosine_logits(emb_warp, emb_cur), weight_mode=3)
@torch.library.custom_op("lsfa::cosine_logits", mutates_args=())
def cosine_logits(emb_warp: torch.Tensor, emb_cur: torch.Tensor) -> torch.Tensor:
    return ops.cosine_logits(emb_warp, emb_cur)


@cosine_logits.register_fake
def _(emb_warp, emb_cur):
    torch._check(emb_warp.dim() == 4 and emb_cur.shape == emb_warp.shape, lambda: "emb_warp, emb_cur (N,E,H,W)")
    return emb_warp.new_empty((emb_warp.shape[0], 2, emb_warp.shape[2], emb_warp.shape[3]))


@torch.library.custom_op("lsfa::cosine_logits_backward", mutates_args=())
def cosine_logits_backward(emb_warp: torch.Tensor, emb_cur: torch.Tensor, grad_logits: torch.Tensor) -> tuple[torch.Tensor, torch.Tensor]:
    return ops.cosine_logits_backward(emb_warp, emb_cur, grad_logits.contiguous())


@cosine_logits_backward.register_fake
def _(emb_warp, emb_cur, grad_logits):
    return torch.empty_like(emb_warp), torch.empty_like(emb_cur)


def _cos_setup(ctx, inputs, output):
    ctx.save_for_backward(*inputs)


def _cos_backward(ctx, grad_logits):
    emb_warp, emb_cur = ctx.saved_tensors
    return cosine_logits_backward(emb_warp, emb_cur, grad_logits)


cosine_logits.register_autograd(_cos_backward, setup_context=_cos_setup)
