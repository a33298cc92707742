"""Backward of Fgfa_net's cosine weights (SYM:111-116,132-148): lsfa_cosine_logits_backward_f32_nchw on its own and
the fused operator's COSINE mode (lsfa_warp_scale_aggregate_backward_f32_nchw).

CPU: the oracle's chain rule (oracle/cosine_backward.py) against torch float64 autograd (tests/golden/fused_backward_cosine_small.npz, minted by
     tools/make_golden_cosine_backward.py), the ref64 gate against the float32 oracle and planted bugs, argument
     validation and workspace sizes, and the previous LsfaAggGrads size.
GPU: the op against the ref64 gate at the Fgfa sizes and on the fallback shapes, bit-level agreement of its two
     kernels and across runs, the fused COSINE mode against the oracle, the fixture and the composition of LOGITS mode
     with the op, the adjoint identity at full size, and torch autograd through lsfa::cosine_logits."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from oracle import lsfa_oracle as O
from oracle import cosine_backward as CB
from oracle import ref64 as R
from tests._util import make_case

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden", "fused_backward_cosine_small.npz")


def _close(got, want, what, rtol=1e-5, atol_frac=4e-6):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    tol = rtol * np.abs(want) + atol_frac * max(np.abs(want).max(), 1e-30)
    err = np.abs(got - want)
    assert (err <= tol).all(), "%s: worst abs err %.3g at scale %.3g (%d outside)" % (what, err.max(), np.abs(want).max(), int((err > tol).sum()))


def _f32_backward(ew, ec, gl, eps=1e-10, keep_g2=True, alpha_ulp=0):
    """The backward in float32 numpy, the way the kernels compute it (optionally with a planted bug)."""
    with np.errstate(invalid="ignore", divide="ignore"):       # eps = 0 on the all-zero pixel
        return _f32_backward_body(np.float32, ew, ec, gl, eps, keep_g2, alpha_ulp)


def _f32_backward_body(f, ew, ec, gl, eps, keep_g2, alpha_ulp):
    a, b = np.asarray(ew, f), np.asarray(ec, f)
    saa, sbb, sab = (np.sum(x, axis=1, keepdims=True, dtype=f) for x in (a * a, b * b, a * b))
    na, nb = np.sqrt(saa + f(eps)), np.sqrt(sbb + f(eps))
    l1, l2 = sab / (na * nb), sbb / (nb * nb)
    g1, g2 = np.asarray(gl[:, 0:1], f), np.asarray(gl[:, 1:2], f)
    al = g1 / (na * nb)
    if alpha_ulp:
        al = np.nextafter(al, np.inf * np.sign(al), dtype=f)
    be = -(g1 * l1) / (na * na)
    ga = ((f(2) * g2 * (f(1) - l2) if keep_g2 else f(0)) - g1 * l1) / (nb * nb)
    return al * b + be * a, al * a + ga * b


def _case(seed, N, E, H, W):
    rng = np.random.default_rng(seed)
    ew = rng.standard_normal((N, E, H, W), dtype=np.float32)
    ec = rng.standard_normal((N, E, H, W), dtype=np.float32)
    ew[:, :, 0, 0] = 0.0
    ec[:, :, 0, 0] = 0.0                                   # all-zero pixel: the eps path
    ec[:, :, 0, 1] *= np.float32(1e-6)                     # tiny norm: eps and the d l2 term matter
    ew[:, :, 0, 1] *= np.float32(1e-6)
    gl = rng.standard_normal((N, 2, H, W), dtype=np.float32)
    return ew, ec, gl


# ------------------------------------------------------------------------------------------------------------- CPU
def test_oracle_equals_torch_autograd_fixture():
    g = np.load(GOLD)
    gw, gc = CB.cosine_logits_backward(g["cos_emb_warp"], g["cos_emb_cur"], g["cos_grad_logits"])
    _close(gw, g["cos_grad_emb_warp"], "op grad_emb_warp")
    _close(gc, g["cos_grad_emb_cur"], "op grad_emb_cur")
    kw = dict(cur=g["fused_cur"], scale_map=g["fused_scale"], weight_mode=O.W_COSINE, emb_warp=g["fused_emb_warp"],
              emb_cur=g["fused_emb_cur"], bypass=g["fused_bypass"])
    _close(O.warp_scale_aggregate(g["fused_key"], g["fused_flow"], **kw), g["fused_out"], "fused forward")
    got = CB.warp_scale_aggregate_backward(g["fused_out_grad"], g["fused_key"], g["fused_flow"], g["fused_emb_warp"], g["fused_emb_cur"],
                                           cur=g["fused_cur"], scale_map=g["fused_scale"], bypass=g["fused_bypass"])
    assert "logits" not in got
    for nme in ("key", "flow", "scale", "cur", "emb_warp", "emb_cur"):
        _close(got[nme], g["fused_grad_%s" % nme], "fused grad_%s" % nme)
    assert not got["emb_warp"][1].any() and not got["emb_cur"][1].any()      # the bypass frame


def test_gate_passes_float32_oracle_and_rejects_planted_bugs():
    ew, ec, gl = _case(5, 2, 64, 6, 7)
    ref = CB.ref64_backward(torch.from_numpy(ew), torch.from_numpy(ec), torch.from_numpy(gl), device="cpu")
    gw, gc = _f32_backward(ew, ec, gl)
    worst = max(R.check(torch.from_numpy(gw), *ref["emb_warp"][:2], n_addends=ref["emb_warp"][2], what="grad_emb_warp"),
                R.check(torch.from_numpy(gc), *ref["emb_cur"][:2], n_addends=ref["emb_cur"][2], what="grad_emb_cur"))
    assert worst < 1.0
    for bug in (dict(eps=0.0), dict(keep_g2=False)):
        bw, bc = _f32_backward(ew, ec, gl, **bug)
        with pytest.raises(AssertionError):
            R.check(torch.from_numpy(bw), *ref["emb_warp"][:2], n_addends=ref["emb_warp"][2], what="planted")
            R.check(torch.from_numpy(bc), *ref["emb_cur"][:2], n_addends=ref["emb_cur"][2], what="planted")
    # a one-ulp error in alpha is below the float32 rounding of the result itself: no per-element bound that the
    # correct float32 computation meets can see it.  It changes the bits, which the GPU tests compare between the two
    # kernels and against the LOGITS-mode composition.
    bw, _ = _f32_backward(ew, ec, gl, alpha_ulp=1)
    assert not np.array_equal(bw, gw)


def test_argument_validation_and_workspace_without_gpu(lib):
    from lsfa_b200 import _cabi as A
    N, E, H, W = 4, 2048, 38, 63
    ws = lib.lsfa_cosine_logits_backward_workspace_bytes(N, E, H, W)
    coef = -(-N * 3 * H * W * 4 // 256) * 256
    part = -(-lib.lsfa_cosine_logits_workspace_bytes(N, E, H, W, 0) // 256) * 256
    assert ws == coef + part and part > 0
    assert lib.lsfa_cosine_logits_backward_workspace_bytes(0, E, H, W) == 0
    f = lib.lsfa_cosine_logits_backward_f32_nchw
    p = 1 << 40
    eb = N * E * H * W * 4
    assert f(p, p + eb, p + 2 * eb, p + 3 * eb, p + 4 * eb, N, E, H, W, 1, 1, p + 6 * eb, ws, 5, None) == A.E_BADARG
    assert f(p, p + eb, p + 2 * eb, p + 3 * eb, p + 4 * eb, N, E, H, W, 7, 1, p + 6 * eb, ws, 0, None) == A.E_BADARG
    assert f(p, p + eb, p + 2 * eb, p + 3 * eb, p + 4 * eb, N, 0, H, W, 1, 1, p + 6 * eb, ws, 0, None) == A.E_SHAPE
    assert f(p, p + eb, p + 2 * eb, p + 3 * eb, p + 4 * eb, N, E, H, W, 1, 1, p + 6 * eb, ws - 1, 0, None) == A.E_BADARG
    assert b"workspace too small" in lib.lsfa_last_error()
    assert f(p, p + eb, p + 2 * eb, p + 3 * eb, p + 4 * eb, N, E, H, W, 1, 1, p + 6 * eb + 4, ws, 0, None) == A.E_ALIGN
    assert f(p, p + eb, p + 2 * eb, p + eb + 64, p + 4 * eb, N, E, H, W, 1, 1, p + 6 * eb, ws, 0, None) == A.E_BADARG
    assert b"overlap" in lib.lsfa_last_error()
    assert f(None, p + eb, p + 2 * eb, p + 3 * eb, p + 4 * eb, N, E, H, W, 1, 1, p + 6 * eb, ws, 0, None) == A.E_BADARG
    assert f(None, None, None, None, None, N, E, H, W, 0, 0, None, 0, 0, None) == A.OK        # nothing requested


def _cosine_args(A, N=2, C=8, E=16, H=5, W=6):
    p = 1 << 40
    return A.new_args(layout=A.LAYOUT_NCHW_F32, N=N, C=C, H=H, W=W, key=p, flow=p, cur=p, out=p, req=A.REQ_WRITE,
                      flow_kind=A.FLOW_PREPOOLED, weight_mode=A.W_COSINE, emb_warp=p, emb_cur=p, E=E)


def test_fused_cosine_validation_and_workspace_without_gpu(lib):
    from lsfa_b200 import _cabi as A
    a = _cosine_args(A)
    g = A.LsfaAggGrads()
    g.struct_bytes = ctypes.sizeof(A.LsfaAggGrads)
    g.out_grad, g.grad_cur, g.req_cur = 1 << 40, 1 << 41, A.REQ_WRITE
    base = lib.lsfa_warp_scale_aggregate_backward_workspace_bytes(a, g)
    assert base > 0
    g.grad_emb_warp, g.grad_emb_cur, g.req_emb = 1 << 42, 1 << 43, A.REQ_WRITE
    assert lib.lsfa_warp_scale_aggregate_backward_workspace_bytes(a, g) > base      # + d/d(logits) partial sums
    g.grad_logits, g.req_logits = 1 << 44, A.REQ_WRITE
    assert lib.lsfa_warp_scale_aggregate_backward_f32_nchw(a, g, None) == A.E_BADARG
    assert b"COSINE" in lib.lsfa_last_error()
    g.grad_logits, g.req_logits = None, A.REQ_NULL
    a.weight_mode = A.W_ADD
    assert lib.lsfa_warp_scale_aggregate_backward_f32_nchw(a, g, None) == A.E_BADARG
    assert b"embedding gradients" in lib.lsfa_last_error()
    g.req_emb = 9
    a.weight_mode = A.W_COSINE
    assert lib.lsfa_warp_scale_aggregate_backward_f32_nchw(a, g, None) == A.E_BADARG


def test_previous_grads_struct_size_is_accepted(lib):
    """A binary built against the header before the embedding fields: struct_bytes = offsetof(grad_emb_warp)."""
    from lsfa_b200 import _cabi as A
    old = A.LsfaAggGrads.grad_emb_warp.offset
    src = open(os.path.join(ROOT, "include", "lsfa_ops.h")).read()
    assert re.search(r"size_t workspace_bytes;\s*\n\s*float\* grad_emb_warp;", src)
    a = _cosine_args(A)
    a.weight_mode, a.logits = A.W_LOGITS, 1 << 40
    g = A.LsfaAggGrads()
    g.struct_bytes = old
    g.out_grad, g.grad_logits, g.req_logits = 1 << 40, 1 << 41, A.REQ_WRITE
    g.grad_emb_warp, g.req_emb = 1 << 42, 77          # past the old size: must not be read
    ws_old = lib.lsfa_warp_scale_aggregate_backward_workspace_bytes(a, g)
    assert ws_old > 0
    g.struct_bytes = ctypes.sizeof(A.LsfaAggGrads)
    g.grad_emb_warp, g.req_emb = None, 0
    assert lib.lsfa_warp_scale_aggregate_backward_workspace_bytes(a, g) == ws_old
    g.struct_bytes = old + 8
    assert lib.lsfa_warp_scale_aggregate_backward_workspace_bytes(a, g) == 0


def test_tma_kernel_does_not_spill(lib):
    from lsfa_b200 import _build
    log = open(os.path.join(os.path.dirname(_build.LIB_PATH), "build.log")).read()
    hits = re.findall(r"Compiling entry function '(\S*cosine_backward_tma_kernel\S*)' for 'sm_100a'\s*\n.*?\n\s*\d+ bytes stack frame, "
                      r"(\d+) bytes spill stores, (\d+) bytes spill loads", log)
    assert hits
    assert all(st == "0" and ld == "0" for _, st, ld in hits), hits


# ------------------------------------------------------------------------------------------------------------- GPU
def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _gate(got, ref, what):
    r, m, na = ref
    return R.check(got.double().cpu(), r, m, n_addends=na, what=what)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(2, 256, 38, 63), (4, 2048, 38, 63), (2, 2048, 68, 120), (2, 40, 17, 23)])
def test_gpu_op_against_ref64_gate(cuda, shape):
    from lsfa_b200 import ops
    N, E, H, W = shape
    ew, ec, gl = (_t(x, cuda) for x in _case(E + H, N, E, H, W))
    gw, gc = ops.cosine_logits_backward(ew, ec, gl)
    torch.cuda.synchronize()
    assert torch.isfinite(gw).all() and torch.isfinite(gc).all()
    ref = CB.ref64_backward(ew, ec, gl)
    worst = max(_gate(gw, ref["emb_warp"], "grad_emb_warp %s" % (shape,)), _gate(gc, ref["emb_cur"], "grad_emb_cur %s" % (shape,)))
    print("max err/tol %s: %.3f" % (shape, worst))


@pytest.mark.gpu
def test_gpu_op_req_add_and_one_gradient_skipped(cuda):
    from lsfa_b200 import ops
    N, E, H, W = 2, 256, 38, 63
    ew, ec, gl = (_t(x, cuda) for x in _case(3, N, E, H, W))
    gw, gc = ops.cosine_logits_backward(ew, ec, gl)
    for kern in ("tma", "plain"):
        base_w, base_c = torch.randn_like(ew), torch.randn_like(ec)
        aw, _ = ops.cosine_logits_backward(ew, ec, gl, grad_emb_warp=base_w.clone(), req_warp="add", req_cur="null", kernel=kern)
        _, ac = ops.cosine_logits_backward(ew, ec, gl, grad_emb_cur=base_c.clone(), req_cur="add", req_warp="null", kernel=kern)
        assert torch.equal(aw, base_w + gw), kern
        assert torch.equal(ac, base_c + gc), kern
        only_w, none_c = ops.cosine_logits_backward(ew, ec, gl, req_cur="null", kernel=kern)
        assert none_c is None and torch.equal(only_w, gw)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(4, 2048, 38, 63), (3, 64, 17, 24)])
def test_gpu_op_kernels_bit_equal_and_deterministic(cuda, shape):
    from lsfa_b200 import ops
    N, E, H, W = shape
    ew, ec, gl = (_t(x, cuda) for x in _case(11, N, E, H, W))
    tw, tc = ops.cosine_logits_backward(ew, ec, gl, kernel="tma")
    pw, pc = ops.cosine_logits_backward(ew, ec, gl, kernel="plain")
    assert torch.equal(tw, pw) and torch.equal(tc, pc)
    for _ in range(3):
        aw, ac = ops.cosine_logits_backward(ew, ec, gl, kernel="tma")
        assert torch.equal(aw, tw) and torch.equal(ac, tc)


@pytest.mark.gpu
def test_gpu_op_tma_kernel_refuses_what_it_cannot_serve(cuda):
    from lsfa_b200 import ops
    from lsfa_b200._cabi import LsfaError
    ew, ec, gl = (_t(x, cuda) for x in _case(1, 1, 8, 68, 120))
    with pytest.raises(LsfaError, match="UNSUPPORTED"):
        ops.cosine_logits_backward(ew, ec, gl, kernel="tma")


def _fused_kw(d, dev):
    return dict(cur=_t(d["cur"], dev), scale_map=_t(d["scale_map"], dev), weight_mode="cosine", emb_warp=_t(d["emb_warp"], dev),
                emb_cur=_t(d["emb_cur"], dev), bypass=_t(d["bypass"], dev), flow_kind="flow")


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(3, 64, 38, 63), (2, 40, 17, 23), (1, 8, 68, 120)])
def test_gpu_fused_cosine_backward_matches_oracle(cuda, shape):
    from lsfa_b200 import ops
    N, C, H, W = shape
    d = make_case(950 + C, N, C, H, W, E=48, with_bypass=True)
    og = np.random.default_rng(C).standard_normal((N, C, H, W), dtype=np.float32)
    flow = np.ascontiguousarray(d["flow"])
    want = CB.warp_scale_aggregate_backward(og, d["key"], flow, d["emb_warp"], d["emb_cur"], cur=d["cur"], scale_map=d["scale_map"],
                                            bypass=d["bypass"])
    kw = _fused_kw(d, cuda)
    got = ops.warp_scale_aggregate_backward(_t(og, cuda), _t(d["key"], cuda), _t(flow, cuda), **kw)
    again = ops.warp_scale_aggregate_backward(_t(og, cuda), _t(d["key"], cuda), _t(flow, cuda), **kw)
    torch.cuda.synchronize()
    assert set(got) == set(want), (sorted(got), sorted(want))
    for nme in want:
        _close(got[nme].cpu().numpy(), want[nme], "cosine grad_%s" % nme, rtol=2e-5, atol_frac=2e-5)
    for nme in ("scale", "cur", "emb_warp", "emb_cur"):
        assert torch.equal(got[nme], again[nme]), "grad_%s is not deterministic" % nme
    byp = torch.from_numpy(d["bypass"]).bool()
    assert not got["emb_warp"][byp].any() and not got["emb_cur"][byp].any()
    # req = add leaves the bypass frames' embedding gradients untouched
    import lsfa_b200._cabi as A
    from lsfa_b200.ops import _build_args
    base = torch.randn_like(kw["emb_warp"])
    acc_w, acc_c = base.clone(), base.clone() + 1
    kw2 = dict(kw)
    kw2["workspace"] = False
    args, _out, _keep = _build_args(_t(d["key"], cuda), _t(flow, cuda), **kw2)
    g = A.LsfaAggGrads()
    g.struct_bytes = ctypes.sizeof(A.LsfaAggGrads)
    ogt = _t(og, cuda)
    g.out_grad = ogt.data_ptr()
    g.grad_emb_warp, g.grad_emb_cur, g.req_emb = acc_w.data_ptr(), acc_c.data_ptr(), A.REQ_ADD
    lib = A.load()
    need = lib.lsfa_warp_scale_aggregate_backward_workspace_bytes(args, g)
    ws = torch.empty(need + 256, dtype=torch.uint8, device=cuda)
    g.workspace, g.workspace_bytes = ws.data_ptr() + (-ws.data_ptr()) % 256, need
    A.check(lib.lsfa_warp_scale_aggregate_backward_f32_nchw(args, g, torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    assert torch.equal(acc_w[byp.to(cuda)], base[byp.to(cuda)]) and torch.equal(acc_c[byp.to(cuda)], base[byp.to(cuda)] + 1)
    live = ~byp.to(cuda)
    assert torch.equal(acc_w[live], base[live] + got["emb_warp"][live])
    assert torch.equal(acc_c[live], base[live] + 1 + got["emb_cur"][live])


@pytest.mark.gpu
def test_gpu_fused_cosine_backward_equals_fixture(cuda):
    from lsfa_b200 import ops
    g = np.load(GOLD)
    kw = dict(cur=_t(g["fused_cur"], cuda), scale_map=_t(g["fused_scale"], cuda), weight_mode="cosine", emb_warp=_t(g["fused_emb_warp"], cuda),
              emb_cur=_t(g["fused_emb_cur"], cuda), bypass=_t(g["fused_bypass"], cuda), flow_kind="flow")
    got = ops.warp_scale_aggregate_backward(_t(g["fused_out_grad"], cuda), _t(g["fused_key"], cuda), _t(g["fused_flow"], cuda), **kw)
    for nme in ("key", "flow", "scale", "cur", "emb_warp", "emb_cur"):
        _close(got[nme].cpu().numpy(), g["fused_grad_%s" % nme], "fused grad_%s" % nme, rtol=2e-5, atol_frac=1e-5)
    gw, gc = ops.cosine_logits_backward(_t(g["cos_emb_warp"], cuda), _t(g["cos_emb_cur"], cuda), _t(g["cos_grad_logits"], cuda))
    _close(gw.cpu().numpy(), g["cos_grad_emb_warp"], "op grad_emb_warp", rtol=2e-5, atol_frac=1e-5)
    _close(gc.cpu().numpy(), g["cos_grad_emb_cur"], "op grad_emb_cur", rtol=2e-5, atol_frac=1e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(3, 64, 2048, 38, 63), (2, 16, 40, 17, 23)])
def test_gpu_fused_cosine_is_logits_mode_composed_with_the_op(cuda, shape):
    """Bit for bit: the fused COSINE backward = the LOGITS-mode backward fed with ops.cosine_logits (full workspace),
    followed by ops.cosine_logits_backward.  So the backward's logits are the forward's bits."""
    from lsfa_b200 import ops
    N, C, E, H, W = shape
    d = make_case(77 + C, N, C, H, W, E=E, with_bypass=True)
    og, key, flow = _t(np.random.default_rng(2).standard_normal((N, C, H, W), dtype=np.float32), cuda), _t(d["key"], cuda), _t(d["flow"], cuda)
    kw = _fused_kw(d, cuda)
    fused = ops.warp_scale_aggregate_backward(og, key, flow, **kw)
    lg = ops.cosine_logits(kw["emb_warp"], kw["emb_cur"])
    lkw = dict(kw, weight_mode="logits", logits=lg)
    ew, ec = lkw.pop("emb_warp"), lkw.pop("emb_cur")
    ref = ops.warp_scale_aggregate_backward(og, key, flow, **lkw)
    gw, gc = ops.cosine_logits_backward(ew, ec, ref["logits"])
    # the fused output with those logits is the COSINE forward
    assert torch.equal(ops.warp_scale_aggregate(key, flow, **kw), ops.warp_scale_aggregate(key, flow, **lkw))
    for nme in ("scale", "cur"):
        assert torch.equal(fused[nme], ref[nme]), nme
    # d/d(key) and d/d(flow) come from the a7/a8 backward, which adds atomically on planes its gather kernel cannot hold
    for nme in ("key", "flow"):
        _close(fused[nme].cpu().numpy(), ref[nme].cpu().numpy(), "grad_%s" % nme)
    assert torch.equal(fused["emb_warp"], gw) and torch.equal(fused["emb_cur"], gc)


@pytest.mark.gpu
def test_gpu_fused_cosine_against_ref64_gate_at_full_size(cuda):
    """Fused COSINE embedding gradients at 2 x 1024 x 38x63, E = 2048, against ref64 with the error of d/d(l1) (a C-term
    sum of the tail) folded into the gate."""
    from lsfa_b200 import ops
    N, C, E, H, W = 2, 1024, 2048, 38, 63
    gen = torch.Generator(device=cuda).manual_seed(4)
    rn = lambda *s: torch.randn(s, device=cuda, generator=gen)  # noqa: E731
    key, cur, sm, flow, og = rn(N, C, H, W).clamp_(min=0), rn(N, C, H, W).clamp_(min=0), 1 + 0.1 * rn(N, C, H, W), 2.0 * rn(N, 2, H, W), rn(N, C, H, W)
    ew, ec = rn(N, E, H, W), rn(N, E, H, W)
    byp = torch.tensor([0, 1], dtype=torch.uint8, device=cuda)
    got = ops.warp_scale_aggregate_backward(og, key, flow, flow_kind="flow", cur=cur, scale_map=sm, weight_mode="cosine",
                                            emb_warp=ew, emb_cur=ec, bypass=byp)
    lg = ops.cosine_logits(ew, ec)
    co = R.coords(flow=flow.cpu())
    tail = R.backward(og, key, co, cur=cur, scale_map=sm, mode="logits", logits=lg, bypass=byp, want=("logits",))
    d, m, na = tail["logits"]
    g_err = ((na + 8) * R.U * m[:, 0:1]).to(cuda)
    ref = CB.ref64_backward(ew, ec, d.to(cuda), g_err=g_err)
    worst = max(_gate(got["emb_warp"], ref["emb_warp"], "fused grad_emb_warp"), _gate(got["emb_cur"], ref["emb_cur"], "fused grad_emb_cur"))
    print("fused cosine max err/tol %.3f" % worst)


@pytest.mark.gpu
def test_gpu_op_full_size_adjoint_identity(cuda):
    """<g, d logits> == <grad_e, d e> at 4 x 2048 x 38x63, with a finite-difference step of the forward."""
    from lsfa_b200 import ops
    N, E, H, W = 4, 2048, 38, 63
    gen = torch.Generator(device=cuda).manual_seed(0)
    rn = lambda *s: torch.randn(s, device=cuda, generator=gen)  # noqa: E731
    ew, ec, gl = rn(N, E, H, W), rn(N, E, H, W), rn(N, 2, H, W)
    gw, gc = ops.cosine_logits_backward(ew, ec, gl)
    eps = 1e-2
    for nme in ("emb_warp", "emb_cur"):
        dx = rn(N, E, H, W)
        if nme == "emb_warp":
            lp, lm = ops.cosine_logits(ew + eps * dx, ec), ops.cosine_logits(ew - eps * dx, ec)
            rhs = (gw.double() * dx.double()).sum().item()
        else:
            lp, lm = ops.cosine_logits(ew, ec + eps * dx), ops.cosine_logits(ew, ec - eps * dx)
            rhs = (gc.double() * dx.double()).sum().item()
        lhs = ((lp.double() - lm.double()) * gl.double()).sum().item() / (2 * eps)
        assert abs(lhs - rhs) <= 2e-3 * max(abs(lhs), abs(rhs), 1.0), (nme, lhs, rhs)


@pytest.mark.gpu
def test_torch_autograd_through_cosine_logits_equals_fused_cosine_backward(cuda):
    import lsfa_b200.torch_ops  # noqa: F401  (registers lsfa::*)
    from lsfa_b200 import ops
    N, C, E, H, W = 3, 64, 256, 38, 63
    d = make_case(5, N, C, H, W, E=E, with_bypass=True)
    leaf = lambda a: _t(a, cuda).requires_grad_(True)  # noqa: E731
    key, flow, cur, sm, ew, ec = (leaf(d[k]) for k in ("key", "flow", "cur", "scale_map", "emb_warp", "emb_cur"))
    byp = _t(d["bypass"], cuda)
    og = torch.randn((N, C, H, W), device=cuda)
    lg = torch.ops.lsfa.cosine_logits(ew, ec)
    out = torch.ops.lsfa.warp_scale_aggregate(key, flow, cur, sm, lg, byp, 3, 0, 1.0, 0)
    out.backward(og)
    want = ops.warp_scale_aggregate_backward(og, key.detach(), flow.detach(), flow_kind="flow", cur=cur.detach(), scale_map=sm.detach(),
                                             weight_mode="cosine", emb_warp=ew.detach(), emb_cur=ec.detach(), bypass=byp)
    for nme, x in (("key", key), ("cur", cur), ("scale", sm), ("emb_warp", ew), ("emb_cur", ec)):
        assert torch.equal(x.grad, want[nme]), nme
