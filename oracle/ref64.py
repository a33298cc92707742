"""Float64 reference of the fused operator and of its backward, with a per-element error gate.

THIS IS TEST INFRASTRUCTURE, NOT PRODUCT CODE (like ``lsfa_oracle``): only ``tests/`` and ``tools/`` import it.

Coordinates.  ``coords`` computes the sampling coordinates with the oracle's own float32 functions
(``mv_pool`` one frame at a time, ``grid_generator_warp``, ``sampler_coords``), so ``x0, y0, wx, wy`` are exactly
the bits MXNet stores and the kernels are pinned to.  Recomputing them in float64 would move every tap weight by
about ``W * 2^-24``, which is larger than the gate below; recomputing them with torch on a device is not bit-exact
either (a division by a scalar may be carried out as a multiply by the reciprocal).

Values.  Everything after the coordinates is float64 torch (CPU or CUDA), processed in chunks of at most
``CHUNK`` frames.  The tap weights are the float32 weights promoted to float64 (``wy*wx``, ``wy*(1-wx)``, ...);
a tap outside the key plane counts as 0.  ``forward`` also returns ``mag``, the float64 sum of the absolute values of
every term of that output element: ``sum_t w_t|v_t|*|s| + sum_k |w_k r_k| + |b|`` for the warped source, blended with
the same weights as the value plus the ``|cur|`` term.

The gate (``check``), with u = 2^-24 the unit roundoff of float32:

* float32 output: ``|got - ref| <= K u mag``, K = 16.  A float32 evaluation of a sum of m terms in any order is
  within ``(m - 1) u sum|term|`` of the exact sum, each product of j float32 factors adds ``(j - 1) u`` of its own
  magnitude, and the blend weight is ``1 / (1 + exp(dl))`` with ``expf`` (<= 2 ulp) and an IEEE division: its
  relative error is at most about 4u, which moves the output by at most ``4u (w1 |src| + w2 |cur|) <= 4u mag``.
  The warped source has 4 taps (3 additions, products of 3 factors: 5u), times the scale map (1u), plus the
  residual product of 3 terms and a bias (4u), blended (2 products and an addition: 2u) - 12u for the longest chain
  in the worst case; with the 4u of the blend weights, K = 16.  Measured on the CPU (the shapes and modes of
  tests/test_ref64_cpu.py) the MXNet-faithful float32 oracle stays within 8 u mag in logits mode and within 3.3 u mag
  in the other modes; rounded to bf16 it reaches 0.996 of the bf16 bound (the rounding alone can reach 1).
* bf16 output: ``|got - ref| <= 2^-8 |ref| + 2 K u mag``.  The kernel rounds a float32 value v (within K u mag of
  ref) to bf16 once: ``|bf16(v) - v| <= 2^-8 |v| <= 2^-8 (|ref| + K u mag)``; the sum is below the bound.  Unlike a
  gate of ``2^-8 max|ref|`` on every element, it notices a one-ulp error on an element much smaller than the largest.
* cosine mode: the two cosines ``l1 = <e_w^, e_c^>``, ``l2 = <e_c^, e_c^>`` lie in [-1, 1] and each is a sum of E
  products of normalised factors: its float32 error is at most ``(E + 2) u``.  ``d out / d l1 = -d out / d l2 =
  w1 w2 (src - cur)``, so the output moves by ``2 (E + 2) u w1 w2 |src - cur|``.  ``forward`` adds that term to mag,
  divided by K, so that ``K u mag`` grows by exactly that amount.
* reductions (the gradients): ``|got - ref| <= (n + 8) u mag`` with n the number of addends of that element and mag
  the sum of their absolute values: the worst-case bound of an n-term float32 sum in any order, plus 8u for the
  products that form each addend (at most 4 float32 factors and the grid scale factors).
* an element with ``mag == 0`` must equal ``ref`` bit for bit: a frame with ``bypass`` set returns ``cur`` itself
  (``ref = cur``, ``mag = 0``), and an output with no term at all is an exact 0.

``check`` reports how many elements are outside, the worst element as (frame, channel, y, x) with got, ref and tol,
and the frames that have failures, and returns the largest ``err / tol``.
"""
from __future__ import annotations

import numpy as np
import torch

from oracle import lsfa_oracle as O

U = 2.0 ** -24           # float32 unit roundoff
K = 16                   # float32 forward gate, in units of u * mag (derivation above)
CHUNK = 8                # frames of float64 intermediates alive at a time

MODES = {"none": O.W_NONE, "add": O.W_ADD, "mean": O.W_MEAN, "logits": O.W_LOGITS, "cosine": O.W_COSINE}


def _mode(m):
    return MODES[m] if isinstance(m, str) else int(m)


# ----------------------------------------------------------------------------------------------------------------
# coordinates: the oracle's float32 index math, bit for bit
# ----------------------------------------------------------------------------------------------------------------
def coords(mv=None, flow=None, key_hw=None):
    """x0, y0 (int32) and wx, wy (float32), each (N, H, W) numpy, from raw motion vectors ``mv`` (N, h, w, 2) int32
    (pooled one frame at a time) or from a pooled ``flow`` (N, 2, H, W) float32.  ``key_hw``: the key plane's
    (H, W) when it differs from the flow's."""
    if (mv is None) == (flow is None):
        raise ValueError("pass exactly one of mv and flow")
    if mv is not None:
        mv = mv.numpy() if isinstance(mv, torch.Tensor) else np.asarray(mv)
        flow = np.concatenate([O.mv_pool(mv[n:n + 1]) for n in range(mv.shape[0])])
    flow = flow.numpy() if isinstance(flow, torch.Tensor) else np.asarray(flow, np.float32)
    Hk, Wk = key_hw if key_hw is not None else flow.shape[2:]
    return O.sampler_coords(O.grid_generator_warp(flow), Hk, Wk)


def _taps(co, frames, Hk, Wk, device):
    """For ``frames``: four (flat index (n, HW) int64, weight (n, 1, HW) float64, in-plane mask (n, HW)) triples,
    out-of-plane taps weighted 0, plus wx, wy as float64 (n, HW)."""
    x0, y0, wx, wy = co
    sl = slice(frames.start, frames.stop)
    x0 = torch.from_numpy(np.ascontiguousarray(x0[sl])).to(device).long().flatten(1)
    y0 = torch.from_numpy(np.ascontiguousarray(y0[sl])).to(device).long().flatten(1)
    wx = torch.from_numpy(np.ascontiguousarray(wx[sl])).to(device).double().flatten(1)
    wy = torch.from_numpy(np.ascontiguousarray(wy[sl])).to(device).double().flatten(1)
    taps = []
    for dy, dx, w in ((0, 0, wy * wx), (0, 1, wy * (1.0 - wx)), (1, 0, (1.0 - wy) * wx), (1, 1, (1.0 - wy) * (1.0 - wx))):
        yy, xx = y0 + dy, x0 + dx
        ok = (xx >= 0) & (xx <= Wk - 1) & (yy >= 0) & (yy <= Hk - 1)
        idx = yy.clamp(0, Hk - 1) * Wk + xx.clamp(0, Wk - 1)
        taps.append((idx, torch.where(ok, w, torch.zeros_like(w)).unsqueeze(1), ok))
    return taps, wx, wy


def _f64(t, frames, device):
    return None if t is None else t[frames.start:frames.stop].to(device).double().contiguous()


def _keys(key, key_index, frames, device):
    if key_index is None:
        k = key[frames.start:frames.stop]
    else:
        ki = torch.as_tensor(np.asarray(key_index.cpu() if isinstance(key_index, torch.Tensor) else key_index))
        k = key[ki[frames.start:frames.stop].to(key.device).long()]
    return k.to(device).double().contiguous()


def _chunks(frames):
    for n0 in range(frames.start, frames.stop, CHUNK):
        yield range(n0, min(n0 + CHUNK, frames.stop))


def _frames(frames, n):
    if frames is None:
        return range(0, n)
    return range(*frames.indices(n)) if isinstance(frames, slice) else frames


def _blend_weights(mode, logits, emb_warp, emb_cur, fr, device, HW):
    """(ww, wc) float64 (n, 1, HW) and, in cosine mode, the cosine-error factor w1 w2 (else None)."""
    n = len(fr)
    one = torch.ones((n, 1, HW), dtype=torch.float64, device=device)
    if mode == O.W_NONE:
        return one, 0 * one, None
    if mode == O.W_ADD:
        return one, one, None
    if mode == O.W_MEAN:
        return 0.5 * one, 0.5 * one, None
    if mode == O.W_LOGITS:
        lg = _f64(logits, fr, device).reshape(n, 2, HW)
        lw, lc = lg[:, 0:1], lg[:, 1:2]
    elif mode == O.W_COSINE:
        ew, ec = _f64(emb_warp, fr, device), _f64(emb_cur, fr, device)
        nw = ew / torch.sqrt((ew * ew).sum(1, keepdim=True) + O.L2NORM_EPS)
        nc = ec / torch.sqrt((ec * ec).sum(1, keepdim=True) + O.L2NORM_EPS)
        lw = (nw * nc).sum(1, keepdim=True).reshape(n, 1, HW)
        lc = (nc * nc).sum(1, keepdim=True).reshape(n, 1, HW)
    else:
        raise ValueError(mode)
    ww = 1.0 / (1.0 + torch.exp(lc - lw))
    wc = 1.0 / (1.0 + torch.exp(lw - lc))
    return ww, wc, (ww * wc if mode == O.W_COSINE else None)


# ----------------------------------------------------------------------------------------------------------------
# forward
# ----------------------------------------------------------------------------------------------------------------
def forward(key, co, *, cur=None, scale_map=None, res=None, rnet_w=None, rnet_b=None, mode="none", logits=None,
            emb_warp=None, emb_cur=None, bypass=None, key_index=None, frames=None, device=None):
    """(ref, mag) float64 (n, C, H, W) for ``frames`` (a range or slice of the batch; default all) of
    ``warp_scale_aggregate``.  Feature tensors are torch tensors in logical NCHW (a permuted view of a channels-last
    tensor will do), any float dtype, on any device; ``co`` = ``coords(...)`` for the whole batch.  The arithmetic
    runs on ``device`` (default: the key's)."""
    mode = _mode(mode)
    device = key.device if device is None else torch.device(device)
    N, H, W = co[0].shape
    Hk, Wk = key.shape[2], key.shape[3]
    HW = H * W
    C = key.shape[1]
    fr = _frames(frames, N)
    refs, mags = [], []
    for ch in _chunks(fr):
        n = len(ch)
        taps, _, _ = _taps(co, ch, Hk, Wk, device)
        kv = _keys(key, key_index, ch, device).reshape(n, C, Hk * Wk)
        src = torch.zeros((n, C, HW), dtype=torch.float64, device=device)
        msrc = torch.zeros_like(src)
        for idx, w, _ok in taps:
            v = kv.gather(2, idx.unsqueeze(1).expand(n, C, HW))
            src += w * v
            msrc += w * v.abs()
        del kv
        if scale_map is not None:
            s = _f64(scale_map, ch, device).reshape(n, C, HW)
            src *= s
            msrc *= s.abs()
        if res is not None:
            rw = rnet_w.to(device).double().reshape(C, 3)
            rb = rnet_b.to(device).double().reshape(1, C, 1)
            r = _f64(res, ch, device).reshape(n, 3, HW)
            src += torch.einsum("cj,njp->ncp", rw, r) + rb
            msrc += torch.einsum("cj,njp->ncp", rw.abs(), r.abs()) + rb.abs()
        ww, wc, cosf = _blend_weights(mode, logits, emb_warp, emb_cur, ch, device, HW)
        if mode == O.W_NONE:
            ref, mag = src, msrc
        else:
            c = _f64(cur, ch, device).reshape(n, C, HW)
            ref = ww * src + wc * c
            mag = ww * msrc + wc * c.abs()
            if cosf is not None:
                E = emb_warp.shape[1]
                mag = mag + (2.0 * (E + 2) / K) * cosf * (src - c).abs()
            if bypass is not None:
                live = torch.as_tensor(np.asarray(bypass.cpu() if isinstance(bypass, torch.Tensor) else bypass)
                                       )[ch.start:ch.stop].to(device) == 0
                live = live.reshape(n, 1, 1)
                ref = torch.where(live, ref, c)
                mag = torch.where(live, mag, torch.zeros_like(mag))
        refs.append(ref.reshape(n, C, H, W))
        mags.append(mag.reshape(n, C, H, W))
    return torch.cat(refs), torch.cat(mags)


# ----------------------------------------------------------------------------------------------------------------
# backward
# ----------------------------------------------------------------------------------------------------------------
def backward(out_grad, key, co, *, cur=None, scale_map=None, mode="none", logits=None, bypass=None, frames=None,
             device=None, want=("key", "flow", "scale", "cur", "logits")):
    """Gradients of ``warp_scale_aggregate`` (modes none/add/mean/logits, optional scale map and bypass) w.r.t. the
    inputs in ``want`` that exist, for ``frames``: {name: (ref, mag, n_addends)}, float64, ``n_addends`` an int or an
    integer tensor of the gradient's shape.  The chain rule is the one of ``lsfa_oracle.warp_scale_aggregate_backward``
    on the same float32 coordinates; ``mode='none'`` without scale map is ``warp_backward`` (grad_key, grad_flow).
    grad_key is an ``index_add_`` in float64 over the taps of every output pixel of the same frame."""
    mode = _mode(mode)
    if mode == O.W_COSINE:
        raise ValueError("the backward has no cosine mode")
    device = out_grad.device if device is None else torch.device(device)
    N, H, W = co[0].shape
    Hk, Wk = key.shape[2], key.shape[3]
    HW, C = H * W, key.shape[1]
    fr = _frames(frames, N)
    outs = {k: ([], [], []) for k in want}
    for ch in _chunks(fr):
        n = len(ch)
        taps, wx, wy = _taps(co, ch, Hk, Wk, device)
        g = _f64(out_grad, ch, device).reshape(n, C, HW)
        kv = _keys(key, None, ch, device).reshape(n, C, Hk * Wk)
        vals = [torch.where(ok.unsqueeze(1), kv.gather(2, idx.unsqueeze(1).expand(n, C, HW)), torch.zeros((), dtype=torch.float64, device=device))
                for idx, _w, ok in taps]
        wp = sum(w * v for (_i, w, _o), v in zip(taps, vals))
        mwp = sum(w * v.abs() for (_i, w, _o), v in zip(taps, vals))
        s = _f64(scale_map, ch, device).reshape(n, C, HW) if scale_map is not None else None
        src0, msrc0 = (wp * s, mwp * s.abs()) if s is not None else (wp, mwp)
        ww, wc, _ = _blend_weights(mode, logits, None, None, ch, device, HW)
        live = torch.ones((n, 1, 1), dtype=torch.float64, device=device)
        if bypass is not None:
            b = torch.as_tensor(np.asarray(bypass.cpu() if isinstance(bypass, torch.Tensor) else bypass))[ch.start:ch.stop]
            live = (b.to(device) == 0).double().reshape(n, 1, 1)
        gs0 = ww * g * live                                     # d/d(src0)
        gw = gs0 * s if s is not None else gs0                  # d/d(warp)
        res = {}
        if "cur" in want and cur is not None and mode != O.W_NONE:
            r = wc * g * live + g * (1.0 - live)
            res["cur"] = (r, (wc * g * live).abs(), 1)          # bypass frames: cur's gradient is out_grad itself
        if "scale" in want and s is not None:
            res["scale"] = (gs0 * wp, (gs0 * mwp).abs(), 4)
        if "key" in want:
            gk = torch.zeros((n, C, Hk * Wk), dtype=torch.float64, device=device)
            mk = torch.zeros_like(gk)
            cnt = torch.zeros((n, 1, Hk * Wk), dtype=torch.float64, device=device)
            for idx, w, ok in taps:
                for i in range(n):
                    gk[i].index_add_(1, idx[i], gw[i] * w[i])
                    mk[i].index_add_(1, idx[i], (gw[i] * w[i]).abs())
                    cnt[i].index_add_(1, idx[i], ok[i].double().unsqueeze(0))
            res["key"] = (gk, mk, cnt.expand(n, C, Hk * Wk))
        if "flow" in want:
            v00, v01, v10, v11 = vals
            t = v00 - v01 - v10 + v11
            wxb, wyb = wx.unsqueeze(1), wy.unsqueeze(1)
            gy = -(gw * (v01 - v11 + t * wxb)).sum(1)
            gx = -(gw * (v10 - v11 + t * wyb)).sum(1)
            ay, ax = v01.abs() + v11.abs(), v10.abs() + v11.abs()
            at = v00.abs() + v01.abs() + v10.abs() + v11.abs()
            my = (gw.abs() * (ay + at * wxb)).sum(1)
            mx = (gw.abs() * (ax + at * wyb)).sum(1)
            half_w, half_h = float(np.float32((W - 1) / 2.0)), float(np.float32((H - 1) / 2.0))
            fy, fx = ((Hk - 1) / 2.0) / half_h, ((Wk - 1) / 2.0) / half_w
            res["flow"] = (torch.stack([gx * fx, gy * fy], 1), torch.stack([mx * abs(fx), my * abs(fy)], 1), 6 * C)
        if "logits" in want and mode == O.W_LOGITS:
            c = _f64(cur, ch, device).reshape(n, C, HW)
            t1 = (g * src0).sum(1, keepdim=True)
            t2 = (g * c).sum(1, keepdim=True)
            m = ww * wc * live * ((g.abs() * msrc0).sum(1, keepdim=True) + (g * c).abs().sum(1, keepdim=True))
            d = ww * wc * (t1 - t2) * live
            res["logits"] = (torch.cat([d, -d], 1), torch.cat([m, m], 1), 5 * C)
        for k, (r, m, na) in res.items():
            shp = (n, -1, Hk, Wk) if k == "key" else (n, -1, H, W)
            outs[k][0].append(r.reshape(shp))
            outs[k][1].append(m.reshape(shp))
            outs[k][2].append(na.reshape(shp) if isinstance(na, torch.Tensor) else na)
    done = {}
    for k, (rs, ms, ns) in outs.items():
        if rs:
            done[k] = (torch.cat(rs), torch.cat(ms), torch.cat(ns) if isinstance(ns[0], torch.Tensor) else ns[0])
    return done


# ----------------------------------------------------------------------------------------------------------------
# the gate
# ----------------------------------------------------------------------------------------------------------------
def _frame_ranges(frames):
    out, start, prev = [], None, None
    for f in frames:
        if start is None:
            start = prev = f
        elif f == prev + 1:
            prev = f
        else:
            out.append((start, prev))
            start = prev = f
    if start is not None:
        out.append((start, prev))
    return ", ".join(str(a) if a == b else "%d-%d" % (a, b) for a, b in out)


def tolerance(ref, mag, out="f32", K=K, n_addends=None):
    """Per-element bound of the gate (0 where mag == 0: those elements must be exact)."""
    if n_addends is not None:
        na = n_addends.to(mag.device).double() if isinstance(n_addends, torch.Tensor) else float(n_addends)
        tol = (na + 8.0) * U * mag
    elif out == "f32":
        tol = K * U * mag
    elif out == "bf16":
        tol = 2.0 ** -8 * ref.abs() + 2.0 * K * U * mag
    else:
        raise ValueError("out must be 'f32' or 'bf16'")
    return torch.where(mag == 0, torch.zeros_like(tol), tol)


def check(got, ref, mag, out="f32", K=K, n_addends=None, what="", frame0=0):
    """Assert ``got`` (any dtype/device, ref's logical shape) is within the gate of ``ref``; return max err/tol.
    ``frame0``: index of ref's first frame in the batch, for the report."""
    ref = torch.as_tensor(ref)
    mag = torch.as_tensor(mag).to(ref.device)
    got = torch.as_tensor(got).to(ref.device).double()
    if tuple(got.shape) != tuple(ref.shape):
        raise AssertionError("%s: shape %s, reference %s" % (what, tuple(got.shape), tuple(ref.shape)))
    tol = tolerance(ref, mag, out, K, n_addends)
    err = (got - ref).abs()
    ok = err <= tol                                      # NaN fails
    ratio = torch.where(ok, err / torch.where(tol > 0, tol, torch.ones_like(tol)), torch.full_like(err, float("inf")))
    ratio = torch.where(ok & (tol == 0), torch.zeros_like(ratio), ratio)
    if not bool(ok.all()):
        bad = ~ok
        nbad = int(bad.sum())
        score = torch.where(bad, torch.nan_to_num(err - tol, nan=float("inf")), torch.full_like(err, -1.0))
        i = tuple(int(p) for p in np.unravel_index(int(score.flatten().argmax()), tuple(ref.shape)))
        pos = (i[0] + frame0,) + i[1:]
        frames = (torch.nonzero(bad.flatten(1).any(1)).flatten() + frame0).tolist()
        raise AssertionError(
            "%s: %d/%d elements outside the %s gate; worst at (frame, c, y, x) = %s: got %.9g ref %.9g tol %.3g "
            "(mag %.3g); frames with failures: %s"
            % (what, nbad, ref.numel(), "reduction" if n_addends is not None else out, pos, float(got[i]), float(ref[i]),
               float(tol[i]), float(mag[i]), _frame_ranges(frames)))
    return float(ratio.max()) if ratio.numel() else 0.0
