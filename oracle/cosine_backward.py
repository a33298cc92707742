"""Backward of Fgfa_net's cosine weights (SYM:111-116,132-148): the float64 chain rule and the float64 reference with its
per-element gate.

THIS IS TEST INFRASTRUCTURE, NOT PRODUCT CODE (like ``lsfa_oracle`` and ``ref64``, whose helpers it uses): only
``tests/`` and ``tools/`` import it.

Logits: l1 = <l2n(emb_warp), l2n(emb_cur)>, l2 = <l2n(emb_cur), l2n(emb_cur)>, l2n(x) = x / sqrt(sum_c x^2 + eps)
(``lsfa_oracle.cosine_weight``).

The gate of ``ref64_backward``, with u = 2^-24 the unit roundoff of float32.  With a = emb_warp[n,:,p],
b = emb_cur[n,:,p], na = sqrt(sum a^2 + eps), nb = sqrt(sum b^2 + eps), l1 = <a,b>/(na nb), l2 = sum b^2/nb^2 and
g1, g2 = d/d(l1), d/d(l2), the gradients are ``alpha b + beta a`` and ``alpha a + gamma b`` with alpha = g1/(na nb),
beta = -g1 l1/na^2, gamma = (-g1 l1 + 2 g2 (1 - l2))/nb^2.  The kernel forms the three sums in float32 over E channels:
each is within ``E u`` times the sum of its absolute terms.  That moves na and nb by at most ``E u / 2`` relative, hence
alpha, beta and each part of gamma by at most ``(E + 4) u`` relative (the extra terms: the divisions, products and the
final fma, at most 8 roundings); l1 moves by at most ``E u sum_k|a_k b_k| / (na nb)`` through <a,b>, which moves
beta a_c by ``|g1| |a_c| sum_k|a_k b_k| / (na^3 nb)`` times E u.  l2 moves by at most ``(E + 2) u l2`` and enters only
as (1 - l2), which float32 cannot resolve below that: the term ``2 |g2| |b_c| (l2 + |1 - l2|) / nb^2`` covers it.  So
the gate is ``ref64.check`` in its reduction form with n = E + 8 (``(E + 16) u mag``) and
    mag(grad_emb_warp) = |alpha b| + |beta a| + |g1| |a| sum|ab| / (na^3 nb)
    mag(grad_emb_cur)  = |alpha a| + |g1 l1 b| / nb^2 + |g1| |b| sum|ab| / (na nb^3) + 2 |g2| |b| (l2 + |1 - l2|) / nb^2.
In the fused operator g1 = -g2 is itself a C-term sum of the tail: an absolute error bound ``g_err`` of g1 adds
``g_err`` times the sensitivity of each gradient to g1 and g2 (the sum of the absolute values of d grad / d g1 and
d grad / d g2) to the allowed error; ``ref64_backward`` folds it into mag.  An element with mag == 0 (both embeddings
zero at that pixel, or g = 0) must be an exact 0.
"""
from __future__ import annotations

import numpy as np
import torch

from oracle import lsfa_oracle as O
from oracle import ref64 as R

F32, F64 = np.float32, np.float64


def cosine_logits_backward(emb_warp, emb_cur, grad_logits):
    """d/d(emb_warp), d/d(emb_cur) of [cosine_weight(emb_warp, emb_cur), cosine_weight(emb_cur, emb_cur)] given
    d/d(logits) (N,2,H,W): float64 chain rule through l2norm_channel (x^ = x / sqrt(sum x^2 + eps)), the product and the
    channel sum: d x = (d x^ - x^ <d x^, x^>) / sqrt(sum x^2 + eps).  float32 results."""
    a, b = np.asarray(emb_warp, F64), np.asarray(emb_cur, F64)
    g = np.asarray(grad_logits, F64)
    g1, g2 = g[:, 0:1], g[:, 1:2]
    na = np.sqrt(np.sum(a * a, axis=1, keepdims=True) + O.L2NORM_EPS)
    nb = np.sqrt(np.sum(b * b, axis=1, keepdims=True) + O.L2NORM_EPS)
    ah, bh = a / na, b / nb
    gah = g1 * bh                                       # d l1 / d a^ = b^
    gbh = g1 * ah + 2.0 * g2 * bh                       # d l1 / d b^ = a^, d l2 / d b^ = 2 b^
    ga = (gah - ah * np.sum(gah * ah, axis=1, keepdims=True)) / na
    gb = (gbh - bh * np.sum(gbh * bh, axis=1, keepdims=True)) / nb
    return ga.astype(F32), gb.astype(F32)


def warp_scale_aggregate_backward(out_grad, key, flow, emb_warp, emb_cur, **kw):
    """Gradients of ``lsfa_oracle.warp_scale_aggregate(..., weight_mode=W_COSINE)``: the LOGITS-mode chain rule of
    ``lsfa_oracle.warp_scale_aggregate_backward`` on the oracle's cosine logits, then ``cosine_logits_backward`` of
    its d/d(logits).  Returns the same dict with 'emb_warp' and 'emb_cur' in place of 'logits'."""
    logits = np.concatenate([O.cosine_weight(emb_warp, emb_cur), O.cosine_weight(emb_cur, emb_cur)], axis=1)
    out = O.warp_scale_aggregate_backward(out_grad, key, flow, weight_mode=O.W_LOGITS, logits=logits, **kw)
    out["emb_warp"], out["emb_cur"] = cosine_logits_backward(emb_warp, emb_cur, out.pop("logits"))
    return out


def ref64_backward(emb_warp, emb_cur, grad_logits, g_err=None, frames=None, device=None):
    """Float64 reference of the gradients w.r.t. emb_warp and emb_cur for ``frames``: {name: (ref, mag, n_addends)}
    for ``ref64.check``, the gate of the module docstring.  Torch tensors on any device; ``grad_logits`` (N,2,H,W);
    ``g_err`` (N,1,H,W) or None: an absolute error bound of the float32 d/d(l1) = -d/d(l2) that the gradients were
    computed from (fused operator)."""
    device = emb_warp.device if device is None else torch.device(device)
    N, E = emb_warp.shape[0], emb_warp.shape[1]
    fr = R._frames(frames, N)
    outs = {"emb_warp": ([], []), "emb_cur": ([], [])}
    for ch in R._chunks(fr):
        a, b = R._f64(emb_warp, ch, device), R._f64(emb_cur, ch, device)
        g = R._f64(grad_logits, ch, device)
        g1, g2 = g[:, 0:1], g[:, 1:2]
        saa, sbb = (a * a).sum(1, keepdim=True), (b * b).sum(1, keepdim=True)
        na, nb = torch.sqrt(saa + O.L2NORM_EPS), torch.sqrt(sbb + O.L2NORM_EPS)
        l1, l2 = (a * b).sum(1, keepdim=True) / (na * nb), sbb / (nb * nb)
        sab = (a * b).abs().sum(1, keepdim=True)
        al, be = g1 / (na * nb), -g1 * l1 / (na * na)
        ga1, ga2 = -g1 * l1 / (nb * nb), 2.0 * g2 * (1.0 - l2) / (nb * nb)
        mw = (al * b).abs() + (be * a).abs() + g1.abs() * a.abs() * sab / (na ** 3 * nb)
        mc = ((al * a).abs() + (ga1 * b).abs() + g1.abs() * b.abs() * sab / (na * nb ** 3)
              + 2.0 * g2.abs() * b.abs() * (l2 + (1.0 - l2).abs()) / (nb * nb))
        if g_err is not None:
            ge = R._f64(g_err, ch, device)
            scale = ge / ((E + 16) * R.U)
            mw = mw + scale * (b.abs() / (na * nb) + (l1 * a).abs() / (na * na))
            mc = mc + scale * (a.abs() / (na * nb) + (l1 * b).abs() / (nb * nb) + 2.0 * b.abs() * (1.0 - l2).abs() / (nb * nb))
        for k, r, m in (("emb_warp", al * b + be * a, mw), ("emb_cur", al * a + (ga1 + ga2) * b, mc)):
            outs[k][0].append(r)
            outs[k][1].append(m)
    return {k: (torch.cat(r), torch.cat(m), E + 8) for k, (r, m) in outs.items()}
