#!/usr/bin/env python
"""Mint tests/golden/fused_backward_cosine_small.npz: gradients of Fgfa_net's cosine weights (SYM:111-116,132-148)
    l1 = <l2n(emb_warp), l2n(emb_cur)>, l2 = <l2n(emb_cur), l2n(emb_cur)>,  l2n(x) = x / sqrt(sum_c x^2 + 1e-10)
on their own ("cos_*": d/d(emb_warp), d/d(emb_cur) from a given d/d(logits)) and inside the fused operator in COSINE
mode ("fused_*": out = w1*(grid_sample(key, grid(flow)) * scale) + w2*cur, (w1,w2) = softmax(l1, l2), bypass -> cur),
from an implementation independent of this repo's oracle: torch autograd in float64 on the CPU.  The embeddings hold
an all-zero pixel (the eps path) and a pixel of norm ~1e-5 (where eps and the d l2 term matter)."""
import os

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def l2n(x):
    return x / torch.sqrt((x * x).sum(1, keepdim=True) + 1e-10)


def logits_of(ew, ec):
    return torch.cat([(l2n(ew) * l2n(ec)).sum(1, keepdim=True), (l2n(ec) * l2n(ec)).sum(1, keepdim=True)], 1)


def main():
    rng = np.random.default_rng(20261022)
    f = lambda *s: rng.standard_normal(s)  # noqa: E731
    out = {}

    def embeddings(N, E, H, W):
        ew, ec = f(N, E, H, W), f(N, E, H, W)
        ew[:, :, 0, 0] = 0.0
        ec[:, :, 0, 0] = 0.0
        ec[:, :, 1, 2] *= 1e-5 / np.sqrt(E)
        ew[:, :, 1, 2] *= 1e-5 / np.sqrt(E)
        return ew.astype(np.float32).astype(np.float64), ec.astype(np.float32).astype(np.float64)

    # the op on its own
    N, E, H, W = 2, 6, 5, 7
    ew, ec = embeddings(N, E, H, W)
    gl = f(N, 2, H, W).astype(np.float32).astype(np.float64)
    t = {k: torch.tensor(v, requires_grad=True) for k, v in dict(ew=ew, ec=ec).items()}
    lg = logits_of(t["ew"], t["ec"])
    lg.backward(torch.tensor(gl))
    out.update(cos_emb_warp=ew.astype(np.float32), cos_emb_cur=ec.astype(np.float32), cos_grad_logits=gl.astype(np.float32),
               cos_logits=lg.detach().numpy().astype(np.float32),
               cos_grad_emb_warp=t["ew"].grad.numpy().astype(np.float32), cos_grad_emb_cur=t["ec"].grad.numpy().astype(np.float32))

    # the fused operator in COSINE mode
    N, C, E, H, W = 3, 5, 6, 9, 11
    key, cur, sm = np.maximum(f(N, C, H, W), 0), np.maximum(f(N, C, H, W), 0), 1 + 0.1 * f(N, C, H, W)
    flow = 1.7 * f(N, 2, H, W)
    flow[0, :, :2] = 30.0
    ew, ec = embeddings(N, E, H, W)
    og = f(N, C, H, W)
    byp = np.array([0, 1, 0], np.uint8)
    inputs = {k: v.astype(np.float32) for k, v in dict(key=key, cur=cur, scale=sm, flow=flow, emb_warp=ew, emb_cur=ec,
                                                       out_grad=og).items()}
    t = {k: torch.tensor(v, dtype=torch.float64, requires_grad=True) for k, v in inputs.items() if k != "out_grad"}
    ys, xs = torch.meshgrid(torch.arange(H, dtype=torch.float64), torch.arange(W, dtype=torch.float64), indexing="ij")
    gx = (t["flow"][:, 0] + xs) / ((W - 1) / 2.0) - 1
    gy = (t["flow"][:, 1] + ys) / ((H - 1) / 2.0) - 1
    wp = torch.nn.functional.grid_sample(t["key"], torch.stack([gx, gy], -1), mode="bilinear", padding_mode="zeros", align_corners=True)
    w = torch.softmax(logits_of(t["emb_warp"], t["emb_cur"]), dim=1)
    o = w[:, 0:1] * (wp * t["scale"]) + w[:, 1:2] * t["cur"]
    live = torch.tensor((byp == 0).astype(np.float64)).reshape(N, 1, 1, 1)
    o = live * o + (1 - live) * t["cur"]
    o.backward(torch.tensor(inputs["out_grad"], dtype=torch.float64))
    for k, v in t.items():
        out["fused_grad_%s" % k] = v.grad.numpy().astype(np.float32)
    out["fused_out"] = o.detach().numpy().astype(np.float32)
    for k, v in inputs.items():
        out["fused_%s" % k] = v
    out["fused_bypass"] = byp
    dst = os.path.join(ROOT, "tests", "golden", "fused_backward_cosine_small.npz")
    np.savez_compressed(dst, **out)
    print("wrote", dst, os.path.getsize(dst))


if __name__ == "__main__":
    main()
