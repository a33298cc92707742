#!/usr/bin/env python
"""Kernel-level numbers for every BASELINE.json config and variant (device-resident inputs,
generated on the device; CUDA events; one JSON line per row).  Not the driver's bench - see
bench.py for the contract line.  Usage: python tools/bench_configs.py [--quick]"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from lsfa_b200 import ops  # noqa: E402


def peak():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        return 6650.0


def tflops_peak():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops_sustained"])
    except Exception:
        return 1400.0


def time_ms(fn, warmup=5, steps=30):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def synth(N, C, H, W, mvh, mvw, dev, max_px=32, E=0):
    g = torch.Generator(device=dev).manual_seed(0)
    d = {
        "key": torch.randn((N, C, H, W), device=dev, generator=g).clamp_(min=0),
        "cur": torch.randn((N, C, H, W), device=dev, generator=g).clamp_(min=0),
        "scale_map": 1 + 0.1 * torch.randn((N, C, H, W), device=dev, generator=g),
        "logits": torch.randn((N, 2, H, W), device=dev, generator=g),
    }
    bh, bw = -(-mvh // 16), -(-mvw // 16)
    blk = torch.randint(-max_px, max_px + 1, (N, bh, bw, 2), device=dev, generator=g, dtype=torch.int32)
    blk[torch.rand((N, bh, bw), device=dev, generator=g) < 0.5] = 0
    d["mv"] = blk.repeat_interleave(16, 1).repeat_interleave(16, 2)[:, :mvh, :mvw].contiguous()
    d["res"] = torch.randn((N, 3, H, W), device=dev, generator=g) * 30
    d["rnet_w"] = 0.01 * torch.randn((C, 3), device=dev, generator=g)
    d["rnet_b"] = torch.zeros((C,), device=dev)
    if E:
        d["emb_warp"] = torch.randn((N, E, H, W), device=dev, generator=g)
        d["emb_cur"] = torch.randn((N, E, H, W), device=dev, generator=g)
    return d


def row(name, frames, alg_bytes_per_frame, ms, pk, note=""):
    gbs = frames * alg_bytes_per_frame / (ms / 1e3) / 1e9      # 0 for rows that are not byte-bound (library GEMMs)
    r = {"config": name, "frames": frames, "ms_per_step": round(ms, 4), "frames_per_s": round(frames / (ms / 1e3), 1),
         "alg_bytes_per_frame": alg_bytes_per_frame, "achieved_gbs": round(gbs, 1), "frac_of_measured_peak": round(gbs / pk, 4),
         "frac_of_8TBs": round(gbs / 8000.0, 4), "note": note}
    print(json.dumps(r), flush=True)
    return r


def backward_rows(dev, pk, quick):
    """Backward of GridGenerator(warp)+BilinearSampler (8f rank 4) at the headline shape.  Algorithmic bytes per
    frame: out_grad + grad_key (+ key when d/d(flow) is wanted) = 2F / 3F, + 8*HW flow + 8*HW grad_flow."""
    C, H, W = 1024, 38, 63
    HW, F4 = H * W, C * H * W * 4
    N = 16 if quick else 64
    d = synth(N, C, H, W, 600, 1000, dev, max_px=96)
    flow = ops.mv_pool(d["mv"])
    og = torch.randn_like(d["key"])
    gk = torch.empty_like(d["key"])
    gf = torch.empty_like(flow)
    ws = torch.empty(ops.A.load().lsfa_bilinear_sampler_backward_workspace_bytes(N, C, H, W, H, W), dtype=torch.uint8, device=dev)
    for kern in ("gather", "scatter"):
        st = 10 if kern == "gather" else 3
        row("bwd warp: grad_key + grad_flow, fp32 NCHW (%s)" % kern, N, 3 * F4 + 16 * HW,
            time_ms(lambda: ops.warp_backward(d["key"], flow, og, grad_key=gk, grad_flow=gf, workspace=ws, kernel=kern), 2, st), pk)
        row("bwd warp: grad_key only (SYM:320-321), fp32 NCHW (%s)" % kern, N, 2 * F4 + 8 * HW,
            time_ms(lambda: ops.warp_backward(d["key"], flow, og, grad_key=gk, req_flow="null", workspace=ws, kernel=kern), 2, st), pk)
    # backward of the fused operator (SYM:306-338): tails (agg_tail_backward_kernel) + the a7/a8 gather on its d/d(warp)
    lg = d["logits"]
    for nm, kw, alg in (("V2 (x scale, logits blend): key, flow, scale, cur, logits", dict(cur=d["cur"], scale_map=d["scale_map"], weight_mode="logits", logits=lg), 10 * F4),
                        ("V1 (+ rnet(res) + cur): key, flow, cur, res, rnet", dict(cur=d["cur"], res=d["res"], rnet_w=d["rnet_w"], rnet_b=d["rnet_b"], weight_mode="add"), 7 * F4)):
        row("bwd fused " + nm, N, alg,
            time_ms(lambda: ops.warp_scale_aggregate_backward(og, d["key"], flow, flow_kind="flow", **kw), 2, 5), pk,
            "bytes: every stream once incl. the d/d(warp) intermediate")
    # smooth motion (every block moves by the same sub-cell vector): short, even lists
    flow2 = torch.full_like(flow, 0.37)
    row("bwd warp: grad_key + grad_flow, uniform flow (gather)", N, 3 * F4 + 16 * HW,
        time_ms(lambda: ops.warp_backward(d["key"], flow2, og, grad_key=gk, grad_flow=gf, workspace=ws, kernel="gather"), 2, 10), pk)


def single_frame_rows(dev, pk):
    """BASELINE configs[0]: ONE non-key frame (1024x38x63 fp32 + a 600x1000 MV field): latency of the two drop-in
    operators and of the fused op, eager launches and replayed from a CUDA graph."""
    C, H, W = 1024, 38, 63
    HW, F4 = H * W, C * H * W * 4
    d = synth(1, C, H, W, 600, 1000, dev)
    s = torch.cuda.current_stream().cuda_stream
    flow = ops.mv_pool(d["mv"])
    grid = torch.empty_like(flow)
    out = torch.empty_like(d["key"])
    row("cfg1 single frame: mv_pool + GridGenerator + BilinearSampler (3 ops)", 1, 2 * F4 + 32 * HW,
        time_ms(lambda: ops.BilinearSampler(d["key"], ops.GridGenerator(ops.mv_pool(d["mv"]), out=grid), out=out), 10, 200), pk,
        "latency, eager")
    p0 = ops.PreparedAggregate(d["key"], d["mv"], flow_kind="raw")
    row("cfg1 single frame: fused warp, raw MV", 1, 2 * F4 + 32 * HW, time_ms(lambda: p0.run(s), 10, 200), pk, "latency, eager")
    p2 = ops.PreparedAggregate(d["key"], d["mv"], flow_kind="raw", cur=d["cur"], scale_map=d["scale_map"],
                               weight_mode="logits", logits=d["logits"])
    row("single frame: fused V2", 1, 4 * F4 + 40 * HW, time_ms(lambda: p2.run(s), 10, 200), pk, "latency, eager")
    p0s = ops.PreparedAggregate(d["key"], d["mv"], flow_kind="raw", workspace=False)
    row("cfg1 single frame: fused warp, raw MV, no scratch (1 launch)", 1, 2 * F4 + 32 * HW, time_ms(lambda: p0s.run(s), 10, 200), pk, "latency, eager")
    p2s = ops.PreparedAggregate(d["key"], d["mv"], flow_kind="raw", cur=d["cur"], scale_map=d["scale_map"],
                                weight_mode="logits", logits=d["logits"], workspace=False)
    row("single frame: fused V2, no scratch (1 launch)", 1, 4 * F4 + 40 * HW, time_ms(lambda: p2s.run(s), 10, 200), pk, "latency, eager")
    # flow / grid given (the drop-in BilinearSampler): records are two coalesced loads per pixel
    gridt = ops.GridGenerator(flow)
    pf = ops.PreparedAggregate(d["key"], flow, flow_kind="flow")
    row("single frame: fused warp, flow given (cooperative records)", 1, 2 * F4 + 8 * HW, time_ms(lambda: pf.run(s), 10, 200), pk, "latency, eager")
    pfs = ops.PreparedAggregate(d["key"], flow, flow_kind="flow", workspace=False)
    row("single frame: fused warp, flow given, records built inside every CTA (1 plain launch)", 1, 2 * F4 + 8 * HW,
        time_ms(lambda: pfs.run(s), 10, 200), pk, "latency, eager")
    pg = ops.PreparedAggregate(d["key"], gridt, flow_kind="grid")
    pgs = ops.PreparedAggregate(d["key"], gridt, flow_kind="grid", workspace=False)

    class _Chain:      # the three drop-in operators back to back (for the graph rows)
        @staticmethod
        def run(st):
            with torch.cuda.stream(torch.cuda.ExternalStream(st)):
                ops.BilinearSampler(d["key"], ops.GridGenerator(ops.mv_pool(d["mv"]), out=grid), out=out)
    for name, p, b in (("cfg1 single frame: fused warp, raw MV", p0, 2 * F4 + 32 * HW), ("single frame: fused V2", p2, 4 * F4 + 40 * HW),
                       ("single frame: fused V2, no scratch", p2s, 4 * F4 + 40 * HW),
                       ("single frame: fused warp, flow given (cooperative records)", pf, 2 * F4 + 8 * HW),
                       ("single frame: fused warp, flow given, records inside every CTA", pfs, 2 * F4 + 8 * HW),
                       ("single frame: BilinearSampler alone, grid given (cooperative)", pg, 2 * F4 + 8 * HW),
                       ("single frame: BilinearSampler alone, grid given, records inside every CTA", pgs, 2 * F4 + 8 * HW),
                       ("cfg1 single frame: mv_pool + GridGenerator + BilinearSampler (3 ops)", _Chain, 2 * F4 + 32 * HW)):
        side = torch.cuda.Stream()
        with torch.cuda.stream(side):
            for _ in range(3):
                p.run(side.cuda_stream)
            side.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                for _ in range(20):
                    p.run(side.cuda_stream)
        torch.cuda.synchronize()
        row(name + " (CUDA graph of 20)", 1, b, time_ms(g.replay, 3, 20) / 20, pk, "latency per frame inside a graph")


def cosine_rows(dev, pk, Nc):
    C, H, W, E = 1024, 38, 63, 2048
    HW, F4 = H * W, C * H * W * 4
    d = synth(Nc, C, H, W, 600, 1000, dev)
    g = torch.Generator(device=dev).manual_seed(1)
    ew = torch.randn((Nc, E, H, W), device=dev, generator=g)
    ec = torch.randn((Nc, E, H, W), device=dev, generator=g)
    s = torch.cuda.current_stream().cuda_stream
    p = ops.PreparedAggregate(d["key"], d["mv"], flow_kind="raw", cur=d["cur"], scale_map=d["scale_map"],
                              weight_mode="cosine", emb_warp=ew, emb_cur=ec)
    row("V3 cosine (Fgfa) fp32 NCHW batch %d: all-TMA cosine pre-pass + fused" % Nc, Nc, 4 * F4 + 40 * HW + 2 * E * HW * 4,
        time_ms(lambda: p.run(s)), pk, "%d launches" % p.launches)
    lg = torch.empty((Nc, 2, H, W), device=dev)
    row("cosine logits alone (LDG kernel, lsfa_cosine_logits)", Nc, 2 * E * HW * 4 + 8 * HW,
        time_ms(lambda: ops.cosine_logits(ew, ec, workspace=False)), pk, "ablation")
    wsc = torch.empty(ops.A.load().lsfa_cosine_logits_workspace_bytes(Nc, E, H, W, 0), dtype=torch.uint8, device=dev)
    row("cosine logits alone (all-TMA pre-pass, lsfa_cosine_logits_ws)", Nc, 2 * E * HW * 4 + 8 * HW,
        time_ms(lambda: ops.cosine_logits(ew, ec, workspace=wsc)), pk)


def cosine_backward_rows(dev):
    """Backward of the cosine logits, 64 frames x E = 2048 x 38x63, seeded inputs.  Each row is reported as a fraction of
    the device-to-device copy bandwidth measured here (read + write bytes of a 2 GiB copy), with the card's name and
    power limit read in the same run."""
    import subprocess
    name = torch.cuda.get_device_name(dev)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", str(dev.index or 0)],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                         # noqa: BLE001 - reported, not hidden
        power = "unknown (%s)" % e
    src = torch.empty(2 << 30, dtype=torch.uint8, device=dev)
    dst = torch.empty_like(src)
    copy_ms = time_ms(lambda: dst.copy_(src), 3, 20)
    copy_gbs = 2 * src.numel() / (copy_ms / 1e3) / 1e9
    del src, dst
    print(json.dumps({"config": "device copy (read + write)", "gpu": name, "power_limit": power, "achieved_gbs": round(copy_gbs, 1)}), flush=True)
    N, C, E, H, W = 64, 1024, 2048, 38, 63
    HW = H * W
    g = torch.Generator(device=dev).manual_seed(2)
    ew = torch.randn((N, E, H, W), device=dev, generator=g)
    ec = torch.randn((N, E, H, W), device=dev, generator=g)
    gl = torch.randn((N, 2, H, W), device=dev, generator=g)
    gw, gc = torch.empty_like(ew), torch.empty_like(ec)
    ws = torch.empty(ops.A.load().lsfa_cosine_logits_backward_workspace_bytes(N, E, H, W), dtype=torch.uint8, device=dev)

    def out(config, alg, ms, note=""):
        gbs = N * alg / (ms / 1e3) / 1e9
        print(json.dumps({"config": config, "frames": N, "ms_per_step": round(ms, 4), "alg_bytes_per_frame": alg, "achieved_gbs": round(gbs, 1),
                          "frac_of_copy": round(gbs / copy_gbs, 4), "gpu": name, "power_limit": power, "note": note}), flush=True)
    for kern in ("tma", "plain"):
        out("cosine logits backward (%s)" % kern, 6 * E * HW * 4 + 8 * HW,
            time_ms(lambda: ops.cosine_logits_backward(ew, ec, gl, grad_emb_warp=gw, grad_emb_cur=gc, workspace=ws, kernel=kern), 3, 20))
    out("cosine pre-pass alone (sums + logits, all-TMA)", 2 * E * HW * 4 + 8 * HW,
        time_ms(lambda: ops.cosine_logits(ew, ec), 3, 20), "the backward's sums pass; the gradient pass is the difference")
    d = synth(N, C, H, W, 600, 1000, dev)
    flow = ops.mv_pool(d["mv"])
    og = torch.randn_like(d["key"])
    F4 = C * HW * 4
    out("bwd fused V2 (x scale, logits blend): key, flow, scale, cur, logits", 10 * F4,
        time_ms(lambda: ops.warp_scale_aggregate_backward(og, d["key"], flow, flow_kind="flow", cur=d["cur"], scale_map=d["scale_map"],
                                                          weight_mode="logits", logits=d["logits"]), 2, 5))
    out("bwd fused V3 (x scale, cosine blend): key, flow, scale, cur, emb_warp, emb_cur", 10 * F4 + 6 * E * HW * 4,
        time_ms(lambda: ops.warp_scale_aggregate_backward(og, d["key"], flow, flow_kind="flow", cur=d["cur"], scale_map=d["scale_map"],
                                                          weight_mode="cosine", emb_warp=ew, emb_cur=ec), 2, 5),
        "bytes: the V2 row's + the standalone backward's; the logits are recomputed (another 2 E HW 4)")


def nhwc_rows(dev, pk, quick, only_tma=False):
    """Channels-last rows (configs 3 and 4 in bf16, fp32 NHWC, the shipped non-key path and the warp alone in bf16):
    the all-TMA kernel (default), its static batch stride (no claim counter) and the LDG/STG tile kernel."""
    s = torch.cuda.current_stream().cuda_stream
    C, H, W = 1024, 38, 63
    HW = H * W
    F4, F2 = C * HW * 4, C * HW * 2
    kinds = ((0, None, ""), (0, False, ", static batch stride"), (1, None, ", LDG/STG tile kernel"),
             (3, None, ", gather-by-bulk-copy kernel"), (5, None, ", window-resident kernel"))
    if only_tma:
        kinds = (kinds[0], kinds[3], kinds[3], kinds[3], kinds[4])
    N = 64
    d = synth(N, C, H, W, 600, 1000, dev)
    Nb = 128 if quick else 512
    reps = Nb // N
    nh = {k: ops.to_nhwc(d[k], torch.bfloat16).repeat(reps, 1, 1, 1) for k in ("key", "cur", "scale_map")}
    mvb = d["mv"].repeat(reps, 1, 1, 1)
    lgb = d["logits"].repeat(reps, 1, 1, 1)
    resb = d["res"].repeat(reps, 1, 1, 1)
    for fg, ws, nm in kinds:
        p = ops.PreparedAggregate(nh["key"], mvb, flow_kind="raw", cur=nh["cur"], scale_map=nh["scale_map"],
                                  weight_mode="logits", logits=lgb, layout="nhwc_bf16", force_generic=fg, workspace=ws)
        row("cfg3 V2 bf16 NHWC batch %d%s" % (Nb, nm), Nb, 4 * F2 + 40 * HW, time_ms(lambda: p.run(s), 3, 10), pk, "ablation" if nm else "")
    for fg, ws, nm in (kinds[0], kinds[2], kinds[3], kinds[4]):
        p = ops.PreparedAggregate(nh["key"], mvb, flow_kind="raw", cur=nh["cur"], res=resb, rnet_w=d["rnet_w"], rnet_b=d["rnet_b"],
                                  weight_mode="add", layout="nhwc_bf16", force_generic=fg, workspace=ws)
        row("V1 shipped non-key path bf16 NHWC batch %d%s" % (Nb, nm), Nb, 3 * F2 + 44 * HW + 16384, time_ms(lambda: p.run(s), 3, 10), pk,
            "ablation" if nm else "")
        p = ops.PreparedAggregate(nh["key"], mvb, flow_kind="raw", layout="nhwc_bf16", force_generic=fg, workspace=ws)
        row("V0 warp only bf16 NHWC batch %d%s" % (Nb, nm), Nb, 2 * F2 + 32 * HW, time_ms(lambda: p.run(s), 3, 10), pk, "ablation" if nm else "")
    if not only_tma:
        # config 3's ablation arm: the same computation op by op in the library a user would reach for (PyTorch eager,
        # bf16 channels-last): grid_sample + mul + softmax + 2 mul + add = 6+ kernels and every intermediate through HBM
        import torch.nn.functional as F
        nb = min(Nb, 128)
        kc, sc, cc = (nh[k][:nb].permute(0, 3, 1, 2) for k in ("key", "scale_map", "cur"))     # logical NCHW, channels-last
        flow = ops.mv_pool(mvb[:nb])
        grid = ops.GridGenerator(flow).permute(0, 2, 3, 1).contiguous().to(torch.bfloat16)     # (N,H,W,2) as grid_sample wants
        lg = lgb[:nb]

        def torch_chain():
            w = F.grid_sample(kc, grid, mode="bilinear", padding_mode="zeros", align_corners=True) * sc
            a = torch.softmax(lg, dim=1).to(torch.bfloat16)
            return a[:, 0:1] * w + a[:, 1:2] * cc

        row("cfg3 V2 bf16 NHWC batch %d, UNFUSED: PyTorch eager op by op (grid_sample, mul, softmax, blend)" % nb, nb,
            4 * F2 + 40 * HW, time_ms(torch_chain, 2, 5), pk, "ablation: algorithmic bytes of the fused op")
        del kc, sc, cc, flow, grid, lg
    del nh, p, mvb, lgb, resb
    torch.cuda.empty_cache()
    nf = {k: ops.to_nhwc(d[k], torch.float32) for k in ("key", "cur", "scale_map")}
    for fg, ws, nm in kinds:
        p = ops.PreparedAggregate(nf["key"], d["mv"], flow_kind="raw", cur=nf["cur"], scale_map=nf["scale_map"],
                                  weight_mode="logits", logits=d["logits"], layout="nhwc_f32", force_generic=fg, workspace=ws)
        row("V2 fp32 NHWC batch 64%s" % nm, N, 4 * F4 + 40 * HW, time_ms(lambda: p.run(s)), pk, "ablation" if nm else "")
    del nf, p, d
    torch.cuda.empty_cache()
    H4, W4 = 68, 120
    N4 = 32 if quick else 128
    d4 = synth(N4, C, H4, W4, 1080, 1920, dev, max_px=96)
    nh = {k: ops.to_nhwc(d4[k], torch.bfloat16) for k in ("key", "cur", "scale_map")}
    for fg, ws, nm in (kinds[0], kinds[2], kinds[3], kinds[4]):
        p = ops.PreparedAggregate(nh["key"], d4["mv"], flow_kind="raw", cur=nh["cur"], scale_map=nh["scale_map"],
                                  weight_mode="logits", logits=d4["logits"], layout="nhwc_bf16", force_generic=fg, workspace=ws)
        row("cfg4 V2 bf16 NHWC 68x120 batch %d%s" % (N4, nm), N4, 4 * C * H4 * W4 * 2 + 40 * H4 * W4, time_ms(lambda: p.run(s), 3, 10), pk,
            "ablation" if nm else "")
    del d4, nh, p


def nhwc_win_rows(dev, pk):
    """The window-resident channels-last kernel (force_generic=5, opt-in) beside the gather-by-bulk-copy kernel (3) on the
    variants that are not HBM bound, bf16, batch 64: same DRAM traffic, 36 % less L2 -> SM traffic, the same speed."""
    s = torch.cuda.current_stream().cuda_stream
    C, H, W, N = 1024, 38, 63, 64
    HW, F2 = H * W, C * H * W * 2
    d = synth(N, C, H, W, 600, 1000, dev)
    nh = {k: ops.to_nhwc(d[k], torch.bfloat16) for k in ("key", "cur", "scale_map")}
    for fg, nm in ((5, "window-resident kernel"), (3, "gather-by-bulk-copy kernel")):
        p = ops.PreparedAggregate(nh["key"], d["mv"], flow_kind="raw", layout="nhwc_bf16", force_generic=fg)
        row("V0 warp only bf16 NHWC batch 64, %s" % nm, N, 2 * F2 + 32 * HW, time_ms(lambda: p.run(s), 3, 20), pk)
        p = ops.PreparedAggregate(nh["key"], d["mv"], flow_kind="raw", cur=nh["cur"], res=d["res"], rnet_w=d["rnet_w"], rnet_b=d["rnet_b"],
                                  weight_mode="add", layout="nhwc_bf16", force_generic=fg)
        row("V1 shipped non-key path bf16 NHWC batch 64, %s" % nm, N, 3 * F2 + 44 * HW, time_ms(lambda: p.run(s), 3, 20), pk)
        p = ops.PreparedAggregate(nh["key"], d["mv"], flow_kind="raw", cur=nh["cur"], scale_map=nh["scale_map"], weight_mode="logits",
                                  logits=d["logits"], layout="nhwc_bf16", force_generic=fg)
        row("V2 bf16 NHWC batch 64, %s" % nm, N, 4 * F2 + 40 * HW, time_ms(lambda: p.run(s), 3, 20), pk)


def nocur_rows(dev, pk):
    """The NCHW variants without a current feature (the two drop-in operators, the fused warp, warp x scale)."""
    s = torch.cuda.current_stream().cuda_stream
    C, H, W, N = 1024, 38, 63, 64
    HW, F4 = H * W, C * H * W * 4
    d = synth(N, C, H, W, 600, 1000, dev)
    flow = ops.mv_pool(d["mv"])
    grid = ops.GridGenerator(flow)
    out = torch.empty_like(d["key"])
    row("cfg1 V0 GridGenerator+BilinearSampler (2 ops, fp32 NCHW)", N, 2 * F4 + 8 * HW,
        time_ms(lambda: ops.BilinearSampler(d["key"], ops.GridGenerator(flow, out=grid), out=out)), pk, "drop-in operators")
    p = ops.PreparedAggregate(d["key"], d["mv"], flow_kind="raw")
    row("cfg1 V0 fused warp only, raw MV pooled in-kernel", N, 2 * F4 + 32 * HW, time_ms(lambda: p.run(s)), pk)
    p = ops.PreparedAggregate(d["key"], flow, flow_kind="flow", scale_map=d["scale_map"])
    row("batch path: warp x scale (SYM:678-680), flow given", N, 3 * F4 + 8 * HW, time_ms(lambda: p.run(s)), pk)
    d4 = synth(32, C, 68, 120, 1080, 1920, dev, max_px=96)
    p = ops.PreparedAggregate(d4["key"], d4["mv"], flow_kind="raw")
    row("V0 fused warp only 68x120 batch 32", 32, 2 * C * 68 * 120 * 4 + 32 * 68 * 120, time_ms(lambda: p.run(s), 3, 10), pk)


def upstream_rows(dev, pk, quick):
    """Upstream (8f rank 3): coviar MV accumulation, 64 GOPs x 11 P-frames at 720p."""
    Na, T, ha, wa = (16 if quick else 64), 11, 720, 1280
    bx, by = wa // 16, ha // 16
    M = bx * by
    g = torch.Generator(device=dev).manual_seed(3)
    cx = (torch.arange(bx, device=dev, dtype=torch.int32) * 16 + 8).view(1, 1, 1, bx).expand(Na, T, by, bx)
    cy = (torch.arange(by, device=dev, dtype=torch.int32) * 16 + 8).view(1, 1, by, 1).expand(Na, T, by, bx)
    off = torch.randint(-16, 17, (Na, T, by, bx, 2), device=dev, generator=g, dtype=torch.int32)
    off[torch.rand((Na, T, by, bx), device=dev, generator=g) < 0.5] = 0
    mvs = torch.stack([torch.full_like(cx, 16), torch.full_like(cx, 16), cx + off[..., 0], cy + off[..., 1], cx, cy], -1)
    mvs = mvs.reshape(Na, T, M, 6).contiguous()
    counts = torch.full((Na, T), M, dtype=torch.int32, device=dev)
    ws = torch.empty(Na * ha * wa * 20, dtype=torch.uint8, device=dev)
    # algorithmic bytes per GOP in the REFERENCE's formulation: per P-frame read + write the (x,y) int2 field once, plus the
    # vector list; the back-trace form needs only the lists and one write of the result
    alg = T * (2 * ha * wa * 8 + M * 24) + ha * wa * 8
    alg_trace = T * M * 24 + ha * wa * 8
    ms = time_ms(lambda: ops.mv_accumulate(mvs, counts, ha, wa, workspace=ws, algo="field"), 2, 5)
    row("upstream: coviar MV accumulation, per-frame field form (round 1), %d GOPs x 11 P-frames @720p" % Na, Na, alg, ms, pk, "unit = GOPs")
    ms = time_ms(lambda: ops.mv_accumulate(mvs, counts, ha, wa, workspace=ws, algo="trace"), 2, 5)
    row("upstream: coviar MV accumulation, cell-index back-trace, %d GOPs x 11 P-frames @720p (reference-formulation bytes)" % Na, Na, alg, ms, pk, "unit = GOPs")
    r = row("upstream: coviar MV accumulation, cell-index back-trace (its own bytes: lists + one write of the field)", Na, alg_trace, ms, pk, "unit = GOPs")
    del mvs, counts, ws, off



def motion_rows(dev, pk, quick):
    """Shared-memory-bound variants under the two motion distributions: the synthetic i.i.d. per-macroblock vectors of
    SURVEY 8d (half the blocks static, the rest uniform in [-32,32] px - neighbouring cells move independently: the worst
    case for bank conflicts on the tap gathers) and vectors block-matched from the reference's demo video
    (tests/golden/demo_block_mvs.npz, tools/make_demo_block_mvs.py: camera motion, neighbouring blocks move together)."""
    import numpy as np
    C, H, W, mvh, mvw = 1024, 38, 63, 600, 1000
    HW, F4 = H * W, C * H * W * 4
    N = 32 if quick else 64
    d = synth(N, C, H, W, mvh, mvw, dev)
    g = np.load(os.path.join(ROOT, "tests", "golden", "demo_block_mvs.npz"))["block_mv"].astype(np.int32)
    blk = torch.from_numpy(g[np.arange(N) % g.shape[0]]).to(dev)
    demo = blk.repeat_interleave(16, 1).repeat_interleave(16, 2)[:, :mvh, :mvw].contiguous()
    s = torch.cuda.current_stream().cuda_stream
    nh = {k: ops.to_nhwc(d[k], torch.bfloat16) for k in ("key", "cur", "scale_map")}
    zero = torch.zeros_like(d["mv"])
    shift = torch.zeros_like(d["mv"]); shift[..., 0] = 56; shift[..., 1] = -24     # every cell moves by (3.5, -1.5) cells
    for tag, mv in (("synthetic i.i.d. blocks", d["mv"]), ("demo video (block matched)", demo),
                    ("zero motion (conflict-free gathers)", zero), ("uniform translation by (3.5,-1.5) cells", shift)):
        for name, alg, mk in (
                ("V0 warp only, fp32 NCHW", 2 * F4 + 32 * HW, lambda: ops.PreparedAggregate(d["key"], mv, flow_kind="raw")),
                ("V1 shipped non-key path (warp + rnet(res) + cur), fp32 NCHW", 3 * F4 + 44 * HW,
                 lambda: ops.PreparedAggregate(d["key"], mv, flow_kind="raw", cur=d["cur"], res=d["res"], rnet_w=d["rnet_w"], rnet_b=d["rnet_b"], weight_mode="add")),
                ("V2 headline (warp x scale, logits blend), fp32 NCHW", 4 * F4 + 40 * HW,
                 lambda: ops.PreparedAggregate(d["key"], mv, flow_kind="raw", cur=d["cur"], scale_map=d["scale_map"], weight_mode="logits", logits=d["logits"])),
                ("V0 warp only, bf16 NHWC", F4 + 32 * HW, lambda: ops.PreparedAggregate(nh["key"], mv, flow_kind="raw", layout="nhwc_bf16")),
                ("V1 shipped non-key path, bf16 NHWC", 3 * F4 // 2 + 44 * HW,
                 lambda: ops.PreparedAggregate(nh["key"], mv, flow_kind="raw", cur=nh["cur"], res=d["res"], rnet_w=d["rnet_w"], rnet_b=d["rnet_b"], weight_mode="add", layout="nhwc_bf16"))):
            if mv is zero or mv is shift:
                if "NHWC" in name or "V2" in name:
                    continue                      # the conflict-free bounds are reported for the two fp32 NCHW variants they explain
            p = mk()
            row("motion = %s: %s" % (tag, name), N, alg, time_ms(lambda: p.run(s), 3, 20), pk)


def keyframe_rows(dev, pk, quick):
    """Key-frame graphs end to end (SYM:468-477): K1 (lsfa warp x scale) -> embedding / Nq convolutions (LIBRARY GEMMs:
    cuDNN through torch, as north_star prescribes) -> K2 (lsfa cosine + blend).  Answers SURVEY 8f rank 2's question
    "do the GEMMs matter": per-phase times; the convolutions in fp32 (TF32 tensor cores) and in bf16."""
    import torch.nn.functional as F
    from lsfa_b200 import graphs
    C, H, W, E = 1024, 38, 63, 2048
    HW, F4 = H * W, C * H * W * 4
    N = 8 if quick else 16
    d = synth(N, C, H, W, 600, 1000, dev)
    flow = ops.mv_pool(d["mv"])
    g = torch.Generator(device=dev).manual_seed(5)
    rn = lambda *sh: 0.01 * torch.randn(sh, device=dev, generator=g)
    emb = (rn(512, C, 1, 1), rn(512), rn(512, 512, 3, 3), rn(512), rn(E, 512, 1, 1), rn(E))
    nq = (rn(256, C, 3, 3), rn(256), rn(16, 256, 1, 1), rn(16), rn(1, 16, 1, 1), rn(1))
    gflop_emb = 2 * N * 2 * HW * (C * 512 + 9 * 512 * 512 + 512 * E) / 1e9
    gflop_nq = 2 * N * 2 * HW * (9 * C * 256 + 256 * 16 + 16) / 1e9
    torch.backends.cudnn.allow_tf32 = True
    torch.backends.cuda.matmul.allow_tf32 = True
    warp = ops.warp_scale_aggregate(d["key"], flow, scale_map=d["scale_map"])
    x2 = torch.cat([d["cur"], warp], dim=0)
    row("key frame: K1 warp x scale (lsfa)", N, 3 * F4 + 8 * HW,
        time_ms(lambda: ops.warp_scale_aggregate(d["key"], flow, scale_map=d["scale_map"], out=warp)), pk)
    ms = time_ms(lambda: graphs.embed_net(x2, *emb), 2, 5)
    row("key frame: embedding convs, library, fp32/TF32 (%.0f GFLOP = %.0f TFLOP/s)" % (gflop_emb, gflop_emb / ms), N, 0, ms, pk, "library GEMMs")
    x2b = graphs._lowp_input([d["cur"], warp], torch.bfloat16)
    embb = graphs.prepare_params(emb, torch.bfloat16)
    nqb = graphs.prepare_params(nq, torch.bfloat16)
    ms = time_ms(lambda: graphs.embed_net(x2b, *embb), 2, 5)
    row("key frame: embedding convs, library, bf16 channels-last (%.0f TFLOP/s)" % (gflop_emb / ms), N, 0, ms, pk, "library GEMMs")
    e = graphs.embed_net(x2, *emb)
    ec, ew = e[:N].contiguous(), e[N:].contiguous()
    lg = ops.cosine_logits(ew, ec)
    row("key frame: K2a cosine logits of the 2048-ch embeddings (lsfa)", N, 2 * E * HW * 4 + 8 * HW, time_ms(lambda: ops.cosine_logits(ew, ec)), pk)
    outb = torch.empty_like(warp)
    row("key frame: K2b softmax blend (lsfa)", N, 3 * F4 + 8 * HW, time_ms(lambda: ops.blend_logits(warp, d["cur"], lg, out=outb)), pk)
    row("key frame: Fgfa graph end to end (K1 + fp32/TF32 convs + K2)", N, 0,
        time_ms(lambda: graphs.key_frame_fgfa(d["key"], flow, d["scale_map"], d["cur"], emb), 2, 5), pk)
    row("key frame: Fgfa graph end to end (K1 + bf16 channels-last convs + K2)", N, 0,
        time_ms(lambda: graphs.key_frame_fgfa(d["key"], flow, d["scale_map"], d["cur"], embb, conv_dtype=torch.bfloat16), 2, 5), pk)
    ms = time_ms(lambda: graphs.nq_net(x2, *nq), 2, 5)
    row("key frame: Nq convs, library, fp32/TF32 (%.0f GFLOP = %.0f TFLOP/s)" % (gflop_nq, gflop_nq / ms), N, 0, ms, pk, "library GEMMs")
    row("key frame: Nq graph end to end (K1 + fp32/TF32 convs + blend), as shipped", N, 0,
        time_ms(lambda: graphs.key_frame_nq(d["key"], flow, d["scale_map"], d["cur"], nq), 2, 5), pk)
    row("key frame: Nq graph end to end (K1 + bf16 channels-last convs + blend)", N, 0,
        time_ms(lambda: graphs.key_frame_nq(d["key"], flow, d["scale_map"], d["cur"], nqb, conv_dtype=torch.bfloat16), 2, 5), pk)
    # ---- this package's tcgen05 convolutions (csrc/conv_gemm_tc.cu): same operands, same box ----
    tf_peak = tflops_peak()
    xb = x2b.permute(0, 2, 3, 1)                       # the contiguous (2N,H,W,C) bf16 buffer
    pe = graphs.pack_embed_params(emb)
    pq = graphs.pack_nq_params(nq)
    xq = graphs._lowp_input([warp, d["cur"]], torch.bfloat16).permute(0, 2, 3, 1)
    h1 = torch.empty((2 * N, H, W, 512), dtype=torch.bfloat16, device=dev)
    h2 = torch.empty_like(h1)
    for name, fn, gf in (
            ("em_conv1 1x1 1024->512 +ReLU", lambda: ops.conv_bf16_nhwc(xb, pe[0], pe[1], relu=True, out=h1), 2 * N * 2 * HW * C * 512 / 1e9),
            ("em_conv2 3x3 512->512 +ReLU", lambda: ops.conv_bf16_nhwc(h1, pe[2], pe[3], relu=True, out=h2), 2 * N * 2 * HW * 9 * 512 * 512 / 1e9),
            ("embedding net + cosine logits (em_conv1,2,3 + compute_weight fused)", lambda: ops.embed_cosine_logits(xb, pe), gflop_emb),
            ("Nq net -> logits (Nq_conv1 + fused 256->16->1 tail)", lambda: ops.nq_logits(xq, pq), gflop_nq)):
        ms = time_ms(fn, 3, 10)
        r = row("key frame tcgen05: %s (%.0f GFLOP = %.0f TFLOP/s = %.2f of the sustained bf16 peak %.0f)" % (
            name, gf, gf / ms, gf / ms / tf_peak, tf_peak), N, 0, ms, pk, "hand-written tcgen05 implicit GEMM")
    row("key frame: Fgfa graph end to end (K1 + tcgen05 convs with fused cosine + blend)", N, 0,
        time_ms(lambda: graphs.key_frame_fgfa(d["key"], flow, d["scale_map"], d["cur"], emb, conv_dtype="tc", packed=pe), 2, 5), pk)
    row("key frame: Nq graph end to end (K1 + tcgen05 convs + blend)", N, 0,
        time_ms(lambda: graphs.key_frame_nq(d["key"], flow, d["scale_map"], d["cur"], nq, conv_dtype="tc", packed=pq), 2, 5), pk)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quick", action="store_true")
    ap.add_argument("--only-backward", action="store_true")
    ap.add_argument("--only-cosine", action="store_true")
    ap.add_argument("--only-single", action="store_true")
    ap.add_argument("--only-nhwc", action="store_true")
    ap.add_argument("--only-nhwc-tma", action="store_true")
    ap.add_argument("--only-nhwc-win", action="store_true")
    ap.add_argument("--only-nocur", action="store_true")
    ap.add_argument("--only-upstream", action="store_true")
    ap.add_argument("--only-keyframe", action="store_true")
    ap.add_argument("--only-motion", action="store_true")
    ap.add_argument("--only-cosine-backward", action="store_true")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    pk = peak()
    if args.only_cosine_backward:
        cosine_backward_rows(dev)
        return
    if args.only_backward:
        backward_rows(dev, pk, args.quick)
        return
    if args.only_single:
        single_frame_rows(dev, pk)
        return
    if args.only_motion:
        motion_rows(dev, pk, args.quick)
        return
    if args.only_keyframe:
        keyframe_rows(dev, pk, args.quick)
        return
    if args.only_upstream:
        upstream_rows(dev, pk, args.quick)
        return
    if args.only_nocur:
        nocur_rows(dev, pk)
        return
    if args.only_nhwc_win:
        nhwc_win_rows(dev, pk)
        return
    if args.only_nhwc or args.only_nhwc_tma:
        nhwc_rows(dev, pk, args.quick, args.only_nhwc_tma)
        return
    if args.only_cosine:
        cosine_rows(dev, pk, 64)
        return
    s = torch.cuda.current_stream().cuda_stream
    C, H, W = 1024, 38, 63
    HW = H * W
    F4, F2 = C * HW * 4, C * HW * 2

    # ---- configs 1/2: fp32 NCHW, 38x63 ----
    N = 64
    d = synth(N, C, H, W, 600, 1000, dev, E=0)
    flow = ops.mv_pool(d["mv"])
    grid = ops.GridGenerator(flow)
    out = torch.empty_like(d["key"])
    row("cfg1 V0 GridGenerator+BilinearSampler (2 ops, fp32 NCHW)", N, 2 * F4 + 8 * HW,
        time_ms(lambda: ops.BilinearSampler(d["key"], ops.GridGenerator(flow, out=grid), out=out)), pk, "drop-in operators")
    p = ops.PreparedAggregate(d["key"], d["mv"], flow_kind="raw")
    row("cfg1 V0 fused warp only, raw MV pooled in-kernel", N, 2 * F4 + 32 * HW, time_ms(lambda: p.run(s)), pk)
    p = ops.PreparedAggregate(d["key"], d["mv"], flow_kind="raw", workspace=False)
    row("cfg1 V0 fused warp only, raw MV, static split (no scratch)", N, 2 * F4 + 32 * HW, time_ms(lambda: p.run(s)), pk, "ablation")
    p = ops.PreparedAggregate(d["key"], flow, flow_kind="flow")
    row("cfg1 V0 fused warp only, flow given", N, 2 * F4 + 8 * HW, time_ms(lambda: p.run(s)), pk, "ablation")
    p = ops.PreparedAggregate(d["key"], flow, flow_kind="flow", workspace=False)
    row("cfg1 V0 fused warp only, flow given, static split", N, 2 * F4 + 8 * HW, time_ms(lambda: p.run(s)), pk, "ablation")
    p = ops.PreparedAggregate(d["key"], grid, flow_kind="grid")
    row("cfg1 V0 fused warp only, grid given", N, 2 * F4 + 8 * HW, time_ms(lambda: p.run(s)), pk, "ablation")
    p = ops.PreparedAggregate(d["key"], flow, flow_kind="flow", scale_map=d["scale_map"])
    row("batch path: warp x scale (SYM:678-680), flow given", N, 3 * F4 + 8 * HW, time_ms(lambda: p.run(s)), pk)
    p = ops.PreparedAggregate(d["key"], flow, flow_kind="flow", scale_map=d["scale_map"], workspace=False)
    row("batch path: warp x scale, static split", N, 3 * F4 + 8 * HW, time_ms(lambda: p.run(s)), pk, "ablation")
    p = ops.PreparedAggregate(d["key"], d["mv"], flow_kind="raw", cur=d["cur"], res=d["res"], rnet_w=d["rnet_w"],
                              rnet_b=d["rnet_b"], weight_mode="add")
    row("V1 shipped non-key path: warp + rnet(res) + cur", N, 3 * F4 + 32 * HW + 12 * HW + 16384, time_ms(lambda: p.run(s)), pk)
    p = ops.PreparedAggregate(d["key"], d["mv"], flow_kind="raw", cur=d["cur"], scale_map=d["scale_map"],
                              weight_mode="logits", logits=d["logits"])
    row("cfg2 V2 fused warp*scale + logits blend (headline, all-TMA)", N, 4 * F4 + 40 * HW, time_ms(lambda: p.run(s)), pk)
    for fk, fl in (("flow", flow), ("grid", grid)):
        p = ops.PreparedAggregate(d["key"], fl, flow_kind=fk, cur=d["cur"], scale_map=d["scale_map"],
                                  weight_mode="logits", logits=d["logits"])
        row("cfg2 V2 all-TMA, %s given (no in-kernel MV pooling)" % fk, N, 4 * F4 + 16 * HW, time_ms(lambda: p.run(s)), pk, "ablation")
    p = ops.PreparedAggregate(d["key"], d["mv"], flow_kind="raw", cur=d["cur"], scale_map=d["scale_map"],
                              weight_mode="logits", logits=d["logits"], workspace=False)
    row("cfg2 V2 all-TMA, static work split (no scratch)", N, 4 * F4 + 40 * HW, time_ms(lambda: p.run(s)), pk, "ablation")
    for fg, nm in ((2, "plane-resident LDG/STG kernel"), (1, "generic gather kernel")):
        p = ops.PreparedAggregate(d["key"], d["mv"], flow_kind="raw", cur=d["cur"], scale_map=d["scale_map"],
                                  weight_mode="logits", logits=d["logits"], force_generic=fg)
        row("cfg2 V2 " + nm, N, 4 * F4 + 40 * HW, time_ms(lambda: p.run(s)), pk, "ablation")
    tmp = torch.empty(5 * d["key"].numel(), dtype=torch.float32, device=dev)
    row("cfg2 V2 UNFUSED op-by-op chain (9 kernels)", N, 4 * F4 + 40 * HW,
        time_ms(lambda: ops.unfused_chain(d["key"], flow, d["scale_map"], d["cur"], d["logits"], tmp), 3, 10), pk,
        "algorithmic bytes of the fused op; real traffic is 16F")
    del tmp
    cosine_rows(dev, pk, 16 if args.quick else 64)
    single_frame_rows(dev, pk)

    del d
    torch.cuda.empty_cache()
    nhwc_rows(dev, pk, args.quick)
    torch.cuda.empty_cache()

    upstream_rows(dev, pk, args.quick)

    # ---- config 4: 1080p -> 68x120 ----
    H4, W4 = 68, 120
    N4 = 32 if args.quick else 128
    d4 = synth(N4, C, H4, W4, 1080, 1920, dev, max_px=96)
    p = ops.PreparedAggregate(d4["key"], d4["mv"], flow_kind="raw", cur=d4["cur"], scale_map=d4["scale_map"],
                              weight_mode="logits", logits=d4["logits"])
    row("cfg4 V2 fp32 NCHW 68x120 batch %d" % N4, N4, 4 * C * H4 * W4 * 4 + 40 * H4 * W4, time_ms(lambda: p.run(s), 3, 10), pk)
    del d4, p
    torch.cuda.empty_cache()
    backward_rows(dev, pk, args.quick)


if __name__ == "__main__":
    main()
