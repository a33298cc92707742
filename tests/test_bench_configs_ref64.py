"""Every configuration bench.py times, at its own sizes and from its own input recipes, against the float64 reference
of oracle/ref64.py with per-element error bounds (see that module for the gate and its derivation).

The float64 reference runs on the device in chunks of ``ref64.CHUNK`` frames; the coordinates come from the oracle's
float32 index math on the host.  Each test prints its largest err/tol (run with -s to see them)."""
import numpy as np
import pytest
import torch

import bench
from oracle import ref64 as R

pytestmark = pytest.mark.gpu

C, H, W = bench.C, bench.H, bench.W
FRAMES = bench.FRAMES_PER_GPU


@pytest.fixture(scope="module")
def ops(cuda):
    from lsfa_b200 import ops as _ops
    return _ops


@pytest.fixture(scope="module")
def inputs(cuda):
    """bench's value/extra inputs: make_host_inputs(64, seed=1000), resident on the device, and their coordinates."""
    host = bench.make_host_inputs(FRAMES, seed=1000)
    d = {k: v.to(cuda) for k, v in host.items()}
    co = R.coords(mv=host["mv"])
    yield host, d, co
    del d
    torch.cuda.empty_cache()


@pytest.fixture(autouse=True)
def peak_memory(cuda, request):
    torch.cuda.reset_peak_memory_stats()
    yield
    print("\n[ref64] %-44s peak device memory %.1f GB" % (request.node.name, torch.cuda.max_memory_allocated() / 1e9))


def gate(what, got, key, co, out="f32", frames=None, show=True, chunk=R.CHUNK, **kw):
    """Check ``got`` (logical NCHW, any layout view) ``chunk`` frames at a time; print and return the largest err/tol."""
    torch.cuda.synchronize()
    fr = range(co[0].shape[0]) if frames is None else frames
    worst = 0.0
    for n0 in range(fr.start, fr.stop, chunk):
        ch = range(n0, min(n0 + chunk, fr.stop))
        ref, mag = R.forward(key, co, frames=ch, device=torch.device("cuda"), **kw)
        g = got[ch.start - fr.start:ch.stop - fr.start]
        worst = max(worst, R.check(g, ref, mag, out, what=what, frame0=ch.start))
        del ref, mag
    if show:
        print("\n[ref64] %-44s max err/tol %.3g" % (what, worst))
    return worst


def v2(d, **over):
    kw = dict(cur=d["cur"], scale_map=d["scale_map"], mode="logits", logits=d["logits"])
    kw.update(over)
    return kw


def test_headline_prepared_aggregate_repeated(ops, inputs):
    _, d, co = inputs
    prep = ops.PreparedAggregate(d["key"], d["mv"], flow_kind="raw", cur=d["cur"], scale_map=d["scale_map"],
                                 weight_mode="logits", logits=d["logits"])
    first = prep.run().clone()
    for _ in range(3):
        prep.run()
        torch.cuda.synchronize()
        assert torch.equal(prep.out, first)
    del first
    gate("value: PreparedAggregate x4", prep.out, d["key"], co, **v2(d))


def test_plane_ldg_kernel(ops, inputs):
    _, d, co = inputs
    prep = ops.PreparedAggregate(d["key"], d["mv"], flow_kind="raw", cur=d["cur"], scale_map=d["scale_map"],
                                 weight_mode="logits", logits=d["logits"], force_generic=2)
    gate("extra.fused_fp32_nchw_plane_ldg", prep.run(), d["key"], co, **v2(d))


def test_unfused_chain(ops, inputs):
    _, d, co = inputs
    flow = ops.mv_pool(d["mv"])
    got = ops.unfused_chain(d["key"], flow, d["scale_map"], d["cur"], d["logits"])
    del flow
    gate("extra.unfused_fp32_nchw", got, d["key"], co, **v2(d))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_channels_last_64_frames(ops, inputs, dtype):
    _, d, co = inputs
    nh = {k: ops.to_nhwc(d[k], dtype) for k in ("key", "cur", "scale_map")}
    lay = "nhwc_bf16" if dtype == torch.bfloat16 else "nhwc_f32"
    prep = ops.PreparedAggregate(nh["key"], d["mv"], flow_kind="raw", cur=nh["cur"], scale_map=nh["scale_map"],
                                 weight_mode="logits", logits=d["logits"], layout=lay)
    got = prep.run().permute(0, 3, 1, 2)
    nc = {k: v.permute(0, 3, 1, 2) for k, v in nh.items()}          # the reference reads the bf16 values themselves
    gate("extra.fused_%s" % ("bf16_nhwc" if dtype == torch.bfloat16 else "fp32_nhwc"), got, nc["key"], co,
         "bf16" if dtype == torch.bfloat16 else "f32", **v2(d, cur=nc["cur"], scale_map=nc["scale_map"]))


def test_bf16_channels_last_512_distinct_frames(ops, cuda):
    """extra.fused_bf16_nhwc_batch512's size (2.5 GB per bf16 tensor) with 512 distinct frames, so that a frame-offset
    bug past frame 64 cannot hide behind a repeated batch."""
    N = 512
    g = torch.Generator(device=cuda).manual_seed(512)
    rng = np.random.default_rng(512)

    def feat(relu):
        t = torch.empty((N, H, W, C), dtype=torch.bfloat16, device=cuda)
        for n0 in range(0, N, 64):
            x = torch.randn((64, H, W, C), device=cuda, generator=g)
            t[n0:n0 + 64] = (x.clamp_(min=0) if relu else 1 + 0.1 * x).to(torch.bfloat16)
        return t

    key, cur, sm = feat(True), feat(True), feat(False)
    logits = torch.randn((N, 2, H, W), device=cuda, generator=g)
    mv = torch.empty((N, bench.MV_H, bench.MV_W, 2), dtype=torch.int32, device=cuda)
    bh, bw = -(-bench.MV_H // 16), -(-bench.MV_W // 16)
    cos = []
    for n0 in range(0, N, 64):
        blk = rng.integers(-32, 33, size=(64, bh, bw, 2), dtype=np.int32)
        blk[rng.random((64, bh, bw)) < 0.5] = 0
        m = np.ascontiguousarray(np.repeat(np.repeat(blk, 16, axis=1), 16, axis=2)[:, :bench.MV_H, :bench.MV_W])
        mv[n0:n0 + 64] = torch.from_numpy(m).to(cuda)
        cos.append(R.coords(mv=m))
    co = tuple(np.concatenate([c[i] for c in cos]) for i in range(4))
    prep = ops.PreparedAggregate(key, mv, flow_kind="raw", cur=cur, scale_map=sm, weight_mode="logits", logits=logits,
                                 layout="nhwc_bf16")
    got = prep.run().permute(0, 3, 1, 2)
    p = lambda t: t.permute(0, 3, 1, 2)  # noqa: E731
    gate("extra.fused_bf16_nhwc_batch512 (distinct)", got, p(key), co, "bf16", cur=p(cur), scale_map=p(sm), mode="logits",
         logits=logits)
    del key, cur, sm, mv, prep, got
    torch.cuda.empty_cache()


def test_cfg1_single_frame(ops, inputs):
    """extra.cfg1_single_frame: the three drop-in operators, the fused warp and the fused V2, each eager and the two
    fused forms replayed from a RecordedGraph into a poisoned output."""
    _, d, co = inputs
    key, mv = d["key"][:1].contiguous(), d["mv"][:1].contiguous()
    one = {k: d[k][:1].contiguous() for k in ("cur", "scale_map", "logits")}
    co1 = tuple(a[:1] for a in co)
    out = ops.BilinearSampler(key, ops.GridGenerator(ops.mv_pool(mv)))
    gate("cfg1: three drop-in operators", out, key, co1)
    p0 = ops.PreparedAggregate(key, mv, flow_kind="raw")
    p2 = ops.PreparedAggregate(key, mv, flow_kind="raw", cur=one["cur"], scale_map=one["scale_map"], weight_mode="logits",
                               logits=one["logits"])
    for tag, p, kw in (("fused warp", p0, {}), ("fused V2", p2, v2(one))):
        eager = p.run().clone()
        gate("cfg1: %s" % tag, eager, key, co1, **kw)
        side = torch.cuda.Stream()
        with torch.cuda.stream(side):
            p.run(side.cuda_stream)
            side.synchronize()
            graph = ops.RecordedGraph(side.cuda_stream)
            with graph:
                p.run(side.cuda_stream)
            p.out.fill_(float("nan"))
            side.synchronize()
            graph.launch()
            side.synchronize()
        graph.close()
        assert torch.equal(p.out, eager), tag
        gate("cfg1: %s, graph replay" % tag, p.out, key, co1, **kw)


def test_cfg4_hires_128_frames(ops, cuda):
    """extra.cfg4_hires_68x120 with bench's recipe (generator seed 4, same order): 4.3 GB fp32 tensors, so byte offsets
    pass 2^32, and 1080-row MV fields whose last block row keeps row 16k+7 only."""
    N4, H4, W4 = 128, 68, 120
    g = torch.Generator(device=cuda).manual_seed(4)
    blk = torch.randint(-96, 97, (N4, H4, W4, 2), device=cuda, generator=g, dtype=torch.int32)
    blk[torch.rand((N4, H4, W4), device=cuda, generator=g) < 0.5] = 0
    mv = blk.repeat_interleave(16, 1).repeat_interleave(16, 2)[:, :1080, :1920].contiguous()
    del blk
    lg = torch.randn((N4, 2, H4, W4), device=cuda, generator=g)
    mvh = mv.cpu()
    co = R.coords(mv=mvh)
    del mvh
    for tag, dt, lay in (("fp32_nchw", torch.float32, "nchw"), ("bf16_nhwc", torch.bfloat16, "nhwc_bf16")):
        shape = (N4, C, H4, W4) if lay == "nchw" else (N4, H4, W4, C)
        key = torch.randn(shape, device=cuda, generator=g, dtype=torch.float32).clamp_(min=0).to(dt)
        cur = torch.randn(shape, device=cuda, generator=g, dtype=torch.float32).clamp_(min=0).to(dt)
        sm = (1 + 0.1 * torch.randn(shape, device=cuda, generator=g, dtype=torch.float32)).to(dt)
        prep = ops.PreparedAggregate(key, mv, flow_kind="raw", cur=cur, scale_map=sm, weight_mode="logits", logits=lg,
                                     layout=lay)
        got = prep.run()
        if lay != "nchw":
            got, key, cur, sm = (t.permute(0, 3, 1, 2) for t in (got, key, cur, sm))
        gate("extra.cfg4_hires_68x120.%s" % tag, got, key, co, "bf16" if dt == torch.bfloat16 else "f32", cur=cur,
             scale_map=sm, mode="logits", logits=lg, chunk=2)        # 68x120 frames: keep the float64 chunks small
        del key, cur, sm, prep, got
        torch.cuda.empty_cache()


def test_cfg5_multi_stream(ops, inputs, cuda):
    """extra.cfg5_multi_stream with bench's recipe: 256 streams through StreamScheduler, every frame checked against its
    stream's slot of the key table (get_cur_test_symbol: warp + rnet_conv0(res) + current feature)."""
    from lsfa_b200 import streams
    from lsfa_b200.driver import StreamScheduler
    _, d, co = inputs
    S, B = 256, 80
    g = torch.Generator(device=cuda).manual_seed(5)
    cur = d["cur"][:min(B, d["cur"].shape[0])]
    reps = -(-B // cur.shape[0])
    cur = cur.repeat(reps, 1, 1, 1)[:B].contiguous()
    mv = d["mv"].repeat(reps, 1, 1, 1)[:B].contiguous()
    cob = tuple(np.concatenate([a] * reps)[:B] for a in co)
    res = torch.randn((B, 3, H, W), device=cuda, generator=g) * 30
    rnet_w = 0.01 * torch.randn((C, 3), device=cuda, generator=g)
    rnet_b = torch.zeros((C,), device=cuda)
    out = torch.empty_like(cur)
    sch = StreamScheduler([streams.KEY_FRAME_INTERVAL] * S, C, (H, W), cuda)
    sch.key_table.normal_(generator=g).clamp_(min=0)
    worst, seen = 0.0, 0
    for sid, _fid, slot in sch.batches(B):
        m = len(slot)
        sl = torch.as_tensor(slot, dtype=torch.int32, device=cuda)
        sch.run_non_key_batch(sl, mv[:m], cur[:m], res=res[:m], rnet_w=rnet_w, rnet_b=rnet_b, out=out[:m])
        assert np.array_equal(slot, [sch.slot_of[int(s)] for s in sid])
        worst = max(worst, gate("extra.cfg5_multi_stream frames %d-%d" % (seen, seen + m - 1), out[:m], sch.key_table,
                                tuple(a[:m] for a in cob), cur=cur[:m], res=res[:m], rnet_w=rnet_w, rnet_b=rnet_b,
                                mode="add", key_index=slot, show=False))
        seen += m
    assert seen == S * sum(1 for f in streams.key_frame_flags(streams.KEY_FRAME_INTERVAL) if f == 2)
    print("\n[ref64] %-44s max err/tol %.3g" % ("extra.cfg5_multi_stream (all %d frames)" % seen, worst))
    del sch, out, cur, mv, res
    torch.cuda.empty_cache()


@pytest.mark.parametrize("gop", [False, True])
def test_e2e_host_aggregator(ops, inputs, cuda, gop):
    """e2e (private keys) and e2e.gop_contract (6 key slots, key_index = i // 11) as bench builds them, two calls each:
    the second call reuses every staging slot and, in the GOP form, re-uploads the key table."""
    from lsfa_b200.host import HostAggregator
    host, d, co = inputs
    gop_len = 11
    n_keys = (FRAMES + gop_len - 1) // gop_len
    agg = HostAggregator(FRAMES, C, H, W, (bench.MV_H, bench.MV_W), cuda, chunk=8, depth=3, num_slots=n_keys if gop else 0)
    hin = host
    if gop:
        hin = {k: host[k] for k in ("scale_map", "cur", "mv", "logits")}
        hin["key_index"] = (torch.arange(FRAMES, dtype=torch.int32) // gop_len).pin_memory()
        hin["new_keys"] = host["key"][:n_keys]
        hin["key_slot"] = torch.arange(n_keys, dtype=torch.int32).pin_memory()
    out_host = torch.empty((FRAMES, C, H, W), dtype=torch.float32).pin_memory()
    for call in range(2):
        out_host.fill_(float("nan"))
        agg(hin, out_host)
        agg.synchronize()
        gate("e2e%s call %d" % (".gop_contract" if gop else "", call + 1), out_host, d["key"], co,
             key_index=hin["key_index"] if gop else None, **v2(d))
    del agg, out_host


@pytest.mark.parametrize("form", ["gather_key_and_flow", "gather_key_only", "fused_v2_all_gradients"])
def test_backward_64_frames(ops, inputs, cuda, form):
    """extra.backward_training_path at 64 frames: the gather backward of the warp (key + flow, key only) and the fused
    V2 backward (key, flow, scale, cur, logits), each gradient against the float64 chain rule with the reduction gate."""
    _, d, co = inputs
    flow = ops.mv_pool(d["mv"])
    g = torch.Generator(device=cuda).manual_seed(64)
    og = torch.randn(d["key"].shape, device=cuda, generator=g)
    if form == "fused_v2_all_gradients":
        got = ops.warp_scale_aggregate_backward(og, d["key"], flow, flow_kind="flow", cur=d["cur"], scale_map=d["scale_map"],
                                                weight_mode="logits", logits=d["logits"])
        kw = v2(d)
    else:
        gk, gf = ops.warp_backward(d["key"], flow, og, req_flow="null" if form == "gather_key_only" else "write",
                                   kernel="gather")
        got = {"key": gk} if gf is None else {"key": gk, "flow": gf}
        kw = {}
    assert set(got) == ({"key", "flow", "scale", "cur", "logits"} if kw else
                        {"key"} if form == "gather_key_only" else {"key", "flow"})
    torch.cuda.synchronize()
    worst = dict.fromkeys(got, 0.0)
    step = 2                                   # float64 intermediates of 2 frames at a time
    for n0 in range(0, FRAMES, step):
        ch = range(n0, n0 + step)
        ref = R.backward(og, d["key"], co, frames=ch, want=tuple(got), **kw)
        assert set(ref) == set(got)
        for k, (r, mag, na) in ref.items():
            worst[k] = max(worst[k], R.check(got[k][n0:n0 + step], r, mag, n_addends=na, what="%s grad_%s" % (form, k),
                                             frame0=n0))
        del ref
    for k, v in worst.items():
        print("\n[ref64] %-44s max err/tol %.3g" % ("extra.backward %s grad_%s" % (form, k), v))
    del got, og, flow
    torch.cuda.empty_cache()
