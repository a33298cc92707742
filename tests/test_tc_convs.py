"""SURVEY 8f rank 2: the embedding / quality networks on Blackwell tensor cores (csrc/conv_gemm_tc.cu),
through the C ABI.  Stated-tolerance variant: bf16 operands, fp32 accumulation (the reference computes
these convolutions in fp32).

Gates
  * single convolutions vs a float64-accumulating NumPy convolution of the SAME bf16-rounded operands:
    |a-b| <= 2^-8 |b| + 2^-8 * 1e-2 * max|b|   (one bf16 rounding of the output + fp32 accumulation order);
  * logits vs the oracle's bf16 restatement (oracle.embed_cosine_logits_bf16 / nq_logits_bf16, same rounding
    points): cosine logits |a-b| <= 2e-3 (they live in [-1,1]); quality logits 2e-3 * max|logit| + 1e-3;
  * end-to-end key-frame graphs vs the float32 oracle (O.key_frame_*_full): 1e-2 * max|feature|, the
    same gate the cuDNN-bf16 arm of the graphs is held to.
"""
import numpy as np
import pytest
import torch

from oracle import lsfa_oracle as O
from tests._util import make_case

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops(cuda):
    from lsfa_b200 import ops as _ops
    return _ops


def dev(x, cuda):
    return torch.from_numpy(np.ascontiguousarray(x)).to(cuda)


def to_bf16_nhwc(x, cuda):
    """(N,C,H,W) float32 -> (N,H,W,C) bf16 device tensor (round to nearest even, as the kernels' producers do)."""
    return dev(x, cuda).permute(0, 2, 3, 1).contiguous().to(torch.bfloat16)


def conv_ref_f64(x, w, b, pad, relu):
    """Independent of the oracle's einsum: torch float64 conv2d on the CPU."""
    y = torch.nn.functional.conv2d(torch.from_numpy(x).double(), torch.from_numpy(w).double(), torch.from_numpy(b).double(),
                                   padding=pad)
    return (y.clamp_min(0) if relu else y).numpy()


@pytest.mark.parametrize("relu", [False, True])
@pytest.mark.parametrize("NB,H,W,Cin,Cout,k", [
    (2, 38, 63, 128, 256, 1), (2, 38, 63, 64, 256, 3), (4, 7, 9, 64, 512, 3), (2, 68, 120, 64, 256, 1),
    (2, 5, 130, 64, 256, 3), (6, 17, 23, 192, 256, 3), (2, 1, 1, 64, 256, 3), (1, 12, 14, 64, 256, 3), (5, 17, 23, 64, 512, 1),
    (11, 38, 63, 64, 256, 3)])
def test_conv_bf16_nhwc_matches_float64_conv(ops, cuda, NB, H, W, Cin, Cout, k, relu):
    rng = np.random.default_rng(NB * 1000 + H * 10 + k)
    x = O.bf16_round(O.synth_features(rng, (NB, Cin, H, W)))
    w = O.bf16_round((rng.standard_normal((Cout, Cin, k, k)) / np.sqrt(Cin * k * k)).astype(np.float32))
    b = (0.1 * rng.standard_normal(Cout)).astype(np.float32)
    want = conv_ref_f64(x, w, b, k // 2, relu)
    wp = ops.pack_conv_weight(dev(w, cuda))
    got = ops.conv_bf16_nhwc(to_bf16_nhwc(x, cuda), wp, dev(b, cuda), relu=relu)
    torch.cuda.synchronize()
    got = got.float().permute(0, 3, 1, 2).cpu().numpy()
    tol = 2.0 ** -8 * np.abs(want) + 2.0 ** -8 * 1e-2 * np.abs(want).max()
    err = np.abs(got - want)
    assert (err <= tol).all(), "worst abs err %.3g at scale %.3g (%d outside)" % (err.max(), np.abs(want).max(), int((err > tol).sum()))


def test_pack_conv_weight_layout(ops, cuda):
    rng = np.random.default_rng(0)
    w = rng.standard_normal((8, 6, 3, 3)).astype(np.float32)
    got = ops.pack_conv_weight(dev(w, cuda)).float().cpu().numpy()
    want = O.bf16_round(w.transpose(0, 2, 3, 1).reshape(8, 54))      # K index = (ky*3 + kx)*Cin + cin
    assert np.array_equal(got, want)


def _embed_params(rng, C, C1, C2, E):
    mk = lambda *s: (rng.standard_normal(s) / np.sqrt(np.prod(s[1:]))).astype(np.float32)  # noqa: E731
    return (mk(C1, C, 1, 1), (0.1 * rng.standard_normal(C1)).astype(np.float32),
            mk(C2, C1, 3, 3), (0.1 * rng.standard_normal(C2)).astype(np.float32),
            mk(E, C2, 1, 1), (0.1 * rng.standard_normal(E)).astype(np.float32))


def _nq_params(rng, C):
    mk = lambda *s: (rng.standard_normal(s) / np.sqrt(np.prod(s[1:]))).astype(np.float32)  # noqa: E731
    return (mk(256, C, 3, 3), (0.1 * rng.standard_normal(256)).astype(np.float32),
            mk(16, 256, 1, 1), (0.1 * rng.standard_normal(16)).astype(np.float32),
            mk(1, 16, 1, 1), (0.1 * rng.standard_normal(1)).astype(np.float32))


@pytest.mark.parametrize("N,C,H,W,C1,C2,E", [(1, 64, 12, 14, 256, 256, 512), (2, 128, 9, 20, 256, 256, 256), (1, 64, 38, 63, 256, 256, 512)])
def test_embed_cosine_logits_against_oracle_bf16_restatement(ops, cuda, N, C, H, W, C1, C2, E):
    from lsfa_b200 import graphs
    rng = np.random.default_rng(C + H)
    x = O.synth_features(rng, (2 * N, C, H, W))
    x[N:] = 0.7 * x[:N] + 0.3 * x[N:]                    # warped feature correlated with the current one, as in a video
    params = _embed_params(rng, C, C1, C2, E)
    want = O.embed_cosine_logits_bf16(x, *params)
    packed = graphs.pack_embed_params([dev(p, cuda) for p in params])
    got = ops.embed_cosine_logits(to_bf16_nhwc(x, cuda), packed)
    torch.cuda.synchronize()
    err = np.abs(got.cpu().numpy() - want)
    assert err.max() <= 2e-3, "cosine logits: worst abs err %.3g" % err.max()
    assert np.abs(got.cpu().numpy()[:, 1] - 1.0).max() <= 1e-5      # <e_cur^, e_cur^> = sum e^2 / (sum e^2 + eps)


@pytest.mark.parametrize("N,C,H,W", [(1, 64, 12, 14), (2, 128, 9, 20), (1, 64, 38, 63)])
def test_nq_logits_against_oracle_bf16_restatement(ops, cuda, N, C, H, W):
    from lsfa_b200 import graphs
    rng = np.random.default_rng(C + W)
    x = O.synth_features(rng, (2 * N, C, H, W))
    params = _nq_params(rng, C)
    want = O.nq_logits_bf16(x, *params)
    packed = graphs.pack_nq_params([dev(p, cuda) for p in params])
    got = ops.nq_logits(to_bf16_nhwc(x, cuda), packed)
    torch.cuda.synchronize()
    err = np.abs(got.cpu().numpy() - want)
    assert err.max() <= 2e-3 * np.abs(want).max() + 1e-3, "quality logits: worst abs err %.3g (scale %.3g)" % (err.max(), np.abs(want).max())


def test_full_size_embedding_and_quality_networks_against_torch_fp32(ops, cuda):
    """The reference's sizes (SYM:97,119-128: 1024 -> 512 -> 512 -> 2048 and 1024 -> 256 -> 16 -> 1 at 38x63), 2 key frames
    and bench.py's 16 (32 images: enough work items per CTA that the double-buffered TMEM accumulators are reused and their
    phase bit flips), against torch float32 convolutions (TF32 off) of the same bf16-rounded operands with the hidden
    activations rounded at the kernel's rounding points."""
    for N in (2, 16):
        _full_size_networks(ops, cuda, N)


def _full_size_networks(ops, cuda, N):
    from lsfa_b200 import graphs
    rng = np.random.default_rng(1)
    C, H, W = 1024, 38, 63
    x = O.bf16_round(O.synth_features(rng, (2 * N, C, H, W)))
    x[N:] = O.bf16_round(0.6 * x[:N] + 0.4 * x[N:])
    ep = _embed_params(rng, C, 512, 512, 2048)
    nq = _nq_params(rng, C)
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        F = torch.nn.functional
        r = lambda t: t.to(torch.bfloat16).float()  # noqa: E731
        xt = dev(x, cuda)
        e1, e2, e3 = (r(dev(ep[i], cuda)) for i in (0, 2, 4))
        h1 = r(F.relu(F.conv2d(xt, e1, dev(ep[1], cuda))))
        h2 = r(F.relu(F.conv2d(h1, e2, dev(ep[3], cuda), padding=1)))
        e = F.conv2d(h2, e3, dev(ep[5], cuda)).double()
        nrm = lambda t: t / torch.sqrt((t * t).sum(1, keepdim=True) + 1e-10)  # noqa: E731
        want_cos = torch.cat([(nrm(e[N:]) * nrm(e[:N])).sum(1, keepdim=True), (nrm(e[:N]) * nrm(e[:N])).sum(1, keepdim=True)], 1)
        q = F.relu(F.conv2d(xt, r(dev(nq[0], cuda)), dev(nq[1], cuda), padding=1))
        q = F.conv2d(F.relu(F.conv2d(q, dev(nq[2], cuda), dev(nq[3], cuda))), dev(nq[4], cuda), dev(nq[5], cuda))
        want_q = torch.cat([q[:N], q[N:]], 1)
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
    xb = to_bf16_nhwc(x, cuda)
    got_cos = ops.embed_cosine_logits(xb, graphs.pack_embed_params([dev(p, cuda) for p in ep]))
    got_q = ops.nq_logits(xb, graphs.pack_nq_params([dev(p, cuda) for p in nq]))
    torch.cuda.synchronize()
    err_c = (got_cos.double() - want_cos).abs().max().item()
    err_q = (got_q - want_q).abs().max().item()
    assert err_c <= 2e-3, "cosine logits at full size, %d key frames: %.3g" % (N, err_c)
    assert err_q <= 2e-3 * want_q.abs().max().item() + 1e-3, "quality logits at full size, %d key frames: %.3g" % (N, err_q)
    # run-to-run determinism (fixed summation order everywhere)
    again = ops.embed_cosine_logits(xb, graphs.pack_embed_params([dev(p, cuda) for p in ep]))
    assert torch.equal(again, got_cos), "%d key frames: embed_cosine_logits not deterministic" % N


def test_key_frame_graphs_on_tensor_cores_against_fp32_oracle(ops, cuda):
    """get_key_test_symbol end to end (SYM:468-477) with this package's tensor-core convolutions (conv_dtype='tc') against
    the float32 oracle (NumPy convolutions): only the blend weights move, by the bf16 rounding inside the networks."""
    from lsfa_b200 import graphs
    rng = np.random.default_rng(4)
    N, C, H, W = 2, 64, 12, 14
    d = make_case(4, N, C, H, W)
    first = np.array([0, 1], np.uint8)
    emb = _embed_params(rng, C, 256, 256, 512)
    nq = _nq_params(rng, C)
    t = lambda a: dev(a, cuda)  # noqa: E731
    got_f = graphs.key_frame_fgfa(t(d["key"]), t(d["mv"]), t(d["scale_map"]), t(d["cur"]), [t(a) for a in emb],
                                  is_first_frame=t(first), flow_kind="raw", conv_dtype="tc")
    got_q = graphs.key_frame_nq(t(d["key"]), t(d["mv"]), t(d["scale_map"]), t(d["cur"]), [t(a) for a in nq],
                                is_first_frame=t(first), flow_kind="raw", conv_dtype="tc")
    torch.cuda.synchronize()
    want_f = O.key_frame_fgfa_full(d["key"], d["flow"], d["scale_map"], d["cur"], emb, first)
    want_q = O.key_frame_nq_full(d["key"], d["flow"], d["scale_map"], d["cur"], nq, first)
    scale = max(np.abs(d["key"]).max(), np.abs(d["cur"]).max())
    assert np.abs(got_f.cpu().numpy() - want_f).max() <= 1e-2 * scale
    assert np.abs(got_q.cpu().numpy() - want_q).max() <= 1e-2 * scale
    assert np.array_equal(got_f.cpu().numpy()[1], d["cur"][1])          # ChooseFeat: first frame of a video keeps conv_feat


def test_tc_errors_are_loud(ops, cuda):
    from lsfa_b200 import LsfaError
    b = torch.zeros(256, device=cuda)
    z = lambda *sh, dt=torch.float32: torch.zeros(sh, dtype=dt, device=cuda)  # noqa: E731
    with pytest.raises(ValueError):                                             # the fused entries need Concat_0 of two batches
        ops.nq_logits(z(3, 4, 4, 64, dt=torch.bfloat16), (z(256, 576, dt=torch.bfloat16), z(256), z(16, 256), z(16), z(16), z(1)))
    x = torch.zeros((2, 4, 4, 32), dtype=torch.bfloat16, device=cuda)          # Cin not a multiple of 64
    with pytest.raises(LsfaError):
        ops.conv_bf16_nhwc(x, torch.zeros((256, 32), dtype=torch.bfloat16, device=cuda), b)
    x = torch.zeros((2, 4, 4, 64), dtype=torch.bfloat16, device=cuda)          # Cout not a multiple of 256
    with pytest.raises(LsfaError):
        ops.conv_bf16_nhwc(x, torch.zeros((128, 64), dtype=torch.bfloat16, device=cuda), torch.zeros(128, device=cuda))


@pytest.mark.parametrize("fuse_type", ["add", "addv2", "concat", "concatv1", "concatv2"])
@pytest.mark.parametrize("rnet_num_conv,res_fuse", [(0, "add"), (1, "add"), (0, "concat")])
def test_non_key_step_with_every_graph_switch(ops, cuda, fuse_type, rnet_num_conv, res_fuse):
    """get_cur_test_symbol's tail (SYM:570-586) with the switches the shipped yaml does not select: small_net_fuse_type
    addv2 / concat / concatv1 / concatv2 (SYM:237-272), rnet_num_conv > 0 (SYM:62-64), fuse_type 'concat' (SYM:326-328) -
    bf16 tensor-core convolutions + the fused warp against the float64-convolution oracle, 2e-2 * max|out| (several
    bf16-rounded layers deep)."""
    from lsfa_b200 import graphs
    rng = np.random.default_rng(len(fuse_type) * 10 + rnet_num_conv)
    N, C, H, W, NF = 3, 256, 10, 13, 64                  # C stands in for 1024, NF for the small net's 256
    mk = lambda co, ci, k: ((rng.standard_normal((co, ci, k, k)) / np.sqrt(ci * k * k)).astype(np.float32),  # noqa: E731
                            (0.1 * rng.standard_normal(co)).astype(np.float32))
    key = O.synth_features(rng, (N, C, H, W))
    flow = (rng.standard_normal((N, 2, H, W)) * 1.5).astype(np.float32)
    res = (rng.standard_normal((N, 3, H, W)) * 2).astype(np.float32)
    small = O.synth_features(rng, (N, NF, H, W))
    rnet = ([mk(256, 3, 3)] if rnet_num_conv else []) + [mk(C, 256 if rnet_num_conv else 3, 1)]
    sp = {"fuse_reduce_add": mk(C, NF, 3), "fuse_reduce_add_conv1": mk(256, NF, 3), "fuse_reduce_add_conv2": mk(C, 256, 1),
          "fuse_reduce_c1": mk(C if fuse_type == "concatv2" else 256, NF, 3), "fuse_reduce_c2": mk(256, C, 3), "fuse_reduce": mk(C, 512, 3),
          "s_feat_conv1": mk(C, 2 * C if fuse_type == "concatv2" else C, 1), "s_feat_conv2": mk(C, C, 1)}
    if fuse_type == "addv2":
        small = O.synth_features(rng, (N, 256, H, W))    # addv2 keeps the small net's width in its first convolution
        sp["fuse_reduce_add_conv1"] = mk(256, 256, 3)
    down = mk(C, 2 * C, 1)
    want = O.cur_frame_step(key, flow, res, rnet, small, sp, fuse_type, res_fuse, down)
    t = lambda a: dev(a, cuda)  # noqa: E731
    tp = lambda wb: (t(wb[0]), t(wb[1]))  # noqa: E731
    got = graphs.cur_frame_step(t(key), t(flow), t(res), [tp(x) for x in rnet], t(small), {k: tp(v) for k, v in sp.items()},
                                fuse_type, res_fuse, tp(down))
    torch.cuda.synchronize()
    got = got.float().permute(0, 3, 1, 2).cpu().numpy()
    err = np.abs(got - want)
    assert err.max() <= 2e-2 * np.abs(want).max(), "%s/%s: worst abs err %.3g at scale %.3g" % (fuse_type, res_fuse, err.max(), np.abs(want).max())
