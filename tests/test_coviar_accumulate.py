"""Upstream widening (SURVEY.md 8f rank 3): coviar's accumulated MV field + residual.
CPU: the two oracle forms (pure-Python literal loop, C restatement of coviar_data_loader.c:71-177)
agree and satisfy the reference's own reconstruction identity (lib/utils/image.py:79-89).
GPU: lsfa_mv_accumulate_i32 / lsfa_coviar_residual_u8 are bit-exact, and the whole chain
lists -> accumulated MV -> (sign, resize, pool, warp, aggregate) matches the oracle chain."""
import numpy as np
import pytest

from oracle import c_port as P
from oracle import lsfa_oracle as O


def test_oracles_agree_and_known_answers():
    P.build()
    rng = np.random.default_rng(0)
    for (T, h, w) in [(1, 32, 48), (3, 48, 80), (5, 40, 56)]:
        mvs, counts = O.synth_mv_lists(rng, T, h, w)
        a = O.coviar_accumulate(mvs, counts, h, w)
        assert np.array_equal(a, P.mv_accumulate(mvs, counts, h, w))
    # no vectors / static vectors -> zero field
    z = np.zeros((2, 4, 6), np.int32); z[:, :, :2] = 16; z[:, :, 2:] = 8
    assert not P.mv_accumulate(z, np.array([4, 4], np.int32), 32, 32).any()
    assert not P.mv_accumulate(z, np.array([0, 0], np.int32), 32, 32).any()
    # one 16x16 block moved by (+3,-2): mv = dst - src inside the block, 0 elsewhere
    one = np.array([[[16, 16, 8 + 16 - 3, 8 + 16 + 2, 8 + 16, 8 + 16]]], np.int32)
    f = P.mv_accumulate(one, np.array([1], np.int32), 64, 64)
    assert (f[16:32, 16:32] == (3, -2)).all() and not f[:16].any() and not f[32:].any()
    # two frames compose: frame 2 moves the same block again by (+1,+1) -> back-trace through frame 1
    two = np.concatenate([one, np.array([[[16, 16, 24 - 1, 24 - 1, 24, 24]]], np.int32)])
    f2 = P.mv_accumulate(two, np.array([1, 1], np.int32), 64, 64)
    assert (f2[17:32, 17:32] == (4, -1)).all()        # pixels whose frame-1 source was itself inside the moved block
    # later vector overwrites an earlier one on the overlap
    ov = np.array([[[16, 16, 20, 24, 24, 24], [8, 8, 30, 30, 28, 28]]], np.int32)
    f3 = P.mv_accumulate(ov, np.array([2], np.int32), 64, 64)
    assert (f3[24:32, 24:32] == (-2, -2)).all() and (f3[16:24, 16:24] == (4, 0)).all()


def test_reconstruction_identity_of_the_reference():
    """lib/utils/image.py:79-89 check_reconstruction: ref_im[y - mv_y, x - mv_x] + res == im[y, x]."""
    rng = np.random.default_rng(1)
    h, w = 48, 64
    mvs, counts = O.synth_mv_lists(rng, 4, h, w)
    mv = P.mv_accumulate(mvs, counts, h, w)
    iframe = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    cur = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    res = P.coviar_residual(iframe, cur, mv)
    assert np.array_equal(res, O.coviar_residual(iframe, cur, mv))
    ys, xs = np.mgrid[0:h, 0:w]
    assert np.array_equal(iframe[ys - mv[..., 1], xs - mv[..., 0]].astype(np.int32) + res, cur.astype(np.int32))


@pytest.mark.gpu
@pytest.mark.parametrize("algo", ["auto", "field", "trace"])
@pytest.mark.parametrize("N,T,h,w", [(1, 1, 32, 48), (3, 4, 48, 80), (2, 11, 96, 160), (2, 3, 45, 77),
                                     (1, 11, 720, 1280)])       # a full-size GOP: 11 P-frames at 720p
def test_gpu_mv_accumulate_bit_exact(cuda, N, T, h, w, algo):
    import torch
    from lsfa_b200 import ops
    rng = np.random.default_rng(N * 100 + T)
    lists = [O.synth_mv_lists(rng, T, h, w, extra=6) for _ in range(N)]
    mvs = np.stack([l[0] for l in lists]); counts = np.stack([l[1] for l in lists])
    counts[0, 0] = max(0, counts[0, 0] - 3)            # ragged counts
    want = np.stack([P.mv_accumulate(mvs[n], counts[n], h, w) for n in range(N)])
    got = ops.mv_accumulate(torch.from_numpy(mvs).to(cuda), torch.from_numpy(counts).to(cuda), h, w, algo=algo)
    torch.cuda.synchronize()
    assert np.array_equal(got.cpu().numpy(), want)
    iframe = rng.integers(0, 256, (N, h, w, 3), dtype=np.uint8)
    cur = rng.integers(0, 256, (N, h, w, 3), dtype=np.uint8)
    res = ops.coviar_residual(torch.from_numpy(iframe).to(cuda), torch.from_numpy(cur).to(cuda), got)
    want_res = np.stack([P.coviar_residual(iframe[n], cur[n], want[n]) for n in range(N)])
    assert np.array_equal(res.cpu().numpy(), want_res)


@pytest.mark.gpu
def test_gpu_chain_from_motion_vector_lists_to_aggregated_feature(cuda):
    """lists -> accumulated MV (coviar) -> sign/resize/pool -> warp -> x scale -> logits blend, all on the GPU,
    against the oracle chain."""
    import torch
    from lsfa_b200 import ops
    from tests._util import assert_close_f32
    rng = np.random.default_rng(9)
    N, T, h, w, scale = 2, 5, 180, 240, 600.0 / 180.0 / 2.0
    lists = [O.synth_mv_lists(rng, T, h, w) for _ in range(N)]
    mvs = np.stack([l[0] for l in lists]); counts = np.stack([l[1] for l in lists])
    field = np.stack([P.mv_accumulate(mvs[n], counts[n], h, w) for n in range(N)])
    flow = O.mv_pool(np.stack([O.resize_linear_f32(O.mv_sign_flip(f), scale) for f in field]), scale)
    _, _, H, W = flow.shape
    C = 16
    key = O.synth_features(rng, (N, C, H, W)); cur = O.synth_features(rng, (N, C, H, W))
    sm = O.synth_scale_map(rng, (N, C, H, W)); lg = rng.standard_normal((N, 2, H, W), dtype=np.float32)
    want = O.warp_scale_aggregate(key, flow, cur=cur, scale_map=sm, weight_mode=O.W_LOGITS, logits=lg)
    t = lambda a: torch.from_numpy(a).to(cuda)  # noqa: E731
    gfield = ops.mv_accumulate(t(mvs), t(counts), h, w)
    got = ops.warp_scale_aggregate(t(key), gfield, flow_kind="coviar", im_scale=scale, negate=True,
                                   cur=t(cur), scale_map=t(sm), weight_mode="logits", logits=t(lg))
    torch.cuda.synchronize()
    assert_close_f32(got.cpu().numpy(), want, scale=max(np.abs(key).max(), np.abs(cur).max()), what="chain")


@pytest.mark.gpu
def test_gpu_back_trace_adversarial_lists(cuda):
    """The cell-index back-trace on lists that defeat its fast path: unaligned blocks of odd sizes, vectors that overlap
    earlier ones, static vectors (skipped, coviar_data_loader.c:92) sitting on top of moving ones, sources and
    destinations leaving the frame on every side, an empty frame, and a frame that is not a multiple of the 8x8 cell."""
    import torch
    from lsfa_b200 import ops
    rng = np.random.default_rng(99)
    N, T, h, w, M = 3, 6, 53, 71, 90
    mvs = np.zeros((N, T, M, 6), np.int32)
    counts = np.full((N, T), M, np.int32)
    for n in range(N):
        for t in range(T):
            for i in range(M):
                bw, bh = (int(v) for v in rng.choice([3, 4, 5, 8, 15, 16, 17], 2))
                dx, dy = int(rng.integers(-6, w + 6)), int(rng.integers(-6, h + 6))
                ox, oy = (0, 0) if rng.random() < 0.25 else (int(v) for v in rng.integers(-20, 21, 2))
                mvs[n, t, i] = (bw, bh, dx + ox, dy + oy, dx, dy)
    counts[1, 2] = 0
    counts[2, 4] = 7
    want = np.stack([P.mv_accumulate(mvs[n], counts[n], h, w) for n in range(N)])
    for algo in ("trace", "field"):
        got = ops.mv_accumulate(torch.from_numpy(mvs).to(cuda), torch.from_numpy(counts).to(cuda), h, w, algo=algo)
        torch.cuda.synchronize()
        assert np.array_equal(got.cpu().numpy(), want), algo
