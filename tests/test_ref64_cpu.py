"""The float64 reference and its gate (oracle/ref64.py), on the CPU: the reference's coordinates are the oracle's
bits, the MXNet-faithful float32 oracle meets the gate in every mode, and the gate fails on small, realistic bugs."""
import numpy as np
import pytest
import torch

from oracle import lsfa_oracle as O
from oracle import ref64 as R
from tests._util import assert_close_bf16, make_case, oracle_fused

SHAPES = [(3, 64, 38, 63), (2, 8, 68, 120), (4, 16, 7, 9)]
BF16_KEYS = ("key", "cur", "scale_map", "emb_warp", "emb_cur")


def _t(d, k):
    return torch.from_numpy(d[k]) if k in d else None


def ref_of(d, mode, co=None, use_res=False, **over):
    """ref64.forward on the arrays of a make_case dict (``over`` replaces some of them)."""
    d = dict(d, **over)
    co = R.coords(mv=d["mv"], key_hw=d["key"].shape[2:]) if co is None else co
    return R.forward(_t(d, "key"), co, cur=_t(d, "cur"), scale_map=_t(d, "scale_map"),
                     res=_t(d, "res") if use_res else None, rnet_w=_t(d, "rnet_w"), rnet_b=_t(d, "rnet_b"), mode=mode,
                     logits=_t(d, "logits"), emb_warp=_t(d, "emb_warp"), emb_cur=_t(d, "emb_cur"), bypass=d.get("bypass"),
                     key_index=d.get("key_index"))


def case(shape, mode, seed=7, **kw):
    E = (2048 if shape[2] * shape[3] < 3000 else 256) if mode == "cosine" else 0
    return make_case(seed, *shape, E=E, max_px=64, **kw)


@pytest.mark.parametrize("raw,max_px", [(True, 32), ("ragged", 64), ("ragged", 4000)])
def test_coordinates_are_the_oracle_bits(raw, max_px):
    d = make_case(3, 5, 4, 12, 9, raw=raw, max_px=max_px)
    want = O.sampler_coords(O.grid_generator_warp(O.mv_pool(d["mv"])), 12, 9)
    for a, b in zip(R.coords(mv=d["mv"]), want):
        assert a.dtype == b.dtype and np.array_equal(a.view(np.uint32), b.view(np.uint32))
    for a, b in zip(R.coords(flow=d["flow"]), want):
        assert np.array_equal(a, b)
    if max_px == 4000:
        x0, y0 = want[0], want[1]
        assert ((x0 < -1) | (x0 > 8) | (y0 < -1) | (y0 > 11)).any()          # some pixels sample outside the plane


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("mode", ["none", "add", "mean", "logits", "cosine"])
@pytest.mark.parametrize("extra", ["plain", "res_bypass", "shared_key", "no_scale"])
def test_oracle_meets_the_gate(shape, mode, extra):
    kw = {"res_bypass": dict(with_res=True, with_bypass=True), "shared_key": dict(shared_key=True)}.get(extra, {})
    d = case(shape, mode, raw="ragged", **kw)
    use_res = extra == "res_bypass"
    if extra == "no_scale":
        d.pop("scale_map")
    m = R.MODES[mode]
    co = R.coords(mv=d["mv"], key_hw=d["key"].shape[2:])
    want = oracle_fused(d, m, use_scale="scale_map" in d, use_res=use_res)
    ref, mag = ref_of(d, mode, co, use_res=use_res)
    R.check(want, ref, mag, "f32", what=mode)             # measured <= 8 u mag in logits mode, K = 16
    # bf16 kernels read bf16 features and round their float32 result once
    db = dict(d, **{k: O.bf16_round(d[k]) for k in BF16_KEYS if k in d})
    want_b = O.bf16_round(oracle_fused(db, m, use_scale="scale_map" in d, use_res=use_res))
    ref_b, mag_b = ref_of(db, mode, co, use_res=use_res)
    assert R.check(want_b, ref_b, mag_b, "bf16", what=mode + " bf16") <= 1.0
    if "bypass" in d and mode != "none":
        b = d["bypass"].astype(bool)
        assert torch.equal(ref[b], torch.from_numpy(d["cur"][b]).double()) and not bool(mag[b].any())


@pytest.mark.parametrize("mode", ["none", "add", "mean", "logits"])
@pytest.mark.parametrize("shape", [(3, 16, 38, 63), (2, 6, 12, 20)])
def test_oracle_backward_meets_the_gate(shape, mode):
    d = make_case(11, *shape, max_px=64, with_bypass=mode != "none")
    rng = np.random.default_rng(5)
    og = rng.standard_normal(d["key"].shape).astype(np.float32)
    m = R.MODES[mode]
    cur = d["cur"] if m != O.W_NONE else None
    want = O.warp_scale_aggregate_backward(og, d["key"], d["flow"], cur=cur, scale_map=d["scale_map"], weight_mode=m,
                                           logits=d["logits"], bypass=d.get("bypass"))
    got = R.backward(torch.from_numpy(og), torch.from_numpy(d["key"]), R.coords(flow=d["flow"]),
                     cur=None if cur is None else torch.from_numpy(cur), scale_map=torch.from_numpy(d["scale_map"]),
                     mode=mode, logits=torch.from_numpy(d["logits"]), bypass=d.get("bypass"))
    expect = {"key", "flow", "scale"} | ({"cur"} if cur is not None else set()) | ({"logits"} if mode == "logits" else set())
    assert set(got) == expect
    for k, (ref, mag, na) in got.items():
        assert R.check(want[k], ref, mag, n_addends=na, what=k) <= 1.0
    # the sampler's own backward (warp_backward: grad_key, grad_flow)
    gk, gf = O.warp_backward(d["key"], d["flow"], og)
    got = R.backward(torch.from_numpy(og), torch.from_numpy(d["key"]), R.coords(flow=d["flow"]))
    assert set(got) == {"key", "flow"}
    assert R.check(gk, *got["key"][:2], n_addends=got["key"][2], what="warp_backward key") <= 1.0
    assert R.check(gf, *got["flow"][:2], n_addends=got["flow"][2], what="warp_backward flow") <= 1.0


def test_chunks_and_frame_ranges_compose():
    d = make_case(9, 19, 4, 10, 11, max_px=64, with_bypass=True)
    co = R.coords(mv=d["mv"])
    ref, mag = ref_of(d, "logits", co)
    part = R.forward(_t(d, "key"), co, cur=_t(d, "cur"), scale_map=_t(d, "scale_map"), mode="logits",
                     logits=_t(d, "logits"), bypass=d["bypass"], frames=range(9, 17))
    assert torch.equal(part[0], ref[9:17]) and torch.equal(part[1], mag[9:17])


# ------------------------------------------------------------------------------------------------------------------
# the gate bites: each mutation below is a plausible kernel bug and must fail it
# ------------------------------------------------------------------------------------------------------------------
def _fails(got, ref, mag, match=None, **kw):
    with pytest.raises(AssertionError, match=match):
        R.check(got, ref, mag, **kw)


@pytest.fixture(scope="module")
def logits_case():
    d = make_case(21, 4, 16, 38, 63, max_px=64)
    co = R.coords(mv=d["mv"])
    ref, mag = ref_of(d, "logits", co)
    R.check(oracle_fused(d, O.W_LOGITS), ref, mag)
    return d, co, ref, mag


def test_gate_catches_one_pixel_with_mirrored_weights(logits_case):
    d, co, ref, mag = logits_case
    x0, y0, wx, wy = (a.copy() for a in co)
    inside = (x0 >= 0) & (x0 < 62) & (y0 >= 0) & (y0 < 37)
    n, y, x = np.argwhere(inside & (np.abs(wx - 0.5) > 0.4))[0]
    wx[n, y, x] = np.float32(1) - wx[n, y, x]
    got, _ = ref_of(d, "logits", (x0, y0, wx, wy))
    _fails(got, ref, mag, match=r"frames with failures: %d$" % n)


def test_gate_catches_last_row_and_column_treated_as_outside(logits_case):
    d, co, ref, mag = logits_case
    key = d["key"].copy()          # a tap on row H-1 or column W-1 read as 0: what '< W-1' instead of '<= W-1' does
    key[:, :, -1, :] = 0
    key[:, :, :, -1] = 0
    got, _ = ref_of(d, "logits", co, key=key)
    _fails(got, ref, mag)


def test_gate_catches_logits_swapped_in_one_frame(logits_case):
    d, co, ref, mag = logits_case
    lg = d["logits"].copy()
    lg[2] = lg[2, ::-1]
    _fails(oracle_fused(dict(d, logits=lg), O.W_LOGITS), ref, mag, match=r"frames with failures: 2$")


def test_gate_catches_the_next_frames_scale_map(logits_case):
    d, co, ref, mag = logits_case
    sm = d["scale_map"].copy()
    sm[1] = sm[2]
    _fails(oracle_fused(dict(d, scale_map=sm), O.W_LOGITS), ref, mag, match=r"frames with failures: 1$")


def test_gate_catches_one_channel_plane_shifted_by_one_pixel(logits_case):
    d, co, ref, mag = logits_case
    got = oracle_fused(d, O.W_LOGITS)
    got[3, 5] = np.roll(got[3, 5], 1, axis=-1)
    _fails(got, ref, mag, match=r"frames with failures: 3$")


def test_gate_catches_cosine_without_its_eps(monkeypatch):
    d = make_case(22, 2, 8, 7, 9, E=64, max_px=64)            # emb_cur has an all-zero pixel
    ref, mag = ref_of(d, "cosine")
    R.check(oracle_fused(d, O.W_COSINE), ref, mag)
    l2n = O.l2norm_channel
    monkeypatch.setattr(O, "l2norm_channel", lambda e, eps=0.0: l2n(e, 0.0))
    with np.errstate(invalid="ignore", divide="ignore"):
        got = oracle_fused(d, O.W_COSINE)
    _fails(got, ref, mag)


def test_gate_catches_one_bf16_ulp_on_a_small_element():
    d = make_case(23, 2, 64, 38, 63, max_px=64)
    db = dict(d, **{k: O.bf16_round(d[k]) for k in ("key", "cur", "scale_map")})
    ref, mag = ref_of(db, "logits")
    got = O.bf16_round(oracle_fused(db, O.W_LOGITS))
    assert R.check(got, ref, mag, "bf16") <= 1.0
    r = ref.numpy()
    small = (np.abs(r) < np.abs(r).max() / 16) & (np.abs(r) > 1e-3)
    i = tuple(np.argwhere(small)[0])
    u = got.view(np.uint32).copy()
    away = 1 if (got[i] >= r[i]) == (got[i] >= 0) else -1        # one ulp further from ref (toward larger |x| or smaller)
    u[i] = np.uint32(int(u[i]) + away * (1 << 16))
    bad = u.view(np.float32)
    assert_close_bf16(bad, r)                                    # the max-relative gate of tests/_util.py accepts it
    _fails(bad, ref, mag, out="bf16")


def test_gate_catches_one_dropped_addend_in_grad_key():
    d = make_case(24, 2, 8, 12, 20, max_px=64)
    rng = np.random.default_rng(1)
    og = rng.standard_normal(d["key"].shape).astype(np.float32)
    got = R.backward(torch.from_numpy(og), torch.from_numpy(d["key"]), R.coords(flow=d["flow"]))
    ref, mag, na = got["key"]
    x0, y0, wx, wy = R.coords(flow=d["flow"])
    inside = (x0 >= 0) & (x0 < 19) & (y0 >= 0) & (y0 < 11) & (np.abs(wx - 0.5) < 0.3) & (np.abs(wy - 0.5) < 0.3)
    n, y, x = np.argwhere(inside)[0]
    og2 = og.copy()
    og2[n, 3, y, x] = 0                    # the four key elements this pixel samples each lose one addend
    gk, _ = O.warp_backward(d["key"], d["flow"], og2)
    assert R.check(O.warp_backward(d["key"], d["flow"], og)[0], ref, mag, n_addends=na) <= 1.0
    _fails(gk, ref, mag, n_addends=na, match=r"frames with failures: %d$" % n)


def test_check_reports_nan_and_frames():
    ref = torch.ones((6, 2, 3, 3), dtype=torch.float64)
    mag = torch.ones_like(ref)
    got = ref.clone()
    got[4:, 0, 1, 1] = float("nan")
    _fails(got, ref, mag, match=r"frames with failures: 4-5")
