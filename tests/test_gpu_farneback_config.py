"""GPU tests of the configurable Farneback model (tobac_flow_b200/farneback.py, tf_farneback_config_pairs and the
general-window iteration kernel csrc/fb_iter_general.cu) against cv2.FarnebackOpticalFlow and the oracle."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

cv2 = pytest.importorskip("cv2")
torch = pytest.importorskip("torch")

import tobac_flow_b200 as tfb  # noqa: E402
from oracle import farneback_np, flow_ops  # noqa: E402
from tobac_flow_b200 import _lib, distributed as D, synthetic as S  # noqa: E402
from tobac_flow_b200.farneback import FarnebackOpticalFlow, polyexp, pyramid_level  # noqa: E402
from tests.test_oracle_farneback_config import GRID, cv2_farneback  # noqa: E402

MOTIONS = {"shift": S.shift_motion(-1.7, 0.6), "large": S.shift_motion(6.3, -4.2), "rotation": S.rotation_motion(3.0),
           "zoom": S.zoom_motion(1.03), "split": S.split_motion(2.0)}
LEGACY = dict(flags=256, win_size=16, num_iters=3)


def _epe(a, b):
    return np.sqrt(((np.asarray(a, np.float64) - b) ** 2).sum(-1))


def _check(mine, want):
    """Mean EPE <= 1e-3 px, p99 <= 1e-2 px, and mean <= 5e-3 px in each 8-px border band."""
    e = _epe(mine, want)
    assert e.mean() <= 1e-3 and np.percentile(e, 99) <= 1e-2, (e.mean(), np.percentile(e, 99), e.max())
    for band in (e[:8], e[-8:], e[:, :8], e[:, -8:]):
        assert band.mean() <= 5e-3, band.mean()


def _pairs(q0s, q1s, model, max_value=0.0):
    """tf_farneback_config_pairs on (n, H, W) u8 pairs -> (fwd, bwd) numpy (n, H, W, 2)."""
    dev = torch.device("cuda")
    a = torch.from_numpy(np.ascontiguousarray(q0s)).to(dev)
    b = torch.from_numpy(np.ascontiguousarray(q1s)).to(dev)
    n, H, W = a.shape
    nbytes = model.workspace_bytes(n, H, W)
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
    f = torch.empty((n, H, W, 2), dtype=torch.float32, device=dev)
    g = torch.empty((n, H, W, 2), dtype=torch.float32, device=dev)
    _lib.check(_lib.load().tf_farneback_config_pairs(
        a.data_ptr(), b.data_ptr(), f.data_ptr(), H * W * 2, g.data_ptr(), H * W * 2, n, H, W,
        ctypes.byref(model.params(max_value)), ws.data_ptr(), nbytes,
        ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)), "tf_farneback_config_pairs")
    return f.cpu().numpy(), g.cpu().numpy()


def _u8_pair(H, W, seed):
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:H, 0:W]
    base = 120 + 80 * np.sin(xx / 17.0 + seed) * np.cos(yy / 11.0) + 20 * rng.standard_normal((H, W))
    return np.clip(base, 0, 255).astype(np.uint8), np.clip(np.roll(base, (1, 2), (0, 1)), 0, 255).astype(np.uint8)


# ---- stages -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("pyr_scale,shape", [(0.3, (375, 625)), (0.7, (300, 500)), (0.48, (1300, 1400))])
def test_pyramid_levels_vs_oracle(pyr_scale, shape):
    q0, q1 = _u8_pair(*shape, seed=int(pyr_scale * 100))
    model = FarnebackOpticalFlow(num_levels=15, pyr_scale=pyr_scale)
    plan = farneback_np.level_plan(*shape, 15, pyr_scale)
    assert model.level_plan(*shape) == [(p["h"], p["w"]) for p in plan]
    if pyr_scale == 0.48:
        assert max(p["ksize"] for p in plan) > 96          # the two-pass path with the wide taps
        levels = [i for i, p in enumerate(plan) if p["ksize"] > 96] + [len(plan) - 2]
    else:
        levels = range(len(plan))
    for li in levels:
        got = pyramid_level(q0, q1, model, li)
        for k, q in enumerate((q0, q1)):
            ref = farneback_np.pyramid_level(q, plan[li])
            assert np.abs(got[k] - ref).max() <= 2e-4, (li, plan[li]["ksize"], k, np.abs(got[k] - ref).max())


@pytest.mark.parametrize("h,w", [(47, 78), (375, 625), (33, 130), (200, 119)])
def test_polyexp7_vs_oracle(h, w):
    rng = np.random.default_rng(h * 1000 + w)
    yy, xx = np.mgrid[0:h, 0:w]
    img = (128 + 90 * np.sin(xx / 9.0) * np.cos(yy / 7.0) + 10 * rng.standard_normal((h, w))).astype(np.float32)
    img2 = rng.uniform(0, 255, (h, w)).astype(np.float32)
    out = polyexp(np.stack([img, img2]), FarnebackOpticalFlow(poly_n=7, poly_sigma=1.5))
    for k, im in enumerate((img, img2)):
        ref = farneback_np.poly_exp(im, 7, 1.5)
        err = np.abs(out[k] - ref).max(axis=(0, 1)) / np.abs(ref).max(axis=(0, 1))
        assert (err <= 2e-5).all(), err


def test_polyexp5_through_config_equals_default():
    rng = np.random.default_rng(5)
    img = rng.uniform(0, 255, (2, 94, 156)).astype(np.float32)
    assert np.array_equal(polyexp(img, FarnebackOpticalFlow()), tfb.flow.fb_polyexp(img))


# ---- whole flow against cv2 ----------------------------------------------------------------------------------------
# The smallest windows (box 3, Gaussian 4: radius 1 and 2) solve nearly singular systems at some pixels, where the
# last-bit differences of any two fp32 orderings grow to pixels: on the sharp synthetic textures the numpy oracle is
# as far from cv2 there as the GPU (mean up to 2e-2 px, isolated pixels up to 28 px).  They are checked on a smooth
# pair instead; for the Gaussian 4 the bulk (p99, median) is gated, a few isolated pixels still differ by pixels.
SMALLEST = ("box3", "gauss4")


@pytest.mark.parametrize("motion", sorted(MOTIONS))
@pytest.mark.parametrize("name,kw", [g for g in GRID if g[0] not in SMALLEST],
                         ids=[g[0] for g in GRID if g[0] not in SMALLEST])
def test_config_pairs_match_cv2(name, kw, motion):
    fr = S.moving_texture(201, 263, [MOTIONS[motion]], seed=11)
    q0, q1 = flow_ops.pair_to_u8(fr[0], fr[1])
    model = FarnebackOpticalFlow(**kw)
    f, b = _pairs(q0[None], q1[None], model)
    _check(f[0], cv2_farneback(q0, q1, **kw))
    _check(b[0], cv2_farneback(q1, q0, **kw))


@pytest.mark.parametrize("name,kw", [g for g in GRID if g[0] in SMALLEST], ids=list(SMALLEST))
def test_smallest_windows_match_cv2(name, kw):
    from tests.test_oracle_farneback_config import textured_pair
    q0, q1 = textured_pair(201, 263)
    f, b = _pairs(q0[None], q1[None], FarnebackOpticalFlow(**kw))
    for mine, want in ((f[0], cv2_farneback(q0, q1, **kw)), (b[0], cv2_farneback(q1, q0, **kw))):
        if name == "box3":
            _check(mine, want)
        else:
            e = _epe(mine, want)
            assert np.percentile(e, 99) <= 1e-2 and np.median(e) <= 1e-4, (np.percentile(e, 99), np.median(e))


@pytest.mark.parametrize("kw", [LEGACY, dict(win_size=21), dict(poly_n=7, poly_sigma=1.5, pyr_scale=0.7)])
def test_batch_equals_one_by_one(kw):
    bt = S.bt_sequence(6, 120, 160, seed=9, nans=True)
    pairs = [flow_ops.pair_to_u8(bt[i], bt[i + 1]) for i in range(5)]
    q0 = np.stack([p[0] for p in pairs])
    q1 = np.stack([p[1] for p in pairs])
    model = FarnebackOpticalFlow(**kw)
    f, b = _pairs(q0, q1, model)
    for i in range(5):
        fi, bi = _pairs(q0[i:i + 1], q1[i:i + 1], model)
        assert np.array_equal(f[i], fi[0]) and np.array_equal(b[i], bi[0])


def test_default_model_bit_identical_to_string_model():
    bt = S.bt_sequence(6, 130, 170, seed=4, nans=True)
    a = tfb.create_flow(bt, model="Farneback")
    m = tfb.create_flow(bt, model=FarnebackOpticalFlow())
    assert np.array_equal(a.forward_flow, m.forward_flow, equal_nan=True)
    assert np.array_equal(a.backward_flow, m.backward_flow, equal_nan=True)


def _cv2_create_flow(data, kw, smoothing_passes=0, interp_method="linear", max_value=20, vr_steps=0):
    """flow_ops.create_flow with cv2.FarnebackOpticalFlow at the settings `kw` as the model."""
    T = data.shape[0]
    fwd = np.full(data.shape + (2,), np.nan, dtype=np.float32)
    bwd = np.full(data.shape + (2,), np.nan, dtype=np.float32)
    for i in range(T - 1):
        q0, q1 = flow_ops.pair_to_u8(data[i], data[i + 1])
        f, b = cv2_farneback(q0, q1, **kw), cv2_farneback(q1, q0, **kw)
        if vr_steps > 0:
            f, b = flow_ops.refine_pair(q0, q1, f, b, "cv2")
        for _ in range(smoothing_passes):
            f, b = flow_ops.smooth_flow_step(f, b, interp_method, "cv2")
        fwd[i], bwd[i + 1] = f, b
    fwd[-1], bwd[0] = -bwd[-1], -fwd[0]
    return np.clip(fwd, -max_value, max_value), np.clip(bwd, -max_value, max_value)


def test_legacy_create_flow_refined_smoothed_matches_cv2():
    bt = S.bt_sequence(5, 96, 128, seed=3, nans=True)
    flow = tfb.create_flow(bt, model=FarnebackOpticalFlow(**LEGACY), vr_steps=1, smoothing_passes=1,
                           interp_method="cubic")
    ref_f, ref_b = _cv2_create_flow(bt, LEGACY, smoothing_passes=1, interp_method="cubic", vr_steps=1)
    for mine, ref in ((flow.forward_flow, ref_f), (flow.backward_flow, ref_b)):
        e = _epe(mine, ref)
        assert e.mean() <= 1e-3 and np.percentile(e, 99) <= 1e-2, (e.mean(), e.max())


def test_legacy_host_path_fused_clamp_and_device_input():
    # > 16 frames of host input take the chunked upload path with per-batch events and the fused clamp
    bt = S.bt_sequence(20, 64, 96, seed=5, nans=True)
    model = FarnebackOpticalFlow(**LEGACY)
    flow = tfb.create_flow(bt, model=model, max_value=0.5)
    ref_f, ref_b = _cv2_create_flow(bt, LEGACY, max_value=0.5)
    for mine, ref in ((flow.forward_flow, ref_f), (flow.backward_flow, ref_b)):
        assert np.abs(mine).max() <= 0.5
        e = _epe(mine, ref)
        assert e.mean() <= 1e-3 and np.percentile(e, 99) <= 1e-2, (e.mean(), e.max())
    d = tfb.create_flow(torch.from_numpy(bt).cuda(), model=model, max_value=0.5)
    assert np.array_equal(flow.forward_flow, d.forward_flow) and np.array_equal(flow.backward_flow, d.backward_flow)
    f2, b2 = tfb.calculate_flow_2(bt[:-1], bt[1:], model=model)
    f1, b1 = tfb.calculate_flow(bt, model=model)
    assert np.array_equal(f2[:18], f1[:18]) and np.array_equal(b2[1:19], b1[1:19])


def test_legacy_full_size_pair_matches_cv2():
    bt = S.bt_sequence(2, 1500, 2500, seed=7, nans=True)
    q0, q1 = flow_ops.pair_to_u8(bt[0], bt[1])
    f, b = _pairs(q0[None], q1[None], FarnebackOpticalFlow(**LEGACY))
    _check(f[0], cv2_farneback(q0, q1, **LEGACY))
    _check(b[0], cv2_farneback(q1, q0, **LEGACY))


def test_calc_matches_cv2_numpy_and_device():
    fr = S.moving_texture(96, 128, [S.rotation_motion(2.0)], seed=6)
    q0, q1 = flow_ops.pair_to_u8(fr[0], fr[1])
    model = FarnebackOpticalFlow(**LEGACY)
    host = model.calc(q0, q1)
    dev = model.calc(torch.from_numpy(q0).cuda(), torch.from_numpy(q1).cuda())
    assert isinstance(host, np.ndarray) and dev.is_cuda and np.array_equal(host, dev.cpu().numpy())
    _check(host, cv2_farneback(q0, q1, **LEGACY))
    with pytest.raises(NotImplementedError):
        model.calc(q0, q1, np.zeros(q0.shape + (2,), np.float32))


@pytest.mark.parametrize("model", [FarnebackOpticalFlow(**LEGACY), tfb.DISOpticalFlow(1)], ids=["legacy", "dis_fast"])
def test_two_shard_emulation_equals_unsharded(model, monkeypatch):
    """create_flow_sharded(model=...) of two time shards run one after the other on one GPU, the halo frames set by
    hand and the one point-to-point hand-over (rank 0's backward flow of rank 1's first frame) emulated: bit-identical
    to create_flow."""
    from types import SimpleNamespace
    mailbox = []

    def p2p(ops, group):
        for o in ops:
            if o.op is D.dist.isend:
                mailbox.append(o.tensor.clone())
            else:
                o.tensor.copy_(mailbox.pop())
    monkeypatch.setattr(D.dist, "P2POp", lambda op, tensor, peer, group=None: SimpleNamespace(op=op, tensor=tensor))
    monkeypatch.setattr(D, "_p2p", p2p)
    bt = S.bt_sequence(9, 96, 128, seed=8, nans=True)
    frames = torch.from_numpy(bt).cuda()
    whole = tfb.create_flow(frames, model=model)
    T = frames.shape[0]
    shards = [D.make_shard(frames[slice(*D.shard_bounds(T, 2, r))], r, 2) for r in range(2)]
    shards[0].buf[-1] = shards[1].buf[1]
    shards[1].buf[0] = shards[0].buf[-2]
    parts = [D.create_flow_sharded(sh, exchange=False, model=model) for sh in shards]
    fwd = torch.cat([p.fwd for p in parts]).cpu().numpy()
    bwd = torch.cat([p.bwd for p in parts]).cpu().numpy()
    assert np.array_equal(fwd, whole.forward_flow) and np.array_equal(bwd, whole.backward_flow)
