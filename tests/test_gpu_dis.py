"""GPU tests of the DIS model (tobac_flow_b200/csrc/dis.cu, tobac_flow_b200/dis.py) against cv2.DISOpticalFlow."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

cv2 = pytest.importorskip("cv2")
torch = pytest.importorskip("torch")

import tobac_flow_b200 as tfb  # noqa: E402
from oracle import dis_np, flow_ops  # noqa: E402
from tobac_flow_b200 import _lib, synthetic as S  # noqa: E402
from tobac_flow_b200.dis import DISOpticalFlow, scale_images  # noqa: E402

MOTIONS = {"neg": S.shift_motion(-1.7, 0.6), "large": S.shift_motion(6.3, -4.2), "rotation": S.rotation_motion(3.0),
           "zoom": S.zoom_motion(1.03), "split": S.split_motion(2.0)}


def _epe(a, b):
    return np.sqrt(((np.asarray(a, np.float64) - b) ** 2).sum(-1))


def _dis_pairs(q0s, q1s, model, max_value=0.0):
    """tf_dis_pairs on a batch of (n, H, W) u8 pairs -> (fwd, bwd) numpy (n, H, W, 2)."""
    dev = torch.device("cuda")
    a = torch.from_numpy(np.ascontiguousarray(q0s)).to(dev)
    b = torch.from_numpy(np.ascontiguousarray(q1s)).to(dev)
    n, H, W = a.shape
    nbytes = model.workspace_bytes(n, H, W)
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
    f = torch.empty((n, H, W, 2), dtype=torch.float32, device=dev)
    g = torch.empty((n, H, W, 2), dtype=torch.float32, device=dev)
    _lib.check(_lib.load().tf_dis_pairs(a.data_ptr(), b.data_ptr(), f.data_ptr(), H * W * 2, g.data_ptr(), H * W * 2,
                                        n, H, W, ctypes.byref(model.params(max_value)), ws.data_ptr(), nbytes,
                                        ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)), "tf_dis_pairs")
    return f.cpu().numpy(), g.cpu().numpy()


def _check(mine, want, model, shape):
    """Mean EPE <= 1e-3, p99 <= 1e-2, and mean EPE <= 5e-3 in each 8-px border band and along the stripe seams."""
    e = _epe(mine, want)
    assert e.mean() <= 1e-3 and np.percentile(e, 99) <= 1e-2, (e.mean(), np.percentile(e, 99), e.max())
    for band in (e[:8], e[-8:], e[:, :8], e[:, -8:]):
        assert band.mean() <= 5e-3, band.mean()
    finest, _, sizes = model.scale_plan(*shape)
    h, _ = sizes[finest]
    hs = 1 + (h - 8) // model.patch_stride
    stripe = -(-hs // 8)
    for k in range(1, 8):
        r = k * stripe * model.patch_stride << finest
        if 8 <= r < shape[0] - 8:
            assert e[r - 8:r + 8].mean() <= 5e-3, (k, e[r - 8:r + 8].mean())


@pytest.mark.parametrize("shape", [(375, 625), (201, 263), (96, 128)])
@pytest.mark.parametrize("preset", [1, 2])
def test_scale_images_bit_exact(shape, preset):
    rng = np.random.default_rng(sum(shape) + preset)
    q = rng.integers(0, 256, (3,) + shape, dtype=np.uint8)
    model = DISOpticalFlow(preset)
    finest, coarsest, _ = model.scale_plan(*shape)
    for scale in range(finest, coarsest + 1):
        img, gx, gy = scale_images(q, model, scale)
        for k in range(q.shape[0]):
            want = dis_np.pyramid(q[k], finest, coarsest)[scale]
            ref = q[k]
            h, w = shape
            h, w = h >> finest, w >> finest
            ref = cv2.resize(ref, (w, h), interpolation=cv2.INTER_AREA) if finest else ref
            for _ in range(scale - finest):
                ref = cv2.resize(ref, (ref.shape[1] // 2, ref.shape[0] // 2), interpolation=cv2.INTER_AREA)
            assert np.array_equal(want, ref)
            assert np.array_equal(img[k], ref), (scale, k)
            cx, cy = cv2.spatialGradient(ref)
            assert np.array_equal(gx[k], cx) and np.array_equal(gy[k], cy)


@pytest.mark.parametrize("preset", [0, 1, 2])
@pytest.mark.parametrize("motion", sorted(MOTIONS))
def test_dis_pairs_match_cv2(preset, motion):
    shape = (201, 263)
    fr = S.moving_texture(*shape, [MOTIONS[motion]], seed=11)
    q0, q1 = flow_ops.pair_to_u8(fr[0], fr[1])
    model = DISOpticalFlow(preset)
    f, b = _dis_pairs(q0[None], q1[None], model)
    _check(f[0], dis_np.dis_cv2(q0, q1, preset), model, shape)
    _check(b[0], dis_np.dis_cv2(q1, q0, preset), model, shape)


@pytest.mark.parametrize("shape", [(10, 15), (16, 16), (40, 40), (100, 100), (375, 625)])
def test_dis_tiny_and_medium_frames_match_cv2(shape):
    fr = S.moving_texture(*shape, [S.rotation_motion(2.0)], seed=12)
    q0, q1 = flow_ops.pair_to_u8(fr[0], fr[1])
    for preset in (0, 1, 2):
        got = DISOpticalFlow(preset).calc(q0, q1)
        e = _epe(got, dis_np.dis_cv2(q0, q1, preset))
        assert e.mean() <= 1e-3 and np.percentile(e, 99) <= 1e-2, (preset, e.mean(), e.max())


def test_batch_equals_one_by_one():
    bt = S.bt_sequence(6, 120, 160, seed=9, nans=True)
    pairs = [flow_ops.pair_to_u8(bt[i], bt[i + 1]) for i in range(5)]
    q0 = np.stack([p[0] for p in pairs])
    q1 = np.stack([p[1] for p in pairs])
    model = DISOpticalFlow()
    f, b = _dis_pairs(q0, q1, model)
    for i in range(5):
        fi, bi = _dis_pairs(q0[i:i + 1], q1[i:i + 1], model)
        assert np.array_equal(f[i], fi[0]) and np.array_equal(b[i], bi[0])


def test_create_flow_with_dis_matches_oracle():
    bt = S.bt_sequence(5, 96, 128, seed=3, nans=True)
    model = DISOpticalFlow()
    flow = tfb.create_flow(bt, model=model, vr_steps=1, smoothing_passes=1, interp_method="cubic")
    ref_f, ref_b = dis_np.create_flow(bt, model, smoothing_passes=1, interp_method="cubic", backend="cv2", vr_steps=1)
    for mine, ref in ((flow.forward_flow, ref_f), (flow.backward_flow, ref_b)):
        e = _epe(mine, ref)
        assert e.mean() <= 1e-3 and np.percentile(e, 99) <= 1e-2, (e.mean(), e.max())


def test_create_flow_dis_clamp_and_host_path():
    # > 16 frames of host input take the chunked upload path with per-batch events and the fused clamp
    bt = S.bt_sequence(20, 64, 96, seed=5, nans=True)
    model = DISOpticalFlow(0)
    flow = tfb.create_flow(bt, model=model, max_value=0.5)
    ref_f, ref_b = dis_np.create_flow(bt, model, max_value=0.5, backend="cv2")
    for mine, ref in ((flow.forward_flow, ref_f), (flow.backward_flow, ref_b)):
        assert np.abs(mine).max() <= 0.5
        e = _epe(mine, ref)
        assert e.mean() <= 1e-3 and np.percentile(e, 99) <= 1e-2, (e.mean(), e.max())
    assert np.array_equal(flow.diff(bt), tfb.Flow(flow.forward_flow, flow.backward_flow).diff(bt), equal_nan=True)


def test_numpy_input_equals_device_input():
    bt = S.bt_sequence(4, 80, 112, seed=2, nans=True)
    model = DISOpticalFlow(2)
    a = tfb.create_flow(bt, model=model)
    d = tfb.create_flow(torch.from_numpy(bt).cuda(), model=model)
    assert np.array_equal(a.forward_flow, d.forward_flow) and np.array_equal(a.backward_flow, d.backward_flow)
    # calculate_flow_2(a, b) over T = 3 frames computes the pairs (a[i], b[i]) for i < T - 1: fwd[0:2], bwd[1:3]
    f2, b2 = tfb.calculate_flow_2(bt[:-1], bt[1:], model=model)
    f1, b1 = tfb.calculate_flow(bt, model=model)
    assert np.array_equal(f2[:2], f1[:2]) and np.array_equal(b2[1:3], b1[1:3])
    q0, q1 = flow_ops.pair_to_u8(bt[0], bt[1])
    host = model.calc(q0, q1)
    dev = model.calc(torch.from_numpy(q0).cuda(), torch.from_numpy(q1).cuda())
    assert isinstance(host, np.ndarray) and dev.is_cuda and np.array_equal(host, dev.cpu().numpy())
    with pytest.raises(NotImplementedError):
        model.calc(q0, q1, np.zeros(q0.shape + (2,), np.float32))


def _paraboloid():
    x, y = np.meshgrid(np.arange(15), np.arange(10))
    return ((7 ** 2 - (x - 7) ** 2) * (4.5 ** 2 - (y - 4.5) ** 2)).astype(np.float32)


@pytest.mark.parametrize("shift,axis", [(1, 1), (-1, 1), (1, 0), (-1, 0)])
def test_reference_dis_paraboloid(shift, axis):
    """The reference's DIS tests: a 15 x 10 paraboloid rolled by +-1 px in x or y (atol 0.05, rounded where the
    reference rounds).  The flow is checked against cv2 on the same frames, not against the ideal +-1 px (cv2 FAST
    gives 0.96-0.97 px for the +1 px x roll)."""
    blob = _paraboloid()
    frames = np.stack([blob, np.roll(blob, shift, axis)])
    model = DISOpticalFlow()
    fwd, bwd = tfb.calculate_flow(frames, model=model)
    ref_f, ref_b = dis_np.calculate_flow(frames, model, backend="cv2")
    assert np.allclose(fwd, ref_f, atol=0.05) and np.allclose(bwd, ref_b, atol=0.05)
    assert np.array_equal(np.round(fwd), np.round(ref_f)) and np.array_equal(np.round(bwd), np.round(ref_b))
    flow = tfb.create_flow(frames, model=model)
    assert np.allclose(flow.forward_flow, np.clip(ref_f, -20, 20), atol=0.05)


@pytest.mark.parametrize("kw", [dict(finest_scale=1), dict(patch_stride=2), dict(gradient_descent_iterations=7),
                                dict(variational_refinement_iterations=2)])
def test_constructor_overrides(kw):
    fr = S.moving_texture(96, 128, [S.rotation_motion(2.0)], seed=6)
    q0, q1 = flow_ops.pair_to_u8(fr[0], fr[1])
    model = DISOpticalFlow(1, **kw)
    for k, v in kw.items():
        assert getattr(model, k) == v
    e = _epe(model.calc(q0, q1), dis_np.dis_cv2(q0, q1, 1, **kw))
    assert e.mean() <= 1e-3 and np.percentile(e, 99) <= 1e-2, (kw, e.mean(), e.max())
