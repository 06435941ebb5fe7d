"""CPU tests of the DIS oracle (oracle/dis_np.py) and of the native scale plan against cv2.DISOpticalFlow."""
import numpy as np
import pytest

cv2 = pytest.importorskip("cv2")

from oracle import dis_np, flow_ops  # noqa: E402
from tobac_flow_b200 import synthetic as S  # noqa: E402

PLAN_SHAPES = [(10, 15), (16, 16), (40, 40), (100, 100), (11, 11), (8, 8), (1, 70), (3, 400), (200, 264), (201, 263),
               (375, 625), (1500, 2500)]
MOTIONS = {"neg": S.shift_motion(-1.7, 0.6), "large": S.shift_motion(6.3, -4.2), "rotation": S.rotation_motion(3.0),
           "zoom": S.zoom_motion(1.03), "split": S.split_motion(2.0)}


def _epe(a, b):
    return np.sqrt(((a.astype(np.float64) - b) ** 2).sum(-1))


def _within(a, b, mean=1e-3, p99=1e-2):
    e = _epe(a, b)
    assert e.mean() <= mean and np.percentile(e, 99) <= p99, (e.mean(), np.percentile(e, 99), e.max())


@pytest.mark.parametrize("shape", [(375, 625), (201, 263), (200, 264), (187, 312), (100, 100), (93, 156)])
def test_pyramid_and_gradients_bit_exact(shape):
    rng = np.random.default_rng(sum(shape))
    img = rng.integers(0, 256, shape, dtype=np.uint8)
    h, w = shape
    for hh, ww in ((h // 2, w // 2), (h // 4, w // 4)):
        assert np.array_equal(dis_np.resize_area_u8(img, hh, ww), cv2.resize(img, (ww, hh), interpolation=cv2.INTER_AREA))
    gx, gy = dis_np.spatial_gradient(img)
    cx, cy = cv2.spatialGradient(img)
    assert np.array_equal(gx, cx) and np.array_equal(gy, cy)


def _cv2_plan(shape, preset):
    m = cv2.DISOpticalFlow_create(preset)
    a = np.zeros(shape, np.uint8)
    try:
        m.calc(a, a, None)
    except cv2.error:
        return None
    return m.getFinestScale()


@pytest.mark.parametrize("shape", PLAN_SHAPES)
def test_scale_plan_matches_cv2(shape):
    from tobac_flow_b200 import DISOpticalFlow, NativeError
    for preset in (0, 1, 2):
        want = _cv2_plan(shape, preset)
        model = DISOpticalFlow(preset)
        if want is None:
            with pytest.raises(ValueError):
                dis_np.scale_plan(*shape, dis_np.PRESETS[preset][0])
            with pytest.raises(NativeError):
                model.scale_plan(*shape)
            continue
        finest, coarsest, sizes = model.scale_plan(*shape)
        assert finest == want
        assert (finest, coarsest) == dis_np.scale_plan(*shape, dis_np.PRESETS[preset][0])
        assert sizes == dis_np.scale_sizes(*shape, finest, coarsest)


@pytest.mark.parametrize("preset", [0, 1, 2])
@pytest.mark.parametrize("motion", sorted(MOTIONS))
@pytest.mark.parametrize("shape", [(96, 128), (75, 101)])
def test_oracle_matches_cv2_on_motions(preset, motion, shape):
    fr = S.moving_texture(*shape, [MOTIONS[motion]], seed=3)
    q0, q1 = flow_ops.pair_to_u8(fr[0], fr[1])
    for a, b in ((q0, q1), (q1, q0)):
        _within(dis_np.dis(a, b, preset), dis_np.dis_cv2(a, b, preset))


@pytest.mark.parametrize("preset", [0, 1, 2])
@pytest.mark.parametrize("shape", [(10, 15), (16, 16), (40, 40), (24, 40)])
def test_oracle_matches_cv2_on_tiny_frames(preset, shape):
    fr = S.moving_texture(*shape, [S.shift_motion(0.8, -0.4)], seed=5)
    q0, q1 = flow_ops.pair_to_u8(fr[0], fr[1])
    _within(dis_np.dis(q0, q1, preset), dis_np.dis_cv2(q0, q1, preset))


@pytest.mark.parametrize("preset", [0, 1, 2])
def test_oracle_matches_cv2_with_nan_patched_frames(preset):
    bt = S.bt_sequence(3, 72, 96, seed=4, nans=True)
    bt[2, 10:30, 5:40] = np.nan
    bt[2, :, 90:] = np.nan
    q0, q1 = flow_ops.pair_to_u8(bt[1], bt[2])
    for a, b in ((q0, q1), (q1, q0)):
        _within(dis_np.dis(a, b, preset), dis_np.dis_cv2(a, b, preset))


def test_oracle_overrides_match_cv2():
    fr = S.moving_texture(64, 96, [S.rotation_motion(2.0)], seed=6)
    q0, q1 = flow_ops.pair_to_u8(fr[0], fr[1])
    for kw in (dict(finest_scale=1), dict(patch_stride=2), dict(gradient_descent_iterations=7),
               dict(variational_refinement_iterations=2)):
        _within(dis_np.dis(q0, q1, 1, **kw), dis_np.dis_cv2(q0, q1, 1, **kw))
