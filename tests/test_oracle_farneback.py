"""Pin the numpy Farneback restatement (oracle/farneback_np.py) against cv2 and the reference goldens."""
import numpy as np
import pytest

from oracle import farneback_np as fb
from oracle import flow_ops
import make_golden as cases
from tobac_flow_b200 import synthetic

cv2 = pytest.importorskip("cv2") if flow_ops.have_cv2() else None


def epe(a, b):
    return np.sqrt(((a.astype(np.float64) - b) ** 2).sum(-1))


def test_level_plan_matches_survey_sizes():
    # SURVEY.md §8(a7) step 1
    plan = fb.level_plan(1500, 2500)
    assert [(p["h"], p["w"]) for p in plan] == [(47, 78), (94, 156), (188, 312), (375, 625), (750, 1250), (1500, 2500)]
    assert [p["ksize"] for p in plan] == [79, 39, 19, 9, 3, 3]
    assert [(p["h"], p["w"]) for p in fb.level_plan(500, 500)] == [(62, 62), (125, 125), (250, 250), (500, 500)]
    assert len(fb.level_plan(3712, 3712)) == 6 and len(fb.level_plan(5424, 5424)) == 6
    assert [(p["h"], p["w"]) for p in fb.level_plan(100, 100)] == [(50, 50), (100, 100)]
    assert len(fb.level_plan(10, 15)) == 1
    assert [(p["h"], p["w"]) for p in fb.level_plan(130, 170)] == [(32, 42), (65, 85), (130, 170)]


def test_polyexp_constants():
    g, xg, xxg, ig11, ig03, ig33, ig55 = fb.prepare_gaussian(5, 1.1)
    # SURVEY.md §8(a7) step 4 (probed on cv2 4.13)
    assert abs(ig11 - 0.8264522919) < 1e-8 and abs(ig03 + 0.4132632753) < 1e-8
    assert abs(ig33 - 0.3415423840) < 1e-8 and abs(ig55 - 0.6830233968) < 1e-8
    assert np.allclose(g[:6], [1.1830532e-05, 4.8769583e-04, 8.7977722e-03, 6.9450498e-02, 2.3991476e-01,
                               3.6267489e-01], rtol=1e-6)


@pytest.mark.skipif(not flow_ops.have_cv2(), reason="cv2 not importable")
@pytest.mark.parametrize("shape", [(10, 15), (64, 96), (100, 100), (130, 170), (300, 420)])
def test_farneback_matches_cv2(shape):
    import cv2
    h, w = shape
    bt = synthetic.bt_sequence(2, h, w, seed=h * 1000 + w, nans=False)
    q0, q1 = flow_ops.pair_to_u8(bt[0], bt[1])
    ref = cv2.calcOpticalFlowFarneback(q0, q1, None, 0.5, 5, 13, 10, 5, 1.1, 0)
    ref2 = cv2.FarnebackOpticalFlow_create().calc(q0, q1, None)
    assert np.array_equal(ref, ref2)
    mine = fb.farneback(q0, q1)
    e = epe(mine, ref)
    assert e.mean() < 2e-5 and e.max() < 1e-3, (e.mean(), e.max())


@pytest.mark.skipif(not flow_ops.have_cv2(), reason="cv2 not importable")
def test_farneback_matches_cv2_on_tiny_frames():
    """Every side 1..15 against a side of 40, both ways round: one pyramid level, the box window and the polynomial
    expansion wider than the frame, and OpenCV's border band test, which on sides of 6..9 px leaves some pixels
    within 5 px of an edge unattenuated."""
    import cv2
    shapes = [(s, 40) for s in range(1, 16)] + [(40, s) for s in range(1, 16)] + [(7, 7), (6, 13)]
    for h, w in shapes:
        bt = synthetic.moving_texture(h, w, [synthetic.rotation_motion(2.0)], seed=h * 100 + w)
        q0, q1 = flow_ops.pair_to_u8(bt[0], bt[1])
        for a, b in ((q0, q1), (q1, q0)):
            ref = cv2.FarnebackOpticalFlow_create().calc(a, b, None)
            e = epe(fb.farneback(a, b), ref)
            assert e.mean() < 1e-5 and e.max() < 1e-4, ((h, w), e.mean(), e.max())


def test_border_scale_band_rule():
    """FarnebackUpdateMatrices attenuates where (unsigned)(x - 5) >= (unsigned)(w - 10) or the same holds for y."""
    s = fb.border_scale(40, 7)                    # w = 7: only columns 2..4 pass the x test
    assert (s[20, 2:5] < 1).all() and s[20, 0] == 1 and s[20, 1] == 1 and s[20, 5] == 1 and s[20, 6] == 1
    assert s[0, 0] == np.float32(np.float32(np.float32(0.14) * np.float32(1)) * np.float32(0.14))
    s = fb.border_scale(3, 3)                     # every factor applies: ((x0 * x1) * y0) * y1 in fp32
    f = [np.float32(v) for v in (0.14, 0.14, 0.4472)]
    assert s[1, 1] == np.float32(np.float32(np.float32(f[1] * f[1]) * f[1]) * f[1])
    s = fb.border_scale(20, 30)
    assert (s[5:15, 5:25] == 1).all() and s[4, 10] == np.float32(0.4472) and s[10, 29] == np.float32(0.14)


@pytest.mark.skipif(not flow_ops.have_cv2(), reason="cv2 not importable")
def test_stages_match_cv2():
    import cv2
    img = (synthetic.base_field(200, 300, 3) * 255).astype(np.float32)
    for k, s in [(3, 0.0), (3, 0.5), (9, 1.5), (19, 3.5), (39, 7.5), (79, 15.5)]:
        assert np.abs(cv2.GaussianBlur(img, (k, k), s) - fb.gaussian_blur(img, k, s)).max() < 5e-4
    for (h, w) in [(100, 150), (50, 75), (25, 38), (67, 91)]:
        assert np.abs(cv2.resize(img, (w, h), interpolation=cv2.INTER_LINEAR) - fb.resize_linear(img, h, w)).max() < 2e-4
    fl = np.stack([img, img[::-1]], -1)[:50, :75]
    assert np.abs(cv2.resize(fl, (150, 100), interpolation=cv2.INTER_LINEAR) - fb.resize_linear(fl, 100, 150)).max() < 2e-4


def test_farneback_matches_reference_golden(golden):
    g = golden("three_level")
    bt = cases.three_level()
    q0, q1 = flow_ops.pair_to_u8(bt[0], bt[1])
    f = np.clip(fb.farneback(q0, q1), -20, 20)
    b = np.clip(fb.farneback(q1, q0), -20, 20)
    for mine, ref in ((f, g["fwd_0"]), (b, g["bwd_1"])):
        e = epe(mine, ref)
        assert e.mean() < 2e-5 and e.max() < 1e-3, (e.mean(), e.max())


def test_blob_known_answers(golden):
    """SURVEY.md §8(c) known-answer values on G1 (cv2 4.13.0)."""
    g = golden("blob100")
    data = synthetic.blob_stack()
    fwd, bwd = flow_ops.create_flow(data, backend="numpy")
    assert epe(fwd[[0, 4, 9]], g["fwd_0_4_9"]).max() < 1e-3
    assert epe(bwd[4], g["bwd_4"]).max() < 1e-3
    assert np.allclose(fwd[4, 50, 50], (0.10432175, 0.10432258), atol=2e-5)
    assert np.allclose(bwd[4, 50, 50], (-0.10804594, -0.10804673), atol=2e-5)
    assert np.allclose(fwd[0, 0, 0], (0.00212546, 0.00212546), atol=2e-5)


@pytest.mark.parametrize("shape", [(300, 500), (129, 260), (97, 1100)])
def test_combined_taps_equal_blur_then_resize(shape):
    """The algebra behind the row / half pyramid kernels (csrc/pyramid.cu): GaussianBlur followed by the bilinear resize is
    one separable filter per destination pixel with taps cw[c] = g[c] + f * (g[c - 1] - g[c]) (f = the resize weight of the
    second source row / column, g[-1] = g[ksize] = 0), REFLECT_101 applied to the source index.  Checked here in float64
    against the oracle's blur -> resize on every down-sampled level."""
    H, W = shape
    rng = np.random.default_rng(H * W)
    img = rng.integers(0, 256, (H, W)).astype(np.uint8)
    for lvl in fb.level_plan(H, W):
        if (lvl["h"], lvl["w"]) == (H, W):
            continue
        g = fb.gaussian_kernel(lvl["ksize"], lvl["sigma"]).astype(np.float64)
        ks, rad = lvl["ksize"], lvl["ksize"] // 2
        gext = np.concatenate([g, [0.0]])                       # g[ksize] = 0
        dg = np.concatenate([[0.0], g]) - gext                  # g[c - 1] - g[c]
        y0, _, fy = fb._linear_coords(lvl["h"], H)
        x0, _, fx = fb._linear_coords(lvl["w"], W)
        src = img.astype(np.float64)
        rows = fb._reflect101((y0[:, None] - rad) + np.arange(ks + 1)[None, :], H)          # (h, ks + 1)
        cv = gext[None, :] + fy.astype(np.float64)[:, None] * dg[None, :]
        V = np.einsum("jr,jrx->jx", cv, src[rows])                                           # vertical pass: (h, W)
        cols = fb._reflect101((x0[:, None] - rad) + np.arange(ks + 1)[None, :], W)          # (w, ks + 1)
        ch = gext[None, :] + fx.astype(np.float64)[:, None] * dg[None, :]
        out = np.einsum("ic,jic->ji", ch, V[:, cols])
        ref = fb.pyramid_level(img, lvl)
        assert out.shape == ref.shape
        assert np.abs(out - ref).max() <= 2e-4, (lvl["k"], np.abs(out - ref).max())
