"""CPU checks of the configurable Farneback model: the oracle's restatement against cv2 over OpenCV's settings, the
native level plan of tf_fb_config against the oracle's, and the constructor's range checks."""
import ctypes

import numpy as np
import pytest

from oracle import farneback_config_np as fbc, farneback_np as fb

# (name, FarnebackOpticalFlow keyword arguments): box and Gaussian windows, pyramid scales and depths, poly_n 7,
# iteration counts, and the legacy tobac-flow setting (Gaussian 16, 3 iterations)
GRID = [
    ("box3", dict(win_size=3)),
    ("box4", dict(win_size=4)),
    ("box15", dict(win_size=15)),
    ("box16", dict(win_size=16)),
    ("box63", dict(win_size=63)),
    ("gauss4", dict(win_size=4, flags=256)),
    ("gauss13", dict(win_size=13, flags=256)),
    ("gauss16", dict(win_size=16, flags=256)),
    ("gauss63", dict(win_size=63, flags=256)),
    ("scale03", dict(pyr_scale=0.3)),
    ("scale07_l15", dict(pyr_scale=0.7, num_levels=15)),
    ("scale08_l15", dict(pyr_scale=0.8, num_levels=15)),
    ("polyn7", dict(poly_n=7, poly_sigma=1.5)),
    ("iters1", dict(num_iters=1)),
    ("iters3", dict(num_iters=3)),
    ("legacy", dict(flags=256, win_size=16, num_iters=3)),
    ("gauss31_polyn7_scale07", dict(flags=256, win_size=31, poly_n=7, poly_sigma=1.5, pyr_scale=0.7, num_levels=6)),
]

SHAPES = [(1500, 2500), (500, 500), (3712, 3712), (5424, 5424), (100, 100), (10, 15), (130, 170), (63, 64)]


def cv2_farneback(q0, q1, num_levels=5, pyr_scale=0.5, win_size=13, num_iters=10, poly_n=5, poly_sigma=1.1, flags=0):
    import cv2
    return cv2.FarnebackOpticalFlow_create(num_levels, pyr_scale, False, win_size, num_iters, poly_n, poly_sigma,
                                           flags).calc(np.ascontiguousarray(q0), np.ascontiguousarray(q1), None)


def textured_pair(H=96, W=128, dy=2, dx=3, seed=0):
    """A smooth random texture and the same texture shifted by (+dx, +dy) px, as u8."""
    from scipy import ndimage
    rng = np.random.default_rng(seed)
    base = ndimage.gaussian_filter(rng.random((H + 2 * 8, W + 2 * 8)) * 255, 2)
    a, b = base[8:8 + H, 8:8 + W], base[8 - dy:8 - dy + H, 8 - dx:8 - dx + W]
    lo, hi = base.min(), base.max()
    return tuple(np.clip((x - lo) / (hi - lo) * 255, 0, 255).astype(np.uint8) for x in (a, b))


@pytest.mark.parametrize("name,kw", GRID, ids=[g[0] for g in GRID])
def test_oracle_matches_cv2(name, kw):
    pytest.importorskip("cv2")
    q0, q1 = textured_pair()
    # The Gaussian window of 4 (radius 2, sigma 0.6) is the smallest accepted one: its solves amplify the last-bit
    # differences of the fp32 sums (OpenCV's SIMD order vs numpy's), a few isolated pixels differ by up to ~4e-3 px
    max_gate = 1e-2 if name == "gauss4" else 1e-3
    for a, b in ((q0, q1), (q1, q0)):
        e = np.sqrt(((fbc.farneback(a, b, **kw) - cv2_farneback(a, b, **kw)) ** 2).sum(-1))
        assert e.mean() <= 1e-5 and e.max() <= max_gate, (name, e.mean(), e.max())


def test_config_oracle_defaults_equal_farneback_np():
    q0, q1 = textured_pair(seed=1)
    assert np.array_equal(fbc.farneback(q0, q1), fb.farneback(q0, q1))
    assert np.array_equal(fbc.farneback(q0, q1, win_size=15, num_iters=3), fb.farneback(q0, q1, win_size=15, num_iters=3))
    with pytest.raises(ValueError):
        fbc.farneback(q0, q1, flags=4)


@pytest.fixture(scope="module")
def lib():
    from tobac_flow_b200 import build, _lib
    build.build_library()
    return _lib


@pytest.mark.parametrize("pyr_scale,num_levels", [(0.5, 5), (0.3, 5), (0.48, 5), (0.7, 15), (0.8, 15), (0.5, 15),
                                                  (0.5, 0), (0.006, 3)])
def test_config_level_plan_matches_oracle(lib, pyr_scale, num_levels):
    from tobac_flow_b200 import FarnebackOpticalFlow
    model = FarnebackOpticalFlow(num_levels=num_levels, pyr_scale=pyr_scale)
    for H, W in SHAPES:
        want = fb.level_plan(H, W, num_levels, pyr_scale)
        assert model.level_plan(H, W) == [(p["h"], p["w"]) for p in want], (H, W)
        # every blur width such a plan needs is built (the widest, 421 taps, is one level at 32 / 5424)
        assert max(p["ksize"] for p in want) <= 511


def test_default_model_is_default_params(lib):
    from tobac_flow_b200 import FarnebackOpticalFlow
    c = lib.FbConfig()
    lib.load().tf_fb_config_default(ctypes.byref(c))
    p = lib.default_params()
    assert [getattr(c, f) for f, _ in lib.FbParams._fields_] == [getattr(p, f) for f, _ in lib.FbParams._fields_]
    assert c.flags == 0
    m = FarnebackOpticalFlow()
    assert [getattr(m.params(20.0), f) for f, _ in lib.FbConfig._fields_] == [getattr(c, f) for f, _ in lib.FbConfig._fields_]
    for H, W in SHAPES:
        assert m.level_plan(H, W) == lib.level_plan(H, W)
        assert m.workspace_bytes(3, H, W) == lib.workspace_bytes(3, H, W)


@pytest.mark.parametrize("kw,name", [
    (dict(num_levels=-1), "num_levels"), (dict(num_levels=16), "num_levels"), (dict(num_levels=2.5), "num_levels"),
    (dict(pyr_scale=0.0), "pyr_scale"), (dict(pyr_scale=1.0), "pyr_scale"),
    (dict(num_iters=0), "num_iters"),
    (dict(poly_n=6), "poly_n"), (dict(poly_n=3), "poly_n"),
    (dict(poly_sigma=0.0), "poly_sigma"),
    (dict(flags=4), "flags"), (dict(flags=257), "flags"),
    (dict(win_size=2), "win_size"), (dict(win_size=1), "win_size"), (dict(win_size=64), "win_size"),
    (dict(win_size=3, flags=256), "win_size"), (dict(win_size=2, flags=256), "win_size"),
    (dict(win_size=64, flags=256), "win_size"),
])
def test_constructor_rejects(lib, kw, name):
    from tobac_flow_b200 import FarnebackOpticalFlow
    with pytest.raises(ValueError, match=name):
        FarnebackOpticalFlow(**kw)


def test_native_config_rejects_with_parameter_name(lib):
    from tobac_flow_b200 import FarnebackOpticalFlow
    for field, value in (("win_size", 2), ("pyr_scale", 1.0), ("poly_n", 9), ("flags", 4), ("num_levels", 16)):
        c = FarnebackOpticalFlow().params()
        setattr(c, field, value)
        assert lib.load().tf_fb_config_level_plan(100, 100, ctypes.byref(c), None, None) < 0
        assert field.encode() in lib.load().tf_last_error()
        assert lib.load().tf_fb_config_workspace_bytes(1, 100, 100, ctypes.byref(c)) == 0
    c = FarnebackOpticalFlow(win_size=4, flags=256).params()
    c.win_size = 3
    assert lib.load().tf_fb_config_level_plan(100, 100, ctypes.byref(c), None, None) < 0


def test_accepted_edges(lib):
    from tobac_flow_b200 import FarnebackOpticalFlow
    for kw in (dict(win_size=3), dict(win_size=63), dict(win_size=4, flags=256), dict(win_size=63, flags=256),
               dict(num_levels=0), dict(num_levels=15, pyr_scale=0.8), dict(poly_n=7), dict(num_iters=1)):
        m = FarnebackOpticalFlow(**kw)
        assert m.level_plan(96, 128)
        assert repr(m).startswith("FarnebackOpticalFlow(") and m.key()[0] == "Farneback"
