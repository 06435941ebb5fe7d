"""Pin oracle/flow_ops.py (normalisation, calculate_flow, convolve, diff, sobel, smoothing) against golden
vectors produced by the unmodified reference (tests/golden/make_golden.py)."""
from functools import partial

import numpy as np
import pytest
from scipy import ndimage as ndi

from oracle import flow_ops as ops
import make_golden as cases

BACKENDS = ["numpy"] + (["cv2"] if ops.have_cv2() else [])


def close(a, b, rtol=1e-4):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    if not np.array_equal(np.isnan(a), np.isnan(b)):
        return False
    m = ~np.isnan(b)
    return bool(np.all(np.abs(a[m] - b[m]) <= rtol * np.maximum(np.abs(b[m]), 1.0)))


@pytest.fixture(scope="module")
def bt():
    return cases.small_bt()


@pytest.fixture(scope="module")
def g(golden):
    return golden("bt_small")


def test_pair_quantisation_bit_exact(bt, g):
    for i in range(bt.shape[0] - 1):
        q0, q1 = ops.pair_to_u8(bt[i], bt[i + 1])
        assert np.array_equal(q0, g["q"][i, 0]) and np.array_equal(q1, g["q"][i, 1])


@pytest.mark.parametrize("backend", BACKENDS)
def test_create_flow(bt, g, backend):
    fwd, bwd = ops.create_flow(bt, backend=backend)
    if backend == "cv2":
        assert np.array_equal(fwd, g["fwd"]) and np.array_equal(bwd, g["bwd"])
    else:
        for a, b in ((fwd, g["fwd"]), (bwd, g["bwd"])):
            e = np.sqrt(((a - b) ** 2).sum(-1))
            assert e.mean() < 2e-5 and e.max() < 2e-3


@pytest.mark.parametrize("backend", BACKENDS)
def test_smoothed_flow(bt, g, backend):
    if backend == "numpy":
        # feed the reference's own un-smoothed pair flow so only smooth_flow_step is under test
        f, b = ops.smooth_flow_step(g["fwd"][0], g["bwd"][1], "cubic", backend)
        f, b = np.clip(f, -20, 20), np.clip(b, -20, 20)
        assert close(f, g["fwd_smooth1_cubic"][0]) and close(b, g["bwd_smooth1_cubic"][1])
    else:
        fwd, bwd = ops.create_flow(bt, smoothing_passes=1, interp_method="cubic", backend=backend)
        assert np.array_equal(fwd, g["fwd_smooth1_cubic"], equal_nan=True)
        assert np.array_equal(bwd, g["bwd_smooth1_cubic"], equal_nan=True)


@pytest.mark.parametrize("backend", BACKENDS)
def test_stencils_on_reference_flow(bt, g, backend):
    fwd, bwd = g["fwd"], g["bwd"]
    eq = partial(np.array_equal, equal_nan=True)
    assert eq(ops.diff(bt, fwd, bwd, backend=backend), g["diff"])
    assert eq(ops.diff(bt, fwd, bwd, method="nearest", backend=backend), g["diff_nearest"])
    assert close(ops.sobel(bt, fwd, bwd, dtype=None, backend=backend), g["sobel"], 1e-12)
    assert ops.sobel(bt, fwd, bwd, dtype=None, backend=backend).dtype == np.float64
    assert close(ops.sobel(bt, fwd, bwd, dtype=np.float32, backend=backend), g["sobel_f32"], 1e-6)
    assert close(ops.sobel(bt, fwd, bwd, method="cubic", dtype=None, direction="uphill", backend=backend),
                 g["sobel_uphill_cubic"], 1e-12)
    assert close(ops.sobel(bt, fwd, bwd, dtype=None, direction="downhill", backend=backend),
                 g["sobel_downhill"], 1e-12)
    assert eq(ops.convolve(bt, fwd, bwd, backend=backend)[:, [1, 3]], g["conv7_t13"])
    assert eq(ops.convolve(bt, fwd, bwd, method="cubic", fill_value=0.0, backend=backend)[:, [1, 3]],
              g["conv7_cubic_fill0_t13"])
    t_struct = np.zeros([3, 3, 3])
    t_struct[:, 1, 1] = 1
    raw64 = g["diff"] / np.full(bt.shape[0], 5.0)[:, None, None]
    assert eq(ops.convolve(raw64, fwd, bwd, t_struct, func=ops.nanmean_reducer, backend=backend), g["tmean_f64src"])
    s_struct = ndi.generate_binary_structure(3, 1)
    s_struct[0] = 0
    s_struct[2] = 0
    assert eq(ops.convolve(g["diff"], fwd, bwd, s_struct, func=ops.nanmean_reducer, backend=backend), g["smean"])
    mask = (np.nan_to_num(bt, nan=300.0) < 250).astype(np.int32)
    assert eq(ops.convolve(mask, fwd, bwd, t_struct.astype(bool), "nearest", np.int32, False, ops.any_reducer,
                           backend=backend), g["any_nearest"])
    labels = ndi.label(mask)[0].astype(np.int32)
    l_struct = ndi.generate_binary_structure(3, 1)
    l_struct[1] = 0
    assert eq(ops.convolve(labels, fwd, bwd, l_struct, "nearest", np.int32, 0, backend=backend), g["labels_nearest"])


def test_blob_stencil_known_answers(golden):
    """SURVEY.md §8(c): diff / sobel known answers on G1 fed with the reference's flow."""
    from tobac_flow_b200 import synthetic
    g1 = golden("blob100")
    data = synthetic.blob_stack()
    # only frames 0, 4, 9 of the reference flow are stored; frame 4 needs fwd[4], bwd[4]
    fwd = np.zeros(data.shape + (2,), np.float32)
    bwd = np.zeros(data.shape + (2,), np.float32)
    fwd[4] = g1["fwd_0_4_9"][1]
    bwd[4] = g1["bwd_4"]
    d = ops.diff(data, fwd, bwd)[4]
    assert np.array_equal(d, g1["diff_4"], equal_nan=True) and d[50, 50] == -30920.5
    s = ops.sobel(data, fwd, bwd, dtype=None)[4]
    assert close(s, g1["sobel_4"], 1e-12) and abs(s[50, 50] - 1254683.1562226177) < 1e-6
    assert close(ops.sobel(data, fwd, bwd, "cubic", None, direction="uphill")[4], g1["sobel_up_cubic_4"], 1e-12)
    assert close(ops.sobel(data, fwd, bwd, "nearest", None)[4], g1["sobel_near_4"], 1e-12)


def test_error_conventions():
    z = np.zeros((2, 4, 5, 2), np.float32)
    d = np.zeros((2, 4, 5), np.float32)
    with pytest.raises(AssertionError):
        ops.convolve(d, z, z, np.ones((3, 3)))
    with pytest.raises(ValueError):
        ops.convolve(d, z, z, method="bogus")


def test_float64_and_integer_normalisation_against_the_unmodified_reference(golden):
    """The oracle's pair quantisation for float64 / integer frames (numpy keeps float64 and promotes integers, so the
    reference normalises in float64) against stored results that match the reference's (reference_checks.npz) and,
    where the reference is installed, against its own to_8bit(linear_norm(.))."""
    import sys
    import refshim
    import make_golden_reference_checks as rc
    stored = golden("reference_checks")
    for name, got in rc.pair_quantisation().items():
        rc.assert_matches(stored, name, got)
    if not refshim.reference_available():
        return
    from oracle import flow_ops as ops
    saved_path, saved_modules = list(sys.path), set(sys.modules)
    try:
        refshim.load_reference()
        from tobac_flow.utils import to_8bit, linear_norm
        for stack in rc.quantisation_stacks():
            r = to_8bit(linear_norm(stack), 0, 1)
            o = ops.pair_to_u8(stack[0], stack[1])
            assert np.array_equal(r[0], o[0]) and np.array_equal(r[1], o[1])
    finally:
        sys.path[:] = saved_path
        for name in set(sys.modules) - saved_modules:
            if name.split(".")[0] in ("tobac_flow", "xarray", "pyproj", "skimage"):
                del sys.modules[name]
        refshim._loaded = None
