"""CPU: the detection / labelling oracle (oracle/detection_ops.py) against golden vectors produced by the unmodified
reference (tests/golden/make_golden.py: detect_growth_markers, flat_label, Flow.label, flow_label with overlap,
filter_labels_by_length), plus the linking walk and the C-ABI host function tf_label_link_groups."""
import ctypes

import numpy as np
import pytest

from oracle import detection_ops as det
from oracle import flow_ops as ops

import make_golden as mg
import make_golden_reference_checks as rc

BACKEND = "cv2" if ops.have_cv2() else "numpy"


def unpack(bits, shape):
    return np.unpackbits(bits)[:int(np.prod(shape))].reshape(shape).astype(bool)


@pytest.fixture(scope="module")
def multi(golden):
    g = golden("growth_multi")
    wvd = mg.growth_multi_case()
    fwd = g["fwd_q256"].astype(np.float32) / 256
    bwd = g["bwd_q256"].astype(np.float32) / 256
    dt = np.full(wvd.shape[0], 5.0)
    inter = det.detect_growth_markers(wvd, dt, fwd, bwd, backend=BACKEND, intermediates=True)
    return g, wvd, fwd, bwd, inter


def test_growth_single_marker(golden):
    g = golden("growth")
    wvd = mg.growth_case()
    fwd = g["fwd_q256"].astype(np.float32) / 256
    bwd = g["bwd_q256"].astype(np.float32) / 256
    r = det.detect_growth_markers(wvd, np.full(wvd.shape[0], 5.0), fwd, bwd, backend=BACKEND, intermediates=True)
    assert np.array_equal(r["smoothed"][::2], g["smoothed_even"], equal_nan=True)
    assert np.array_equal(r["filtered"] >= 0.25, unpack(g["mask025"], wvd.shape))
    assert np.array_equal(r["filtered"] >= 0.5, unpack(g["mask05"], wvd.shape))
    assert np.array_equal(r["markers"], g["markers"])
    assert int(r["markers"].max()) == int(g["n_markers"])


def test_growth_multi_intermediates(multi):
    g, wvd, fwd, bwd, r = multi
    shape = wvd.shape
    assert np.array_equal(r["smoothed"][::2], g["smoothed_even"], equal_nan=True)
    assert np.array_equal(det.get_curvature_filter(wvd), unpack(g["curv"], shape))
    assert np.array_equal(r["filtered"] >= 0.25, unpack(g["mask025"], shape))
    assert np.array_equal(r["filtered"] >= 0.5, unpack(g["mask05"], shape))
    assert np.array_equal(r["seeds"], unpack(g["seeds"], shape))


def test_growth_multi_labels(multi):
    g, wvd, fwd, bwd, r = multi
    seeds = r["seeds"]
    assert np.array_equal(det.flat_label(seeds), g["flat"])
    assert np.array_equal(r["linked"], g["linked"])
    assert np.array_equal(det.flow_label(seeds, fwd, bwd, overlap=0.5, absolute_overlap=4, backend=BACKEND), g["linked_ov"])
    assert np.array_equal(det.filter_labels_by_length(r["linked"], 3), g["by_len"])
    assert np.array_equal(r["markers"], g["markers"])
    # the fixture exercises every filter: one label lost to the length filter, two to the mask filters
    assert g["linked"].max() == 5 and g["by_len"].max() == 4 and g["markers"].max() == 2


def test_link_overlap_equals_label_from_flat(multi):
    g, wvd, fwd, bwd, r = multi
    flat = g["flat"].astype(np.int32)
    assert np.array_equal(det.flow_link_overlap(flat, fwd, bwd, absolute_overlap=1, backend=BACKEND), g["linked"])


def _link_groups_c(flat, back, fwd_l, overlap, absolute_overlap):
    """Drive the HOST function tf_label_link_groups with a histogram built in numpy (no GPU needed)."""
    from tobac_flow_b200 import _lib
    lib = _lib.load()
    n_labels = int(flat.max())
    sizes = np.bincount(flat.ravel(), minlength=n_labels + 1).astype(np.int32)
    keys, counts = [], []
    for d, nb in ((0, fwd_l), (1, back)):
        sel = (flat > 0) & (nb > 0)
        k = (np.uint64(d) << np.uint64(62)) | (flat[sel].astype(np.uint64) << np.uint64(31)) | nb[sel].astype(np.uint64)
        u, c = np.unique(k, return_counts=True)
        keys.append(u)
        counts.append(c)
    keys = np.concatenate(keys)
    counts = np.concatenate(counts).astype(np.int32)
    cap = 64
    while cap < 2 * len(keys):
        cap *= 2
    tk = np.full(cap, np.uint64(0xFFFFFFFFFFFFFFFF), np.uint64)
    tc = np.zeros(cap, np.int32)
    rng = np.random.default_rng(0)
    slots = rng.permutation(cap)[:len(keys)]          # any slot order must give the same answer
    tk[slots] = keys
    tc[slots] = counts
    out = np.zeros(n_labels + 1, np.int32)
    n = lib.tf_label_link_groups(tk.ctypes.data, tc.ctypes.data, cap, sizes.ctypes.data, n_labels,
                                 ctypes.c_double(overlap), absolute_overlap, out.ctypes.data)
    assert n >= 0
    return out[flat], n


@pytest.mark.parametrize("overlap,absolute", [(0.0, 1), (0.5, 4), (0.0, 0), (0.9, 0)])
def test_link_groups_host_function(multi, overlap, absolute):
    g, wvd, fwd, bwd, r = multi
    flat = g["flat"].astype(np.int32)
    back, fwd_l = det.label_taps(flat, fwd, bwd, backend=BACKEND)
    want = det.link_flat_labels(flat, back, fwd_l, np.int32, overlap, absolute)
    got, n = _link_groups_c(flat, back, fwd_l, overlap, absolute)
    assert np.array_equal(got, want)
    assert n == want.max()


def test_link_groups_random_graph():
    """Random sparse label fields with hand-made 'warped' neighbours: order-dependent linking must match."""
    rng = np.random.default_rng(11)
    for trial in range(5):
        flat = rng.integers(0, 40, (6, 30, 30)).astype(np.int32)
        flat[rng.random(flat.shape) < 0.5] = 0
        flat[flat == 7] = 0                              # a label number with no pixels
        back = np.roll(flat, 1, 0)
        back[0] = 0
        fwd_l = np.roll(flat, -1, 0)
        fwd_l[-1] = 0
        back[rng.random(flat.shape) < 0.3] = 0
        fwd_l[rng.random(flat.shape) < 0.3] = 0
        for overlap, absolute in ((0.0, 0), (0.05, 2), (0.2, 5)):
            want = det.link_flat_labels(flat, back, fwd_l, np.int32, overlap, absolute)
            got, n = _link_groups_c(flat, back, fwd_l, overlap, absolute)
            assert np.array_equal(got, want), (trial, overlap, absolute)


def test_growth_rate_and_anvil_markers_against_the_unmodified_reference(multi, golden):
    """The oracle's get_growth_rate and get_anvil_markers against stored results that match the reference's
    (reference_checks.npz) and, where the reference is installed, against its own functions run under the dependency
    stubs."""
    g, wvd, fwd, bwd, r = multi
    stored = golden("reference_checks")
    for name, got in rc.growth_rate_and_anvil(wvd, fwd, bwd).items():
        rc.assert_matches(stored, name, got)
    import refshim
    if not refshim.reference_available():
        return
    import sys
    import pandas as pd
    saved_path, saved_modules = list(sys.path), set(sys.modules)
    try:
        refshim.load_reference()
        from tobac_flow.flow import Flow
        from tobac_flow import detection
        fl = Flow(fwd, bwd)
        t = pd.date_range("2020-01-01", periods=wvd.shape[0], freq="5min")
        da = refshim.DataArray(wvd, coords={"t": t}, dims=("t", "y", "x"), t=t)
        dt = np.full(wvd.shape[0], 5.0)
        for m in ("linear", "cubic"):
            assert np.array_equal(detection.get_growth_rate(fl, da, method=m),
                                  det.get_growth_rate(wvd, dt, fwd, bwd, method=m, backend="cv2"), equal_nan=True)
        anvil = getattr(detection.get_anvil_markers, "__wrapped__", detection.get_anvil_markers)
        for kw in rc.ANVIL_KW:
            assert np.array_equal(np.asarray(anvil(fl, wvd, **kw)),
                                  det.get_anvil_markers(wvd, fwd, bwd, backend="cv2", **kw))
    finally:
        # the reference's path entry (it has its own `tests` package) and the dependency stubs must not leak into
        # the rest of the session
        sys.path[:] = saved_path
        for name in set(sys.modules) - saved_modules:
            if name.split(".")[0] in ("tobac_flow", "xarray", "pyproj", "skimage"):
                del sys.modules[name]
        refshim._loaded = None


def test_multichannel_markers_and_nan_gaussian_against_the_unmodified_reference(multi, golden):
    """The oracle's detect_growth_markers_multichannel, its legacy multi-mask label filter and nan_gaussian_filter
    against stored results that match the reference's (reference_checks.npz) and, where the reference is installed,
    against its own functions run under the dependency stubs."""
    g, wvd, fwd, bwd, r = multi
    stored = golden("reference_checks")
    mine = rc.multichannel_and_nan_gaussian(wvd, fwd, bwd)
    for name, a in mine.items():
        rc.assert_matches(stored, name, a)
    assert mine["multichannel_0_2"].max() >= 1 and mine["multichannel_1_2"].max() >= 1
    import refshim
    if not refshim.reference_available():
        return
    import sys
    import pandas as pd
    saved_path, saved_modules = list(sys.path), set(sys.modules)
    try:
        refshim.load_reference()
        from tobac_flow.flow import Flow
        from tobac_flow import detection
        bt = rc.bt_companion(wvd)
        fl = Flow(fwd, bwd)
        t = pd.date_range("2020-01-01", periods=wvd.shape[0], freq="5min")
        da_w = refshim.DataArray(wvd, coords={"t": t}, dims=("t", "y", "x"), t=t)
        da_b = refshim.DataArray(bt, coords={"t": t}, dims=("t", "y", "x"), t=t)
        dt = np.full(wvd.shape[0], 5.0)
        for kw in rc.MULTICHANNEL_KW:
            want = detection.detect_growth_markers_multichannel(fl, da_w, da_b, **kw)
            got = det.detect_growth_markers_multichannel(wvd, bt, dt, dt, fwd, bwd, backend="cv2", **kw)
            for a, b in zip(want, got):
                a = np.asarray(a.data if hasattr(a, "data") and not isinstance(a, np.ndarray) else a)
                assert np.array_equal(a, b, equal_nan=True)
            assert got[2].max() >= 1
        x = rc.nan_gaussian_input(wvd)
        for sigma in rc.GAUSS_SIGMAS:
            assert np.array_equal(detection.nan_gaussian_filter(x, sigma), det.nan_gaussian_filter(x, sigma), equal_nan=True)
            assert np.array_equal(detection.nan_gaussian_filter(x, sigma, propagate_nan=False),
                                  det.nan_gaussian_filter(x, sigma, propagate_nan=False), equal_nan=True)
    finally:
        sys.path[:] = saved_path
        for name in set(sys.modules) - saved_modules:
            if name.split(".")[0] in ("tobac_flow", "xarray", "pyproj", "skimage"):
                del sys.modules[name]
        refshim._loaded = None
