"""GPU parity for the "next" rows (SURVEY.md 8f ranks 2-3): detection filters and semi-Lagrangian labelling through the
C ABI, against scipy.ndimage / the oracle (bit-exact: masks, labels and label numbers; float filters bit-exact too) and
against the goldens of the unmodified reference."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from scipy import ndimage as ndi  # noqa: E402

from oracle import detection_ops as det  # noqa: E402
from oracle import flow_ops as ops  # noqa: E402
import make_golden as mg  # noqa: E402

BACKEND = "cv2" if ops.have_cv2() else "numpy"


def unpack(bits, shape):
    return np.unpackbits(bits)[:int(np.prod(shape))].reshape(shape).astype(bool)


def blobs(rng, shape, density, smooth):
    f = ndi.gaussian_filter(rng.standard_normal(shape), (0, smooth, smooth))
    return f > np.quantile(f, 1 - density)


CROSS3 = ndi.generate_binary_structure(3, 1)
FULL3 = np.ones((3, 3, 3), bool)


@pytest.mark.parametrize("shape", [(3, 37, 45), (2, 64, 96), (1, 5, 131), (4, 130, 33), (1, 1, 1), (2, 1, 70), (2, 70, 1)])
@pytest.mark.parametrize("conn", [1, 2])
def test_flat_label_matches_scipy(shape, conn):
    from tobac_flow_b200.label import flat_label
    rng = np.random.default_rng(hash((shape, conn)) % 2 ** 31)
    for density, smooth in ((0.5, 0.0), (0.3, 1.5), (0.62, 0.7), (1.0, 0.0), (0.0, 0.0)):
        mask = blobs(rng, shape, density, smooth) if 0 < density < 1 else np.full(shape, bool(density))
        s = CROSS3 if conn == 1 else FULL3
        want = det.flat_label(mask, s)
        got = flat_label(mask, s)
        assert got.dtype == np.int32 and np.array_equal(got, want), (shape, conn, density)


def test_flat_label_spirals_and_long_runs():
    """Worst cases for union-find: a spiral (one component, very long paths), full rows, a comb."""
    from tobac_flow_b200.label import flat_label
    H, W = 97, 203
    m = np.zeros((3, H, W), bool)
    y0, y1, x0, x1 = 0, H - 1, 0, W - 1
    while y1 - y0 > 3 and x1 - x0 > 3:
        m[0, y0, x0:x1 + 1] = m[0, y0:y1 + 1, x1] = m[0, y1, x0 + 2:x1 + 1] = m[0, y0 + 2:y1 + 1, x0 + 2] = True
        y0, y1, x0, x1 = y0 + 2, y1 - 2, x0 + 4, x1 - 2
    m[1, ::2] = True
    m[2, :, ::2] = True
    m[2, H // 2] = True
    for s in (CROSS3, FULL3):
        assert np.array_equal(flat_label(m, s), det.flat_label(m, s))


def test_flat_label_conus_size():
    from tobac_flow_b200.label import flat_label
    rng = np.random.default_rng(3)
    mask = blobs(rng, (2, 1500, 2500), 0.3, 3.0)
    want = det.flat_label(mask)
    got = flat_label(torch.from_numpy(mask).cuda())
    assert got.is_cuda and np.array_equal(got.cpu().numpy(), want)


@pytest.mark.parametrize("shape", [(3, 40, 50), (2, 33, 129), (1, 3, 3), (2, 1, 9)])
def test_fill_holes_and_opening(shape):
    from tobac_flow_b200 import _lib
    from tobac_flow_b200._io import stream as _stream
    lib = _lib.load()
    rng = np.random.default_rng(5)
    T, H, W = shape
    s = CROSS3.copy()
    s[0] = 0
    s[2] = 0
    for density, smooth in ((0.5, 1.0), (0.7, 0.0), (0.35, 2.0)):
        mask = blobs(rng, shape, density, smooth)
        m = torch.from_numpy(mask).cuda().to(torch.uint8)
        out = torch.empty_like(m)
        nb = int(lib.tf_ccl_workspace_bytes(T, H, W))
        ws = torch.empty((nb,), dtype=torch.uint8, device="cuda")
        _lib.check(lib.tf_binary_fill_holes(m.data_ptr(), out.data_ptr(), T, H, W, ws.data_ptr(), nb, _stream()))
        assert np.array_equal(out.cpu().numpy().astype(bool), ndi.binary_fill_holes(mask, structure=s))
        _lib.check(lib.tf_binary_opening_cross(m.data_ptr(), out.data_ptr(), T, H, W, _stream()))
        assert np.array_equal(out.cpu().numpy().astype(bool), ndi.binary_opening(mask, structure=s))


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("shape", [(2, 50, 70), (1, 5, 6), (2, 17, 3), (1, 1, 40)])
def test_gaussian_filter_bit_exact(dtype, shape):
    from tobac_flow_b200.detection import gaussian_filter_yx_device
    rng = np.random.default_rng(9)
    a = (rng.standard_normal(shape) * 20 - 10).astype(dtype)
    for sigma in (2, 1.0, 0.6, 3.3):
        want = ndi.gaussian_filter(a, (0, sigma, sigma))
        got = gaussian_filter_yx_device(torch.from_numpy(a).cuda(), sigma).cpu().numpy()
        assert got.dtype == want.dtype and np.array_equal(got, want), (dtype, shape, sigma)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_grey_opening_bit_exact_with_nans(dtype):
    from tobac_flow_b200.detection import grey_opening_cross_device
    rng = np.random.default_rng(10)
    fp = ndi.generate_binary_structure(2, 1)[np.newaxis, ...]
    for shape in ((3, 31, 47), (1, 2, 2), (2, 1, 5), (1, 64, 1)):
        a = rng.standard_normal(shape).astype(dtype)
        a[rng.random(shape) < 0.05] = np.nan
        want = ndi.grey_opening(a, footprint=fp)
        got = grey_opening_cross_device(torch.from_numpy(a).cuda()).cpu().numpy()
        assert np.array_equal(got, want, equal_nan=True), shape


@pytest.mark.parametrize("direction", ["negative", "positive"])
def test_curvature_filter(direction):
    from tobac_flow_b200.detection import get_curvature_filter
    wvd = mg.growth_multi_case()
    want = det.get_curvature_filter(wvd, direction=direction)
    got = get_curvature_filter(wvd, direction=direction)
    assert got.dtype == np.bool_ and np.array_equal(got, want)
    w64 = wvd.astype(np.float64)[:4]
    assert np.array_equal(get_curvature_filter(w64, sigma=1.5, threshold=0.01, direction=direction),
                          det.get_curvature_filter(w64, sigma=1.5, threshold=0.01, direction=direction))
    with pytest.raises(ValueError):
        get_curvature_filter(wvd, direction="sideways")


@pytest.fixture(scope="module")
def multi(golden):
    import tobac_flow_b200 as tfb
    g = golden("growth_multi")
    wvd = mg.growth_multi_case()
    fwd = g["fwd_q256"].astype(np.float32) / 256
    bwd = g["bwd_q256"].astype(np.float32) / 256
    return g, wvd, fwd, bwd, tfb.Flow(fwd, bwd)


def test_flow_label_against_reference_golden(multi):
    g, wvd, fwd, bwd, flow = multi
    seeds = unpack(g["seeds"], wvd.shape)
    got = flow.label(seeds)
    assert got.dtype == np.int32 and np.array_equal(got, g["linked"])
    from tobac_flow_b200.label import flow_label, flow_link_overlap, flat_label
    assert np.array_equal(flow_label(flow, seeds, overlap=0.5, absolute_overlap=4), g["linked_ov"])
    assert np.array_equal(flat_label(seeds), g["flat"])
    assert np.array_equal(flow.link_overlap(g["flat"].astype(np.int32)), g["linked"])
    assert np.array_equal(flow_link_overlap(flow, g["flat"].astype(np.int64), overlap=0.5, absolute_overlap=4), g["linked_ov"])
    d = flow.label(torch.from_numpy(seeds).cuda())
    assert d.is_cuda and np.array_equal(d.cpu().numpy(), g["linked"])


@pytest.mark.parametrize("overlap,absolute", [(0.0, 0), (0.0, 1), (0.3, 2), (0.8, 0)])
def test_flow_label_random_against_oracle(overlap, absolute):
    import tobac_flow_b200 as tfb
    from tobac_flow_b200.label import flow_label
    rng = np.random.default_rng(21)
    T, H, W = 7, 90, 140
    fwd = (rng.standard_normal((T, H, W, 2)) * 0.3 + np.array([2.0, 1.0])).astype(np.float32)
    bwd = (rng.standard_normal((T, H, W, 2)) * 0.3 - np.array([2.0, 1.0])).astype(np.float32)
    base = blobs(rng, (1, H + 40, W + 40), 0.25, 2.5)[0]
    mask = np.stack([np.roll(base, (t, 2 * t), (0, 1))[20:20 + H, 20:20 + W] for t in range(T)])
    mask[3, 30:50] = False
    flow = tfb.Flow(fwd, bwd)
    want = det.flow_label(mask, fwd, bwd, overlap=overlap, absolute_overlap=absolute, backend=BACKEND)
    got = flow_label(flow, mask, overlap=overlap, absolute_overlap=absolute)
    assert want.max() > 3 and np.array_equal(got, want)


def test_flow_label_errors(multi):
    g, wvd, fwd, bwd, flow = multi
    seeds = unpack(g["seeds"], wvd.shape)
    with pytest.raises(AssertionError):
        flow.label(seeds[1:])
    with pytest.raises(ValueError):
        flow.label(seeds, structure=np.ones((3, 3, 3), bool))      # 18 time taps cannot unpack into (back, forward)
    empty = flow.label(np.zeros_like(seeds))
    assert empty.shape == seeds.shape and not empty.any()


def test_label_filters(multi):
    from tobac_flow_b200 import analysis
    g, wvd, fwd, bwd, flow = multi
    linked = g["linked"].astype(np.int32)
    assert np.array_equal(analysis.filter_labels_by_length(linked, 3), g["by_len"])
    m05 = unpack(g["mask05"], wvd.shape)
    for lab in (linked, g["by_len"].astype(np.int32)):
        assert np.array_equal(analysis.filter_labels_by_mask(lab, m05), det.filter_labels_by_mask(lab, m05))
        assert np.array_equal(analysis.filter_labels_by_mask(lab, wvd >= -5), det.filter_labels_by_mask(lab, wvd >= -5))
        for n in (1, 2, 4, 9, 20):
            assert np.array_equal(analysis.filter_labels_by_length(lab, n), det.filter_labels_by_length(lab, n))
    want = det.filter_labels_by_mask(det.filter_labels_by_length(linked, 3), m05)
    assert np.array_equal(analysis.filter_labels_by_length_and_mask(linked, m05, 3), want)


@pytest.mark.parametrize("case", ["growth", "growth_multi"])
def test_detect_growth_markers_against_reference_golden(golden, case):
    import pandas as pd
    import refshim
    import tobac_flow_b200 as tfb
    from tobac_flow_b200.detection import detect_growth_markers, growth_markers_device
    g = golden(case)
    wvd = mg.growth_case() if case == "growth" else mg.growth_multi_case()
    fwd = g["fwd_q256"].astype(np.float32) / 256
    bwd = g["bwd_q256"].astype(np.float32) / 256
    flow = tfb.Flow(fwd, bwd)
    t = pd.date_range("2020-01-01", periods=wvd.shape[0], freq="5min")
    da = refshim.DataArray(wvd, coords={"t": t}, dims=("t", "y", "x"), t=t)
    smoothed, markers = detect_growth_markers(flow, da)
    markers = np.asarray(markers.data if hasattr(markers, "data") else markers)
    assert smoothed.dtype == np.float32
    assert np.array_equal(smoothed[::2], g["smoothed_even"], equal_nan=True)
    assert np.array_equal(markers, g["markers"])
    r = growth_markers_device(flow, torch.from_numpy(wvd).cuda(), np.full(wvd.shape[0], 5.0))
    filt = r["filtered"].cpu().numpy()
    assert np.array_equal(filt >= 0.25, unpack(g["mask025"], wvd.shape))
    assert np.array_equal(filt >= 0.5, unpack(g["mask05"], wvd.shape))
    if case == "growth_multi":
        assert np.array_equal(r["seeds"].cpu().numpy().astype(bool), unpack(g["seeds"], wvd.shape))
        assert np.array_equal(r["flat"].cpu().numpy(), g["flat"])
        assert np.array_equal(r["linked"].cpu().numpy(), g["linked"])


def test_detect_growth_markers_with_own_flow_and_nans():
    """End to end on the device with the library's own flow and NaN pixels, against the oracle fed the same flow."""
    import tobac_flow_b200 as tfb
    from tobac_flow_b200.detection import growth_markers_device
    wvd = mg.growth_multi_case()
    wvd[5, 40:43, 50:90] = np.nan
    wvd[8, 100, 20] = np.nan
    flow = tfb.create_flow(wvd)
    dt = np.array([5.0] * 6 + [7.5] + [10.0] * 7)
    r = growth_markers_device(flow, torch.from_numpy(wvd).cuda(), dt)
    want = det.detect_growth_markers(wvd, dt, flow.forward_flow, flow.backward_flow, backend=BACKEND, intermediates=True)
    assert np.array_equal(r["raw"].cpu().numpy(), want["raw"], equal_nan=True)
    assert np.array_equal(r["smoothed"].cpu().numpy(), want["smoothed"], equal_nan=True)
    assert np.array_equal(r["filtered"].cpu().numpy(), want["filtered"], equal_nan=True)
    assert np.array_equal(r["seeds"].cpu().numpy().astype(bool), want["seeds"])
    assert np.array_equal(r["linked"].cpu().numpy(), want["linked"])
    assert np.array_equal(r["markers"].cpu().numpy(), want["markers"])
    assert want["markers"].max() >= 1


def test_detect_growth_markers_multichannel_and_nan_gaussian(multi):
    """detection.py:203-254 and :128-146 on the device against the oracle (itself checked against the unmodified
    reference in tests/test_oracle_detection.py): both smoothed rates and the marker labels bit-exact, with NaN pixels in
    both channels and non-default thresholds; the legacy multi-mask label filter on its own."""
    import pandas as pd
    import refshim
    from tobac_flow_b200 import analysis
    from tobac_flow_b200.detection import detect_growth_markers_multichannel, nan_gaussian_filter
    g, wvd, fwd, bwd, flow = multi
    wvd = wvd.copy()
    bt = (250.0 - 2.2 * (wvd + 25.0)).astype(np.float32)
    wvd[6, 40:42, 50:80] = np.nan
    bt[3, 70, 10:40] = np.nan
    t = pd.date_range("2020-01-01", periods=wvd.shape[0], freq="5min")
    da_w = refshim.DataArray(wvd, coords={"t": t}, dims=("t", "y", "x"), t=t)
    da_b = refshim.DataArray(bt, coords={"t": t}, dims=("t", "y", "x"), t=t)
    dt = np.full(wvd.shape[0], 5.0)
    for kw in (dict(), dict(overlap=0.2, min_length=2, lower_threshold=0.2, upper_threshold=0.4)):
        got = detect_growth_markers_multichannel(flow, da_w, da_b, **kw)
        want = det.detect_growth_markers_multichannel(wvd, bt, dt, dt, fwd, bwd, backend=BACKEND, **kw)
        for a, b in zip(got, want):
            a = np.asarray(a.data if hasattr(a, "data") and not isinstance(a, np.ndarray) else a)
            assert a.dtype == b.dtype and np.array_equal(a, b, equal_nan=True)
        assert want[2].max() >= 1
    with pytest.raises(NotImplementedError):
        detect_growth_markers_multichannel(flow, da_w, da_b, subsegment_shrink=0.5)
    # the label filter alone: three masks, odd count
    lab = g["linked"].astype(np.int32)
    rng = np.random.default_rng(3)
    masks = [rng.random(lab.shape) > 0.9995, rng.random(lab.shape) > 0.999, wvd > -12]
    assert np.array_equal(analysis.filter_labels_by_length_and_multimask_legacy(lab, masks, 3),
                          det.filter_labels_by_length_and_multimask_legacy(lab, masks, 3))
    with pytest.raises(ValueError):
        analysis.filter_labels_by_length_and_multimask_legacy(lab, tuple(masks), 3)
    # nan_gaussian_filter
    x = wvd[:4].copy()
    x[2] = np.nan
    x[1, :, 50] = np.nan
    for dtype in (np.float32, np.float64):
        for prop in (True, False):
            got = nan_gaussian_filter(x.astype(dtype), (0, 2, 2), propagate_nan=prop)
            want = det.nan_gaussian_filter(x.astype(dtype), (0, 2, 2), propagate_nan=prop)
            assert got.dtype == want.dtype and np.array_equal(got, want, equal_nan=True)
    got = nan_gaussian_filter(x[0], 1.5)
    assert np.array_equal(got, det.nan_gaussian_filter(x[0], 1.5), equal_nan=True)
    with pytest.raises(NotImplementedError):
        nan_gaussian_filter(x, (0, 2, 2), mode="nearest")


@pytest.mark.parametrize("method", ["linear", "cubic"])
def test_get_growth_rate(multi, method):
    import pandas as pd
    import refshim
    from tobac_flow_b200.detection import get_growth_rate
    g, wvd, fwd, bwd, flow = multi
    t = pd.date_range("2020-01-01", periods=wvd.shape[0], freq="5min")
    da = refshim.DataArray(wvd, coords={"t": t}, dims=("t", "y", "x"), t=t)
    got = get_growth_rate(flow, da, method=method)
    want = det.get_growth_rate(wvd, np.full(wvd.shape[0], 5.0), fwd, bwd, method=method, backend=BACKEND)
    assert got.dtype == np.float32 and np.array_equal(got, want, equal_nan=True)
    w64 = -wvd.astype(np.float64) * 1.000000123                       # a float64 field (detect_cores passes -bt)
    got = get_growth_rate(flow, refshim.DataArray(w64, coords={"t": t}, dims=("t", "y", "x"), t=t), method=method)
    want = det.get_growth_rate(w64, np.full(wvd.shape[0], 5.0), fwd, bwd, method=method, backend=BACKEND)
    assert got.dtype == np.float32 and np.array_equal(got, want, equal_nan=True)


def test_get_anvil_markers(multi):
    from tobac_flow_b200.detection import get_anvil_markers
    g, wvd, fwd, bwd, flow = multi
    for thr, ov, ab, ml in ((-5, 0.5, 5, 3), (-12, 0.2, 1, 1), (5, 0.5, 5, 3)):
        want = det.get_anvil_markers(wvd, fwd, bwd, threshold=thr, overlap=ov, absolute_overlap=ab, min_length=ml,
                                     backend=BACKEND)
        got = get_anvil_markers(flow, wvd, threshold=thr, overlap=ov, absolute_overlap=ab, min_length=ml)
        assert np.array_equal(got, want), (thr, ov, ab, ml)
    assert det.get_anvil_markers(wvd, fwd, bwd, backend=BACKEND).max() >= 1


def test_short_and_degenerate_series():
    """One- and two-frame series, tiny frames, all-true / all-false masks: same answers as the oracle, no crashes."""
    import tobac_flow_b200 as tfb
    from tobac_flow_b200.detection import growth_markers_device
    rng = np.random.default_rng(2)
    for T, H, W in ((1, 20, 30), (2, 9, 7), (3, 33, 65)):
        fwd = (rng.standard_normal((T, H, W, 2)) * 0.7).astype(np.float32)
        bwd = (rng.standard_normal((T, H, W, 2)) * 0.7).astype(np.float32)
        flow = tfb.Flow(fwd, bwd)
        for mask in (rng.random((T, H, W)) < 0.4, np.ones((T, H, W), bool), np.zeros((T, H, W), bool)):
            want = det.flow_label(mask, fwd, bwd, absolute_overlap=1, backend=BACKEND)
            assert np.array_equal(flow.label(mask), want), (T, H, W)
        if T >= 2:
            wvd = (rng.standard_normal((T, H, W)) * 8 - 10).astype(np.float32)
            dt = np.full(T, 5.0)
            r = growth_markers_device(flow, torch.from_numpy(wvd).cuda(), dt)
            want = det.detect_growth_markers(wvd, dt, fwd, bwd, backend=BACKEND, intermediates=True)
            assert np.array_equal(r["smoothed"].cpu().numpy(), want["smoothed"], equal_nan=True)
            assert np.array_equal(r["seeds"].cpu().numpy().astype(bool), want["seeds"])
            assert np.array_equal(r["markers"].cpu().numpy(), want["markers"])


def test_sharded_label_single_rank_cuda_backend(multi):
    """ShardedFlow.label with the CUDA back-end on one rank (the collectives are skipped at world size 1; they are
    covered by the gloo tests and by scratch/label_sharded_check.py under torchrun)."""
    from tobac_flow_b200 import distributed as D
    g, wvd, fwd, bwd, flow = multi
    seeds = unpack(g["seeds"], wvd.shape)
    fl = D.ShardedFlow(torch.from_numpy(fwd).cuda(), torch.from_numpy(bwd).cuda(), 0, 1)
    lab = fl.label(torch.from_numpy(seeds).cuda())
    assert np.array_equal(lab.cpu().numpy(), g["linked"])
    lab = fl.label(torch.from_numpy(seeds).cuda(), overlap=0.5, absolute_overlap=4)
    assert np.array_equal(lab.cpu().numpy(), g["linked_ov"])


def test_sharded_growth_markers_single_rank_cuda_backend(multi):
    """ShardedFlow.detect_growth_markers with the CUDA back-end on one rank equals the single-call pipeline and the
    reference golden (collectives are skipped at world size 1; gloo tests and scratch/detect_sharded_check.py cover them)."""
    from tobac_flow_b200 import distributed as D
    from tobac_flow_b200.detection import growth_markers_device
    g, wvd, fwd, bwd, flow = multi
    dt = np.full(wvd.shape[0], 5.0)
    fl = D.ShardedFlow(torch.from_numpy(fwd).cuda(), torch.from_numpy(bwd).cuda(), 0, 1)
    shard = D.make_shard(torch.from_numpy(wvd).cuda(), 0, 1)
    smoothed, markers = fl.detect_growth_markers(shard, dt, 0)
    ref = growth_markers_device(flow, torch.from_numpy(wvd).cuda(), dt)
    assert torch.equal(torch.nan_to_num(smoothed, nan=-7.0), torch.nan_to_num(ref["smoothed"], nan=-7.0))
    assert np.array_equal(markers.cpu().numpy(), g["markers"])


def test_growth_markers_float64_field(multi):
    """A float64 field is smoothed / thresholded in float64 (scipy keeps the array dtype): same result as the oracle."""
    from tobac_flow_b200.detection import growth_markers_device
    g, wvd, fwd, bwd, flow = multi
    w64 = wvd.astype(np.float64) + 1e-9 * np.arange(wvd.shape[2])[None, None, :]
    dt = np.full(wvd.shape[0], 5.0)
    r = growth_markers_device(flow, torch.from_numpy(w64).cuda(), dt)
    want = det.detect_growth_markers(w64, dt, fwd, bwd, backend=BACKEND, intermediates=True)
    assert np.array_equal(r["smoothed"].cpu().numpy(), want["smoothed"], equal_nan=True)
    assert np.array_equal(r["seeds"].cpu().numpy().astype(bool), want["seeds"])
    assert np.array_equal(r["markers"].cpu().numpy(), want["markers"])


# ------------------------------------------------------------------------------------------------------------------
# watershed inputs: get_combined_edge_field / get_watershed_mask (the reference's tests/test_detection.py:17-60 restated)
# ------------------------------------------------------------------------------------------------------------------
def test_reference_get_combined_edge_field_and_watershed_mask():
    import tobac_flow_b200 as tfb
    from tobac_flow_b200.detection import get_combined_edge_field, get_watershed_mask
    field = np.zeros([1, 5, 5], dtype=np.float32)
    field[:, 3:] = 1
    fl = tfb.Flow(np.zeros([1, 5, 5, 2], np.float32), np.zeros([1, 5, 5, 2], np.float32))
    res = get_combined_edge_field(fl, field)
    assert np.all(res[:, 2] > 0) and np.all(res[:, :2] == 0) and np.all(res[:, 3:] == -1)
    field[:, :, 0] = np.nan
    res = get_combined_edge_field(fl, field)
    assert np.all(np.isnan(field) == np.isinf(res))
    # get_watershed_mask (tests/test_detection.py:17-33): ones from row 2 on, eroded once
    f2 = np.zeros([1, 5, 5], dtype=np.float32)
    f2[:, 3:] = 1
    m = get_watershed_mask(f2, erode_distance=1)
    want = ndi.binary_erosion(np.logical_or(f2 <= 0, np.isnan(f2)), structure=np.ones([3, 3, 3]), iterations=1, border_value=1)
    assert np.array_equal(m, want)
    rng = np.random.default_rng(8)
    f3 = rng.standard_normal((4, 30, 40)).astype(np.float32)
    f3[rng.random(f3.shape) < 0.02] = np.nan
    for it in (1, 2):
        want = ndi.binary_erosion(np.logical_or(f3 <= 0, np.isnan(f3)), structure=np.ones([3, 3, 3]), iterations=it, border_value=1)
        want[np.isnan(f3)] = True
        assert np.array_equal(get_watershed_mask(f3, erode_distance=it), want)
