"""GPU parity tests: the CUDA path (through the C ABI) against the oracle and the reference's golden vectors.

Tolerances (BASELINE.json north_star): flow mean end-point error <= 0.05 px and 99th percentile <= 0.5 px vs
OpenCV Farneback; convolve / sobel / diff within 1e-4 relative with identical NaN masks when fed the reference's
own flow fields (most are in fact bit-exact and asserted so); integer / byte results bit-exact.
"""
from functools import partial

import numpy as np
import pytest
from scipy import ndimage as ndi

pytestmark = pytest.mark.gpu

from oracle import farneback_np, flow_ops as ops  # noqa: E402
import make_golden as cases  # noqa: E402
from tobac_flow_b200 import synthetic  # noqa: E402


@pytest.fixture(scope="module")
def tfb():
    import tobac_flow_b200
    return tobac_flow_b200


def epe(a, b):
    return np.sqrt(((np.asarray(a, np.float64) - np.asarray(b, np.float64)) ** 2).sum(-1))


def assert_flow_close(mine, ref, mean_tol=0.05, p99_tol=0.5):
    e = epe(mine, ref)
    assert np.isfinite(e).all()
    assert e.mean() <= mean_tol and np.percentile(e, 99) <= p99_tol, (e.mean(), np.percentile(e, 99), e.max())
    return e


def assert_close(a, b, rtol=1e-4):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    assert a.shape == b.shape
    assert np.array_equal(np.isnan(a), np.isnan(b)), "NaN masks differ"
    m = ~np.isnan(b)
    err = np.abs(a[m] - b[m]) / np.maximum(np.abs(b[m]), 1.0)
    assert err.size == 0 or err.max() <= rtol, err.max()


def assert_same(a, b):
    assert a.dtype == b.dtype and a.shape == b.shape
    assert np.array_equal(a, b, equal_nan=True), f"max abs diff {np.nanmax(np.abs(a.astype(np.float64) - b))}"


# ------------------------------------------------------------------------------------------------------------------
# K1 normalisation / quantisation: bit-exact
# ------------------------------------------------------------------------------------------------------------------
def test_pair_quantisation_bit_exact(tfb, golden):
    bt = cases.small_bt()
    g = golden("bt_small")
    for i in range(bt.shape[0] - 1):
        q0, q1 = tfb.pair_to_8bit(bt[i], bt[i + 1])
        assert np.array_equal(q0, g["q"][i, 0]) and np.array_equal(q1, g["q"][i, 1])
    data = synthetic.blob_stack()
    rng = np.random.default_rng(5)
    odd = (rng.standard_normal((2, 37, 53)) * 1e3).astype(np.float32)  # odd size -> scalar path
    odd[0, 3, 4] = np.inf
    odd[1, 7, 7] = np.nan
    const = np.full((2, 40, 40), 3.25, np.float32)                      # vmax == vmin -> factor 0
    for a, b in ((data[0], data[1]), (odd[0], odd[1]), (const[0], const[1])):
        q0, q1 = tfb.pair_to_8bit(a, b)
        r0, r1 = ops.pair_to_u8(a, b)
        assert np.array_equal(q0, r0) and np.array_equal(q1, r1)


# ------------------------------------------------------------------------------------------------------------------
# Farneback flow vs the reference (cv2) goldens and the oracle
# ------------------------------------------------------------------------------------------------------------------
def test_flow_small_bt_vs_reference_golden(tfb, golden):
    g = golden("bt_small")
    f = tfb.create_flow(cases.small_bt())
    e1 = assert_flow_close(f.forward_flow, g["fwd"], 1e-3, 1e-2)
    e2 = assert_flow_close(f.backward_flow, g["bwd"], 1e-3, 1e-2)
    print("bt_small EPE mean/max", e1.mean(), e1.max(), e2.mean(), e2.max())


def test_flow_three_levels_vs_reference_golden(tfb, golden):
    g = golden("three_level")
    f = tfb.create_flow(cases.three_level())
    assert_flow_close(f.forward_flow[0], g["fwd_0"], 1e-3, 1e-2)
    assert_flow_close(f.backward_flow[1], g["bwd_1"], 1e-3, 1e-2)


def test_flow_blob_known_answers(tfb, golden):
    g = golden("blob100")
    f = tfb.create_flow(synthetic.blob_stack())
    assert_flow_close(f.forward_flow[[0, 4, 9]], g["fwd_0_4_9"], 1e-3, 1e-2)
    assert_flow_close(f.backward_flow[4], g["bwd_4"], 1e-3, 1e-2)
    assert np.allclose(f.forward_flow[4, 50, 50], (0.10432175, 0.10432258), atol=1e-4)   # SURVEY.md §8(c)
    assert np.allclose(f.backward_flow[4, 50, 50], (-0.10804594, -0.10804673), atol=1e-4)
    # end rules (flow.py:425-426)
    assert np.array_equal(f.forward_flow[-1], -f.backward_flow[-1])
    assert np.array_equal(f.backward_flow[0], -f.forward_flow[0])


# tiny frames: single rows / columns, frames narrower than the 6-column halo of a strip, sides of 6..9 px (OpenCV's
# border band test wraps there), widths on either side of a 116-column strip boundary.  They take the analytic texture:
# bt_sequence's field is noise low-passed at 12 px, and on a side of a few px only one Fourier mode of it is left, a
# one-directional sinusoid on which the flow along the stripes is set by rounding (two float64 restatements of
# OpenCV already differ by 0.1 px at 7 x 12).
TINY_FRAMES = [(1, 1), (1, 40), (40, 1), (2, 3), (5, 5), (7, 12), (12, 7), (6, 40), (40, 9), (13, 13), (31, 33),
               (64, 115), (64, 116), (64, 117), (40, 233)]


@pytest.mark.parametrize("shape", [(10, 15), (33, 47), (64, 64), (100, 259), (257, 130)] + TINY_FRAMES)
def test_flow_vs_oracle_odd_sizes(tfb, shape):
    h, w = shape
    if shape in TINY_FRAMES:
        motions = [synthetic.shift_motion(1.0, 2.0), synthetic.shift_motion(-2.0, 1.0)]
        bt = synthetic.moving_texture(h, w, motions, seed=h * 7 + w)
    else:
        bt = synthetic.bt_sequence(3, h, w, seed=h * 7 + w, nans=False)
    f = tfb.create_flow(bt)
    ref_f, ref_b = ops.create_flow(bt, backend="cv2" if ops.have_cv2() else "numpy")
    assert_flow_close(f.forward_flow, ref_f, 2e-3, 2e-2)
    assert_flow_close(f.backward_flow, ref_b, 2e-3, 2e-2)


def test_identical_frames_match_opencv_and_batching_is_deterministic(tfb):
    bt = synthetic.bt_sequence(1, 96, 128, seed=3, nans=False)
    f = tfb.create_flow(np.repeat(bt, 3, 0))
    # OpenCV itself is not zero here (near the borders its out-of-image branch drops the R1 term); the two pairs
    # of the batch must agree bit for bit
    assert np.array_equal(f.forward_flow[0], f.forward_flow[1])
    q0, q1 = ops.pair_to_u8(bt[0], bt[0])
    # identical frames: h ~ 0 and G ~ 0 in smooth areas, so the flow is a ratio of rounding-level numbers there;
    # fp32 window sums (OpenCV: fp64) and the level images' fp32 association (a few 1e-5 of the 0..255 range) show up at
    # the 1e-3..5e-2 px level in this degenerate case only (north-star gate: mean 0.05 px, p99 0.5 px)
    assert_flow_close(f.forward_flow[0], farneback_np.farneback(q0, q1), 1e-3, 5e-2)


def test_clamp_and_calculate_flow(tfb):
    bt = synthetic.bt_sequence(3, 80, 120, seed=11, nans=False)
    fwd, bwd = tfb.calculate_flow(bt)
    f = tfb.create_flow(bt, max_value=0.25)
    assert np.array_equal(f.forward_flow, np.clip(fwd, -0.25, 0.25))
    assert np.array_equal(f.backward_flow, np.clip(bwd, -0.25, 0.25))


def test_smoothing_passes_vs_reference_golden(tfb, golden):
    g = golden("bt_small")
    # smooth_flow_step itself, fed with the reference's un-smoothed fields
    f, b = tfb.smooth_flow_step(g["fwd"][0], g["bwd"][1], method="cubic")
    rf, rb = ops.smooth_flow_step(g["fwd"][0], g["bwd"][1], "cubic")
    assert_same(f, rf.astype(np.float32))
    assert_same(b, rb.astype(np.float32))
    fl = tfb.create_flow(cases.small_bt(), smoothing_passes=1, interp_method="cubic")
    assert_flow_close(fl.forward_flow, g["fwd_smooth1_cubic"], 1e-3, 1e-2)
    assert_flow_close(fl.backward_flow, g["bwd_smooth1_cubic"], 1e-3, 1e-2)


# ------------------------------------------------------------------------------------------------------------------
# stencil operators fed with the REFERENCE's flow fields
# ------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ref_flow(tfb, golden):
    g = golden("bt_small")
    return tfb.Flow(g["fwd"], g["bwd"]), cases.small_bt(), g


def test_diff(ref_flow):
    fl, bt, g = ref_flow
    assert_same(fl.diff(bt), g["diff"])
    assert_same(fl.diff(bt, method="nearest"), g["diff_nearest"])


def test_sobel(ref_flow):
    fl, bt, g = ref_flow
    s = fl.sobel(bt)
    assert s.dtype == np.float64
    assert_close(s, g["sobel"], 1e-12)
    assert_close(fl.sobel(bt, dtype=np.float32), g["sobel_f32"], 1e-6)
    assert_close(fl.sobel(bt, direction="uphill", method="cubic"), g["sobel_uphill_cubic"], 1e-12)
    assert_close(fl.sobel(bt, direction="downhill"), g["sobel_downhill"], 1e-12)


def test_convolve_stack(ref_flow):
    fl, bt, g = ref_flow
    c = fl.convolve(bt)
    assert c.shape == (7,) + bt.shape and c.dtype == np.float32
    assert_same(c[:, [1, 3]], g["conv7_t13"])
    assert_same(fl.convolve(bt, method="cubic", fill_value=0.0)[:, [1, 3]], g["conv7_cubic_fill0_t13"])


def test_convolve_reducers(ref_flow):
    fl, bt, g = ref_flow
    t_struct = np.zeros([3, 3, 3])
    t_struct[:, 1, 1] = 1
    raw64 = g["diff"] / np.full(bt.shape[0], 5.0)[:, None, None]
    assert raw64.dtype == np.float64
    assert_same(fl.convolve(raw64, structure=t_struct, func=lambda x: np.nanmean(x, 0)), g["tmean_f64src"])
    s_struct = ndi.generate_binary_structure(3, 1)
    s_struct[0] = 0
    s_struct[2] = 0
    assert_same(fl.convolve(g["diff"], structure=s_struct, func=lambda x: np.nanmean(x, 0)), g["smean"])
    mask = (np.nan_to_num(bt, nan=300.0) < 250).astype(int)
    assert_same(fl.convolve(mask, structure=t_struct.astype(bool), method="nearest", fill_value=False,
                            dtype=np.int32, func=partial(np.any, axis=0)), g["any_nearest"])
    labels = ndi.label(mask)[0].astype(np.int32)
    l_struct = ndi.generate_binary_structure(3, 1)
    l_struct[1] = 0
    assert_same(fl.convolve(labels, structure=l_struct, method="nearest", dtype=np.int32, fill_value=0),
                g["labels_nearest"])


def test_unrecognised_python_reducer_uses_stack_path(ref_flow):
    fl, bt, g = ref_flow
    func = lambda x: np.nanmedian(x, 0)  # noqa: E731
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        want = ops.convolve(bt, g["fwd"], g["bwd"], func=func)
        got = fl.convolve(bt, func=func)
    assert_same(got, want)


def test_blob_stencil_known_answers(tfb, golden):
    g1 = golden("blob100")
    data = synthetic.blob_stack()
    fwd = np.zeros(data.shape + (2,), np.float32)
    bwd = np.zeros(data.shape + (2,), np.float32)
    fwd[4] = g1["fwd_0_4_9"][1]
    bwd[4] = g1["bwd_4"]
    fl = tfb.Flow(fwd, bwd)
    d = fl.diff(data)[4]
    assert_same(d, g1["diff_4"])
    assert d[50, 50] == -30920.5
    s = fl.sobel(data)[4]
    assert_close(s, g1["sobel_4"], 1e-12)
    assert abs(s[50, 50] - 1254683.1562226177) < 1e-6
    assert_close(fl.sobel(data, direction="uphill", method="cubic")[4], g1["sobel_up_cubic_4"], 1e-12)
    assert_close(fl.sobel(data, method="nearest")[4], g1["sobel_near_4"], 1e-12)


def test_reference_test_detection_edge_field(tfb):
    """Restates the reference's only Flow.sobel test (tests/test_detection.py:36-60): zero flow, 1x5x5 step
    field, uphill + cubic, NaN where the field is NaN."""
    field = np.zeros((1, 5, 5), np.float32)
    field[..., 3:] = 1
    field[0, 0, 0] = np.nan
    z = np.zeros((1, 5, 5, 2), np.float32)
    fl = tfb.Flow(z, z)
    got = fl.sobel(field, direction="uphill", method="cubic")
    want = ops.sobel(field, z, z, "cubic", None, direction="uphill")
    assert_close(got, want, 1e-12)
    assert np.isnan(got[0, 0, 0])


def test_function_level_mirrors(tfb, golden):
    from tobac_flow_b200 import convolve as cmod, sobel as smod
    g = golden("bt_small")
    bt = cases.small_bt()
    assert_same(cmod.convolve(bt, g["fwd"], g["bwd"])[:, [1, 3]], g["conv7_t13"])
    assert_close(smod.sobel(bt, g["fwd"], g["bwd"]), g["sobel_f32"], 1e-6)
    offs = np.array([[1, 0], [0, -1], [-1, 1]])
    w = cmod.warp_flow(bt[1], g["fwd"][0], offsets=offs)
    for k, (dx, dy) in enumerate(offs):
        assert_same(w[k], ops.warp_image(bt[1], g["fwd"][0], "linear", np.nan, dx, dy))


def test_error_conventions(tfb):
    z = np.zeros((2, 8, 9, 2), np.float32)
    with pytest.raises(ValueError):
        tfb.Flow(z, z[:1])
    with pytest.raises(ValueError):
        tfb.Flow(z[..., :1], z[..., :1])
    fl = tfb.Flow(z, z)
    assert fl.shape == (2, 8, 9)
    with pytest.raises(AssertionError):
        fl.convolve(np.zeros((2, 8, 8), np.float32))
    with pytest.raises(AssertionError):
        fl.convolve(np.zeros((2, 8, 9), np.float32), structure=np.ones((3, 3)))
    with pytest.raises(ValueError):
        fl.convolve(np.zeros((2, 8, 9), np.float32), method="bogus")
    with pytest.raises(ValueError):
        tfb.create_flow(np.zeros((2, 40, 40), np.float32), model="bogus")
    with pytest.raises(NotImplementedError):
        tfb.create_flow(np.zeros((2, 40, 40), np.float32), model="DIS")
    sub = fl[0:1]
    assert sub.shape == (1, 8, 9)


# ------------------------------------------------------------------------------------------------------------------
# downstream: growth markers (detection.py:98-125) up to the thresholds that define the marker masks
# ------------------------------------------------------------------------------------------------------------------
def test_growth_marker_masks_bit_exact(tfb, golden):
    g = golden("growth")
    wvd = cases.growth_case()
    fl = tfb.Flow(g["fwd_q256"].astype(np.float32) / 256, g["bwd_q256"].astype(np.float32) / 256)
    dt = np.full(wvd.shape[0], 5.0)                                   # get_time_diff_from_coord of a 5-min axis
    raw = fl.diff(wvd) / dt[:, None, None]                             # detection.py:99-101 (float64)
    t_struct = np.zeros([3, 3, 3])
    t_struct[:, 1, 1] = 1
    smoothed = fl.convolve(raw, structure=t_struct, func=lambda x: np.nanmean(x, 0))   # detection.py:53-55
    assert_same(smoothed[::2], g["smoothed_even"])
    # detection.py:105-108 + get_curvature_filter :64-94 (scipy, downstream of the hot path)
    s_struct = ndi.generate_binary_structure(2, 1)[np.newaxis, ...]
    sm = ndi.gaussian_filter(wvd, (0, 2, 2))
    x_diff = np.zeros(wvd.shape)
    x_diff[:, :, 1:-1] = np.diff(sm, n=2, axis=2)
    y_diff = np.zeros(wvd.shape)
    y_diff[:, 1:-1] = np.diff(sm, n=2, axis=1)
    s3 = ndi.generate_binary_structure(3, 1)
    s3[0] = 0
    s3[2] = 0
    curv = ndi.binary_opening(ndi.binary_fill_holes(np.logical_and(x_diff < 0, y_diff < 0), structure=s3), structure=s3)
    filtered = ndi.grey_opening(smoothed, footprint=s_struct) * curv
    assert np.array_equal(np.packbits(filtered >= 0.25), g["mask025"])
    assert np.array_equal(np.packbits(filtered >= 0.5), g["mask05"])
    assert (filtered >= 0.5).sum() > 0


# ------------------------------------------------------------------------------------------------------------------
# time sharding on one GPU: two shards computed one after the other with the halos filled by hand (the NCCL
# exchange itself is covered by the gloo tests and by the multi-GPU bench) must reproduce the unsharded result
# ------------------------------------------------------------------------------------------------------------------
def test_two_emulated_shards_equal_unsharded(tfb):
    import torch
    from tobac_flow_b200 import distributed as D, _lib
    bt = synthetic.bt_sequence(7, 96, 140, seed=21, nans=True)
    bt[3, 10:14] = np.nan
    full = tfb.create_flow(bt)
    s_diff = np.zeros((3, 3, 3))
    s_diff[:, 1, 1] = 1
    want_diff = full.diff(bt)
    want_sobel = full.sobel(bt)
    dev = torch.device("cuda")
    frames = torch.from_numpy(bt).to(dev)
    world = 2
    shards = [D.make_shard(frames[slice(*D.shard_bounds(7, world, r))], r, world) for r in range(world)]
    # halo frames (what exchange_halos moves)
    shards[0].buf[-1] = shards[1].buf[1]
    shards[1].buf[0] = shards[0].buf[-2]
    T0 = shards[0].local.shape[0]
    # rank 0 produced backward_flow of rank 1's first frame in its extra slot
    fw0 = torch.full((T0, 96, 140, 2), float("nan"), device=dev)
    bw0 = torch.full((T0 + 1, 96, 140, 2), float("nan"), device=dev)
    D.CudaOps().calculate_flow(shards[0].buf[1:T0 + 2], fw0, bw0, 0, "linear", 20)
    bwd_handover = bw0[T0].clone()
    T1 = shards[1].local.shape[0]
    fw1 = torch.full((T1, 96, 140, 2), float("nan"), device=dev)
    bw1 = torch.full((T1 + 1, 96, 140, 2), float("nan"), device=dev)
    D.CudaOps().calculate_flow(shards[1].buf[1:T1 + 1], fw1, bw1, 0, "linear", 20)
    bw1[0] = bwd_handover
    D.CudaOps().finalise(fw0, bw0[:T0], 20, False, True, False)
    D.CudaOps().finalise(fw1, bw1[:T1], 20, False, False, True)
    got_f = torch.cat([fw0, fw1]).cpu().numpy()
    got_b = torch.cat([bw0[:T0], bw1[:T1]]).cpu().numpy()
    assert np.array_equal(got_f, full.forward_flow) and np.array_equal(got_b, full.backward_flow)
    fl0 = D.ShardedFlow(fw0, bw0[:T0], 0, world)
    fl1 = D.ShardedFlow(fw1, bw1[:T1], 1, world)
    d = torch.cat([fl0.convolve(shards[0], s_diff, reducer=_lib.TF_RED_DIFF, exchange=False),
                   fl1.convolve(shards[1], s_diff, reducer=_lib.TF_RED_DIFF, exchange=False)]).cpu().numpy()
    s = torch.cat([fl0.convolve(shards[0], np.ones((3, 3, 3)), dtype=None, reducer=_lib.TF_RED_SOBEL, exchange=False),
                   fl1.convolve(shards[1], np.ones((3, 3, 3)), dtype=None, reducer=_lib.TF_RED_SOBEL, exchange=False)]
                  ).cpu().numpy()
    assert np.array_equal(d, want_diff, equal_nan=True)
    assert np.array_equal(s, want_sobel, equal_nan=True)
    # world == 1 goes through create_flow_sharded itself
    one = D.create_flow_sharded(D.make_shard(frames, 0, 1))
    assert np.array_equal(one.fwd.cpu().numpy(), full.forward_flow) and np.array_equal(one.bwd.cpu().numpy(), full.backward_flow)


# ------------------------------------------------------------------------------------------------------------------
# variational refinement (vr_steps > 0) and the production flow settings
# ------------------------------------------------------------------------------------------------------------------
def test_variational_refinement_vs_reference_golden(tfb, golden):
    g = golden("bt_small_production")
    bt = cases.small_bt()
    f = tfb.create_flow(bt, vr_steps=1)
    assert_flow_close(f.forward_flow, g["fwd_vr1"], 2e-3, 2e-2)
    assert_flow_close(f.backward_flow, g["bwd_vr1"], 2e-3, 2e-2)
    # the refinement must have changed the Farneback field
    f0 = tfb.create_flow(bt)
    assert np.abs(f.forward_flow - f0.forward_flow).max() > 0.05


def test_production_settings_vs_reference_golden(tfb, golden):
    """scripts/dcc_detect_goes.py:164-166: create_flow(bt, model="Farneback", vr_steps=1, smoothing_passes=1,
    interp_method="cubic")."""
    g = golden("bt_small_production")
    f = tfb.create_flow(cases.small_bt(), model="Farneback", vr_steps=1, smoothing_passes=1, interp_method="cubic")
    assert_flow_close(f.forward_flow, g["fwd_vr1_smooth1_cubic"], 2e-3, 2e-2)
    assert_flow_close(f.backward_flow, g["bwd_vr1_smooth1_cubic"], 2e-3, 2e-2)
    assert np.abs(f.forward_flow).max() <= 20


@pytest.mark.parametrize("shape", [(33, 47), (100, 259)])
def test_variational_refinement_vs_opencv(tfb, shape):
    h, w = shape
    bt = synthetic.bt_sequence(3, h, w, seed=h + w, nans=False)
    f = tfb.create_flow(bt, vr_steps=1)
    rf, rb = ops.create_flow(bt, vr_steps=1, backend="cv2" if ops.have_cv2() else "numpy")
    assert_flow_close(f.forward_flow, rf, 2e-3, 2e-2)
    assert_flow_close(f.backward_flow, rb, 2e-3, 2e-2)


def test_sobel_around_nan_inf_and_wild_flow():
    """Flow.sobel next to NaN pixels, NaN stripes, an all-NaN frame, Inf values, NaN / huge flow vectors and samples far
    outside the image: identical NaN mask and 1e-12 relative agreement with the oracle."""
    import tobac_flow_b200 as tfb
    bt = synthetic.bt_sequence(6, 203, 331, seed=77, nans=True)
    bt[2, 50:53, 100:140] = np.nan
    bt[3, 120, 200] = np.inf
    bt[4] = np.nan
    rng = np.random.default_rng(5)
    fwd = (rng.standard_normal(bt.shape + (2,)) * 1.5).astype(np.float32)
    bwd = (rng.standard_normal(bt.shape + (2,)) * 1.5).astype(np.float32)
    fwd[1, 10, 10] = np.nan
    bwd[1, 20, 20] = 1e9
    fwd[0, :, :5] = 30.0          # samples far outside the image on the left
    got = tfb.Flow(fwd, bwd).sobel(bt)
    assert got.dtype == np.float64
    with np.errstate(all="ignore"):
        want = ops.sobel(bt, fwd, bwd, dtype=None, backend="cv2" if ops.have_cv2() else "numpy")
    assert np.array_equal(np.isnan(got), np.isnan(want))
    assert np.array_equal(np.isinf(got), np.isinf(want))
    ok = np.isfinite(want)
    assert np.max(np.abs(got[ok] - want[ok]) / np.maximum(np.abs(want[ok]), 1.0)) < 1e-12


def test_diff_and_default_convolve_around_nan_inf_and_wild_flow():
    """The lean diff / cross-7 kernels and their out-of-line general path (image border, first / last frame, samples
    outside the image, NaN / huge flow vectors, quantised positions on the half-way points): bit-exact with the oracle."""
    import tobac_flow_b200 as tfb
    bt = synthetic.bt_sequence(6, 203, 331, seed=78, nans=True)
    bt[3, 120, 200] = np.inf
    bt[4] = np.nan
    rng = np.random.default_rng(6)
    fwd = (rng.standard_normal(bt.shape + (2,)) * 1.5).astype(np.float32)
    bwd = (rng.standard_normal(bt.shape + (2,)) * 1.5).astype(np.float32)
    fwd[1, 10, 10] = np.nan
    bwd[1, 20, 20] = 1e9
    bwd[2, 30, 30] = -1e9
    fwd[2, 40, 40] = np.inf
    fwd[0, :, :5] = 30.0
    bwd[3, -4:, :] = 7.0                      # off the bottom edge
    fwd[3, 60:90, 60:90] = (np.arange(30, dtype=np.float32)[None, :, None] + 0.5) / 32   # exact ties of the 1/32 grid
    bwd[5, :, :] = np.float32(1.0) / 64
    flow = tfb.Flow(fwd, bwd)
    backend = "cv2" if ops.have_cv2() else "numpy"
    with np.errstate(all="ignore"):
        assert_same(flow.diff(bt), ops.diff(bt, fwd, bwd, backend=backend))
        assert_same(flow.convolve(bt), ops.convolve(bt, fwd, bwd, backend=backend))
        # non-default fill value (the same-step taps outside the image take it)
        assert_same(flow.convolve(bt, fill_value=-3.5), ops.convolve(bt, fwd, bwd, fill_value=-3.5, backend=backend))


def test_float64_frames_are_normalised_in_float64():
    """float64 (and integer) frames: numpy keeps / promotes the dtype, so the reference quantises them in float64; the
    u8 pair must match that bit for bit (casting to float32 first moves a few per cent of the pixels by one count)."""
    import tobac_flow_b200 as tfb
    bt = synthetic.bt_sequence(3, 120, 160, seed=3, nans=True).astype(np.float64) * 1.0000001
    bt[1, 5:8] = np.nan
    moved = 0
    for i in range(2):
        q0, q1 = tfb.pair_to_8bit(bt[i], bt[i + 1])
        r0, r1 = ops.pair_to_u8(bt[i], bt[i + 1])
        assert np.array_equal(q0, r0) and np.array_equal(q1, r1)
        s0, s1 = ops.pair_to_u8(bt[i].astype(np.float32), bt[i + 1].astype(np.float32))
        moved += int((r0 != s0).sum() + (r1 != s1).sum())
    assert moved > 0                                   # the case does distinguish the two arithmetic paths
    bi = np.nan_to_num(bt * 10).astype(np.int32)
    q0, q1 = tfb.pair_to_8bit(bi[0], bi[1])
    r0, r1 = ops.pair_to_u8(bi[0], bi[1])
    assert np.array_equal(q0, r0) and np.array_equal(q1, r1)
    f = tfb.create_flow(bt)
    rf, rb = ops.create_flow(bt, backend="cv2" if ops.have_cv2() else "numpy")
    for mine, ref in ((f.forward_flow, rf), (f.backward_flow, rb)):
        e = np.sqrt(((mine - ref) ** 2).sum(-1))
        assert e.mean() <= 1e-3 and np.percentile(e, 99) <= 1e-2, (e.mean(), e.max())


# ------------------------------------------------------------------------------------------------------------------
# end rules on one-frame shards (tf_flow_finalise with T == 1: the last rank of a sharded run that owns one frame)
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("first,last", [(0, 1), (1, 0), (1, 1), (0, 0)])
@pytest.mark.parametrize("clamp_all", [False, True])
def test_finalise_single_frame_shard(tfb, first, last, clamp_all):
    import torch
    from tobac_flow_b200.flow import finalise_flow_device
    rng = np.random.default_rng(3)
    f = (rng.standard_normal((1, 9, 11, 2)) * 30).astype(np.float32)
    b = (rng.standard_normal((1, 9, 11, 2)) * 30).astype(np.float32)
    ft, bt_ = torch.from_numpy(f.copy()).cuda(), torch.from_numpy(b.copy()).cuda()
    finalise_flow_device(ft, bt_, 20.0, clamp_all, bool(first), bool(last))
    ef, eb = f.copy(), b.copy()
    if last:
        ef[-1] = -eb[-1]          # flow.py:425
    if first:
        eb[0] = -ef[0]            # flow.py:426 (after :425, as in the reference)
    if clamp_all:
        ef, eb = np.clip(ef, -20, 20), np.clip(eb, -20, 20)
    assert np.array_equal(ft.cpu().numpy(), ef) and np.array_equal(bt_.cpu().numpy(), eb)


# ------------------------------------------------------------------------------------------------------------------
# the default iteration kernel (TMA-staged, tensor-memory ring, packed fp32) against the scalar LDG kernel
# ------------------------------------------------------------------------------------------------------------------
def test_iteration_kernels_agree(tfb):
    """Both kernels form the same window sums bit for bit; they differ only in the reciprocal of the determinant (one
    MUFU.RCP, <= 1 ulp, against an IEEE division), so the flows agree to a few ulp of a pixel; odd sizes exercise the
    general alignment path (WAL = 0 / 1) and strips narrower than the halo."""
    from tobac_flow_b200 import _lib
    lib = _lib.load()
    try:
        for shape in ((3, 100, 100), (3, 97, 131), (2, 150, 258), (2, 64, 1101), (3, 12, 7), (3, 40, 117)):
            bt = synthetic.bt_sequence(shape[0], shape[1], shape[2], seed=77 + shape[2], nans=True)
            res = {}
            for k in (0, 1, 3, 4, 5):
                _lib.check(lib.tf_fb_select_kernel(k), "tf_fb_select_kernel")
                f = tfb.create_flow(bt)
                res[k] = (f.forward_flow.copy(), f.backward_flow.copy())
            assert np.array_equal(res[0][0], res[1][0]) and np.array_equal(res[0][1], res[1][1])   # ring placement only
            assert np.array_equal(res[3][0], res[4][0]) and np.array_equal(res[3][1], res[4][1])   # lookahead depth only
            # the flow up-sampling fused into a level's first iteration gives the bits of the separate kernel
            assert np.array_equal(res[3][0], res[5][0]) and np.array_equal(res[3][1], res[5][1])
            for a, b in zip(res[0], res[3]):
                assert np.abs(a - b).max() <= 4e-5, np.abs(a - b).max()
        assert lib.tf_fb_select_kernel(2) < 0 and lib.tf_fb_select_kernel(6) < 0
    finally:
        lib.tf_fb_select_kernel(3)


def test_host_results_beyond_the_pinned_cap(tfb, golden, monkeypatch):
    """Results larger than TF_PINNED_RESULT_MAX_GB are staged through two pinned chunks into an ordinary numpy array:
    same values as the page-locked path."""
    g = golden("bt_small")
    bt = cases.small_bt()
    fl = tfb.Flow(g["fwd"], g["bwd"])
    want_d, want_c = fl.diff(bt), fl.convolve(bt)
    monkeypatch.setenv("TF_PINNED_RESULT_MAX_GB", "0")
    got_d, got_c = fl.diff(bt), fl.convolve(bt)
    assert_same(got_d, want_d)
    assert_same(got_c, want_c)


def test_host_operators_overlapping_create_flow_equal_the_device_path(tfb, monkeypatch):
    """create_flow on a long host array returns with its pair batches still queued (Flow._ready); the host operators
    then run chunk by chunk on the operator stream behind the batch events.  Same bits as the device-tensor path, in
    either call order, with small chunks so that many chunk / batch boundaries are crossed."""
    import torch
    from tobac_flow_b200 import flow as tflow
    bt = synthetic.bt_sequence(45, 150, 202, seed=21, nans=True)
    dev_t = torch.from_numpy(bt).cuda()
    fd = tfb.create_flow(dev_t)
    want_f, want_b = fd.forward_flow_device.cpu().numpy(), fd.backward_flow_device.cpu().numpy()
    want = [x.cpu().numpy() for x in (fd.convolve(dev_t), fd.sobel(dev_t), fd.diff(dev_t))]
    monkeypatch.setattr(tflow, "_HOST_CHUNK_BYTES", 3 * 150 * 202 * 4)
    monkeypatch.setattr(tflow, "_HOST_PAIR_BATCH", 3)
    for stack_first in (True, False):
        tflow.operand_cache_clear()
        fh = tfb.create_flow(bt)
        assert fh._ready is not None and fh._ready[-1][0] == 45 and len(fh._ready) >= 4
        if stack_first:
            got = [fh.convolve(bt), fh.sobel(bt), fh.diff(bt)]
        else:
            got = [fh.diff(bt), fh.sobel(bt), fh.convolve(bt)][::-1]
        for a, b in zip(got, want):
            assert_same(a, b)
        assert_same(fh.forward_flow, want_f)
        assert_same(fh.backward_flow, want_b)
    # an operand that is NOT the array the flow was made from (its device copy comes from another create_flow, whose
    # upload is not ordered behind this flow's batch events): the operators must take the stream-ordered path
    bt2 = (bt[::-1] * np.float32(0.5) + np.float32(100.0)).copy()
    tflow.operand_cache_clear()
    fa = tfb.create_flow(bt)
    fb = tfb.create_flow(bt2)
    assert fb._ready_frames != fa._ready_frames
    got = fa.diff(bt2)
    assert_same(got, fd.diff(torch.from_numpy(bt2).cuda()).cpu().numpy())
    del fb


# ------------------------------------------------------------------------------------------------------------------
# lanczos interpolation (cv2.INTER_LANCZOS4; convolve.py:46-51): bit-exact against the oracle (itself bit-exact vs cv2)
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_lanczos_gather_bit_exact(tfb, golden, dtype):
    g = golden("bt_small")
    bt = cases.small_bt().astype(dtype)
    fl = tfb.Flow(g["fwd"], g["bwd"])
    for fill in (np.nan, 0.0):
        got = fl.convolve(bt, method="lanczos", fill_value=fill, dtype=dtype)
        want = ops.convolve(bt, g["fwd"], g["bwd"], method="lanczos", dtype=dtype, fill_value=fill)
        assert_same(got, want)
    # wild flows: taps leave the image, whole footprints outside
    rng = np.random.default_rng(17)
    wild_f = (g["fwd"] + rng.standard_normal(g["fwd"].shape).astype(np.float32) * 15).astype(np.float32)
    wild_b = (g["bwd"] + rng.standard_normal(g["bwd"].shape).astype(np.float32) * 15).astype(np.float32)
    fw = tfb.Flow(wild_f, wild_b)
    assert_same(fw.diff(bt.astype(np.float32), method="lanczos"), ops.diff(bt.astype(np.float32), wild_f, wild_b, method="lanczos"))
    f, b = tfb.smooth_flow_step(g["fwd"][0], g["bwd"][1], method="lanczos")
    rf, rb = ops.smooth_flow_step(g["fwd"][0], g["bwd"][1], "lanczos")
    assert_same(f, rf)
    assert_same(b, rb)
