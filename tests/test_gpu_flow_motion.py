"""GPU: Farneback and variational refinement (VR) against OpenCV on prescribed, non-uniform motion.

Frames are an analytic texture (a seeded sum of sinusoids around 250 K) evaluated in float64 at the displaced positions,
so every frame is exact and each pair of a sequence carries its own motion: a uniform shift towards the top-left, a
large one (the +-20 px clamp is active), one beyond the clamp, a rotation, a zoom whose samples leave all four borders,
and a motion discontinuity.  One batch of pairs then mixes all of them.  These reach the parts of the kernels that a
constant +1 / +2 px roll does not: the out-of-image branch of the R1 gather on every edge, non-trivial flow carried up
from the coarse levels, the clamp fused into the last iteration, spatially varying window sums, and VR on its own at
iteration counts and frame sizes around the tiles of its fused SOR kernel.

Besides the image-wide EPE, a fault confined to one place must show: the mean EPE is also checked in each 8-px border
band and in the columns next to the seams of the 116-column iteration strips.
"""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

cv2 = pytest.importorskip("cv2")

from oracle import flow_ops as ops  # noqa: E402
from tobac_flow_b200 import synthetic  # noqa: E402

STRIP_W = 116          # output columns of one iteration strip (fb_iter.cu, TsCfg::OUT_W)
BAND = 8


MOTIONS = {
    "neg": synthetic.shift_motion(-3.4, -5.7),
    "large": synthetic.shift_motion(11.3, -7.6),
    "beyond": synthetic.shift_motion(24.0, 0.0),
    "rotation": synthetic.rotation_motion(2.0),
    "zoom": synthetic.zoom_motion(1.04),
    "split": synthetic.split_motion(3.0),
}
SEQUENCE = ("neg", "large", "beyond", "rotation", "zoom", "split")


# ------------------------------------------------------------------------------------------------------------------
# error measures
# ------------------------------------------------------------------------------------------------------------------
def epe(a, b):
    return np.sqrt(((np.asarray(a, np.float64) - np.asarray(b, np.float64)) ** 2).sum(-1))


def regions(H, W):
    """name -> (row mask, column mask) of the places a localised fault would hide in."""
    ys, xs = np.arange(H), np.arange(W)
    out = {"top": (ys < BAND, xs >= 0), "bottom": (ys >= H - BAND, xs >= 0),
           "left": (ys >= 0, xs < BAND), "right": (ys >= 0, xs >= W - BAND)}
    for s in range(STRIP_W, W, STRIP_W):
        out[f"seam{s}"] = (ys >= 0, np.abs(xs - s) <= 2)
    return out


def check_flow(mine, ref, what, mean_tol=1e-3, p99_tol=1e-2, band_tol=5e-3):
    """Image-wide mean / p99 EPE and the mean EPE of every border band and strip seam; returns the stats line."""
    e = epe(mine, ref)
    H, W = e.shape
    yx = np.unravel_index(np.argmax(e), e.shape)
    stats = f"{what}: mean {e.mean():.2e} p99 {np.percentile(e, 99):.2e} max {e.max():.2e} at (y, x) = {yx}"
    print(stats)
    assert np.isfinite(e).all(), what
    assert e.mean() <= mean_tol and np.percentile(e, 99) <= p99_tol, stats
    for name, (ry, rx) in regions(H, W).items():
        eb = e[np.ix_(ry, rx)]
        assert eb.mean() <= band_tol, f"{stats}; {name} band mean {eb.mean():.2e}"
    return e


# ------------------------------------------------------------------------------------------------------------------
# Farneback
# ------------------------------------------------------------------------------------------------------------------
FB_CASES = [((200, 264), SEQUENCE), ((201, 263), SEQUENCE), ((512, 768), ("beyond", "rotation"))]
FB_IDS = [f"{h}x{w}" for (h, w), _ in FB_CASES]
MOTION_512 = {"beyond": synthetic.shift_motion(24.0, -3.0)}     # OpenCV finds this one at 512 x 768 only


def _case(shape, names):
    """The sequence of one case; its last frame carries NaN pixels and a NaN stripe."""
    H, W = shape
    motions = [MOTION_512.get(n, MOTIONS[n]) if shape == (512, 768) else MOTIONS[n] for n in names]
    bt = synthetic.moving_texture(H, W, motions, seed=H + W)
    rng = np.random.default_rng(H * W)
    bt[-1].reshape(-1)[rng.integers(0, H * W, H * W // 500)] = np.nan
    bt[-1, H // 3:H // 3 + 6] = np.nan
    return bt


@pytest.fixture(scope="module")
def tfb():
    import tobac_flow_b200
    return tobac_flow_b200


@pytest.mark.parametrize("shape,names", FB_CASES, ids=FB_IDS)
def test_farneback_motion_vs_opencv(tfb, shape, names):
    bt = _case(shape, names)
    f = tfb.create_flow(bt)
    rf, rb = ops.create_flow(bt, backend="cv2")
    for i, name in enumerate(names):
        check_flow(f.forward_flow[i], rf[i], f"{shape} {name} forward")
        check_flow(f.backward_flow[i + 1], rb[i + 1], f"{shape} {name} backward")
    assert np.abs(f.forward_flow).max() <= 20 and np.abs(f.backward_flow).max() <= 20
    assert np.array_equal(f.forward_flow[-1], -f.backward_flow[-1])
    assert np.array_equal(f.backward_flow[0], -f.forward_flow[0])
    if shape == (512, 768):
        # OpenCV finds the 24 px motion at this size: the clamp is what bounds the result
        assert (np.abs(rf[0, ..., 0]) >= 20).mean() > 0.05
        assert (np.abs(f.forward_flow[0, ..., 0]) == 20).mean() > 0.05
    else:
        # the generator moves the texture as intended: the shift towards the top-left is found away from the borders
        inner = f.forward_flow[0, 16:-16, 16:-16]
        assert np.allclose(np.median(inner.reshape(-1, 2), 0), (-3.4, -5.7), atol=0.05)


@pytest.mark.parametrize("shape,names", FB_CASES, ids=FB_IDS)
def test_iteration_kernels_agree_on_motion(tfb, shape, names):
    """The contract of test_iteration_kernels_agree (test_gpu_parity.py) on flows that leave the image, vary in space
    and reach the clamp: 0 = 1 and 3 = 4 = 5 bit for bit, |0 - 3| <= 4e-5.

    The exception is the pair moved beyond the clamp.  The pyramid does not lock on to that motion everywhere, the
    iteration is far from converged there, and the one-ulp difference of the two kernels' reciprocals of the
    determinant grows to a few 1e-3 px on 1-2 % of the pixels (measured on a B200: 7e-5 px at 200 x 264, 3e-3 px at
    512 x 768).  OpenCV's own result is as unsettled there.  For that pair each kernel must instead meet the OpenCV
    contract of test_farneback_motion_vs_opencv on its own, and the two must agree within its p99 bound."""
    from tobac_flow_b200 import _lib
    lib = _lib.load()
    bt = _case(shape, names)
    res = {}
    try:
        for k in (0, 1, 3, 4, 5):
            _lib.check(lib.tf_fb_select_kernel(k), "tf_fb_select_kernel")
            f = tfb.create_flow(bt)
            res[k] = (f.forward_flow.copy(), f.backward_flow.copy())
    finally:
        lib.tf_fb_select_kernel(3)
    assert all(np.array_equal(a, b) for a, b in zip(res[0], res[1]))
    for k in (4, 5):
        assert all(np.array_equal(a, b) for a, b in zip(res[3], res[k])), k
    rf, rb = ops.create_flow(bt, backend="cv2")
    for i, name in enumerate(names):
        pairs = ((res[0][0][i], res[3][0][i], rf[i]), (res[0][1][i + 1], res[3][1][i + 1], rb[i + 1]))
        for d, (k0, k3, ref) in enumerate(pairs):
            diff = np.abs(k0 - k3).max()
            print(f"{shape} {name} {'forward' if d == 0 else 'backward'}: |kernel 0 - kernel 3| max {diff:.2e}")
            if name == "beyond":
                check_flow(k0, ref, f"{shape} {name} kernel 0")
                assert diff <= 1e-2, diff
            else:
                assert diff <= 4e-5, (name, d, diff)


# ------------------------------------------------------------------------------------------------------------------
# variational refinement as a stage
# ------------------------------------------------------------------------------------------------------------------
VR_SHAPES = [(32, 64), (31, 63), (33, 65), (64, 128), (97, 129), (375, 625), (1, 70), (70, 1), (5, 5)]
VR_ITERS = [(5, 5), (1, 1), (2, 3), (3, 8), (0, 5), (5, 0)]
VR_MOTIONS = ("neg", "large", "rotation", "zoom", "split")


def vr_inputs(H, W):
    """(q0, q1, fwd, bwd): u8 pairs of the motion cases with OpenCV's Farneback flows, plus a pair whose input flow is
    the outward zoom flow x 1.3 (so samples leave every border)."""
    bt = synthetic.moving_texture(H, W, [MOTIONS[n] for n in VR_MOTIONS], seed=H * 31 + W)
    q0, q1, fw, bw = [], [], [], []
    fb = cv2.FarnebackOpticalFlow_create()
    for i in range(len(VR_MOTIONS)):
        a, b = ops.pair_to_u8(bt[i], bt[i + 1])
        q0.append(a), q1.append(b), fw.append(fb.calc(a, b, None)), bw.append(fb.calc(b, a, None))
    y, x = np.mgrid[0:H, 0:W].astype(np.float64)
    u, v = MOTIONS["zoom"](x, y, H, W)
    z = (np.stack([u, v], -1) * 1.3).astype(np.float32)
    a, b = ops.pair_to_u8(bt[VR_MOTIONS.index("zoom")], bt[VR_MOTIONS.index("zoom") + 1])
    q0.append(a), q1.append(b), fw.append(z), bw.append(-z)
    return np.stack(q0), np.stack(q1), np.stack(fw), np.stack(bw)


def gpu_vr(q0, q1, fwd, bwd, fp, sor):
    """tf_variational_refinement on device u8 pairs, flows at the strides calculate_flow_device uses."""
    import torch
    from tobac_flow_b200 import _lib
    lib = _lib.load()
    n, H, W = q0.shape
    p = _lib.default_vr_params()
    p.fixed_point_iterations, p.sor_iterations = fp, sor
    dq0, dq1 = torch.from_numpy(q0).cuda(), torch.from_numpy(q1).cuda()
    df, db = torch.from_numpy(fwd.copy()).cuda(), torch.from_numpy(bwd.copy()).cuda()
    nbytes = int(lib.tf_vr_workspace_bytes(n, H, W))
    ws = torch.empty((nbytes,), dtype=torch.uint8, device="cuda")
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    _lib.check(lib.tf_variational_refinement(dq0.data_ptr(), dq1.data_ptr(), df.data_ptr(), H * W * 2, db.data_ptr(),
                                             H * W * 2, n, H, W, ctypes.byref(p), ws.data_ptr(), nbytes, st),
               "tf_variational_refinement")
    return df.cpu().numpy(), db.cpu().numpy()


def cv2_vr(q0, q1, flow, fp, sor):
    vr = cv2.VariationalRefinement_create()
    vr.setFixedPointIterations(fp)
    vr.setSorIterations(sor)
    return vr.calc(q0, q1, flow.copy())


@pytest.fixture(scope="module")
def vr_cases():
    cache = {}

    def get(shape):
        if shape not in cache:
            cache[shape] = vr_inputs(*shape)
        return cache[shape]
    return get


@pytest.mark.parametrize("fp,sor", VR_ITERS)
@pytest.mark.parametrize("shape", VR_SHAPES, ids=lambda s: f"{s[0]}x{s[1]}")
def test_variational_refinement_vs_opencv(vr_cases, shape, fp, sor):
    """Fused SOR (1..5 sweeps) and the unfused path (8 sweeps) against cv2.VariationalRefinement at the same counts;
    with no fixed-point or no SOR iteration the flow comes back unchanged (-0.0 may become +0.0)."""
    q0, q1, fwd, bwd = vr_cases(shape)
    gf, gb = gpu_vr(q0, q1, fwd, bwd, fp, sor)
    worst = 0.0
    for i in range(q0.shape[0]):
        for d, (a, b, flow, got) in enumerate(((q0[i], q1[i], fwd[i], gf[i]), (q1[i], q0[i], bwd[i], gb[i]))):
            ref = cv2_vr(a, b, flow, fp, sor)
            if fp == 0 or sor == 0:
                assert np.array_equal(ref, flow) and np.array_equal(got, flow)
                continue
            e = epe(got, ref)
            yx = np.unravel_index(np.argmax(e), e.shape)
            worst = max(worst, e.max())
            assert np.isfinite(e).all()
            assert e.max() <= 1e-3 and e.mean() <= 1e-5, (i, d, e.mean(), e.max(), yx)
    print(f"VR {shape} ({fp},{sor}) max EPE vs OpenCV {worst:.2e}")
    if fp and sor:
        assert np.abs(gf - fwd).max() > 1e-3          # the refinement did change the flows


@pytest.mark.parametrize("shape", [(33, 65), (97, 129), (1, 70)], ids=lambda s: f"{s[0]}x{s[1]}")
@pytest.mark.parametrize("fp,sor", [(5, 5), (3, 8)])
def test_variational_refinement_batch_equals_single_pairs(vr_cases, shape, fp, sor):
    q0, q1, fwd, bwd = (a[:3] for a in vr_cases(shape))
    gf, gb = gpu_vr(q0, q1, fwd, bwd, fp, sor)
    for i in range(3):
        sf, sb = gpu_vr(q0[i:i + 1], q1[i:i + 1], fwd[i:i + 1], bwd[i:i + 1], fp, sor)
        assert np.array_equal(gf[i], sf[0]) and np.array_equal(gb[i], sb[0]), i
