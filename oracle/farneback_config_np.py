"""ORACLE (test infrastructure, never shipped, never on the product path).

``cv2.FarnebackOpticalFlow_create(numLevels, pyrScale, False, winSize, numIters, polyN, polySigma, flags)`` restated
in numpy for the settings beyond the factory defaults that ``farneback_np`` restates: box windows of any size (an
even ``winSize`` included) and ``flags=OPTFLOW_FARNEBACK_GAUSSIAN`` (256), i.e. OpenCV's
``FarnebackUpdateFlow_GaussianBlur``.  The level plan, pyramid, polynomial expansion (``polyN`` 5 or 7) and
``FarnebackUpdateMatrices`` are ``farneback_np``'s; only the window sums and the solve are restated here.

Pinning: ``tests/test_oracle_farneback_config.py`` checks this restatement against cv2 over the settings grid the GPU
tests use.  At the factory defaults it gives the same bits as ``farneback_np.farneback``.
"""
import math

import numpy as np

from . import farneback_np as fb

F32 = np.float32
OPTFLOW_FARNEBACK_GAUSSIAN = 256


def box_sum(M: np.ndarray, win: int) -> np.ndarray:
    """Box SUM over (2m+1) x (2m+1), m = win // 2, with replicate borders, fp64 (OpenCV keeps double running sums).
    For an even ``win`` OpenCV sums win + 1 rows and columns (and still scales by 1 / win**2, see ``solve``)."""
    h, w = M.shape[:2]
    m = win // 2
    n = 2 * m + 1
    Md = M.astype(np.float64)
    ys = np.clip(np.arange(-m, h + m), 0, h - 1)
    cs = np.concatenate([np.zeros((1, w, 5)), np.cumsum(Md[ys], axis=0)], axis=0)
    v = cs[n:] - cs[:-n]
    xs = np.clip(np.arange(-m, w + m), 0, w - 1)
    cs = np.concatenate([np.zeros((h, 1, 5)), np.cumsum(v[:, xs], axis=1)], axis=1)
    return cs[:, n:] - cs[:, :-n]


def gaussian_window(win: int) -> np.ndarray:
    """Taps k[0..m] (m = win // 2, sigma = 0.3 m): float32 exp values normalised by their sum taken in double."""
    m = win // 2
    sigma = m * 0.3
    k = np.ones(m + 1, dtype=F32)
    s = 1.0
    for i in range(1, m + 1):
        k[i] = F32(math.exp(-i * i / (2 * sigma * sigma)))
        s += float(k[i]) * 2
    return (k.astype(np.float64) * (1.0 / s)).astype(F32)


def gaussian_sum(M: np.ndarray, win: int) -> np.ndarray:
    """k0 r[y] + sum_i k_i (r[y+i] + r[y-i]) along y, then the same along x, fp32, replicate borders."""
    k = gaussian_window(win)
    m = len(k) - 1
    h, w = M.shape[:2]
    ys = np.arange(h)
    v = M * k[0]
    for i in range(1, m + 1):
        v = v + (M[np.minimum(ys + i, h - 1)] + M[np.maximum(ys - i, 0)]) * k[i]
    xs = np.arange(w)
    out = v * k[0]
    for i in range(1, m + 1):
        out = out + k[i] * (v[:, np.maximum(xs - i, 0)] + v[:, np.minimum(xs + i, w - 1)])
    return out.astype(F32)


def solve(S: np.ndarray, scale: float) -> np.ndarray:
    """The 2x2 solve of the window sums S (h, w, 5) scaled by ``scale``, in double as OpenCV does."""
    g11, g12, g22, h1, h2 = (S[..., i].astype(np.float64) * scale for i in range(5))
    idet = 1.0 / (g11 * g22 - g12 * g12 + 1e-3)
    out = np.empty(S.shape[:2] + (2,), dtype=F32)
    out[..., 0] = ((g11 * h2 - g12 * h1) * idet).astype(F32)
    out[..., 1] = ((g22 * h1 - g12 * h2) * idet).astype(F32)
    return out


def update_flow(M: np.ndarray, win: int, flags: int) -> np.ndarray:
    if flags == OPTFLOW_FARNEBACK_GAUSSIAN:
        return solve(gaussian_sum(M, win), 1.0)
    return solve(box_sum(M, win), 1.0 / (win * win))


def farneback(prev_u8: np.ndarray, next_u8: np.ndarray, *, num_levels=5, pyr_scale=0.5, win_size=13, num_iters=10,
              poly_n=5, poly_sigma=1.1, flags=0) -> np.ndarray:
    """cv2.FarnebackOpticalFlow_create(num_levels, pyr_scale, False, win_size, num_iters, poly_n, poly_sigma,
    flags).calc(prev, next, None) restated; ``flags`` is 0 or 256.  Returns (H, W, 2) fp32."""
    if flags not in (0, OPTFLOW_FARNEBACK_GAUSSIAN):
        raise ValueError("flags must be 0 or 256 (OPTFLOW_FARNEBACK_GAUSSIAN)")
    prev_u8 = np.ascontiguousarray(prev_u8, dtype=np.uint8)
    next_u8 = np.ascontiguousarray(next_u8, dtype=np.uint8)
    H, W = prev_u8.shape
    flow = None
    for lvl in fb.level_plan(H, W, num_levels, pyr_scale):
        h, w = lvl["h"], lvl["w"]
        if flow is None:
            flow = np.zeros((h, w, 2), dtype=F32)
        else:
            flow = fb.resize_linear(flow, h, w) * F32(1.0 / pyr_scale)
        R0 = fb.poly_exp(fb.pyramid_level(prev_u8, lvl), poly_n, poly_sigma)
        R1 = fb.poly_exp(fb.pyramid_level(next_u8, lvl), poly_n, poly_sigma)
        M = fb.update_matrices(R0, R1, flow)
        for i in range(num_iters):
            flow = update_flow(M, win_size, flags)
            if i < num_iters - 1:
                M = fb.update_matrices(R0, R1, flow)
    return flow
