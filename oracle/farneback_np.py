"""ORACLE (test infrastructure, never shipped, never on the product path).

CPU restatement in numpy of the dense optical flow the reference calls at
``tobac_flow/flow.py:511,516`` (``of_model.calc(prev, next, None)``) through
``tobac_flow/utils/flow_utils.py:52-53`` (``cv2.optflow.createOptFlow_Farneback()``).

The arithmetic lives in a third-party dependency that is NOT vendored under /root/reference:
OpenCV (declared unpinned as ``opencv`` in ``environment.yml:15``; the image has
opencv-python-headless 4.13.0).  This file restates the published CPU algorithm of
``cv::FarnebackOpticalFlow::calc`` (opencv/modules/video/src/optflowgf.cpp: FarnebackPrepareGaussian,
FarnebackPolyExp, FarnebackUpdateMatrices, FarnebackUpdateFlow_Blur, FarnebackOpticalFlowImpl::calc)
with the factory defaults numLevels=5, pyrScale=0.5, fastPyramids=False, winSize=13, numIters=10,
polyN=5, polySigma=1.1, flags=0.

Pinning: ``tests/test_oracle_farneback.py`` checks this restatement against cv2 itself (when cv2 is
importable) and against golden vectors generated from the unmodified reference
(``tests/golden/make_golden.py``).  The reference's own tests do not pin Farneback numerics
(``tests/test_flow.py:14-15`` is an isinstance check only).

Every stage is exposed separately so the CUDA kernels can be checked stage by stage.
"""
import math

import numpy as np

F32 = np.float32

DEFAULTS = dict(
    num_levels=5, pyr_scale=0.5, win_size=13, num_iters=10, poly_n=5, poly_sigma=1.1
)

BORDER_ATTEN = np.array([0.14, 0.14, 0.4472, 0.4472, 0.4472], dtype=F32)


def cv_round(x: float) -> int:
    """cvRound: round half to even (lrint under the default rounding mode)."""
    return int(np.rint(x))


# ----------------------------------------------------------------------------------------------
# pyramid geometry  (FarnebackOpticalFlowImpl::calc, level cropping + per-level sizes)
# ----------------------------------------------------------------------------------------------
def level_plan(height: int, width: int, num_levels: int = 5, pyr_scale: float = 0.5):
    """Return a list (coarsest first) of dicts: k, scale, h, w, sigma, ksize."""
    min_size = 32
    k = 0
    scale = 1.0
    while k < num_levels:
        scale *= pyr_scale
        if width * scale < min_size or height * scale < min_size:
            break
        k += 1
    levels = k
    plan = []
    for k in range(levels, -1, -1):
        scale = 1.0
        for _ in range(k):
            scale *= pyr_scale
        sigma = (1.0 / scale - 1.0) * 0.5
        ksize = cv_round(sigma * 5) | 1
        ksize = max(ksize, 3)
        w = cv_round(width * scale)
        h = cv_round(height * scale)
        plan.append(dict(k=k, scale=scale, h=h, w=w, sigma=sigma, ksize=ksize))
    return plan


# ----------------------------------------------------------------------------------------------
# GaussianBlur (imgproc) on CV_32F, BORDER_REFLECT_101, separable
# ----------------------------------------------------------------------------------------------
def gaussian_kernel(ksize: int, sigma: float) -> np.ndarray:
    """cv::getGaussianKernel(ksize, sigma, CV_32F)."""
    if sigma <= 0:
        if ksize == 3:
            return np.array([0.25, 0.5, 0.25], dtype=F32)
        sigma = 0.3 * ((ksize - 1) * 0.5 - 1) + 0.8
    x = np.arange(ksize, dtype=np.float64) - (ksize - 1) * 0.5
    k = np.exp(-0.5 * x * x / (sigma * sigma))
    k = k / k.sum()
    return k.astype(F32)


def _reflect101(idx: np.ndarray, n: int) -> np.ndarray:
    if n == 1:
        return np.zeros_like(idx)
    period = 2 * (n - 1)
    idx = np.mod(idx, period)
    return np.where(idx >= n, period - idx, idx)


def gaussian_blur(img: np.ndarray, ksize: int, sigma: float) -> np.ndarray:
    """cv::GaussianBlur(img32f, (ksize, ksize), sigma, sigma) — rows first, then columns, fp32."""
    k = gaussian_kernel(ksize, sigma)
    h, w = img.shape
    r = ksize // 2
    xs = _reflect101(np.arange(-r, w + r), w)
    padded = img[:, xs]
    tmp = np.zeros((h, w), dtype=F32)
    for i in range(ksize):
        tmp += k[i] * padded[:, i : i + w]
    ys = _reflect101(np.arange(-r, h + r), h)
    padded = tmp[ys, :]
    out = np.zeros((h, w), dtype=F32)
    for i in range(ksize):
        out += k[i] * padded[i : i + h, :]
    return out


# ----------------------------------------------------------------------------------------------
# cv::resize(..., INTER_LINEAR) for CV_32F (1 or 2 channels)
# ----------------------------------------------------------------------------------------------
def _linear_coords(dst_n: int, src_n: int):
    scale = float(src_n) / float(dst_n)
    d = np.arange(dst_n, dtype=np.float64)
    f = ((d + 0.5) * scale - 0.5).astype(F32)
    i = np.floor(f).astype(np.int64)
    f = (f - i.astype(F32)).astype(F32)
    lo = i < 0
    f[lo] = 0
    i[lo] = 0
    hi = i >= src_n - 1
    f[hi] = 0
    i[hi] = src_n - 1
    i1 = np.minimum(i + 1, src_n - 1)
    return i, i1, f


def resize_linear(img: np.ndarray, h: int, w: int) -> np.ndarray:
    """cv::resize(img, (w, h), INTER_LINEAR); img is (H, W) or (H, W, C) float32."""
    sh, sw = img.shape[:2]
    if (sh, sw) == (h, w):
        return img.astype(F32, copy=True)
    x0, x1, fx = _linear_coords(w, sw)
    y0, y1, fy = _linear_coords(h, sh)
    if img.ndim == 3:
        fx = fx[None, :, None]
        fyb = fy[:, None, None]
    else:
        fx = fx[None, :]
        fyb = fy[:, None]
    one = F32(1)
    rows = img[:, x0] * (one - fx) + img[:, x1] * fx
    out = rows[y0] * (one - fyb) + rows[y1] * fyb
    return out.astype(F32)


def pyramid_level(img_u8: np.ndarray, lvl: dict) -> np.ndarray:
    """convertTo(CV_32F) -> GaussianBlur(ksize, sigma) -> resize(w, h)   (calc(), per level/image)."""
    f = img_u8.astype(F32)
    f = gaussian_blur(f, lvl["ksize"], lvl["sigma"])
    return resize_linear(f, lvl["h"], lvl["w"])


# ----------------------------------------------------------------------------------------------
# FarnebackPrepareGaussian / FarnebackPolyExp
# ----------------------------------------------------------------------------------------------
def prepare_gaussian(n: int = 5, sigma: float = 1.1):
    if sigma < np.finfo(np.float32).eps:
        sigma = n * 0.3
    x = np.arange(-n, n + 1)
    g = np.exp(-(x * x) / (2.0 * sigma * sigma)).astype(F32)
    s = 1.0 / float(np.sum(g.astype(np.float64)))
    g = (g.astype(np.float64) * s).astype(F32)
    xg = (x * g.astype(np.float64)).astype(F32)
    xxg = (x * x * g.astype(np.float64)).astype(F32)
    G = np.zeros((6, 6), dtype=np.float64)
    gd = g.astype(np.float64)
    for yy in range(-n, n + 1):
        for xx in range(-n, n + 1):
            gg = gd[yy + n] * gd[xx + n]
            G[0, 0] += gg
            G[1, 1] += gg * xx * xx
            G[3, 3] += gg * xx * xx * xx * xx
            G[5, 5] += gg * xx * xx * yy * yy
    G[2, 2] = G[0, 3] = G[0, 4] = G[3, 0] = G[4, 0] = G[1, 1]
    G[4, 4] = G[3, 3]
    G[3, 4] = G[4, 3] = G[5, 5]
    inv = np.linalg.inv(G)
    return g, xg, xxg, inv[1, 1], inv[0, 3], inv[3, 3], inv[5, 5]


def poly_exp(img: np.ndarray, n: int = 5, sigma: float = 1.1) -> np.ndarray:
    """FarnebackPolyExp: (h, w) fp32 -> (h, w, 5) fp32; replicate borders; fp64 horizontal sums."""
    g, xg, xxg, ig11, ig03, ig33, ig55 = prepare_gaussian(n, sigma)
    h, w = img.shape
    ys = np.arange(h)
    # vertical pass, fp32
    r0 = img * g[n]
    r1 = np.zeros_like(img)
    r2 = np.zeros_like(img)
    for k in range(1, n + 1):
        s0 = img[np.maximum(ys - k, 0)]
        s1 = img[np.minimum(ys + k, h - 1)]
        p = s0 + s1
        r0 = r0 + g[n + k] * p
        r1 = r1 + xg[n + k] * (s1 - s0)
        r2 = r2 + xxg[n + k] * p
    # horizontal pass, fp64 accumulators on fp32 operands
    xs = np.arange(w)
    gd, xgd, xxgd = g.astype(np.float64), xg.astype(np.float64), xxg.astype(np.float64)

    def col(a, idx):
        return a[:, np.clip(idx, 0, w - 1)]

    b1 = (r0 * g[n]).astype(np.float64)
    b3 = (r1 * g[n]).astype(np.float64)
    b5 = (r2 * g[n]).astype(np.float64)
    b2 = np.zeros((h, w), np.float64)
    b4 = np.zeros((h, w), np.float64)
    b6 = np.zeros((h, w), np.float64)
    for k in range(1, n + 1):
        r0p, r0m = col(r0, xs + k), col(r0, xs - k)
        r1p, r1m = col(r1, xs + k), col(r1, xs - k)
        r2p, r2m = col(r2, xs + k), col(r2, xs - k)
        tg = (r0p + r0m).astype(np.float64)  # fp32 add, then promoted (double tg = float + float)
        b1 += tg * gd[n + k]
        b4 += tg * xxgd[n + k]
        b2 += (r0p - r0m).astype(np.float64) * xgd[n + k]
        b3 += (r1p + r1m).astype(np.float64) * gd[n + k]
        b6 += (r1p - r1m).astype(np.float64) * xgd[n + k]
        b5 += (r2p + r2m).astype(np.float64) * gd[n + k]
    out = np.empty((h, w, 5), dtype=F32)
    out[..., 1] = (b2 * ig11).astype(F32)
    out[..., 0] = (b3 * ig11).astype(F32)
    out[..., 3] = (b1 * ig03 + b4 * ig33).astype(F32)
    out[..., 2] = (b1 * ig03 + b5 * ig33).astype(F32)
    out[..., 4] = (b6 * ig55).astype(F32)
    return out


# ----------------------------------------------------------------------------------------------
# FarnebackUpdateMatrices
# ----------------------------------------------------------------------------------------------
def _border_band(n: int) -> np.ndarray:
    """OpenCV's test ``(unsigned)(x - BORDER) >= (unsigned)(n - BORDER*2)`` along one axis.  For n >= 10 it selects the
    five indices next to either edge.  For n < 10 the right-hand side wraps: it then selects only n - 5 <= x < 5, so on a
    side of 6..9 px some indices within 5 px of an edge are not attenuated (unless the other axis selects the pixel)."""
    i = np.arange(n, dtype=np.int64)
    return ((i - 5) & 0xFFFFFFFF) >= ((n - 10) & 0xFFFFFFFF)


def border_scale(h: int, w: int) -> np.ndarray:
    """The attenuation FarnebackUpdateMatrices applies to (r2..r6): 1 where neither axis' band test holds, else the
    product (x<B ? b[x] : 1)*(x>=w-B ? b[w-x-1] : 1)*(y<B ? b[y] : 1)*(y>=h-B ? b[h-y-1] : 1), left to right in fp32."""
    def factors(n):
        lo = np.ones(n, dtype=F32)
        hi = np.ones(n, dtype=F32)
        for i in range(min(5, n)):
            lo[i] = BORDER_ATTEN[i]
            hi[n - 1 - i] = BORDER_ATTEN[i]
        return lo, hi
    xl, xr = factors(w)
    yt, yb = factors(h)
    prod = ((xl * xr)[None, :] * yt[:, None]).astype(F32) * yb[:, None]
    band = _border_band(w)[None, :] | _border_band(h)[:, None]
    return np.where(band, prod, F32(1)).astype(F32)


def update_matrices(R0: np.ndarray, R1: np.ndarray, flow: np.ndarray) -> np.ndarray:
    """(h,w,5),(h,w,5),(h,w,2) -> M (h,w,5) fp32."""
    h, w = flow.shape[:2]
    x = np.arange(w, dtype=F32)[None, :]
    y = np.arange(h, dtype=F32)[:, None]
    dx = flow[..., 0]
    dy = flow[..., 1]
    fx = (x + dx).astype(F32)
    fy = (y + dy).astype(F32)
    with np.errstate(invalid="ignore"):
        x1 = np.floor(fx).astype(np.int64)
        y1 = np.floor(fy).astype(np.int64)
    fx = (fx - x1.astype(F32)).astype(F32)
    fy = (fy - y1.astype(F32)).astype(F32)
    inside = (x1 >= 0) & (x1 < w - 1) & (y1 >= 0) & (y1 < h - 1)
    xc = np.clip(x1, 0, max(w - 2, 0))
    yc = np.clip(y1, 0, max(h - 2, 0))
    one = F32(1)
    a00 = (one - fx) * (one - fy)
    a01 = fx * (one - fy)
    a10 = (one - fx) * fy
    a11 = fx * fy
    x2 = np.minimum(xc + 1, w - 1)
    y2 = np.minimum(yc + 1, h - 1)

    def samp(c):
        p = R1[..., c]
        return a00 * p[yc, xc] + a01 * p[yc, x2] + a10 * p[y2, xc] + a11 * p[y2, x2]

    r2 = np.where(inside, samp(0), F32(0)).astype(F32)
    r3 = np.where(inside, samp(1), F32(0)).astype(F32)
    r4 = np.where(inside, (R0[..., 2] + samp(2)) * F32(0.5), R0[..., 2]).astype(F32)
    r5 = np.where(inside, (R0[..., 3] + samp(3)) * F32(0.5), R0[..., 3]).astype(F32)
    r6 = np.where(inside, (R0[..., 4] + samp(4)) * F32(0.25), R0[..., 4] * F32(0.5)).astype(F32)
    r2 = (R0[..., 0] - r2) * F32(0.5)
    r3 = (R0[..., 1] - r3) * F32(0.5)
    r2 = r2 + (r4 * dy + r6 * dx)
    r3 = r3 + (r6 * dy + r5 * dx)
    sc = border_scale(h, w)
    r2, r3, r4, r5, r6 = (v * sc for v in (r2, r3, r4, r5, r6))
    M = np.empty((h, w, 5), dtype=F32)
    M[..., 0] = r4 * r4 + r6 * r6
    M[..., 1] = (r4 + r5) * r6
    M[..., 2] = r5 * r5 + r6 * r6
    M[..., 3] = r4 * r2 + r6 * r3
    M[..., 4] = r6 * r2 + r5 * r3
    return M


# ----------------------------------------------------------------------------------------------
# FarnebackUpdateFlow_Blur (box window, replicate borders, Jacobi update)
# ----------------------------------------------------------------------------------------------
def box_sum(M: np.ndarray, win: int) -> np.ndarray:
    """win x win box SUM with replicate borders, fp64 (OpenCV keeps double running sums)."""
    h, w = M.shape[:2]
    m = win // 2
    Md = M.astype(np.float64)
    ys = np.clip(np.arange(-m, h + m), 0, h - 1)
    cs = np.concatenate([np.zeros((1, w, 5)), np.cumsum(Md[ys], axis=0)], axis=0)
    v = cs[win:] - cs[:-win]
    xs = np.clip(np.arange(-m, w + m), 0, w - 1)
    cs = np.concatenate([np.zeros((h, 1, 5)), np.cumsum(v[:, xs], axis=1)], axis=1)
    return cs[:, win:] - cs[:, :-win]


def solve_flow(S: np.ndarray, win: int) -> np.ndarray:
    scale = 1.0 / (win * win)
    g11, g12, g22, h1, h2 = (S[..., i] * scale for i in range(5))
    idet = 1.0 / (g11 * g22 - g12 * g12 + 1e-3)
    out = np.empty(S.shape[:2] + (2,), dtype=F32)
    out[..., 0] = ((g11 * h2 - g12 * h1) * idet).astype(F32)
    out[..., 1] = ((g22 * h1 - g12 * h2) * idet).astype(F32)
    return out


def update_flow_blur(M: np.ndarray, win: int = 13) -> np.ndarray:
    return solve_flow(box_sum(M, win), win)


# ----------------------------------------------------------------------------------------------
# the whole calc()
# ----------------------------------------------------------------------------------------------
def farneback(prev_u8: np.ndarray, next_u8: np.ndarray, *, num_levels=5, pyr_scale=0.5,
              win_size=13, num_iters=10, poly_n=5, poly_sigma=1.1, trace=None) -> np.ndarray:
    """cv2.FarnebackOpticalFlow_create().calc(prev, next, None) restated.  Returns (H, W, 2) fp32.

    ``trace`` (optional list) receives a dict per level with the intermediate arrays.
    """
    prev_u8 = np.ascontiguousarray(prev_u8, dtype=np.uint8)
    next_u8 = np.ascontiguousarray(next_u8, dtype=np.uint8)
    H, W = prev_u8.shape
    flow = None
    for lvl in level_plan(H, W, num_levels, pyr_scale):
        h, w = lvl["h"], lvl["w"]
        if flow is None:
            flow = np.zeros((h, w, 2), dtype=F32)
        else:
            flow = resize_linear(flow, h, w) * F32(1.0 / pyr_scale)
        I0 = pyramid_level(prev_u8, lvl)
        I1 = pyramid_level(next_u8, lvl)
        R0 = poly_exp(I0, poly_n, poly_sigma)
        R1 = poly_exp(I1, poly_n, poly_sigma)
        flow_in = flow
        M = update_matrices(R0, R1, flow)
        for i in range(num_iters):
            flow = update_flow_blur(M, win_size)
            if i < num_iters - 1:
                M = update_matrices(R0, R1, flow)
        if trace is not None:
            trace.append(dict(level=lvl, I0=I0, I1=I1, R0=R0, R1=R1, flow_in=flow_in, flow=flow))
    return flow
