"""ORACLE (test infrastructure, never shipped, never on the product path).

numpy restatement of OpenCV's Dense Inverse Search, ``cv::DISOpticalFlow::calc``
(``opencv/modules/video/src/dis_flow.cpp``), for patch size 8 with mean normalisation and spatial propagation on
(what the three presets use).  Pinned against ``cv2.DISOpticalFlow`` by ``tests/test_oracle_dis.py``.

Every float operation is float32 in the order OpenCV's SSE build evaluates it, so that the patch search takes the
same propagation choices:

* the 8x8 patch sums accumulate in four lanes (lane k takes columns k and k + 4 of every row, row by row) and the
  lanes are reduced as (l0 + l2) + (l1 + l3);
* the structure-tensor box sums are float running sums of exact integer products and differences;
* the patch search visits a stripe's patches in raster order (pass 1: left and upper neighbour as candidates) and in
  reverse raster order (pass 2: right and lower neighbour).  OpenCV splits the patch rows into 8 stripes of
  ceil(hs / 8) rows whatever the thread count, and flow never propagates across a stripe boundary.  Inside a stripe
  the patches of one anti-diagonal (row + column = const) do not depend on each other, which is how both this
  oracle and the CUDA kernel run them.
"""
import math

import numpy as np

from . import farneback_np, varref_np

F32 = np.float32
PATCH = 8
BORDER = 16
N_STRIPES = 8
EPS = F32(0.001)
INF = F32(1e10)

# preset -> (finest_scale, patch_stride, gradient_descent_iterations, variational_refinement_iterations)
PRESETS = {0: (2, 4, 12, 0), 1: (2, 4, 16, 5), 2: (1, 3, 25, 5)}
VR_ALPHA, VR_DELTA, VR_GAMMA, VR_EPSILON = 20.0, 5.0, 10.0, 0.01


def scale_plan(H: int, W: int, finest: int):
    """(finest, coarsest) scales calc() runs for an H x W frame; ValueError where cv2 raises."""
    c = min(int(math.log(max(W, H) / (4.0 * PATCH)) / math.log(2.0) + 0.5),
            int(math.log(min(W, H) // PATCH) / math.log(2.0)) if min(W, H) // PATCH > 0 else -1)
    if c < 0:
        raise ValueError("The input image must have either width or height >= 12")
    if c < finest:
        # autoSelectPatchSizeAndScales (finest 0..2 keep patch size 8): coarsest from the width only
        if finest > 2:
            raise NotImplementedError("finest_scale > 2 on a small frame selects patch size 12")
        c = max(0, int(math.floor(math.log2((2.0 * float(np.float32(W))) / (5.0 * 8.0)))))
        finest = max(c - 2, 0)
    return finest, c


def scale_sizes(H: int, W: int, finest: int, coarsest: int):
    """{scale: (h, w)} of the pyramid (frame size over 2^finest, then halved)."""
    sizes = {finest: (H // (1 << finest), W // (1 << finest))}
    for i in range(finest + 1, coarsest + 1):
        h, w = sizes[i - 1]
        sizes[i] = (h // 2, w // 2)
    return sizes


# ----------------------------------------------------------------------------------------------
# cv::resize(INTER_AREA) for CV_8U (downscale), cv::spatialGradient
# ----------------------------------------------------------------------------------------------
def _area_tab(ssize: int, dsize: int):
    scale = ssize / dsize
    tab = []
    for d in range(dsize):
        fs1 = d * scale
        fs2 = fs1 + scale
        cell = min(scale, ssize - fs1)
        s1, s2 = math.ceil(fs1), math.floor(fs2)
        s2 = min(s2, ssize - 1)
        s1 = min(s1, s2)
        if s1 - fs1 > 1e-3:
            tab.append((d, s1 - 1, F32((s1 - fs1) / cell)))
        for s in range(s1, s2):
            tab.append((d, s, F32(1.0 / cell)))
        if fs2 - s2 > 1e-3:
            tab.append((d, s2, F32(min(min(fs2 - s2, 1.0), cell) / cell)))
    return tab


def resize_area_u8(img: np.ndarray, h: int, w: int) -> np.ndarray:
    sh, sw = img.shape
    if (sh, sw) == (h, w):
        return img.copy()
    sx, sy = sw / w, sh / h
    if abs(sx - round(sx)) < 2.220446049250313e-16 and abs(sy - round(sy)) < 2.220446049250313e-16:
        kx, ky = int(round(sx)), int(round(sy))
        blocks = img[:h * ky, :w * kx].astype(np.int32).reshape(h, ky, w, kx)
        if kx == 2 and ky == 2:
            return ((blocks.sum((1, 3)) + 2) >> 2).astype(np.uint8)
        s = blocks.sum((1, 3)).astype(F32) * F32(1.0 / (kx * ky))
        return np.clip(np.rint(s), 0, 255).astype(np.uint8)
    xt, yt = _area_tab(sw, w), _area_tab(sh, h)
    src = img.astype(F32)
    out = np.zeros((h, w), np.uint8)
    acc = None
    prev = yt[0][0]
    for dy, syy, beta in yt:
        buf = np.zeros(w, F32)
        for dx, sxx, alpha in xt:
            buf[dx] = F32(buf[dx] + F32(src[syy, sxx] * alpha))
        if dy != prev:
            out[prev] = np.clip(np.rint(acc), 0, 255).astype(np.uint8)
            acc = (beta * buf).astype(F32)
            prev = dy
        elif acc is None:
            acc = (beta * buf).astype(F32)
        else:
            acc = (acc + beta * buf).astype(F32)
    out[prev] = np.clip(np.rint(acc), 0, 255).astype(np.uint8)
    return out


def spatial_gradient(img: np.ndarray):
    """cv::spatialGradient (3x3 Sobel, BORDER_REFLECT_101) -> (Ix, Iy) int16."""
    h, w = img.shape
    ry = farneback_np._reflect101(np.arange(-1, h + 1), h)
    rx = farneback_np._reflect101(np.arange(-1, w + 1), w)
    p = img.astype(np.int32)[ry][:, rx]
    c = lambda dy, dx: p[1 + dy:1 + dy + h, 1 + dx:1 + dx + w]  # noqa: E731
    ix = (c(-1, 1) - c(-1, -1)) + 2 * (c(0, 1) - c(0, -1)) + (c(1, 1) - c(1, -1))
    iy = (c(1, -1) - c(-1, -1)) + 2 * (c(1, 0) - c(-1, 0)) + (c(1, 1) - c(-1, 1))
    return ix.astype(np.int16), iy.astype(np.int16)


def pyramid(q: np.ndarray, finest: int, coarsest: int):
    """{scale: u8 image}: INTER_AREA from the frame to the finest scale, then halving."""
    sizes = scale_sizes(*q.shape, finest, coarsest)
    out = {finest: resize_area_u8(q, *sizes[finest])}
    for i in range(finest + 1, coarsest + 1):
        out[i] = resize_area_u8(out[i - 1], *sizes[i])
    return out


# ----------------------------------------------------------------------------------------------
# per-scale stages
# ----------------------------------------------------------------------------------------------
def structure_tensor(ix: np.ndarray, iy: np.ndarray, stride: int):
    """precomputeStructureTensor -> (xx, yy, xy, x, y), each (hs, ws) float32."""
    h, w = ix.shape
    ws = 1 + (w - PATCH) // stride
    hs = 1 + (h - PATCH) // stride
    x = ix.astype(np.int64)
    y = iy.astype(np.int64)
    terms = [x * x, y * y, x * y, x, y]
    aux = []
    for t in terms:
        s = np.zeros(h, F32)
        for j in range(PATCH):
            s = (s + t[:, j].astype(F32)).astype(F32)
        a = np.zeros((h, ws), F32)
        a[:, 0] = s
        js = 1
        for j in range(PATCH, w):
            s = (s + (t[:, j] - t[:, j - PATCH]).astype(F32)).astype(F32)
            if (j - PATCH + 1) % stride == 0:
                a[:, js] = s
                js += 1
        aux.append(a)
    out = []
    for a in aux:
        s = np.zeros(ws, F32)
        for i in range(PATCH):
            s = (s + a[i]).astype(F32)
        o = np.zeros((hs, ws), F32)
        o[0] = s
        is_ = 1
        for i in range(PATCH, h):
            s = (s + (a[i] - a[i - PATCH])).astype(F32)
            if (i - PATCH + 1) % stride == 0:
                o[is_] = s
                is_ += 1
        out.append(o)
    return out


def _lane_reduce(v):
    """v_reduce_sum of a 4-lane float32 accumulator: (l0 + l2) + (l1 + l3)."""
    return (v[..., 0] + v[..., 2]) + (v[..., 1] + v[..., 3])


def _patch_diff(I0, I1e, i, j, ux, uy, h, w):
    """Bilinear I1 patch minus the I0 patch for K patches at (i, j) displaced by (ux, uy): (K, 8, 8) float32."""
    bsz = F32(BORDER)
    i_I1 = np.minimum(np.maximum((i.astype(F32) + uy) + bsz, F32(BORDER - PATCH + 1)), F32(BORDER + h - 1))
    j_I1 = np.minimum(np.maximum((j.astype(F32) + ux) + bsz, F32(BORDER - PATCH + 1)), F32(BORDER + w - 1))
    di = i_I1 - np.floor(i_I1)
    dj = j_I1 - np.floor(j_I1)
    one = F32(1)
    w11 = (di * dj)[:, None, None]
    w10 = (di * (one - dj))[:, None, None]
    w01 = ((one - di) * dj)[:, None, None]
    w00 = ((one - di) * (one - dj))[:, None, None]
    ii = i_I1.astype(np.int64)[:, None, None] + np.arange(PATCH)[None, :, None]
    jj = j_I1.astype(np.int64)[:, None, None] + np.arange(PATCH)[None, None, :]
    a, b = I1e[ii, jj], I1e[ii, jj + 1]
    c, d = I1e[ii + 1, jj], I1e[ii + 1, jj + 1]
    i0 = I0[i[:, None, None] + np.arange(PATCH)[None, :, None], j[:, None, None] + np.arange(PATCH)[None, None, :]]
    return (((w00 * a + w01 * b) + w10 * c) + w11 * d) - i0


def _lane_sums(x):
    """Per-row lane accumulation of an (K, 8, 8) term: lane k += x[row, k] + x[row, k + 4]."""
    acc = np.zeros(x.shape[:1] + (4,), F32)
    for r in range(PATCH):
        acc = acc + (x[:, r, :4] + x[:, r, 4:])
    return _lane_reduce(acc)


def _ssd_mean_norm(d):
    n = F32(PATCH * PATCH)
    s = _lane_sums(d)
    sq = _lane_sums(d * d)
    return sq - s * s / n


def _process_patch(d, gx, gy, x_grad_sum, y_grad_sum):
    n = F32(PATCH * PATCH)
    s = _lane_sums(d)
    sq = _lane_sums(d * d)
    sx = _lane_sums(d * gx)
    sy = _lane_sums(d * gy)
    dux = sx - s * x_grad_sum / n
    duy = sy - s * y_grad_sum / n
    return sq - s * s / n, dux, duy


def patch_inverse_search(I0, I1, Ix, Iy, Ux, Uy, stride, gd_iters):
    """PatchInverseSearch_ParBody over all 8 stripes, two passes -> sparse (Sx, Sy), each (hs, ws)."""
    h, w = I0.shape
    ws = 1 + (w - PATCH) // stride
    hs = 1 + (h - PATCH) // stride
    xx, yy, xy, gxs, gys = structure_tensor(Ix, Iy, stride)
    I1e = np.pad(I1, BORDER, mode="edge").astype(F32)
    I0f = I0.astype(F32)
    gxf, gyf = Ix.astype(F32), Iy.astype(F32)
    psz2 = PATCH // 2
    stripe = int(math.ceil(hs / float(N_STRIPES)))
    Sx = np.zeros((hs, ws), F32)
    Sy = np.zeros((hs, ws), F32)
    for is_ in range(hs):
        for js in range(ws):
            Sx[is_, js] = Ux[is_ * stride + psz2, js * stride + psz2]
            Sy[is_, js] = Uy[is_ * stride + psz2, js * stride + psz2]
    inner = int(math.floor(gd_iters / F32(2)))
    # patches grouped by anti-diagonal of their stripe-local position
    is_all, js_all = np.meshgrid(np.arange(hs), np.arange(ws), indexing="ij")
    s0 = (is_all // stripe) * stripe
    s1 = np.minimum(s0 + stripe, hs)
    for it in range(2):
        if it == 0:
            diag = (is_all - s0) + js_all
        else:
            diag = (s1 - 1 - is_all) + (ws - 1 - js_all)
        step = 1 if it == 0 else -1
        for dg in range(int(diag.max()) + 1):
            sel = np.nonzero(diag == dg)
            pi, pj = sel
            i = pi * stride
            j = pj * stride
            cx, cy = Sx[pi, pj].copy(), Sy[pi, pj].copy()
            best = _ssd_mean_norm(_patch_diff(I0f, I1e, i, j, cx, cy, h, w))
            # horizontal neighbour in the pass direction, then the vertical one (same stripe only)
            for ni, nj, ok in ((pi, pj - step, (pj - step >= 0) & (pj - step < ws)),
                               (pi - step, pj, (pi - step >= s0[sel]) & (pi - step < s1[sel]))):
                k = np.nonzero(ok)[0]
                if k.size == 0:
                    continue
                nx, ny = Sx[ni[k], nj[k]], Sy[ni[k], nj[k]]
                c = _ssd_mean_norm(_patch_diff(I0f, I1e, i[k], j[k], nx, ny, h, w))
                better = c < best[k]
                kb = k[better]
                best[kb] = c[better]
                cx[kb] = nx[better]
                cy[kb] = ny[better]
            sx0, sy0 = cx.copy(), cy.copy()
            a, b, cxy = xx[pi, pj], yy[pi, pj], xy[pi, pj]
            det = a * b - cxy * cxy
            det = np.where(np.abs(det) < EPS, EPS, det)
            h11, h12, h22 = b / det, -cxy / det, a / det
            xg, yg = gxs[pi, pj], gys[pi, pj]
            ii = i[:, None, None] + np.arange(PATCH)[None, :, None]
            jj = j[:, None, None] + np.arange(PATCH)[None, None, :]
            pgx, pgy = gxf[ii, jj], gyf[ii, jj]
            prev = np.full(pi.shape, INF, F32)
            live = np.ones(pi.shape, bool)
            for _ in range(inner):
                k = np.nonzero(live)[0]
                if k.size == 0:
                    break
                ssd, dux, duy = _process_patch(_patch_diff(I0f, I1e, i[k], j[k], cx[k], cy[k], h, w),
                                               pgx[k], pgy[k], xg[k], yg[k])
                cx[k] = cx[k] - (h11[k] * dux + h12[k] * duy)
                cy[k] = cy[k] - (h12[k] * dux + h22[k] * duy)
                stop = ssd >= prev[k]
                live[k[stop]] = False
                prev[k] = np.where(stop, prev[k], ssd)
            dx = (cx - sx0).astype(np.float64)
            dy = (cy - sy0).astype(np.float64)
            keep = np.sqrt(dx * dx + dy * dy) <= PATCH
            Sx[pi, pj] = np.where(keep, cx, sx0)
            Sy[pi, pj] = np.where(keep, cy, sy0)
    return Sx, Sy


def densify(I0, I1, Sx, Sy, stride):
    """Densification_ParBody: per pixel, the patches covering it, weighted by 1 / max(1, |I1(x + u) - I0(x)|)."""
    h, w = I0.shape
    hs, ws = Sx.shape
    I0f, I1f = I0.astype(F32), I1.astype(F32)

    def cover(n, ns):
        lo, hi = np.zeros(n, int), np.zeros(n, int)
        s, e = 0, -1
        for p in range(n):
            if p % stride == 0 and p + PATCH <= n:
                e += 1
            if p - PATCH >= 0 and (p - PATCH) % stride == 0 and s < e:
                s += 1
            lo[p], hi[p] = s, e
        return lo, hi
    ilo, ihi = cover(h, hs)
    jlo, jhi = cover(w, ws)
    Ux = np.zeros((h, w), F32)
    Uy = np.zeros((h, w), F32)
    ii, jj = np.meshgrid(np.arange(h), np.arange(w), indexing="ij")
    sum_x = np.zeros((h, w), F32)
    sum_y = np.zeros((h, w), F32)
    sum_c = np.zeros((h, w), F32)
    one = F32(1)
    for a in range(int((ihi - ilo).max()) + 1):
        for b in range(int((jhi - jlo).max()) + 1):
            is_ = ilo[ii] + a
            js = jlo[jj] + b
            m = (is_ <= ihi[ii]) & (js <= jhi[jj])
            isc, jsc = np.minimum(is_, hs - 1), np.minimum(js, ws - 1)
            sx, sy = Sx[isc, jsc], Sy[isc, jsc]
            j_m = np.minimum(np.maximum(jj.astype(F32) + sx, F32(0)), F32(w) - one - EPS)
            i_m = np.minimum(np.maximum(ii.astype(F32) + sy, F32(0)), F32(h) - one - EPS)
            j_l = j_m.astype(np.int64)
            i_l = i_m.astype(np.int64)
            j_u, i_u = j_l + 1, i_l + 1
            jlf, ilf, juf, iuf = j_l.astype(F32), i_l.astype(F32), j_u.astype(F32), i_u.astype(F32)
            diff = ((((j_m - jlf) * (i_m - ilf)) * I1f[i_u, j_u] + ((juf - j_m) * (i_m - ilf)) * I1f[i_u, j_l])
                    + ((j_m - jlf) * (iuf - i_m)) * I1f[i_l, j_u]) + ((juf - j_m) * (iuf - i_m)) * I1f[i_l, j_l]
            diff = diff - I0f
            coef = one / np.maximum(one, np.abs(diff))
            sum_x = np.where(m, sum_x + coef * sx, sum_x)
            sum_y = np.where(m, sum_y + coef * sy, sum_y)
            sum_c = np.where(m, sum_c + coef, sum_c)
    Ux[:] = sum_x / sum_c
    Uy[:] = sum_y / sum_c
    return Ux, Uy


def resize_linear(img: np.ndarray, h: int, w: int) -> np.ndarray:
    """cv::resize(INTER_LINEAR) of an (sh, sw, 2) float32 flow.  Columns outside the source take the edge value;
    rows outside it take the edge row with the unclamped weights (row 0 * (1 - fy) + row 0 * fy), as OpenCV does."""
    sh, sw = img.shape[:2]
    if (sh, sw) == (h, w):
        return img.copy()

    def coords(dn, sn):
        f = ((np.arange(dn, dtype=np.float64) + 0.5) * (1.0 / (dn / sn)) - 0.5).astype(F32)
        i = np.floor(f).astype(np.int64)
        return i, (f - i.astype(F32)).astype(F32)
    x0, fx = coords(w, sw)
    edge = (x0 < 0) | (x0 >= sw - 1)
    fx[edge] = 0
    x0 = np.clip(x0, 0, sw - 1)
    x1 = np.minimum(x0 + 1, sw - 1)
    y, fy = coords(h, sh)
    y0, y1 = np.clip(y, 0, sh - 1), np.clip(y + 1, 0, sh - 1)
    one = F32(1)
    fx = fx[None, :, None]
    rows = img[:, x0] * (one - fx) + img[:, x1] * fx
    rows[:, edge] = img[:, x0[edge]]
    fy = fy[:, None, None]
    return (rows[y0] * (one - fy) + rows[y1] * fy).astype(F32)


def dis(I0: np.ndarray, I1: np.ndarray, preset: int = 1, finest_scale=None, patch_stride=None,
        gradient_descent_iterations=None, variational_refinement_iterations=None, trace=None):
    """cv2.DISOpticalFlow_create(preset) (with the given overrides) .calc(I0, I1, None) -> (H, W, 2) float32."""
    f0, stride, gd, vr = PRESETS[preset]
    f0 = f0 if finest_scale is None else finest_scale
    stride = stride if patch_stride is None else patch_stride
    gd = gd if gradient_descent_iterations is None else gradient_descent_iterations
    vr = vr if variational_refinement_iterations is None else variational_refinement_iterations
    H, W = I0.shape
    finest, coarsest = scale_plan(H, W, f0)
    p0, p1 = pyramid(I0, finest, coarsest), pyramid(I1, finest, coarsest)
    h, w = p0[coarsest].shape
    U = np.zeros((h, w, 2), F32)
    for s in range(coarsest, finest - 1, -1):
        Ix, Iy = spatial_gradient(p0[s])
        Sx, Sy = patch_inverse_search(p0[s], p1[s], Ix, Iy, U[..., 0], U[..., 1], stride, gd)
        Ux, Uy = densify(p0[s], p1[s], Sx, Sy, stride)
        U = np.stack([Ux, Uy], -1)
        if trace is not None:
            trace[s] = dict(Sx=Sx, Sy=Sy, dense=U.copy())
        if vr > 0:
            U = varref_np.variational_refinement(p0[s], p1[s], U, alpha=VR_ALPHA, delta=VR_DELTA, gamma=VR_GAMMA,
                                                 fixed_point_iterations=vr, sor_iterations=5,
                                                 epsilon=VR_EPSILON).astype(F32)
        if s > finest:
            U = resize_linear(U, *p0[s - 1].shape) * F32(2)
    return (resize_linear(U, H, W) * F32(1 << finest)).astype(F32)


def dis_cv2(I0, I1, preset=1, finest_scale=None, patch_stride=None, gradient_descent_iterations=None,
            variational_refinement_iterations=None):
    """The same through OpenCV (a fresh object per call: calc() lowers the finest scale of its object for a small
    frame, and a reused object would keep that lowered scale)."""
    import cv2
    m = cv2.DISOpticalFlow_create(preset)
    if finest_scale is not None:
        m.setFinestScale(finest_scale)
    if patch_stride is not None:
        m.setPatchStride(patch_stride)
    if gradient_descent_iterations is not None:
        m.setGradientDescentIterations(gradient_descent_iterations)
    if variational_refinement_iterations is not None:
        m.setVariationalRefinementIterations(variational_refinement_iterations)
    return m.calc(np.ascontiguousarray(I0), np.ascontiguousarray(I1), None)


# ----------------------------------------------------------------------------------------------
# calculate_flow / create_flow with DIS as the model (the sequence rules of flow_ops, DIS per pair)
# ----------------------------------------------------------------------------------------------
def dis_pair(q0: np.ndarray, q1: np.ndarray, model, backend: str = "numpy"):
    """Both directions of a pair; ``model`` carries ``preset`` and the overrides (the attribute names of
    ``tobac_flow_b200.DISOpticalFlow``).  backend "numpy": this restatement, "cv2": OpenCV."""
    kw = dict(preset=model.preset, finest_scale=model.finest_scale, patch_stride=model.patch_stride,
              gradient_descent_iterations=model.gradient_descent_iterations,
              variational_refinement_iterations=model.variational_refinement_iterations)
    f = dis_cv2 if backend == "cv2" else dis
    return f(q0, q1, **kw), f(q1, q0, **kw)


def calculate_flow(data, model, smoothing_passes=0, interp_method="linear", backend="numpy", vr_steps=0):
    """``flow_ops.calculate_flow`` with DIS in place of Farneback: per-pair normalisation, the model, the optional
    refinement and smoothing of the reference, then the end rules."""
    from . import flow_ops
    data = np.asarray(data)
    T = data.shape[0]
    fwd = np.full(data.shape + (2,), np.nan, dtype=F32)
    bwd = np.full(data.shape + (2,), np.nan, dtype=F32)
    for i in range(T - 1):
        q0, q1 = flow_ops.pair_to_u8(data[i], data[i + 1])
        f, b = dis_pair(q0, q1, model, backend)
        if vr_steps > 0:
            f, b = flow_ops.refine_pair(q0, q1, f, b, backend)
        for _ in range(smoothing_passes):
            f, b = flow_ops.smooth_flow_step(f, b, interp_method, backend)
        fwd[i], bwd[i + 1] = f, b
    fwd[-1] = -bwd[-1]
    bwd[0] = -fwd[0]
    return fwd, bwd


def create_flow(data, model, smoothing_passes=0, interp_method="linear", max_value=20, backend="numpy", vr_steps=0):
    fwd, bwd = calculate_flow(data, model, smoothing_passes, interp_method, backend, vr_steps)
    return np.minimum(np.maximum(fwd, -max_value), max_value), np.minimum(np.maximum(bwd, -max_value), max_value)
