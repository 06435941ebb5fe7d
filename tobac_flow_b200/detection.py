"""B200-native mirror of the growth-marker detection (``tobac_flow/detection.py:34-125``; SURVEY.md section 8f rank 2).

``filtered_tdiff``, ``get_curvature_filter`` and ``detect_growth_markers`` keep the reference's names, arguments and
results; every array stays in HBM between the Flow operators (diff -> /dt -> 3-frame nanmean -> grey opening x
curvature filter -> thresholds -> binary opening -> Flow.label -> label filters).  The scipy.ndimage filters the
reference calls are re-implemented bit-exactly in ``csrc/morph.cu`` / ``csrc/ccl.cu``.  There is no CPU fallback.
"""
import numpy as np
import torch

from . import _lib
from . import analysis
from . import label as _label
from .flow import Flow, _as_numpy, _device, _stream, _to_device, _to_host

_T_STRUCT = np.zeros([3, 3, 3])
_T_STRUCT[:, 1, 1] = 1


def _nanmean0(x):
    return np.nanmean(x, 0)


_nanmean0._tf_reducer = _lib.TF_RED_NANMEAN


def filtered_tdiff(flow, raw_diff):
    """detection.py:34-60: 3-frame semi-Lagrangian moving average (nanmean) of a time derivative."""
    return flow.convolve(raw_diff, structure=_T_STRUCT, func=_nanmean0)


def gaussian_kernel1d(sigma: float, truncate: float = 4.0):
    """The weights scipy.ndimage.gaussian_filter1d builds for order 0 (``_gaussian_kernel1d``) and their radius."""
    sd = float(sigma)
    radius = int(truncate * sd + 0.5)
    x = np.arange(-radius, radius + 1)
    phi = np.exp(-0.5 / (sd * sd) * x ** 2)
    return phi / phi.sum(), radius


def _float_code(t: torch.Tensor):
    if t.dtype == torch.float32:
        return _lib.TF_F32
    if t.dtype == torch.float64:
        return _lib.TF_F64
    raise NotImplementedError(f"dtype {t.dtype} is not supported (float32 / float64 are)")


def gaussian_filter_yx_device(field: torch.Tensor, sigma: float) -> torch.Tensor:
    """ndi.gaussian_filter(field, (0, sigma, sigma)) on a (T, H, W) CUDA tensor."""
    if sigma <= 1e-15:
        return field.clone()
    w, radius = gaussian_kernel1d(sigma)
    w = np.ascontiguousarray(w[::-1], dtype=np.float64)
    T, H, W = field.shape
    tmp, out = torch.empty_like(field), torch.empty_like(field)
    _lib.check(_lib.load().tf_gaussian_filter_yx(field.data_ptr(), tmp.data_ptr(), out.data_ptr(), _float_code(field),
                                                 T, H, W, w.ctypes.data_as(_lib.ctypes.POINTER(_lib.ctypes.c_double)),
                                                 radius, _stream()), "tf_gaussian_filter_yx")
    return out


def curvature_filter_device(field: torch.Tensor, sigma=2, threshold=0, direction="negative") -> torch.Tensor:
    """``get_curvature_filter`` on a float CUDA tensor -> uint8 mask (T, H, W)."""
    if direction not in ("negative", "positive"):
        raise ValueError("Direction must be either positive or negative")
    lib = _lib.load()
    T, H, W = field.shape
    smoothed = gaussian_filter_yx_device(field, sigma)
    m = torch.empty((T, H, W), dtype=torch.uint8, device=field.device)
    _lib.check(lib.tf_curvature_mask(smoothed.data_ptr(), m.data_ptr(), _float_code(smoothed), T, H, W, float(threshold),
                                     int(direction == "positive"), _stream()), "tf_curvature_mask")
    del smoothed
    filled = torch.empty_like(m)
    done = 0
    while done < T:
        tc = min(T - done, 65535)
        ws_bytes = int(lib.tf_ccl_workspace_bytes(tc, H, W))
        ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=field.device)
        _lib.check(lib.tf_binary_fill_holes(m[done:].data_ptr(), filled[done:].data_ptr(), tc, H, W, ws.data_ptr(),
                                            ws_bytes, _stream()), "tf_binary_fill_holes")
        done += tc
    del m
    return _binary_opening(filled)


def get_curvature_filter(field, sigma=2, threshold=0, direction="negative"):
    """detection.py:64-94: Gaussian-smoothed second differences both beyond the threshold, holes filled, opened."""
    if direction not in ("negative", "positive"):
        raise ValueError("Direction must be either positive or negative")
    t, host = _to_device(field)
    if not t.dtype.is_floating_point:
        raise NotImplementedError("get_curvature_filter: integer fields are not supported")
    if t.dtype not in (torch.float32, torch.float64):
        t = t.to(torch.float32)
    m = curvature_filter_device(t, sigma, threshold, direction)
    return _to_host(m).view(np.bool_) if host else m.to(torch.bool)


def grey_opening_cross_device(field: torch.Tensor) -> torch.Tensor:
    T, H, W = field.shape
    tmp, out = torch.empty_like(field), torch.empty_like(field)
    _lib.check(_lib.load().tf_grey_opening_cross(field.data_ptr(), tmp.data_ptr(), out.data_ptr(), _float_code(field),
                                                 T, H, W, _stream()), "tf_grey_opening_cross")
    return out


def _threshold_ge(x: torch.Tensor, threshold) -> torch.Tensor:
    """uint8 mask of ``x >= threshold`` for a contiguous float CUDA tensor."""
    m = torch.empty(x.shape, dtype=torch.uint8, device=x.device)
    _lib.check(_lib.load().tf_threshold_ge(x.data_ptr(), float(threshold), m.data_ptr(), _float_code(x), x.numel(),
                                           _stream()), "tf_threshold_ge")
    return m


def _mask_multiply(x: torch.Tensor, mask: torch.Tensor) -> torch.Tensor:
    """``x * mask`` for a float CUDA tensor and a uint8 mask of the same shape."""
    out = torch.empty_like(x)
    _lib.check(_lib.load().tf_mask_multiply(x.data_ptr(), mask.data_ptr(), out.data_ptr(), _float_code(x), x.numel(),
                                            _stream()), "tf_mask_multiply")
    return out


def _binary_opening(m: torch.Tensor) -> torch.Tensor:
    """Per-frame binary opening of a (T, H, W) uint8 mask with the 2-D cross."""
    T, H, W = m.shape
    out = torch.empty_like(m)
    _lib.check(_lib.load().tf_binary_opening_cross(m.data_ptr(), out.data_ptr(), T, H, W, _stream()),
               "tf_binary_opening_cross")
    return out


def scale_by_dt_device(raw32: torch.Tensor, dt_minutes) -> torch.Tensor:
    """A (T, H, W) float32 ``Flow.diff`` result divided frame by frame by ``dt_minutes`` (T doubles) -> float64."""
    T, H, W = raw32.shape
    dt = torch.from_numpy(np.ascontiguousarray(np.asarray(dt_minutes, np.float64))).to(raw32.device)
    assert dt.numel() == T
    raw = torch.empty((T, H, W), dtype=torch.float64, device=raw32.device)
    _lib.check(_lib.load().tf_scale_frames(raw32.data_ptr(), dt.data_ptr(), raw.data_ptr(), T, H, W, _stream()),
               "tf_scale_frames")
    return raw


def growth_seed_masks_device(smoothed: torch.Tensor, wvd: torch.Tensor):
    """detection.py:105-112 -> (filtered, filtered >= 0.5, wvd >= -5, seeds): ``filtered`` is the grey opening of
    ``smoothed`` times the curvature filter of ``wvd``, the seeds are ``filtered >= 0.25`` opened; masks are uint8."""
    opened = grey_opening_cross_device(smoothed)                                        # :105-107
    curv = curvature_filter_device(wvd)                                                 # :108
    filtered = _mask_multiply(opened, curv)
    del opened, curv
    seeds = _binary_opening(_threshold_ge(filtered, 0.25))
    return filtered, _threshold_ge(filtered, 0.5), _threshold_ge(wvd, -5.0), seeds


def growth_marker_keep(tmin, tmax, any_a, any_b) -> np.ndarray:
    """detection.py:114-119 from the per-label statistics of the linked labels (``any_a``: touches filtered >= 0.5,
    ``any_b``: touches wvd >= -5): the relabel table that keeps the labels lasting at least 3 frames and touching both
    masks, numbered 1, 2, ... in label order.  The reference renumbers three times; dropping labels commutes with the
    order-preserving renumbering, so one table does."""
    wh = ((tmax[1:] - tmin[1:] + 1) >= 3) & (any_a[1:] != 0) & (any_b[1:] != 0)
    return analysis._keep_table(wh)


def time_diff_minutes(t_coord) -> np.ndarray:
    """``get_time_diff_from_coord`` (tobac_flow/utils/datetime_utils.py:126-166): centred differences in minutes."""
    import pandas as pd
    dts = pd.to_datetime(np.asarray(t_coord)).to_pydatetime().tolist()
    return np.array([(dts[1] - dts[0]).total_seconds() / 60]
                    + [(dts[i + 2] - dts[i]).total_seconds() / 120 for i in range(len(dts) - 2)]
                    + [(dts[-1] - dts[-2]).total_seconds() / 60])


def growth_markers_device(flow: Flow, wvd: torch.Tensor, dt_minutes) -> dict:
    """The whole of detection.py:98-118 on device tensors; returns the intermediates the reference exposes plus the
    markers.  ``wvd`` (T, H, W) float32 or float64 CUDA tensor, ``dt_minutes`` T doubles."""
    raw = scale_by_dt_device(flow.diff(wvd), dt_minutes)                                # detection.py:99-100
    smoothed = filtered_tdiff(flow, raw)                                                # :103, float32
    filtered, m05, warm, seeds = growth_seed_masks_device(smoothed, wvd)                # :105-112
    flat, n_flat = _label.flat_label_device(seeds, 1)                                   # Flow.label -> label.py:125
    linked, _ = _label.link_overlap_device(flow, flat, _label._default_structure(), 0, 1, n_flat)
    _, tmin, tmax, any_a, any_b = analysis.label_stats_device(linked, m05, warm)
    markers = _label.relabel_device(linked, growth_marker_keep(tmin, tmax, any_a, any_b))   # :114-119
    return dict(raw=raw, smoothed=smoothed, filtered=filtered, seeds=seeds, flat=flat, linked=linked, markers=markers)


def _time_coord(field):
    t_coord = getattr(field, "t", None)
    if t_coord is None:
        raise AttributeError("the field needs a time coordinate `.t`")
    return time_diff_minutes(t_coord)


def growth_rate_device(flow: Flow, field: torch.Tensor, dt_minutes, method: str = "linear") -> torch.Tensor:
    """``get_growth_rate`` on a float32 / float64 CUDA tensor: Flow.diff / dt, then the 5-point same-step nanmean
    (float32 result)."""
    raw = scale_by_dt_device(flow.diff(field, method=method), dt_minutes)
    s_struct = np.zeros((3, 3, 3), bool)
    s_struct[1, 1, :] = s_struct[1, :, 1] = True
    return flow.convolve(raw, structure=s_struct, func=_nanmean0, method=method)


def get_growth_rate(flow, field, method: str = "linear"):
    """detection.py:168-198: growth / cooling rate of ``field`` (an array with a ``.t`` time coordinate)."""
    dt = _time_coord(field)
    on_device = isinstance(field, torch.Tensor) and field.is_cuda
    f, _ = _to_device(field if isinstance(field, torch.Tensor) else _as_numpy(field))
    if f.dtype not in (torch.float32, torch.float64):     # the taps are warped in the field's own dtype (cv2.remap)
        f = f.to(torch.float32)
    r = growth_rate_device(flow, f, dt, method)
    return r if on_device else _to_host(r)


def anvil_markers_device(flow: Flow, field: torch.Tensor, threshold=-5, overlap=0.5, absolute_overlap=5,
                         min_length=3) -> torch.Tensor:
    """``get_anvil_markers`` on a float CUDA tensor (subsegment_shrink == 0)."""
    flat, n_flat = _label.flat_label_device(_binary_opening(_threshold_ge(field, threshold)), 1)
    linked, _ = _label.link_overlap_device(flow, flat, _label._default_structure(), overlap, absolute_overlap, n_flat)
    _, tmin, tmax, _, _ = analysis.label_stats_device(linked)
    wh = (tmax[1:] - tmin[1:] + 1) > min_length        # find_object_lengths(...) > min_length, then remap_labels
    return analysis._apply_keep(linked, wh)


def get_anvil_markers(flow, field, threshold=-5, overlap=0.5, absolute_overlap=5, subsegment_shrink=0, min_length=3):
    """detection.py:494-516 (without the DataArray decoration): opened ``field >= threshold`` mask, linked along the
    flow, labels no longer than ``min_length`` steps dropped and the rest renumbered."""
    if subsegment_shrink != 0:
        raise NotImplementedError("subsegment_shrink != 0 (skimage watershed sub-segmentation) is not built here")
    on_device = isinstance(field, torch.Tensor) and field.is_cuda
    f, _ = _to_device(field if isinstance(field, torch.Tensor) else _as_numpy(field))
    if f.dtype not in (torch.float32, torch.float64):
        f = f.to(torch.float32)
    r = anvil_markers_device(flow, f, threshold, overlap, absolute_overlap, min_length)
    return r if on_device else _to_host(r)


def detect_growth_markers(flow, wvd):
    """detection.py:98-125: returns (wvd_diff_smoothed, marker_labels).

    ``wvd`` is an ``xr.DataArray``-like with a ``.t`` time coordinate (results are numpy, wrapped back into the
    input's type when it offers ``coords`` / ``dims``), or a CUDA tensor with a ``t`` attribute (results stay on the
    device).
    """
    t_coord = getattr(wvd, "t", None)
    if t_coord is None:
        raise AttributeError("wvd needs a time coordinate `.t` (detection.py:100)")
    dt = time_diff_minutes(t_coord)
    on_device = isinstance(wvd, torch.Tensor) and wvd.is_cuda
    w, _ = _to_device(wvd if isinstance(wvd, torch.Tensor) else _as_numpy(wvd))
    if w.dtype not in (torch.float32, torch.float64):     # a float64 field is filtered in float64, as scipy would
        w = w.to(torch.float32)
    r = growth_markers_device(flow, w, dt)
    if on_device:
        return r["smoothed"], r["markers"]
    smoothed, markers = _to_host(r["smoothed"]), _to_host(r["markers"])
    if hasattr(wvd, "coords") and hasattr(wvd, "dims") and not isinstance(wvd, np.ndarray):
        try:
            markers = type(wvd)(markers, wvd.coords, wvd.dims)                          # detection.py:121-123
        except Exception:
            pass
    return smoothed, markers


def nan_gaussian_filter(a, *args, propagate_nan=True, **kwargs):
    """detection.py:128-146: Gaussian filter that ignores NaNs (filtered values / filtered weights).  Built for the
    per-frame filter the reference's callers use -- a (t, y, x) field with sigma = (0, s, s), or one (y, x) frame with a
    scalar sigma -- in scipy's default mode; other ``gaussian_filter`` arguments are not built."""
    if kwargs or len(args) != 1:
        raise NotImplementedError("nan_gaussian_filter: only the sigma argument of gaussian_filter is supported")
    sigma = args[0]
    t, host = _to_device(a)
    if t.dtype not in (torch.float32, torch.float64):
        t = t.to(torch.float64)
    squeeze = t.dim() == 2
    if squeeze:
        t = t[None]
        s_yx = (sigma, sigma) if np.isscalar(sigma) else tuple(sigma)
    else:
        if np.isscalar(sigma) or len(sigma) != 3 or sigma[0] != 0:
            raise NotImplementedError("nan_gaussian_filter: a (t, y, x) field needs sigma = (0, s, s)")
        s_yx = (sigma[1], sigma[2])
    if t.dim() != 3 or s_yx[0] != s_yx[1]:
        raise NotImplementedError("nan_gaussian_filter: equal y / x sigmas on (y, x) or (t, y, x) fields only")
    t = t.contiguous()
    wh_nan = torch.isnan(t)
    a0 = torch.where(wh_nan, torch.zeros_like(t), t)
    c = torch.where(wh_nan, torch.zeros_like(t), torch.ones_like(t))
    a0_g = gaussian_filter_yx_device(a0, float(s_yx[0]))
    c_g = gaussian_filter_yx_device(c, float(s_yx[0]))
    c_g = torch.where(c_g == 0, torch.full_like(c_g, float("nan")), c_g)
    result = a0_g / c_g
    if propagate_nan:
        result = torch.where(wh_nan, torch.full_like(result, float("nan")), result)
    if squeeze:
        result = result[0]
    return _to_host(result) if host else result


def growth_markers_multichannel_device(flow: Flow, wvd: torch.Tensor, bt: torch.Tensor, dt_wvd, dt_bt, overlap=0.5,
                                       min_length=4, lower_threshold=0.25, upper_threshold=0.5) -> dict:
    """detection.py:203-254 on device tensors (``subsegment_shrink == 0``): growth of the water-vapour difference OR
    cooling of the window brightness temperature, each inside its curvature filter."""
    wvd_s = filtered_tdiff(flow, scale_by_dt_device(flow.diff(wvd), dt_wvd))           # :214-217
    bt_s = filtered_tdiff(flow, scale_by_dt_device(flow.diff(bt), dt_bt))              # :218-220
    grow = _threshold_ge(_mask_multiply(wvd_s, curvature_filter_device(wvd)), lower_threshold)     # :223
    cool = _threshold_ge(-_mask_multiply(bt_s, curvature_filter_device(bt, direction="positive")),
                         lower_threshold)                                               # :224-225 (x <= -l)
    seeds = _binary_opening(torch.bitwise_or(grow, cool))
    flat, n_flat = _label.flat_label_device(seeds, 1)                                   # Flow.label(overlap=overlap), :227-233
    linked, _ = _label.link_overlap_device(flow, flat, _label._default_structure(), overlap, 1, n_flat)
    markers = linked
    if bool((linked != 0).any()):                                                       # :236-246
        masks = [_threshold_ge(wvd_s, upper_threshold), _threshold_ge(-bt_s, upper_threshold),
                 (wvd > -5).to(torch.uint8)]
        markers = analysis.filter_labels_by_length_and_multimask_legacy(linked, masks, min_length)
    else:
        import warnings
        warnings.warn("No regions detected in labeled array", RuntimeWarning)
    return dict(wvd_diff_smoothed=wvd_s, bt_diff_smoothed=bt_s, seeds=seeds, linked=linked, markers=markers)


def detect_growth_markers_multichannel(flow, wvd, bt, t_sigma=1, overlap=0.5, subsegment_shrink=0, min_length=4,
                                       lower_threshold=0.25, upper_threshold=0.5):
    """detection.py:203-254: returns (wvd_diff_smoothed, bt_diff_smoothed, markers).  ``wvd`` and ``bt`` carry a ``.t``
    time coordinate; CUDA tensors (with a ``t`` attribute) keep the results on the device."""
    if subsegment_shrink != 0:
        raise NotImplementedError("subsegment_shrink != 0 (skimage watershed sub-segmentation) is not built here")
    if getattr(wvd, "t", None) is None or getattr(bt, "t", None) is None:
        raise AttributeError("wvd and bt need a time coordinate `.t` (detection.py:216, 219)")
    on_device = isinstance(wvd, torch.Tensor) and wvd.is_cuda
    w, _ = _to_device(wvd if isinstance(wvd, torch.Tensor) else _as_numpy(wvd))
    b, _ = _to_device(bt if isinstance(bt, torch.Tensor) else _as_numpy(bt))
    if w.dtype not in (torch.float32, torch.float64):
        w = w.to(torch.float32)
    if b.dtype not in (torch.float32, torch.float64):
        b = b.to(torch.float32)
    r = growth_markers_multichannel_device(flow, w.contiguous(), b.contiguous(), time_diff_minutes(wvd.t),
                                           time_diff_minutes(bt.t), overlap, min_length, lower_threshold, upper_threshold)
    if on_device:
        return r["wvd_diff_smoothed"], r["bt_diff_smoothed"], r["markers"]
    out = [_to_host(r["wvd_diff_smoothed"]), _to_host(r["bt_diff_smoothed"]), _to_host(r["markers"])]
    if hasattr(wvd, "coords") and hasattr(wvd, "dims") and not isinstance(wvd, np.ndarray):
        try:
            out = [type(wvd)(out[0], wvd.coords, wvd.dims), type(bt)(out[1], bt.coords, bt.dims),
                   type(wvd)(out[2], wvd.coords, wvd.dims)]                             # detection.py:249-252
        except Exception:
            pass
    return tuple(out)


# ------------------------------------------------------------------------------------------------------------------
# watershed inputs (detection.py:575-642): the edge field the anvil watershed floods, and its mask
# ------------------------------------------------------------------------------------------------------------------
def combined_edge_field_device(flow: Flow, field: torch.Tensor) -> torch.Tensor:
    """``get_combined_edge_field`` (tobac_flow/detection.py:620-642) on a device tensor: uphill cubic flow-Sobel (fused
    gather kernel, float64 like ``Flow.sobel``), ``+1`` where an edge exists, minus the field, ``inf`` where it is NaN."""
    from .sobel import sobel_reducer
    edges = flow.convolve(field, structure=np.ones((3, 3, 3), bool), method="cubic", fill_value=np.nan, dtype=None,
                          func=sobel_reducer("uphill"))
    edges = torch.where(edges > 0, edges + 1, edges)
    edges = edges - field
    return torch.where(torch.isnan(field), torch.full_like(edges, float("inf")), edges)


def get_combined_edge_field(flow: Flow, field, **kwargs):
    """``get_combined_edge_field`` (tobac_flow/detection.py:620-642); numpy in, numpy out."""
    t, host = _to_device(_as_numpy(field) if not isinstance(field, torch.Tensor) else field)
    res = combined_edge_field_device(flow, t)
    return _to_host(res) if host else res


def get_watershed_mask(field, erode_distance: int = 1):
    """``get_watershed_mask`` (tobac_flow/detection.py:581-617): ``field <= 0`` or NaN, eroded ``erode_distance`` times with
    the full 3x3x3 structure (border value 1), NaN pixels forced back to True."""
    t, host = _to_device(_as_numpy(field) if not isinstance(field, torch.Tensor) else field)
    nan = torch.isnan(t)
    m = ((t <= 0) | nan).to(torch.float32)[None, None]
    for _ in range(int(erode_distance)):
        # binary erosion with a full structure and border_value = 1: the minimum over the 3x3x3 neighbourhood, the
        # outside counting as 1 (max_pool3d pads with -inf)
        m = -torch.nn.functional.max_pool3d(-m, kernel_size=3, stride=1, padding=1)
    res = (m[0, 0] > 0.5) | nan
    return res.cpu().numpy() if host else res
