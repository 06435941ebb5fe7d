"""ctypes binding of the C-ABI library (include/tobac_flow_b200.h).

This is the only place the package touches native code.  There is no CPU fallback: if the shared library is
missing or a call fails, an exception is raised.
"""
import ctypes
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
# TF_LIB_PATH: load an alternative build of the same library (kernel A/B experiments)
LIB_PATH = os.environ.get("TF_LIB_PATH") or os.path.join(HERE, "libtobacflow_b200.so")

TF_F32, TF_F64, TF_I32 = 0, 1, 2
TF_NEAREST, TF_LINEAR, TF_CUBIC, TF_LANCZOS4 = 0, 1, 2, 3
(TF_RED_NONE, TF_RED_DIFF, TF_RED_NANMEAN, TF_RED_ANY, TF_RED_SOBEL, TF_RED_SOBEL_UPHILL,
 TF_RED_SOBEL_DOWNHILL, TF_RED_NANMAX, TF_RED_NANMIN) = range(9)

# every symbol include/tobac_flow_b200.h declares
EXPORTS = (
    "tf_version", "tf_last_error", "tf_fb_default_params", "tf_fb_level_plan", "tf_fb_poly_constants",
    "tf_fb_pyramid_level", "tf_fb_r_stride", "tf_fb_polyexp", "tf_fb_select_kernel",
    "tf_farneback_workspace_bytes", "tf_pair_normalise_u8", "tf_pair_normalise_u8_f64", "tf_farneback_pairs", "tf_smooth_flow_step",
    "tf_flow_finalise", "tf_sl_convolve", "tf_profile_enable", "tf_profile_reset", "tf_profile_read",
    "tf_vr_default_params", "tf_vr_workspace_bytes", "tf_variational_refinement",
    "tf_ccl_workspace_bytes", "tf_flat_label", "tf_binary_fill_holes", "tf_gaussian_filter_yx", "tf_curvature_mask",
    "tf_binary_opening_cross", "tf_grey_opening_cross", "tf_scale_frames", "tf_mask_multiply", "tf_threshold_ge",
    "tf_label_max", "tf_label_overlap_count", "tf_label_link_groups", "tf_relabel", "tf_label_stats",
    "tf_watershed_flood_host", "tf_dis_default_params", "tf_dis_scale_plan", "tf_dis_workspace_bytes", "tf_dis_pairs",
    "tf_dis_scale_images", "tf_fb_config_default", "tf_fb_config_level_plan", "tf_fb_config_workspace_bytes",
    "tf_farneback_config_pairs", "tf_fb_config_pyramid_level", "tf_fb_config_polyexp",
)

KERNEL_CLASSES = ("normalise", "pyramid", "polyexp", "flow_upsample", "fb_iter_coarse", "fb_iter_fullres",
                  "sl_gather", "smooth_flow", "finalise", "variational_refinement", "labelling", "detection_filters")


class FbParams(ctypes.Structure):
    _fields_ = [
        ("num_levels", ctypes.c_int), ("pyr_scale", ctypes.c_double), ("win_size", ctypes.c_int),
        ("num_iters", ctypes.c_int), ("poly_n", ctypes.c_int), ("poly_sigma", ctypes.c_double),
        ("max_value", ctypes.c_float),
    ]


class FbConfig(ctypes.Structure):
    _fields_ = FbParams._fields_ + [("flags", ctypes.c_int)]


class VrParams(ctypes.Structure):
    _fields_ = [
        ("alpha", ctypes.c_float), ("delta", ctypes.c_float), ("gamma", ctypes.c_float), ("omega", ctypes.c_float),
        ("fixed_point_iterations", ctypes.c_int), ("sor_iterations", ctypes.c_int), ("zeta", ctypes.c_float),
        ("epsilon", ctypes.c_float),
    ]


class DisParams(ctypes.Structure):
    _fields_ = [
        ("finest_scale", ctypes.c_int), ("patch_stride", ctypes.c_int), ("gradient_descent_iterations", ctypes.c_int),
        ("variational_refinement_iterations", ctypes.c_int), ("vr_alpha", ctypes.c_float),
        ("vr_delta", ctypes.c_float), ("vr_gamma", ctypes.c_float), ("vr_epsilon", ctypes.c_float),
        ("max_value", ctypes.c_float),
    ]


class NativeError(RuntimeError):
    pass


_lib = None


def load():
    """Load libtobacflow_b200.so (built by ``python -m tobac_flow_b200.build``); raises if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeError(
            f"{LIB_PATH} not found: build it with `python -m tobac_flow_b200.build` "
            "(tobac_flow_b200 has no CPU fallback)")
    lib = ctypes.CDLL(LIB_PATH)
    vp, ll, ci, cf, cd = ctypes.c_void_p, ctypes.c_longlong, ctypes.c_int, ctypes.c_float, ctypes.c_double
    pp = ctypes.POINTER(FbParams)
    lib.tf_version.restype = ci
    lib.tf_last_error.restype = ctypes.c_char_p
    lib.tf_fb_default_params.argtypes = [pp]
    lib.tf_fb_default_params.restype = None
    lib.tf_fb_level_plan.argtypes = [ci, ci, pp, ctypes.POINTER(ci), ctypes.POINTER(ci)]
    lib.tf_fb_poly_constants.argtypes = [pp, ctypes.POINTER(cf)]
    lib.tf_farneback_workspace_bytes.argtypes = [ci, ci, ci, pp]
    lib.tf_farneback_workspace_bytes.restype = ctypes.c_size_t
    lib.tf_fb_pyramid_level.argtypes = [vp, vp, ci, ci, ci, pp, ci, vp, vp, ctypes.c_size_t, ci, vp]
    lib.tf_fb_pyramid_level.restype = ci
    lib.tf_fb_r_stride.argtypes = [ci, ci]
    lib.tf_fb_r_stride.restype = ll
    lib.tf_fb_polyexp.argtypes = [vp, ci, ci, ci, pp, vp, vp]
    lib.tf_fb_polyexp.restype = ci
    lib.tf_fb_select_kernel.argtypes = [ci]
    lib.tf_fb_select_kernel.restype = ci
    lib.tf_pair_normalise_u8.argtypes = [vp, vp, ll, vp, vp, ci, ci, ci, vp, vp]
    lib.tf_pair_normalise_u8_f64.argtypes = lib.tf_pair_normalise_u8.argtypes
    lib.tf_pair_normalise_u8_f64.restype = ci
    lib.tf_farneback_pairs.argtypes = [vp, vp, vp, ll, vp, ll, ci, ci, ci, pp, vp, ctypes.c_size_t, vp]
    lib.tf_smooth_flow_step.argtypes = [vp, vp, vp, vp, ll, ci, ci, ci, ci, vp]
    lib.tf_flow_finalise.argtypes = [vp, vp, ci, ci, ci, cf, ci, ci, ci, vp]
    lib.tf_sl_convolve.argtypes = [vp, ci, ci, ci, vp, vp, vp, ll, ci, ci, ci, ci, ci, ci,
                                   ctypes.POINTER(ctypes.c_uint8), cd, vp]
    lib.tf_vr_default_params.argtypes = [ctypes.POINTER(VrParams)]
    lib.tf_vr_default_params.restype = None
    lib.tf_vr_workspace_bytes.argtypes = [ci, ci, ci]
    lib.tf_vr_workspace_bytes.restype = ctypes.c_size_t
    lib.tf_variational_refinement.argtypes = [vp, vp, vp, ll, vp, ll, ci, ci, ci, ctypes.POINTER(VrParams), vp,
                                              ctypes.c_size_t, vp]
    lib.tf_variational_refinement.restype = ci
    sz = ctypes.c_size_t
    lib.tf_ccl_workspace_bytes.argtypes = [ci, ci, ci]
    lib.tf_ccl_workspace_bytes.restype = sz
    lib.tf_flat_label.argtypes = [vp, vp, ci, ci, ci, ci, vp, vp, sz, vp]
    lib.tf_binary_fill_holes.argtypes = [vp, vp, ci, ci, ci, vp, sz, vp]
    lib.tf_gaussian_filter_yx.argtypes = [vp, vp, vp, ci, ci, ci, ci, ctypes.POINTER(cd), ci, vp]
    lib.tf_curvature_mask.argtypes = [vp, vp, ci, ci, ci, ci, cd, ci, vp]
    lib.tf_binary_opening_cross.argtypes = [vp, vp, ci, ci, ci, vp]
    lib.tf_grey_opening_cross.argtypes = [vp, vp, vp, ci, ci, ci, ci, vp]
    lib.tf_scale_frames.argtypes = [vp, vp, vp, ci, ci, ci, vp]
    lib.tf_mask_multiply.argtypes = [vp, vp, vp, ci, ll, vp]
    lib.tf_threshold_ge.argtypes = [vp, cd, vp, ci, ll, vp]
    lib.tf_label_max.argtypes = [vp, ll, vp, vp]
    lib.tf_label_overlap_count.argtypes = [vp, vp, vp, ll, vp, ci, vp, vp, ll, vp, vp]
    lib.tf_label_link_groups.argtypes = [vp, vp, ll, vp, ci, cd, ci, vp]
    lib.tf_relabel.argtypes = [vp, vp, vp, ll, ci, vp]
    lib.tf_label_stats.argtypes = [vp, vp, vp, ci, ll, ci, vp, vp, vp, vp, vp]
    lib.tf_label_stats.restype = ci
    for name in ("tf_flat_label", "tf_binary_fill_holes", "tf_gaussian_filter_yx", "tf_curvature_mask",
                 "tf_binary_opening_cross", "tf_grey_opening_cross", "tf_scale_frames", "tf_mask_multiply",
                 "tf_threshold_ge", "tf_label_max", "tf_label_overlap_count", "tf_label_link_groups", "tf_relabel"):
        getattr(lib, name).restype = ci
    lib.tf_watershed_flood_host.argtypes = [vp, vp, ll, vp, ci, vp, vp, vp, vp, vp, vp, ll]
    lib.tf_watershed_flood_host.restype = ci
    dp = ctypes.POINTER(DisParams)
    lib.tf_dis_default_params.argtypes = [dp, ci]
    lib.tf_dis_default_params.restype = None
    lib.tf_dis_scale_plan.argtypes = [ci, ci, dp, ctypes.POINTER(ci), ctypes.POINTER(ci), ctypes.POINTER(ci),
                                      ctypes.POINTER(ci)]
    lib.tf_dis_scale_plan.restype = ci
    lib.tf_dis_workspace_bytes.argtypes = [ci, ci, ci, dp]
    lib.tf_dis_workspace_bytes.restype = sz
    lib.tf_dis_pairs.argtypes = [vp, vp, vp, ll, vp, ll, ci, ci, ci, dp, vp, sz, vp]
    lib.tf_dis_pairs.restype = ci
    lib.tf_dis_scale_images.argtypes = [vp, ci, ci, ci, dp, ci, vp, vp, vp, vp, sz, vp]
    lib.tf_dis_scale_images.restype = ci
    cp = ctypes.POINTER(FbConfig)
    lib.tf_fb_config_default.argtypes = [cp]
    lib.tf_fb_config_default.restype = None
    lib.tf_fb_config_level_plan.argtypes = [ci, ci, cp, ctypes.POINTER(ci), ctypes.POINTER(ci)]
    lib.tf_fb_config_level_plan.restype = ci
    lib.tf_fb_config_workspace_bytes.argtypes = [ci, ci, ci, cp]
    lib.tf_fb_config_workspace_bytes.restype = sz
    lib.tf_farneback_config_pairs.argtypes = [vp, vp, vp, ll, vp, ll, ci, ci, ci, cp, vp, sz, vp]
    lib.tf_farneback_config_pairs.restype = ci
    lib.tf_fb_config_pyramid_level.argtypes = [vp, vp, ci, ci, ci, cp, ci, vp, vp, sz, ci, vp]
    lib.tf_fb_config_pyramid_level.restype = ci
    lib.tf_fb_config_polyexp.argtypes = [vp, ci, ci, ci, cp, vp, vp]
    lib.tf_fb_config_polyexp.restype = ci
    lib.tf_profile_enable.argtypes = [ci]
    lib.tf_profile_read.argtypes = [ci, ctypes.POINTER(cd), ctypes.POINTER(cd), ctypes.POINTER(ll)]
    for name in ("tf_profile_enable", "tf_profile_reset", "tf_profile_read", "tf_fb_level_plan", "tf_fb_poly_constants", "tf_pair_normalise_u8", "tf_farneback_pairs",
                 "tf_smooth_flow_step", "tf_flow_finalise", "tf_sl_convolve"):
        getattr(lib, name).restype = ci
    if lib.tf_version() != 1:
        raise NativeError("libtobacflow_b200.so ABI version mismatch")
    _lib = lib
    return lib


def check(rc, what=""):
    if rc != 0:
        msg = load().tf_last_error().decode("utf-8", "replace")
        raise NativeError(f"{what} failed with status {rc}: {msg}")


def default_params(max_value=20.0):
    p = FbParams()
    load().tf_fb_default_params(ctypes.byref(p))
    p.max_value = float(max_value) if max_value is not None else 0.0
    return p


def default_vr_params():
    p = VrParams()
    load().tf_vr_default_params(ctypes.byref(p))
    return p


def level_plan(H, W, params=None):
    params = params or default_params()
    hs = (ctypes.c_int * 8)()
    ws = (ctypes.c_int * 8)()
    n = load().tf_fb_level_plan(H, W, ctypes.byref(params), hs, ws)
    if n < 0:
        check(n, "tf_fb_level_plan")
    return [(hs[i], ws[i]) for i in range(n)]


def poly_constants(params=None):
    params = params or default_params()
    out = (ctypes.c_float * 22)()
    check(load().tf_fb_poly_constants(ctypes.byref(params), out), "tf_fb_poly_constants")
    return np.array(out, dtype=np.float32)


def dis_scale_plan(H, W, params):
    """(finest, coarsest, {scale: (h, w)}) of a DIS call on an H x W frame; raises where OpenCV refuses the frame."""
    f, c = ctypes.c_int(), ctypes.c_int()
    hs = (ctypes.c_int * 16)()
    ws = (ctypes.c_int * 16)()
    check(load().tf_dis_scale_plan(H, W, ctypes.byref(params), ctypes.byref(f), ctypes.byref(c), hs, ws),
          "tf_dis_scale_plan")
    return f.value, c.value, {s: (hs[s], ws[s]) for s in range(f.value, c.value + 1)}


def workspace_bytes(n_pairs, H, W, params=None):
    params = params or default_params()
    return int(load().tf_farneback_workspace_bytes(n_pairs, H, W, ctypes.byref(params)))


def structure_bytes(structure):
    s = np.ascontiguousarray(np.asarray(structure) != 0, dtype=np.uint8).reshape(27)
    return (ctypes.c_uint8 * 27)(*s.tolist())


def profile_enable(on=True):
    check(load().tf_profile_enable(int(bool(on))), "tf_profile_enable")


def profile_reset():
    check(load().tf_profile_reset(), "tf_profile_reset")


def profile_read():
    """{kernel class: dict(ms, bytes, launches)} accumulated since the last reset (synchronises)."""
    out = {}
    for i, name in enumerate(KERNEL_CLASSES):
        ms, by, n = ctypes.c_double(), ctypes.c_double(), ctypes.c_longlong()
        check(load().tf_profile_read(i, ctypes.byref(ms), ctypes.byref(by), ctypes.byref(n)), "tf_profile_read")
        out[name] = dict(ms=ms.value, bytes=by.value, launches=n.value)
    return out
