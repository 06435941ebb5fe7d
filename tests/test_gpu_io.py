"""The numpy / tensor boundary of every public wrapper: numpy, CPU-tensor and DataArray-like input give numpy output (a
DataArray-like wrapped back where the reference does that), CUDA-tensor input gives CUDA-tensor output, all with equal
values, and each input dtype gives the result dtype written in the table below."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import make_golden as mg  # noqa: E402
import refshim  # noqa: E402
import tobac_flow_b200 as tfb  # noqa: E402
from tobac_flow_b200 import NativeError, analysis, detection, label  # noqa: E402
from tobac_flow_b200 import convolve as tf_convolve  # noqa: E402

DTYPES = ["int16", "bool", "float16", "float32", "float64"]
F32, F64, I32, U8, B = "float32", "float64", "int32", "uint8", "bool"


def same_for(want):
    return {d: want for d in DTYPES}


OWN = {d: d for d in DTYPES}
NAN_GAUSS = dict(int16=F64, bool=F64, float16=F64, float32=F32, float64=F64)
CURVATURE = dict(int16=NotImplementedError, bool=NotImplementedError, float16=B, float32=B, float64=B)
# the warp kernels take integer operands with nearest interpolation only (as cv2.remap); warp_flow gives a float16 image
# an int32 result, which is refused as well
LINEAR_F32 = dict(int16=NativeError, bool=NativeError, float16=F32, float32=F32, float64=F32)
LINEAR_F64 = dict(int16=NativeError, bool=NativeError, float16=F64, float32=F64, float64=F64)
WARP = dict(int16=NativeError, bool=NativeError, float16=NativeError, float32=F32, float64=F64)


class Inputs:
    def __init__(self, golden):
        g = golden("growth_multi")
        self.wvd = mg.growth_multi_case()
        self.fwd = g["fwd_q256"].astype(np.float32) / 256
        self.bwd = g["bwd_q256"].astype(np.float32) / 256
        self.flat = g["flat"]
        self.markers = np.zeros(self.wvd.shape, np.int32)
        self.markers[1, 20:23, 30:33] = 1
        self.markers[2, 60:63, 90:93] = 2
        self.flow = tfb.Flow(self.fwd, self.bwd)

    def field(self, d):
        return cast(self.wvd, d, cut=-10)

    def mask(self, d):
        return (self.wvd > -10).astype(d)

    def labels(self, d):
        return self.flat.astype(d)


def cast(a, d, cut=0.0):
    if d == "bool":
        return a > cut
    if d == "int16":
        return np.round(a).astype(np.int16)
    return a.astype(d)


# name: (numpy arguments for an input dtype, the call, result dtypes of a host caller, result dtypes of a CUDA caller
# (None: the same), options)
CASES = {
    "Flow.convolve": (lambda c, d: (c.field(d),), lambda c, x: c.flow.convolve(x), LINEAR_F32, None, {}),
    "Flow.diff": (lambda c, d: (c.field(d),), lambda c, x: c.flow.diff(x), LINEAR_F32, None, {}),
    "Flow.sobel": (lambda c, d: (c.field(d),), lambda c, x: c.flow.sobel(x), LINEAR_F64, None, {}),
    "Flow.label": (lambda c, d: (c.mask(d),), lambda c, m: c.flow.label(m), same_for(I32), None, {}),
    "Flow.link_overlap": (lambda c, d: (c.labels(d),), lambda c, x: c.flow.link_overlap(x), same_for(I32), None, {}),
    "Flow.watershed": (lambda c, d: (c.field(d), c.markers), lambda c, f, m: c.flow.watershed(f, m), same_for(I32),
                       None, dict(device_out=False)),
    "flat_label": (lambda c, d: (c.mask(d),), lambda c, m: label.flat_label(m), same_for(I32), None, {}),
    "filter_labels_by_length": (lambda c, d: (c.labels(d),), lambda c, x: analysis.filter_labels_by_length(x, 2), OWN,
                                same_for(I32), {}),
    "filter_labels_by_mask": (lambda c, d: (c.labels(d), c.mask(np.float32)),
                              lambda c, x, m: analysis.filter_labels_by_mask(x, m), OWN, same_for(I32), {}),
    "filter_labels_by_length_and_mask": (lambda c, d: (c.labels(d), c.mask(np.float32)),
                                         lambda c, x, m: analysis.filter_labels_by_length_and_mask(x, m, 2), OWN,
                                         same_for(I32), {}),
    "filter_labels_by_length_and_multimask_legacy": (
        lambda c, d: (c.labels(d), c.mask(np.float32), c.wvd > -20, c.mask(np.int16)),
        lambda c, x, m0, m1, m2: analysis.filter_labels_by_length_and_multimask_legacy(x, [m0, m1, m2], 2), OWN,
        same_for(I32), {}),
    "get_curvature_filter": (lambda c, d: (c.field(d),), lambda c, x: detection.get_curvature_filter(x), CURVATURE,
                             None, {}),
    "get_growth_rate": (lambda c, d: (c.field(d),), lambda c, x: detection.get_growth_rate(c.flow, x), same_for(F32),
                        None, dict(needs_t=True)),
    "get_anvil_markers": (lambda c, d: (c.field(d),), lambda c, x: detection.get_anvil_markers(c.flow, x),
                          same_for(I32), None, {}),
    "detect_growth_markers": (lambda c, d: (c.field(d),), lambda c, x: detection.detect_growth_markers(c.flow, x),
                              same_for((F32, I32)), None, dict(needs_t=True, rewrap=(False, True))),
    "detect_growth_markers_multichannel": (
        lambda c, d: (c.field(d), cast(250.0 - 2.2 * (c.wvd + 25.0), d, cut=250)),
        lambda c, w, b: detection.detect_growth_markers_multichannel(c.flow, w, b), same_for((F32, F32, I32)), None,
        dict(needs_t=True, rewrap=(True, True, True))),
    "nan_gaussian_filter": (lambda c, d: (c.field(d),), lambda c, x: detection.nan_gaussian_filter(x, (0, 2, 2)),
                            NAN_GAUSS, None, {}),
    "get_combined_edge_field": (lambda c, d: (c.field(d),), lambda c, x: detection.get_combined_edge_field(c.flow, x),
                                LINEAR_F64, None, {}),
    "get_watershed_mask": (lambda c, d: (c.field(d) - (5 if d != "bool" else 0),),
                           lambda c, x: detection.get_watershed_mask(x), same_for(B), None, {}),
    "warp_flow": (lambda c, d: (c.field(d)[3], c.fwd[3]), lambda c, x, f: tf_convolve.warp_flow(x, f), WARP, None, {}),
    "pair_to_8bit": (lambda c, d: (c.field(d)[3], c.field(d)[4]), lambda c, a, b: tfb.pair_to_8bit(a, b),
                     same_for((U8, U8)), None, {}),
    "smooth_flow_step": (lambda c, d: (cast(c.fwd[3], d), cast(c.bwd[3], d)), lambda c, f, b: tfb.smooth_flow_step(f, b),
                         same_for((F32, F32)), None, {}),
}


@pytest.fixture(scope="module")
def inputs(golden):
    return Inputs(golden)


def _t_coord(n):
    import pandas as pd
    return pd.date_range("2020-01-01", periods=n, freq="5min")


def _as_kind(a, kind, t):
    if kind == "dataarray":
        return refshim.DataArray(a, coords={"t": t}, dims=("t", "y", "x"), t=t)
    if kind == "numpy":
        return a
    x = torch.from_numpy(np.ascontiguousarray(a).copy())
    if kind == "cuda":
        x = x.cuda()
    x.t = t                      # the time coordinate the growth-rate / marker functions read from `.t`
    return x


def _values(r):
    if isinstance(r, torch.Tensor):
        r = r.cpu().numpy()
    elif isinstance(r, refshim.DataArray):
        r = r.data
    return np.asarray(r, np.float64)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("name", list(CASES))
def test_result_kind_dtype_and_values(inputs, name, dtype):
    make, call, host_want, cuda_want, opt = CASES[name]
    args = make(inputs, dtype)
    t = _t_coord(inputs.wvd.shape[0])
    kinds = ["dataarray", "cpu", "cuda"] if opt.get("needs_t") else ["numpy", "dataarray", "cpu", "cuda"]
    ref = None
    for kind in kinds:
        want = (cuda_want or host_want)[dtype] if kind == "cuda" else host_want[dtype]
        xs = [_as_kind(a, kind, t) for a in args]
        if isinstance(want, type) and issubclass(want, Exception):
            with pytest.raises(want):
                call(inputs, *xs)
            continue
        got = call(inputs, *xs)
        got = got if isinstance(got, tuple) else (got,)
        want = want if isinstance(want, tuple) else (want,)
        rewrap = opt.get("rewrap", (False,) * len(got))
        assert len(got) == len(want), (name, kind)
        for i, (r, w) in enumerate(zip(got, want)):
            if kind == "cuda" and opt.get("device_out", True):
                assert isinstance(r, torch.Tensor) and r.is_cuda and r.dtype == getattr(torch, w), (name, kind, i, r)
            elif kind == "dataarray" and rewrap[i]:
                assert type(r) is refshim.DataArray and r.dims == ("t", "y", "x") and r.t is t, (name, i)
                assert r.data.dtype == np.dtype(w), (name, kind, i, r.data.dtype)
            else:
                assert type(r) is np.ndarray and r.dtype == np.dtype(w), (name, kind, i, type(r), r.dtype)
        vals = [_values(r) for r in got]
        if ref is None:
            ref = vals
        else:
            for i, (a, b) in enumerate(zip(vals, ref)):
                assert np.array_equal(a, b, equal_nan=True), (name, kind, i)
