"""Farneback optical flow on the GPU with any of OpenCV's settings, the arithmetic of ``cv2.FarnebackOpticalFlow``.

``FarnebackOpticalFlow`` is a model object for ``create_flow`` / ``calculate_flow`` / ``calculate_flow_2``
(``model=``) and can also be used on its own through ``calc``.  ``FarnebackOpticalFlow()`` has OpenCV's factory
settings and runs exactly what ``model="Farneback"`` runs.

``cv2.calcOpticalFlowFarneback(prev, next, None, pyr_scale, levels, winsize, iterations, poly_n, poly_sigma, flags)``
is ``FarnebackOpticalFlow(levels, pyr_scale, winsize, iterations, poly_n, poly_sigma, flags).calc(prev, next)``.
"""
import ctypes

import numpy as np
import torch

from . import _lib
from ._io import device, stream

OPTFLOW_FARNEBACK_GAUSSIAN = 256


def _integer(name, v):
    if isinstance(v, bool) or int(v) != v:
        raise ValueError(f"{name} must be an integer")
    return int(v)


class FarnebackOpticalFlow:
    """``cv2.FarnebackOpticalFlow_create(num_levels, pyr_scale, False, win_size, num_iters, poly_n, poly_sigma, flags)``.

    Accepted: ``0 <= num_levels <= 15``, ``0 < pyr_scale < 1``, ``num_iters >= 1``, ``poly_n`` 5 or 7,
    ``poly_sigma > 0``, ``flags`` 0 (box window) or ``OPTFLOW_FARNEBACK_GAUSSIAN`` (256), and ``3 <= win_size <= 63``
    with the box window, ``4 <= win_size <= 63`` with the Gaussian one.  Anything else raises ``ValueError``.

    OpenCV also accepts Gaussian windows of 2 and 3 and a box window of 1.  They are refused here on purpose: with a
    window radius of 1 (sigma 0.3 for the Gaussian) the 2x2 systems are so ill-conditioned that two correct
    implementations in different floating-point orders end up hundreds of pixels apart, so no result could be checked.
    ``OPTFLOW_USE_INITIAL_FLOW`` and ``fastPyramids`` are not supported.
    """

    def __init__(self, num_levels: int = 5, pyr_scale: float = 0.5, win_size: int = 13, num_iters: int = 10,
                 poly_n: int = 5, poly_sigma: float = 1.1, flags: int = 0):
        num_levels = _integer("num_levels", num_levels)
        win_size = _integer("win_size", win_size)
        num_iters = _integer("num_iters", num_iters)
        poly_n = _integer("poly_n", poly_n)
        flags = _integer("flags", flags)
        pyr_scale, poly_sigma = float(pyr_scale), float(poly_sigma)
        if not 0 <= num_levels <= 15:
            raise ValueError("num_levels must be in 0..15")
        if not 0 < pyr_scale < 1:
            raise ValueError("pyr_scale must be in (0, 1)")
        if num_iters < 1:
            raise ValueError("num_iters must be >= 1")
        if poly_n not in (5, 7):
            raise ValueError("poly_n must be 5 or 7")
        if not poly_sigma > 0:
            raise ValueError("poly_sigma must be > 0")
        if flags not in (0, OPTFLOW_FARNEBACK_GAUSSIAN):
            raise ValueError("flags must be 0 or OPTFLOW_FARNEBACK_GAUSSIAN (256)")
        lo = 4 if flags else 3
        if not lo <= win_size <= 63:
            raise ValueError(f"win_size must be in {lo}..63" + (" with the Gaussian window" if flags else ""))
        self.num_levels, self.pyr_scale, self.win_size, self.num_iters = num_levels, pyr_scale, win_size, num_iters
        self.poly_n, self.poly_sigma, self.flags = poly_n, poly_sigma, flags

    def __repr__(self):
        return (f"FarnebackOpticalFlow(num_levels={self.num_levels}, pyr_scale={self.pyr_scale}, "
                f"win_size={self.win_size}, num_iters={self.num_iters}, poly_n={self.poly_n}, "
                f"poly_sigma={self.poly_sigma}, flags={self.flags})")

    def key(self):
        return ("Farneback", self.num_levels, self.pyr_scale, self.win_size, self.num_iters, self.poly_n,
                self.poly_sigma, self.flags)

    def params(self, max_value: float = 0.0) -> _lib.FbConfig:
        c = _lib.FbConfig()
        c.num_levels, c.pyr_scale, c.win_size, c.num_iters = self.num_levels, self.pyr_scale, self.win_size, self.num_iters
        c.poly_n, c.poly_sigma, c.flags = self.poly_n, self.poly_sigma, self.flags
        c.max_value = float(max_value or 0.0)
        return c

    def level_plan(self, H: int, W: int):
        """[(h, w)] of the pyramid levels this model runs for an H x W frame, coarsest first."""
        hs, ws = (ctypes.c_int * 16)(), (ctypes.c_int * 16)()
        n = _lib.load().tf_fb_config_level_plan(H, W, ctypes.byref(self.params()), hs, ws)
        if n < 0:
            _lib.check(n, "tf_fb_config_level_plan")
        return [(hs[i], ws[i]) for i in range(n)]

    def workspace_bytes(self, n_pairs: int, H: int, W: int) -> int:
        n = int(_lib.load().tf_fb_config_workspace_bytes(n_pairs, H, W, ctypes.byref(self.params())))
        if n == 0:
            raise ValueError(f"no Farneback workspace for {n_pairs} pairs of {H} x {W}")
        return n

    def _run_pairs(self, q0, q1, fwd, fwd_stride, bwd, bwd_stride, n_pairs, H, W, params, ws, ws_bytes, st):
        _lib.check(_lib.load().tf_farneback_config_pairs(q0, q1, fwd, fwd_stride, bwd, bwd_stride, n_pairs, H, W,
                                                         ctypes.byref(params), ws, ws_bytes, st),
                   "tf_farneback_config_pairs")

    def calc(self, I0, I1, flow=None):
        """Flow from ``I0`` to ``I1`` ((H, W) uint8 each) as (H, W, 2) float32: numpy in gives numpy out, a CUDA
        tensor in gives a CUDA tensor out.  ``flow`` (an initial flow) is not supported and must be None."""
        if flow is not None:
            raise NotImplementedError("FarnebackOpticalFlow.calc: an initial flow is not supported (pass None)")
        on_device = isinstance(I0, torch.Tensor) and I0.is_cuda
        dev = device() if not on_device else I0.device
        t0 = I0 if isinstance(I0, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(I0))
        t1 = I1 if isinstance(I1, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(I1))
        if t0.dtype != torch.uint8 or t1.dtype != torch.uint8 or t0.dim() != 2 or tuple(t0.shape) != tuple(t1.shape):
            raise ValueError("I0 and I1 must be uint8 images of the same (H, W) shape")
        t0 = t0.to(dev).contiguous()
        t1 = t1.to(dev).contiguous()
        H, W = t0.shape
        nbytes = self.workspace_bytes(1, H, W)
        ws = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
        out = torch.empty((2, H, W, 2), dtype=torch.float32, device=dev)
        self._run_pairs(t0.data_ptr(), t1.data_ptr(), out[0].data_ptr(), 0, out[1].data_ptr(), 0, 1, H, W,
                        self.params(), ws.data_ptr(), nbytes, stream())
        return out[0] if on_device else out[0].cpu().numpy()


def pyramid_level(q0, q1, model: FarnebackOpticalFlow, level: int):
    """Stage entry point: level image ``level`` (index into ``model.level_plan``) of the (H, W) uint8 pair -> (2, h, w)
    float32 (numpy)."""
    q = torch.from_numpy(np.ascontiguousarray(np.stack([q0, q1]), dtype=np.uint8)).to(device())
    _, H, W = q.shape
    h, w = model.level_plan(H, W)[level]
    nbytes = model.workspace_bytes(1, H, W)
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=q.device)
    out = torch.empty((2, h, w), dtype=torch.float32, device=q.device)
    _lib.check(_lib.load().tf_fb_config_pyramid_level(q.data_ptr(), q.data_ptr() + H * W, 1, H, W,
                                                      ctypes.byref(model.params()), int(level), out.data_ptr(),
                                                      ws.data_ptr(), nbytes, 0, stream()), "tf_fb_config_pyramid_level")
    return out.cpu().numpy()


def polyexp(images, model: FarnebackOpticalFlow):
    """Stage entry point: FarnebackPolyExp with the model's (poly_n, poly_sigma) of (n, h, w) float32 images ->
    (n, h, w, 5) float32 (numpy), channels in OpenCV's order."""
    I = torch.from_numpy(np.ascontiguousarray(images, dtype=np.float32)).to(device())
    n, h, w = I.shape
    rs = int(_lib.load().tf_fb_r_stride(h, w))
    R = torch.empty((n, rs), dtype=torch.float32, device=I.device)
    _lib.check(_lib.load().tf_fb_config_polyexp(I.data_ptr(), n, h, w, ctypes.byref(model.params()), R.data_ptr(),
                                                stream()), "tf_fb_config_polyexp")
    out = torch.empty((n, h, w, 5), dtype=torch.float32, device=I.device)
    out[..., :4] = R[:, :4 * h * w].reshape(n, h, w, 4)
    out[..., 4] = R[:, 4 * h * w:5 * h * w].reshape(n, h, w)
    return out.cpu().numpy()
