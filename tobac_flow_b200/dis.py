"""DIS (Dense Inverse Search) optical flow on the GPU, the arithmetic of ``cv2.DISOpticalFlow``.

``DISOpticalFlow`` is a model object for ``create_flow`` / ``calculate_flow`` / ``calculate_flow_2`` (``model=``) and
can also be used on its own through ``calc``.  It is built for patch size 8 with mean normalisation and spatial
propagation, which is what OpenCV's three presets use.
"""
import ctypes

import numpy as np
import torch

from . import _lib
from ._io import device, stream

PRESET_ULTRAFAST, PRESET_FAST, PRESET_MEDIUM = 0, 1, 2


class DISOpticalFlow:
    """``cv2.DISOpticalFlow_create(preset)`` with optional overrides of its settings.

    ``preset``: 0 ULTRAFAST, 1 FAST (OpenCV's default), 2 MEDIUM.  ``None`` overrides keep the preset's value.
    As in ``calc()`` of a freshly created OpenCV object, a frame too small for ``finest_scale`` runs at a lower one
    (the object itself is not changed, so every frame of a sequence gets the same settings).
    """

    def __init__(self, preset: int = PRESET_FAST, finest_scale: int | None = None, patch_stride: int | None = None,
                 gradient_descent_iterations: int | None = None, variational_refinement_iterations: int | None = None):
        if preset not in (PRESET_ULTRAFAST, PRESET_FAST, PRESET_MEDIUM):
            raise ValueError("preset must be 0 (ULTRAFAST), 1 (FAST) or 2 (MEDIUM)")
        self.preset = int(preset)
        p = _lib.DisParams()
        _lib.load().tf_dis_default_params(ctypes.byref(p), self.preset)
        for name, v in (("finest_scale", finest_scale), ("patch_stride", patch_stride),
                        ("gradient_descent_iterations", gradient_descent_iterations),
                        ("variational_refinement_iterations", variational_refinement_iterations)):
            if v is not None:
                if int(v) != v or v < 0:
                    raise ValueError(f"{name} must be a non-negative integer")
                setattr(p, name, int(v))
        if not 1 <= p.patch_stride <= 8:
            raise ValueError("patch_stride must be in 1..8 (patch size 8)")
        self.finest_scale = p.finest_scale
        self.patch_stride = p.patch_stride
        self.gradient_descent_iterations = p.gradient_descent_iterations
        self.variational_refinement_iterations = p.variational_refinement_iterations
        self._p = p

    def __repr__(self):
        return (f"DISOpticalFlow(preset={self.preset}, finest_scale={self.finest_scale}, "
                f"patch_stride={self.patch_stride}, gradient_descent_iterations={self.gradient_descent_iterations}, "
                f"variational_refinement_iterations={self.variational_refinement_iterations})")

    def key(self):
        return ("DIS", self.finest_scale, self.patch_stride, self.gradient_descent_iterations,
                self.variational_refinement_iterations)

    def params(self, max_value: float = 0.0) -> _lib.DisParams:
        p = _lib.DisParams()
        ctypes.memmove(ctypes.byref(p), ctypes.byref(self._p), ctypes.sizeof(p))
        p.max_value = float(max_value or 0.0)
        return p

    def scale_plan(self, H: int, W: int):
        """(finest, coarsest, {scale: (h, w)}) this model runs for an H x W frame."""
        return _lib.dis_scale_plan(H, W, self._p)

    def workspace_bytes(self, n_pairs: int, H: int, W: int) -> int:
        self.scale_plan(H, W)      # raises for a frame OpenCV refuses
        return int(_lib.load().tf_dis_workspace_bytes(n_pairs, H, W, ctypes.byref(self._p)))

    def _run_pairs(self, q0, q1, fwd, fwd_stride, bwd, bwd_stride, n_pairs, H, W, params, ws, ws_bytes, st):
        _lib.check(_lib.load().tf_dis_pairs(q0, q1, fwd, fwd_stride, bwd, bwd_stride, n_pairs, H, W, ctypes.byref(params),
                                            ws, ws_bytes, st), "tf_dis_pairs")

    def calc(self, I0, I1, flow=None):
        """Flow from ``I0`` to ``I1`` ((H, W) uint8 each) as (H, W, 2) float32: numpy in gives numpy out, a CUDA
        tensor in gives a CUDA tensor out.  ``flow`` (an initial flow) is not supported and must be None."""
        if flow is not None:
            raise NotImplementedError("DISOpticalFlow.calc: an initial flow is not supported (pass None)")
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


def scale_images(q, model: DISOpticalFlow, scale: int):
    """Stage entry point: scale image ``scale`` of the DIS pyramid of the (n, H, W) uint8 frames ``q`` and its
    spatialGradient -> (img (n, h, w) uint8, gx, gy (n, h, w) int16), numpy."""
    t = torch.from_numpy(np.ascontiguousarray(q, dtype=np.uint8)).to(device())
    n, H, W = t.shape
    _, _, sizes = model.scale_plan(H, W)
    if scale not in sizes:
        raise ValueError(f"scale {scale} is not in the plan {sorted(sizes)}")
    h, w = sizes[scale]
    nbytes = model.workspace_bytes(n, H, W)
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=t.device)
    img = torch.empty((n, h, w), dtype=torch.uint8, device=t.device)
    gx = torch.empty((n, h, w), dtype=torch.int16, device=t.device)
    gy = torch.empty((n, h, w), dtype=torch.int16, device=t.device)
    _lib.check(_lib.load().tf_dis_scale_images(t.data_ptr(), n, H, W, ctypes.byref(model.params()), int(scale),
                                               img.data_ptr(), gx.data_ptr(), gy.data_ptr(), ws.data_ptr(), nbytes,
                                               stream()), "tf_dis_scale_images")
    return img.cpu().numpy(), gx.cpu().numpy(), gy.cpu().numpy()
