"""Function-level mirror of ``tobac_flow/convolve.py`` (``warp_flow`` :8-86, ``convolve`` :248-348) on the CUDA path."""
from typing import Callable

import numpy as np
import torch

from . import _lib
from ._io import to_device
from .flow import Flow, _default_structure, _interp_code, convolve_device


def convolve(data, forward_flow, backward_flow, structure=None, method: str = "linear", dtype: type = np.float32,
             fill_value: float = np.nan, func: Callable | None = None):
    """``tobac_flow.convolve.convolve`` (convolve.py:248-348) — note the reference's argument order
    (``dtype`` before ``fill_value``)."""
    if structure is None:
        structure = _default_structure()
    structure = np.asarray(structure)
    assert structure.shape == (3, 3, 3), "Structure input must be a 3x3x3 array"
    return Flow(forward_flow, backward_flow).convolve(data, structure=structure, method=method,
                                                      fill_value=fill_value, dtype=dtype, func=func)


def warp_flow(img, flow, method: str = "linear", fill_value: float = np.nan, offsets=np.array([[0, 0]])):
    """``tobac_flow.convolve.warp_flow`` (convolve.py:8-86): ``img`` sampled at grid + flow + offset for each
    (dx, dy) offset; offsets must lie in {-1, 0, 1}^2 (the only ones a 3x3x3 structure produces).
    Returns (n_offsets, H, W) in the dtype of ``img``."""
    _interp_code(method)
    offsets = np.atleast_2d(np.asarray(offsets)).astype(int)
    if np.abs(offsets).max(initial=0) > 1:
        raise NotImplementedError("warp_flow offsets outside {-1, 0, 1} are not built in tobac_flow_b200")
    t, host = to_device(img)
    f, _ = to_device(flow, torch.float32)
    H, W = t.shape
    structure = np.zeros((3, 3, 3), bool)
    for dx, dy in offsets:
        structure[2, dy + 1, dx + 1] = True
    # kernel tap order is row-major (y, x); restore the caller's offset order afterwards
    order = sorted(range(len(offsets)), key=lambda i: (offsets[i][1], offsets[i][0]))
    if len({(int(o[0]), int(o[1])) for o in offsets}) != len(offsets):
        raise NotImplementedError("duplicate offsets are not supported")
    pair = torch.stack([torch.zeros_like(t), t])
    np_dt = {torch.float32: np.float32, torch.float64: np.float64, torch.int32: np.int32}.get(pair.dtype, np.int32)
    out = convolve_device(pair, f[None], torch.zeros_like(f)[None], structure, method, fill_value, np_dt,
                          _lib.TF_RED_NONE, has_prev=False, has_next=True)[:, 0]
    res = torch.empty_like(out)
    for k, i in enumerate(order):
        res[i] = out[k]
    return res.cpu().numpy() if host else res
