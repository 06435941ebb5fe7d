"""The crossing between caller data and device tensors, shared by every public function of the package.

numpy, DataArray-like or CPU-tensor input gives numpy output; CUDA-tensor input gives CUDA-tensor output.  Inputs are
converted here to the dtypes the kernels take, and results go back to host callers through page-locked memory.
"""
import ctypes

import numpy as np
import torch

from ._lib import NativeError


def device():
    if not torch.cuda.is_available():
        raise NativeError("tobac_flow_b200 needs a CUDA device (there is no CPU fallback)")
    return torch.device("cuda", torch.cuda.current_device())


def stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def as_numpy(data) -> np.ndarray:
    """numpy / DataArray-like / tensor -> numpy array (a CPU tensor's storage is shared, not copied)."""
    if isinstance(data, torch.Tensor):
        return data.detach().cpu().numpy()
    if hasattr(data, "compute") and hasattr(data, "data") and not isinstance(data, np.ndarray):
        data = data.compute().data  # xr.DataArray   (flow.py:405-406)
    elif hasattr(data, "to_numpy"):
        data = data.to_numpy()      # convolve.py:293-294
    return np.asarray(data)


def to_device(data, dtype=None):
    """numpy / DataArray-like / tensor -> contiguous CUDA tensor; returns (tensor, came_from_host)."""
    dev = device()
    if isinstance(data, torch.Tensor):
        t = data.to(dev)
        host = not data.is_cuda
    else:
        a = np.ascontiguousarray(as_numpy(data))
        if a.dtype == np.bool_:
            a = a.astype(np.int32)
        t = torch.from_numpy(a).to(dev, non_blocking=False)
        host = True
    if dtype is not None and t.dtype != dtype:
        t = t.to(dtype)
    return t.contiguous(), host


def float_to_device(data, promote: torch.dtype):
    """``to_device`` for a field the kernels read as float32 or float64: those stay, any other dtype becomes
    ``promote``."""
    t, host = to_device(data)
    if t.dtype not in (torch.float32, torch.float64):
        t = t.to(promote)
    return t, host


def mask_to_device(mask, shape=None):
    """-> ((T, H, W) uint8 CUDA tensor of ``mask != 0``, came_from_host).  Host masks are compared on the host, so one
    byte per pixel crosses PCIe."""
    dev = device()
    if isinstance(mask, torch.Tensor):
        host = not mask.is_cuda
        t = mask.to(dev)
        if t.dtype != torch.bool:
            t = t != 0
    else:
        a = as_numpy(mask)
        host = True
        t = torch.from_numpy(np.ascontiguousarray(a != 0)).to(dev)
    if shape is not None:
        assert tuple(t.shape) == tuple(shape), "Labels and mask parameters must have the same shape"
    return t.to(torch.uint8).contiguous(), host


def labels_to_device(labels):
    """-> (int32 CUDA tensor, came_from_host, numpy dtype of the caller's labels; None for a CUDA tensor)."""
    dev = device()
    if isinstance(labels, torch.Tensor):
        np_dtype = None if labels.is_cuda else torch.empty(0, dtype=labels.dtype).numpy().dtype
        return labels.to(dev, torch.int32).contiguous(), not labels.is_cuda, np_dtype
    a = as_numpy(labels)
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).to(dev), True, a.dtype


def to_host(t: torch.Tensor) -> np.ndarray:
    """Device tensor -> numpy through page-locked memory (torch caches the pinned block, so repeated calls neither
    page-fault a fresh pageable array nor re-register memory); the array keeps the pinned storage alive."""
    if not t.is_cuda:
        return t.numpy()
    t = t.contiguous()
    h = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
    h.copy_(t, non_blocking=True)
    torch.cuda.current_stream().synchronize()
    return h.numpy()


def to_caller(t: torch.Tensor, from_host: bool, dtype=None):
    """A result for the caller: numpy (through ``to_host``, cast to ``dtype`` when given) for host input, the tensor
    itself for CUDA input."""
    if not from_host:
        return t
    a = to_host(t)
    return a if dtype is None else a.astype(dtype, copy=False)


def like_input(template, arr):
    """``arr`` wrapped into the type of a DataArray-like ``template`` with its coords and dims, else ``arr``."""
    if hasattr(template, "coords") and hasattr(template, "dims") and not isinstance(template, np.ndarray):
        try:
            return type(template)(arr, template.coords, template.dims)
        except Exception:
            pass
    return arr
