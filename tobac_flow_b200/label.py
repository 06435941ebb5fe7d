"""B200-native drop-in for the labelling half of ``tobac_flow.label`` (SURVEY.md section 8f rank 3).

Mirrors ``flat_label`` (tobac_flow/utils/label_utils.py:143-180), ``flow_label`` (tobac_flow/label.py:84-175) and
``flow_link_overlap`` (tobac_flow/label.py:249-321): same names, arguments, defaults and results (label numbers
included).  The pixel work runs in ``libtobacflow_b200.so`` (connected components, nearest-neighbour gathers of the
labels along the flow, the (label, neighbour) overlap histogram, relabelling); the walk that links a few thousand flat
labels into objects is order-dependent and tiny, so it runs on the host inside the library
(``tf_label_link_groups``) in the reference's visiting order.  numpy in -> numpy out, CUDA tensor in -> CUDA tensor
out.  There is no CPU fallback.
"""
import ctypes

import numpy as np
import torch

from . import _lib
from .flow import _default_structure, _device, _stream, _to_host, convolve_device


def _mask_u8(mask) -> tuple[torch.Tensor, bool]:
    """Anything array-like -> (T, H, W) uint8 CUDA tensor of ``mask != 0``; second value: input lived on the host."""
    dev = _device()
    if isinstance(mask, torch.Tensor):
        host = not mask.is_cuda
        t = mask.to(dev)
    else:
        a = np.asarray(mask.to_numpy() if hasattr(mask, "to_numpy") else mask)
        t = torch.from_numpy(np.ascontiguousarray(a != 0)).to(dev)
        host = True
    if t.dtype != torch.bool:
        t = t != 0
    return t.to(torch.uint8).contiguous(), host


def _connectivity(structure) -> int:
    s = np.asarray(structure)
    if s.shape != (3, 3, 3):
        raise ValueError("structure must be a (3, 3, 3) array")
    mid = s[1] != 0
    cross = np.array([[0, 1, 0], [1, 1, 1], [0, 1, 0]], bool)
    if np.array_equal(mid, cross):
        return 1
    if mid.all():
        return 2
    raise NotImplementedError("flat_label: the middle slab of the structure must be the 2-D cross or the full 3x3")


def flat_label_device(mask_u8: torch.Tensor, connectivity: int = 1) -> tuple[torch.Tensor, int]:
    """tf_flat_label on a (T, H, W) uint8 CUDA tensor -> (int32 labels, number of labels)."""
    lib = _lib.load()
    T, H, W = mask_u8.shape
    labels = torch.empty((T, H, W), dtype=torch.int32, device=mask_u8.device)
    if T == 0 or H * W == 0:
        return labels, 0
    n = torch.zeros((1,), dtype=torch.int32, device=mask_u8.device)
    done = 0
    offset = 0
    while done < T:                                  # the library takes at most 65535 frames per call
        tc = min(T - done, 65535)
        ws_bytes = int(lib.tf_ccl_workspace_bytes(tc, H, W))
        ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=mask_u8.device)
        _lib.check(lib.tf_flat_label(mask_u8[done:].data_ptr(), labels[done:].data_ptr(), tc, H, W, connectivity,
                                     n.data_ptr(), ws.data_ptr(), ws_bytes, _stream()), "tf_flat_label")
        if offset:
            part = labels[done:done + tc]
            part += (part > 0).to(torch.int32) * offset
        offset += int(n.item())
        done += tc
    return labels, offset


def flat_label(mask, structure=None, dtype=np.int32):
    """``flat_label`` (tobac_flow/utils/label_utils.py:143-180): per-frame connected components, scipy's numbering."""
    if structure is None:
        structure = _default_structure()
    m, host = _mask_u8(mask)
    labels, _ = flat_label_device(m, _connectivity(structure))
    if host:
        return _to_host(labels).astype(dtype, copy=False)
    return labels


def _label_struct(structure):
    structure = np.asarray(structure)
    label_struct = structure * np.array([1, 0, 1])[:, np.newaxis, np.newaxis]        # label.py:131
    if int(np.count_nonzero(label_struct)) != 2:
        # the reference unpacks the convolve result into (back_labels, forward_labels) (label.py:133)
        raise ValueError("too many values to unpack (expected 2): the structure may only link the centre pixel in time")
    return label_struct


def overlap_table_device(flat: torch.Tensor, back: torch.Tensor, fwd: torch.Tensor, n_labels: int):
    """tf_label_overlap_count on int32 CUDA tensors -> host arrays (keys uint64, counts int32, sizes int32[n_labels+1]):
    the (direction, label, neighbour) overlap histogram of ``flat`` against its two warped neighbours and
    np.bincount(flat).  Labels may be any values in 0..n_labels (a time shard holds a sub-range of them)."""
    lib = _lib.load()
    dev = flat.device
    n = flat.numel()
    sizes = torch.empty((n_labels + 1,), dtype=torch.int32, device=dev)
    flags = torch.empty((2,), dtype=torch.int32, device=dev)
    cap = 1024
    while cap < 16 * (n_labels + 1):
        cap *= 2
    while True:
        keys = torch.empty((cap,), dtype=torch.int64, device=dev)
        counts = torch.empty((cap,), dtype=torch.int32, device=dev)
        _lib.check(lib.tf_label_overlap_count(flat.data_ptr(), back.data_ptr(), fwd.data_ptr(), n, sizes.data_ptr(),
                                              n_labels, keys.data_ptr(), counts.data_ptr(), cap, flags.data_ptr(),
                                              _stream()), "tf_label_overlap_count")
        fl = flags.cpu()
        if int(fl[1]):
            raise ValueError("flat labels outside 0..max(label)")
        if not int(fl[0]):
            break
        cap *= 4                                                                     # table overflow: retry larger
    used = keys != -1
    k_h = np.ascontiguousarray(keys[used].cpu().numpy().view(np.uint64))
    c_h = np.ascontiguousarray(counts[used].cpu().numpy())
    return k_h, c_h, sizes.cpu().numpy()


def warped_overlap_table_device(flat_view: torch.Tensor, fwd: torch.Tensor, bwd: torch.Tensor, label_struct,
                                n_labels: int, has_prev: bool = False, has_next: bool = False):
    """``overlap_table_device`` of the flat labels against their neighbouring frames warped along the flow (nearest,
    label.py:131-134).  With ``has_prev`` / ``has_next`` the first / last frame of ``flat_view`` is a halo frame of a
    time shard: it is only warped, and the table covers the frames between the halos."""
    taps = convolve_device(flat_view, fwd, bwd, label_struct, "nearest", 0, np.int32, _lib.TF_RED_NONE, has_prev,
                           has_next)
    local = flat_view[int(has_prev):flat_view.shape[0] - int(has_next)].contiguous()
    return overlap_table_device(local, taps[0], taps[1], n_labels)


def link_groups_host(keys: np.ndarray, counts: np.ndarray, sizes: np.ndarray, n_labels: int, overlap: float,
                     absolute_overlap: int):
    """tf_label_link_groups (the order-dependent walk of label.py:139-163, run on the host inside the library) ->
    (relabel table int32[n_labels+1], number of linked objects)."""
    lib = _lib.load()
    keys = np.ascontiguousarray(keys, dtype=np.uint64)
    counts = np.ascontiguousarray(counts, dtype=np.int32)
    sizes = np.ascontiguousarray(sizes, dtype=np.int32)
    mapping = np.zeros(n_labels + 1, np.int32)
    n_obj = lib.tf_label_link_groups(keys.ctypes.data, counts.ctypes.data, len(keys), sizes.ctypes.data, n_labels,
                                     ctypes.c_double(float(overlap)), int(absolute_overlap), mapping.ctypes.data)
    _lib.check(min(n_obj, 0), "tf_label_link_groups")
    return mapping, int(n_obj)


def relabel_device(flat: torch.Tensor, mapping: np.ndarray) -> torch.Tensor:
    """out = mapping[flat] on the device (label.py:165-170)."""
    out = torch.empty_like(flat)                                 # tf_relabel writes every element
    if flat.numel():
        map_d = torch.from_numpy(np.ascontiguousarray(mapping, dtype=np.int32)).to(flat.device)
        _lib.check(_lib.load().tf_relabel(flat.data_ptr(), map_d.data_ptr(), out.data_ptr(), flat.numel(),
                                          len(mapping) - 1, _stream()), "tf_relabel")
    return out


def link_overlap_device(flow, flat: torch.Tensor, structure, overlap: float, absolute_overlap: int,
                        n_labels: int | None = None) -> tuple[torch.Tensor, int]:
    """The body shared by ``flow_label`` and ``flow_link_overlap`` on an int32 CUDA tensor of flat labels."""
    lib = _lib.load()
    dev = flat.device
    n = flat.numel()
    if n == 0:
        return torch.zeros_like(flat), 0
    if n_labels is None:
        mx = torch.zeros((1,), dtype=torch.int32, device=dev)
        _lib.check(lib.tf_label_max(flat.data_ptr(), n, mx.data_ptr(), _stream()), "tf_label_max")
        n_labels = int(mx.item())
        if bool((flat < 0).any()):
            raise ValueError("flat labels must be non-negative")                      # np.bincount raises the same
    keys, counts, sizes = warped_overlap_table_device(flat, flow.forward_flow_device, flow.backward_flow_device,
                                                      _label_struct(structure), n_labels)
    mapping, n_obj = link_groups_host(keys, counts, sizes, n_labels, overlap, absolute_overlap)
    return relabel_device(flat, mapping), n_obj


def flow_label(flow, mask, structure=None, dtype: type = np.int32, overlap: float = 0.0, absolute_overlap: int = 0,
               subsegment_shrink: float = 0.0, peak_min_distance: int = 10):
    """``flow_label`` (tobac_flow/label.py:84-175): connected objects in the semi-Lagrangian frame."""
    if structure is None:
        structure = _default_structure()
    if subsegment_shrink != 0:
        raise NotImplementedError("subsegment_shrink != 0 (skimage watershed sub-segmentation) is not built here")
    if tuple(mask.shape) != tuple(flow.shape):
        raise AssertionError("Data input must have the same shape as the Flow object")
    m, host = _mask_u8(mask)
    flat, n_labels = flat_label_device(m, _connectivity(structure))
    out, _ = link_overlap_device(flow, flat, structure, overlap, absolute_overlap, n_labels)
    if host:
        return _to_host(out).astype(dtype, copy=False)
    return out


def flow_link_overlap(flow, flat_labels, structure=None, dtype: type = np.int32, overlap: float = 0.0,
                      absolute_overlap: int = 0):
    """``flow_link_overlap`` (tobac_flow/label.py:249-321): link existing per-frame labels along the flow."""
    if structure is None:
        structure = _default_structure()
    if tuple(flat_labels.shape) != tuple(flow.shape):
        raise AssertionError("Data input must have the same shape as the Flow object")
    dev = _device()
    if isinstance(flat_labels, torch.Tensor):
        host = not flat_labels.is_cuda
        flat = flat_labels.to(dev, torch.int32).contiguous()
    else:
        host = True
        flat = torch.from_numpy(np.ascontiguousarray(np.asarray(flat_labels), dtype=np.int32)).to(dev)
    out, _ = link_overlap_device(flow, flat, structure, overlap, absolute_overlap)
    if host:
        return _to_host(out).astype(dtype, copy=False)
    return out
