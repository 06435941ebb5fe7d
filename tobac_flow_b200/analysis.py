"""B200-native mirror of the label filters ``detect_growth_markers`` uses (``tobac_flow/analysis.py:66-86``):
``filter_labels_by_length`` and ``filter_labels_by_mask``.  The per-label statistics (time extent, "touches the mask")
come from one pass of ``tf_label_stats`` over the label array; the renumbering table is a few thousand entries and is
built on the host exactly as the reference does (``remap[1:] = cumsum(wh) * wh``); ``tf_relabel`` applies it.
numpy in -> numpy out, CUDA tensor in -> CUDA tensor out.
"""
import numpy as np
import torch

from . import _lib
from ._io import labels_to_device, mask_to_device, stream, to_caller
from .label import relabel_device


def label_stats_device(labels: torch.Tensor, mask_a=None, mask_b=None, n_labels=None):
    """(n_labels, tmin, tmax, any_a, any_b) as host arrays of n_labels + 1 entries for a (T, ...) int32 CUDA tensor
    (tmax = -1 and tmin huge where a label does not occur).  ``n_labels`` defaults to the largest label, which costs a
    device reduction and a host sync."""
    lib = _lib.load()
    dev = labels.device
    T = labels.shape[0]
    hw = labels.numel() // max(T, 1)
    if n_labels is None:
        mx = torch.zeros((1,), dtype=torch.int32, device=dev)
        _lib.check(lib.tf_label_max(labels.data_ptr(), labels.numel(), mx.data_ptr(), stream()), "tf_label_max")
        n_labels = int(mx.item())
    stats = torch.empty((4, n_labels + 1), dtype=torch.int32, device=dev)
    _lib.check(lib.tf_label_stats(labels.data_ptr(), mask_a.data_ptr() if mask_a is not None else None,
                                  mask_b.data_ptr() if mask_b is not None else None, T, hw, n_labels,
                                  stats[0].data_ptr(), stats[1].data_ptr(), stats[2].data_ptr(), stats[3].data_ptr(),
                                  stream()), "tf_label_stats")
    s = stats.cpu().numpy()
    return n_labels, s[0], s[1], s[2], s[3]


def _keep_table(wh: np.ndarray) -> np.ndarray:
    """Relabel table over labels 0..len(wh): drops label i + 1 where ``wh[i]`` is False, numbers the rest 1, 2, ..."""
    remap = np.zeros(len(wh) + 1, np.int32)
    remap[1:] = np.cumsum(wh) * wh                                  # analysis.py:72-73
    return remap


def _apply_keep(labels: torch.Tensor, wh: np.ndarray) -> torch.Tensor:
    return relabel_device(labels, _keep_table(wh))


def filter_labels_by_length(labels, min_length):
    """analysis.py:66-75: keep labels whose extent along axis 0 (ndi.find_objects) is >= min_length; renumber."""
    lab, host, np_dtype = labels_to_device(labels)
    _, tmin, tmax, _, _ = label_stats_device(lab)
    if (tmax[1:] < 0).any():
        raise TypeError("'NoneType' object is not subscriptable")   # ndi.find_objects gives None for absent labels
    wh = (tmax[1:] - tmin[1:] + 1) >= min_length
    return to_caller(_apply_keep(lab, wh), host, np_dtype)


def filter_labels_by_mask(labels, mask):
    """analysis.py:78-86: keep labels with at least one pixel inside ``mask``; renumber."""
    lab, host, np_dtype = labels_to_device(labels)
    m, _ = mask_to_device(mask, lab.shape)
    _, _, _, any_a, _ = label_stats_device(lab, m)
    wh = any_a[1:] != 0
    return to_caller(_apply_keep(lab, wh), host, np_dtype)


def filter_labels_by_length_and_mask(labels, mask, min_length):
    """analysis.py:89-102."""
    lab, host, np_dtype = labels_to_device(labels)
    m, _ = mask_to_device(mask, lab.shape)
    _, tmin, tmax, any_a, _ = label_stats_device(lab, m)
    wh = np.logical_and((tmax[1:] - tmin[1:] + 1) >= min_length, any_a[1:] != 0)
    return to_caller(_apply_keep(lab, wh), host, np_dtype)


def filter_labels_by_length_and_multimask_legacy(labels, masks, min_length):
    """analysis.py:182-201: keep labels whose extent along axis 0 is >= min_length and that touch EVERY mask of the list;
    renumber in ascending label order."""
    if type(masks) is not type(list()):
        raise ValueError("masks input must be a list of masks to process")
    lab, host, np_dtype = labels_to_device(labels)
    wh = None
    ms = [mask_to_device(m, lab.shape)[0] for m in masks]
    for k in range(0, max(len(ms), 1), 2):
        ma = ms[k] if k < len(ms) else None
        mb = ms[k + 1] if k + 1 < len(ms) else None
        _, tmin, tmax, any_a, any_b = label_stats_device(lab, ma, mb)
        ok = (tmax[1:] - tmin[1:] + 1) >= min_length
        if ma is not None:
            ok = np.logical_and(ok, any_a[1:] != 0)
        if mb is not None:
            ok = np.logical_and(ok, any_b[1:] != 0)
        wh = ok if wh is None else np.logical_and(wh, ok)
    return to_caller(_apply_keep(lab, wh), host, np_dtype)
