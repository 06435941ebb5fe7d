"""Semi-Lagrangian watershed (``tobac_flow/watershed.py:17-168``) without the reference package.

Mirror of the reference's ``watershed(forward_flow, backward_flow, field, markers, mask, connectivity)``: the volume is
padded by the structure's reach plus the largest rounded flow displacement, every pixel gets the raveled offset of its
rounded forward / backward flow vector, and a priority flood from the markers labels the volume; the neighbours in the
next / previous time step are displaced by those offsets.  The element-wise preparation (rounding, padding, raveled
offsets; ~10 passes over the volume) runs on the GPU; the flood itself is sequential by construction -- its result depends
on the global (value, age) pop order -- and runs on the host inside the native library (``tf_watershed_flood_host``), as
it does in the reference's Cython.

The two scikit-image helpers the reference imports are restated here: ``_validate_connectivity`` (an integer becomes
``scipy.ndimage.generate_binary_structure(ndim, connectivity)``, the centre is ``shape // 2``) and
``_offsets_to_raveled_neighbors`` (raveled offsets of the footprint's non-zero cells, stably sorted by Euclidean distance
from the centre, the centre itself removed) -- skimage/morphology/_util.py.
"""
import ctypes

import numpy as np
import torch

from . import _lib
from ._io import to_device


def _binary_structure(ndim: int, connectivity: int) -> np.ndarray:
    """``scipy.ndimage.generate_binary_structure``: cells within ``connectivity`` city-block steps of the centre."""
    idx = np.indices((3,) * ndim) - 1
    return np.abs(idx).sum(0) <= connectivity


def validate_connectivity(ndim: int, connectivity):
    if np.isscalar(connectivity):
        footprint = _binary_structure(ndim, int(connectivity))
    else:
        footprint = np.asarray(connectivity, dtype=bool)
        if footprint.ndim != ndim:
            raise ValueError("Connectivity dimension must be same as image")
    if any(s % 2 == 0 for s in footprint.shape):
        raise ValueError("Connectivity array must have an unambiguous center")
    offset = np.array(footprint.shape) // 2
    return footprint, offset


def offsets_to_raveled_neighbors(image_shape, footprint: np.ndarray, center) -> np.ndarray:
    offsets = np.stack([idx - c for idx, c in zip(np.nonzero(footprint), center)], axis=-1)
    ravel_factors = np.cumprod((tuple(image_shape[1:]) + (1,))[::-1])[::-1]
    raveled = (offsets * ravel_factors).sum(axis=1)
    distances = np.sqrt((offsets.astype(np.float64) ** 2).sum(axis=1))
    order = np.argsort(distances, kind="stable")
    return raveled[order][1:].astype(np.int64)      # without the offset to the centre itself


def flood_host(image, marker_locations, structure, forward_offset, backward_offset, forward_offset_locations,
               backward_offset_locations, mask, output):
    """``watershed_raveled`` (``_watershed.pyx:222-344``) on contiguous host arrays; ``output`` is filled in place."""
    image = np.ascontiguousarray(image, np.float32)
    marker_locations = np.ascontiguousarray(marker_locations, np.int64)
    structure = np.ascontiguousarray(structure, np.int64)
    fo = np.ascontiguousarray(forward_offset, np.int32)
    bo = np.ascontiguousarray(backward_offset, np.int32)
    fl = np.ascontiguousarray(forward_offset_locations, np.int32)
    bl = np.ascontiguousarray(backward_offset_locations, np.int32)
    mask = np.ascontiguousarray(mask, np.int8)
    assert output.dtype == np.int32 and output.flags.c_contiguous
    n = image.size
    assert fo.size == n and bo.size == n and mask.size == n and output.size == n and fl.size == structure.size == bl.size
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)  # noqa: E731
    _lib.check(_lib.load().tf_watershed_flood_host(p(image), p(marker_locations), marker_locations.size, p(structure),
                                                   structure.size, p(fo), p(bo), p(fl), p(bl), p(mask), p(output), n),
               "tf_watershed_flood_host")
    return output


def watershed(forward_flow, backward_flow, field, markers, mask=None, connectivity=1) -> np.ndarray:
    """``tobac_flow.watershed.watershed``; flow arguments may be numpy arrays or CUDA tensors (T, H, W, 2)."""
    field = np.asarray(field)
    markers = np.asarray(markers)
    if field.dtype != np.float32:
        field = field.astype(np.float32)
    if markers.shape != field.shape:
        raise ValueError(f"`markers` (shape {markers.shape}) must have same shape as `image` (shape {field.shape})")
    if markers.dtype != np.int32:
        markers = markers.astype(np.int32)
    if mask is None:
        mask = np.ones(field.shape, np.int8)
    else:
        mask = np.asarray(mask)
        if mask.dtype != np.int8:
            mask = mask.astype(np.int8)
        if mask.shape != field.shape:
            raise ValueError(f"`mask` (shape {mask.shape}) must have same shape as `image` (shape {field.shape})")
    footprint, offset = validate_connectivity(field.ndim, connectivity)

    # (raises without a CUDA device: there is no CPU path for the device-side preparation)
    ff, bf = to_device(forward_flow)[0], to_device(backward_flow)[0]
    # np.round = round half to even = torch.round
    rf, rb = torch.round(ff), torch.round(bf)
    pad_offset = offset.copy()
    pad_offset[1] += int(torch.maximum(rf[..., 1].abs().max(), rb[..., 1].abs().max()).item())
    pad_offset[2] += int(torch.maximum(rf[..., 0].abs().max(), rb[..., 0].abs().max()).item())
    pad_width = [(int(p), int(p)) for p in pad_offset]
    tpad = (pad_width[2][0], pad_width[2][1], pad_width[1][0], pad_width[1][1], pad_width[0][0], pad_width[0][1])

    field_p = np.pad(field, pad_width, mode="constant")
    mask_p = np.pad(mask, pad_width, mode="constant").ravel()
    output = np.pad(markers, pad_width, mode="constant")
    flat_neighborhood = offsets_to_raveled_neighbors(field_p.shape, footprint, center=offset)
    marker_locations = np.flatnonzero(output)
    strides = np.array(field_p.strides, dtype=np.int64) // field_p.itemsize

    def raveled_offset(r):
        o = r[..., 0].to(torch.int32) * int(strides[2]) + r[..., 1].to(torch.int32) * int(strides[1])
        return torch.nn.functional.pad(o, tpad).reshape(-1).cpu().numpy()

    forward_offset = raveled_offset(rf)
    backward_offset = raveled_offset(rb)
    forward_offset_locations = (np.round(flat_neighborhood / strides[0]) == 1).astype(np.int32)
    backward_offset_locations = (np.round(flat_neighborhood / strides[0]) == -1).astype(np.int32)

    flood_host(field_p.ravel(), marker_locations, flat_neighborhood, forward_offset, backward_offset,
               forward_offset_locations, backward_offset_locations, mask_p, output.reshape(-1))
    sl = tuple(slice(a, s - b) for (a, b), s in zip(pad_width, output.shape))
    return output[sl].copy()
