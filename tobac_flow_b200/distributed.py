"""Time sharding of a frame series across the GPUs of one box (SURVEY.md §8e).

Rank r of ``world`` owns frames ``[t0, t1)`` of the global series.  Consecutive pairs are independent
(``tobac_flow/flow.py:411-423`` touches only frames i and i+1; the normalisation is per pair) and the stencils at
step i read frames i-1, i, i+1 (``tobac_flow/convolve.py:305-345``), so the only communication is a neighbour
exchange over NCCL point-to-point (NVLink):

* one operand frame in each direction (4*H*W bytes): rank r needs frame ``t1`` to compute the pair
  ``(t1-1, t1)`` and frames ``t0-1`` / ``t1`` as stencil halos;
* one flow field (8*H*W bytes): the pair ``(t1-1, t1)`` computed on rank r yields ``backward_flow[t1]``, which
  belongs to rank r+1.

No collective is involved in the flow / stencil path; the sequence end rules (``flow.py:425-426``) apply on the
first / last rank only.  ``ShardedFlow.label`` (the semi-Lagrangian labelling of a sharded mask) is the one operator
with a real exchange step: per-rank component counts, per-label pixel counts and the (label, neighbour, overlap)
tables are gathered (a few thousand entries) so that every rank can run the same linking walk.
The compute back-end is injectable so the sharding logic can be exercised on CPU with ``gloo`` (tests).
"""
from dataclasses import dataclass

import numpy as np
import torch
import torch.distributed as dist


def shard_bounds(T: int, world: int, rank: int):
    """Frames [t0, t1) owned by ``rank``: t_g = floor(g*T/world)."""
    return (rank * T) // world, ((rank + 1) * T) // world


class CudaOps:
    """The product back-end: the CUDA kernels through the C ABI."""

    def calculate_flow(self, frames, fwd, bwd, smoothing_passes, interp_method, max_value, vr_steps=0, model=None):
        from .flow import calculate_flow_device
        calculate_flow_device(frames, fwd, bwd, smoothing_passes, interp_method, max_value, vr_steps=vr_steps,
                              model=model)

    def finalise(self, fwd, bwd, max_value, clamp_all, mirror_first, mirror_last):
        from .flow import finalise_flow_device
        finalise_flow_device(fwd, bwd, max_value, clamp_all, mirror_first, mirror_last)

    def convolve(self, data, fwd, bwd, structure, method, fill_value, dtype, reducer, has_prev, has_next, out=None):
        from .flow import convolve_device
        return convolve_device(data, fwd, bwd, structure, method, fill_value, dtype, reducer, has_prev, has_next, out)

    # -- labelling (flow_label on a time-sharded mask) --------------------------------------------------------------
    def flat_label(self, mask_u8, connectivity):
        from .label import flat_label_device
        return flat_label_device(mask_u8, connectivity)

    def overlap_table(self, flat_view, fwd, bwd, label_struct, has_prev, has_next, n_labels):
        """(keys, counts, sizes) of this rank's frames; ``flat_view`` carries the halo frames that exist."""
        from .label import warped_overlap_table_device
        return warped_overlap_table_device(flat_view, fwd, bwd, label_struct, n_labels, has_prev, has_next)

    def relabel(self, flat, mapping):
        from .label import relabel_device
        return relabel_device(flat, mapping)

    # -- growth-marker detection (the per-frame filters of detection.py:98-118 are local to a rank) -------------------
    def scale_frames(self, raw32, dt_minutes):
        from .detection import scale_by_dt_device
        return scale_by_dt_device(raw32, dt_minutes)

    def growth_seed_masks(self, smoothed, wvd):
        """(filtered >= 0.5, wvd >= -5, opened(filtered >= 0.25)) as uint8 tensors: detection.py:105-119."""
        from .detection import growth_seed_masks_device
        return growth_seed_masks_device(smoothed, wvd)[1:]

    def label_stats(self, labels, mask_a, mask_b, n_labels):
        """(tmin, tmax, any_a, any_b) host arrays of n_labels + 1 entries over this rank's frames (local frame indices;
        tmax = -1 and tmin huge where the label does not occur here)."""
        from .analysis import label_stats_device
        return label_stats_device(labels, mask_a, mask_b, n_labels)[1:]


_HALO_STREAMS = {}


def _halo_stream(dev):
    key = (dev.type, dev.index)
    if key not in _HALO_STREAMS:
        _HALO_STREAMS[key] = torch.cuda.Stream(dev)
    return _HALO_STREAMS[key]


def _p2p(ops, group):
    if ops:
        for w in dist.batch_isend_irecv(ops):
            w.wait()


@dataclass
class Shard:
    """A rank's slice of a (T, H, W) operand with one halo frame on each side: ``buf`` is (T_loc + 2, H, W);
    ``buf[1:-1]`` are the owned frames, ``buf[0]`` / ``buf[-1]`` the neighbours' boundary frames."""
    buf: torch.Tensor
    rank: int
    world: int

    @property
    def local(self):
        return self.buf[1:-1]

    @property
    def has_prev(self):
        return self.rank > 0

    @property
    def has_next(self):
        return self.rank < self.world - 1

    def stencil_view(self):
        """The contiguous slice the stencil kernels read: owned frames plus the halos that exist."""
        a = 0 if self.has_prev else 1
        b = self.buf.shape[0] if self.has_next else self.buf.shape[0] - 1
        return self.buf[a:b]

    def exchange_halos(self, group=None):
        """Fill ``buf[0]`` with the previous rank's last frame and ``buf[-1]`` with the next rank's first."""
        if self.world == 1:
            return
        ops = []
        if self.has_prev:
            ops.append(dist.P2POp(dist.isend, self.buf[1], self.rank - 1, group))
            ops.append(dist.P2POp(dist.irecv, self.buf[0], self.rank - 1, group))
        if self.has_next:
            ops.append(dist.P2POp(dist.isend, self.buf[-2], self.rank + 1, group))
            ops.append(dist.P2POp(dist.irecv, self.buf[-1], self.rank + 1, group))
        _p2p(ops, group)


def make_shard(local: torch.Tensor, rank: int, world: int) -> Shard:
    T, H, W = local.shape
    buf = torch.empty((T + 2, H, W), dtype=local.dtype, device=local.device)
    buf[1:-1] = local
    return Shard(buf, rank, world)


class ShardedFlow:
    """The flow vectors of one rank's frames plus the operators on sharded operands."""

    def __init__(self, fwd, bwd, rank, world, ops=None, group=None):
        self.fwd, self.bwd = fwd, bwd
        self.rank, self.world = rank, world
        self.ops = ops or CudaOps()
        self.group = group

    def convolve(self, shard: Shard, structure, method="linear", fill_value=np.nan, dtype=np.float32, reducer=0,
                 exchange=True, out=None):
        if exchange:
            shard.exchange_halos(self.group)
        return self.ops.convolve(shard.stencil_view(), self.fwd, self.bwd, structure, method, fill_value, dtype,
                                 reducer, shard.has_prev, shard.has_next, out)

    def label(self, mask_local, structure=None, overlap: float = 0.0, absolute_overlap: int = 1, return_count=False):
        """``Flow.label`` (tobac_flow/flow.py:281-330 -> label.py:84-175) on a time-sharded mask: every rank passes the
        (T_loc, H, W) mask of its own frames and gets the labels of those frames, numbered exactly as the unsharded
        call numbers them.

        Per-frame components are local.  The exchange steps are: an all-gather of the per-rank component counts (the
        global numbering continues from rank to rank, as scipy's does from frame to frame), the one-frame halos of the
        numbered components (point to point), a sum of the per-label pixel counts and an all-gather of the
        (label, neighbour, overlap) tables; a few thousand entries each.  The order-dependent linking walk then runs
        redundantly on every rank, so no label map has to be broadcast."""
        from .label import _connectivity, _default_structure, _label_struct, link_groups_host
        if structure is None:
            structure = _default_structure()
        dev = mask_local.device
        m = (mask_local != 0).to(torch.uint8).contiguous()
        flat, n_loc = self.ops.flat_label(m, _connectivity(structure))
        flat = flat.to(torch.int32)
        if self.world > 1:
            counts = [torch.zeros(1, dtype=torch.int64, device=dev) for _ in range(self.world)]
            dist.all_gather(counts, torch.tensor([n_loc], dtype=torch.int64, device=dev), group=self.group)
            counts = [int(c.item()) for c in counts]
        else:
            counts = [int(n_loc)]
        offset, total = sum(counts[:self.rank]), sum(counts)
        if offset:
            flat = flat + (flat > 0).to(torch.int32) * offset
        shard = make_shard(flat, self.rank, self.world)
        shard.buf[0] = 0
        shard.buf[-1] = 0
        shard.exchange_halos(self.group)
        keys, cnts, sizes = self.ops.overlap_table(shard.stencil_view(), self.fwd, self.bwd, _label_struct(structure),
                                                   shard.has_prev, shard.has_next, total)
        if self.world > 1:
            sz = torch.from_numpy(np.ascontiguousarray(sizes, dtype=np.int64)).to(dev)
            dist.all_reduce(sz, op=dist.ReduceOp.SUM, group=self.group)
            sizes = sz.cpu().numpy().astype(np.int32)
            n_e = torch.tensor([len(keys)], dtype=torch.int64, device=dev)
            lens = [torch.zeros(1, dtype=torch.int64, device=dev) for _ in range(self.world)]
            dist.all_gather(lens, n_e, group=self.group)
            lens = [int(v.item()) for v in lens]
            pad = max(max(lens), 1)
            table = torch.zeros((2, pad), dtype=torch.int64, device=dev)
            table[0, :len(keys)] = torch.from_numpy(keys.view(np.int64)).to(dev)
            table[1, :len(keys)] = torch.from_numpy(cnts.astype(np.int64)).to(dev)
            tables = [torch.zeros_like(table) for _ in range(self.world)]
            dist.all_gather(tables, table, group=self.group)
            keys = np.concatenate([t[0, :n].cpu().numpy().view(np.uint64) for t, n in zip(tables, lens)])
            cnts = np.concatenate([t[1, :n].cpu().numpy().astype(np.int32) for t, n in zip(tables, lens)])
        mapping, n_obj = link_groups_host(keys, cnts, sizes, total, overlap, absolute_overlap)
        out = self.ops.relabel(shard.local.contiguous(), mapping)
        return (out, n_obj) if return_count else out

    def detect_growth_markers(self, wvd: "Shard", dt_minutes_local, t0: int = 0):
        """``detect_growth_markers`` (tobac_flow/detection.py:98-125) on a time-sharded field: returns
        (wvd_diff_smoothed, marker_labels) for this rank's frames, identical to the unsharded call.

        ``wvd`` is this rank's Shard of the float32 field, ``dt_minutes_local`` the centred time differences of its
        frames (get_time_diff_from_coord evaluated on the whole series, sliced), ``t0`` its first global frame index.
        Exchanges: one-frame halos of the field and of the raw derivative (point to point), the labelling exchange of
        ``label``, and a min / max reduction of the per-label time extent and mask hits (one int per label)."""
        from . import _lib
        from .detection import _T_STRUCT, growth_marker_keep
        ops = self.ops
        raw32 = self.convolve(wvd, _T_STRUCT, reducer=_lib.TF_RED_DIFF)                # Flow.diff       (:99)
        raw = make_shard(ops.scale_frames(raw32, dt_minutes_local), self.rank, self.world)   # / dt      (:100)
        smoothed = self.convolve(raw, _T_STRUCT, reducer=_lib.TF_RED_NANMEAN)          # filtered_tdiff  (:103)
        m05, warm, seeds = ops.growth_seed_masks(smoothed, wvd.local.contiguous())     # :105-112
        linked, n_obj = self.label(seeds, overlap=0.0, absolute_overlap=1, return_count=True)
        tmin, tmax, any_a, any_b = ops.label_stats(linked, m05, warm, n_obj)
        dev = linked.device
        present = tmax >= 0
        lo = torch.from_numpy(np.where(present, tmin.astype(np.int64) + t0, np.iinfo(np.int32).max)).to(dev)
        hi = torch.from_numpy(np.stack([np.where(present, tmax.astype(np.int64) + t0, -1), any_a.astype(np.int64),
                                        any_b.astype(np.int64)])).to(dev)
        if self.world > 1:
            dist.all_reduce(lo, op=dist.ReduceOp.MIN, group=self.group)
            dist.all_reduce(hi, op=dist.ReduceOp.MAX, group=self.group)
        lo, hi = lo.cpu().numpy(), hi.cpu().numpy()
        return smoothed, ops.relabel(linked, growth_marker_keep(lo, hi[0], hi[1], hi[2]))   # :114-119


def create_flow_sharded(shard: Shard, smoothing_passes=0, interp_method="linear", max_value=20, ops=None, group=None,
                        exchange=True, fwd=None, bwd=None, vr_steps=0, model=None) -> ShardedFlow:
    """``create_flow`` for one rank of a time-sharded series; ``shard.buf[1:-1]`` holds the rank's frames.
    ``model``: as for ``create_flow`` (None is "Farneback")."""
    ops = ops or CudaOps()
    rank, world = shard.rank, shard.world
    T_loc, H, W = shard.local.shape
    dev = shard.buf.device
    if fwd is None:
        fwd = torch.full((T_loc, H, W, 2), float("nan"), dtype=torch.float32, device=dev)
    if bwd is None:
        # one extra slot: backward_flow of the next rank's first frame, produced here, sent on below
        bwd = torch.full((T_loc + 1, H, W, 2), float("nan"), dtype=torch.float32, device=dev)
    else:
        assert fwd.dtype == torch.float32 and bwd.dtype == torch.float32 and fwd.is_contiguous() and bwd.is_contiguous()
        assert tuple(fwd.shape) == (T_loc, H, W, 2) and tuple(bwd.shape) == (T_loc + 1, H, W, 2), "fwd (T_loc,..) / bwd (T_loc+1,..)"
    kw = dict(vr_steps=vr_steps) if vr_steps else {}
    if model is not None:        # (passed only when given: a back-end may have no `model` parameter)
        from .flow import _check_model
        _check_model(model, vr_steps)
        kw["model"] = model
    halo_ready = None
    if exchange and world > 1 and dev.type == "cuda":
        # the one-frame halos travel on a side stream (NCCL p2p over NVLink) while the interior pairs, which only read
        # this rank's own frames, are computed; the stream rejoins before the boundary pair (T_loc - 1, T_loc)
        cur = torch.cuda.current_stream(dev)
        side = _halo_stream(dev)
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            shard.exchange_halos(group)
            halo_ready = torch.cuda.Event()
            halo_ready.record(side)
        shard.buf.record_stream(side)
    elif exchange:
        shard.exchange_halos(group)
    if halo_ready is not None and T_loc >= 2:
        ops.calculate_flow(shard.buf[1:T_loc + 1], fwd, bwd, smoothing_passes, interp_method, max_value, **kw)
        torch.cuda.current_stream(dev).wait_event(halo_ready)
        if shard.has_next:
            ops.calculate_flow(shard.buf[T_loc:T_loc + 2], fwd[T_loc - 1:], bwd[T_loc - 1:], smoothing_passes,
                               interp_method, max_value, **kw)
    else:
        if halo_ready is not None:
            torch.cuda.current_stream(dev).wait_event(halo_ready)
        frames = shard.buf[1:T_loc + 2] if shard.has_next else shard.buf[1:T_loc + 1]
        ops.calculate_flow(frames, fwd, bwd, smoothing_passes, interp_method, max_value, **kw)
    if world > 1:
        p2p = []
        if shard.has_next:
            p2p.append(dist.P2POp(dist.isend, bwd[T_loc], rank + 1, group))
        if shard.has_prev:
            p2p.append(dist.P2POp(dist.irecv, bwd[0], rank - 1, group))
        _p2p(p2p, group)
    clamp_all = max_value is not None and (smoothing_passes > 0 or bool(vr_steps))
    ops.finalise(fwd, bwd[:T_loc], max_value, clamp_all, rank == 0, rank == world - 1)
    return ShardedFlow(fwd, bwd[:T_loc], rank, world, ops, group)
