"""B200-native drop-in for ``tobac_flow.flow`` — the dense-flow hot path only.

Mirrors the reference interface (``tobac_flow/flow.py:23-65`` ``create_flow``, ``:68-355`` ``Flow``,
``:362-428`` ``calculate_flow``, ``:530-568`` ``smooth_flow_step``; contract ``tobac_flow/core/abstracts.py:10-84``):
same names, argument meaning, defaults and exception types.  All arithmetic runs in the hand-written CUDA
kernels of ``libtobacflow_b200.so`` through its C ABI (``include/tobac_flow_b200.h``); PyTorch is used only for
device memory and streams.  There is no CPU fallback.

Differences by design (device residency):
* ``Flow`` keeps its vectors as CUDA tensors; ``.forward_flow`` / ``.backward_flow`` materialise numpy copies
  lazily (the downstream ``watershed.py`` / ``label.py`` read them as numpy).
* ``convolve`` / ``diff`` / ``sobel`` return numpy for numpy input and CUDA tensors for CUDA-tensor input, so
  chained operators (``diff`` -> ``filtered_tdiff``) stay on the device.
"""
import ctypes
import os
from functools import partial
from typing import Callable

import numpy as np
import torch

from . import _lib
from ._lib import NativeError  # noqa: F401  (re-export)

_INTERP = {"nearest": _lib.TF_NEAREST, "linear": _lib.TF_LINEAR, "cubic": _lib.TF_CUBIC, "lanczos": _lib.TF_LANCZOS4}
_REFERENCE_INTERP_NAMES = ["nearest", "linear", "cubic", "lanczos"]  # convolve.py:46-51
_REFERENCE_MODELS = ["Farneback", "DeepFlow", "PCA", "SimpleFlow", "SparseToDense", "DIS", "DenseRLOF", "DualTVL1"]
_NORMALISATIONS = ["linear", "log", "inverse_log", "z_score", "uniform", "local_linear"]

_TORCH_DT = {torch.float32: _lib.TF_F32, torch.float64: _lib.TF_F64, torch.int32: _lib.TF_I32}


def _default_structure():
    s = np.zeros((3, 3, 3), bool)  # == ndi.generate_binary_structure(3, 1)
    s[1, 1, :] = s[1, :, 1] = s[:, 1, 1] = True
    return s


def _device():
    if not torch.cuda.is_available():
        raise NativeError("tobac_flow_b200 needs a CUDA device (there is no CPU fallback)")
    return torch.device("cuda", torch.cuda.current_device())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _interp_code(method: str) -> int:
    if method not in _REFERENCE_INTERP_NAMES:
        raise ValueError(f"method must be one of {_REFERENCE_INTERP_NAMES}")  # convolve.py:52-53
    if method not in _INTERP:
        raise NotImplementedError(f"interpolation '{method}' is not built in tobac_flow_b200 (nearest/linear/cubic are)")
    return _INTERP[method]


def _as_numpy(data):
    if isinstance(data, torch.Tensor):
        return None
    if hasattr(data, "compute") and hasattr(data, "data") and not isinstance(data, np.ndarray):
        data = data.compute().data  # xr.DataArray   (flow.py:405-406)
    elif hasattr(data, "to_numpy"):
        data = data.to_numpy()      # convolve.py:293-294
    return np.asarray(data)


def _to_device(data, dtype=None):
    """numpy / DataArray-like / tensor -> contiguous CUDA tensor; returns (tensor, came_from_host)."""
    dev = _device()
    if isinstance(data, torch.Tensor):
        t = data.to(dev)
        host = not data.is_cuda
    else:
        a = np.ascontiguousarray(_as_numpy(data))
        if a.dtype == np.bool_:
            a = a.astype(np.int32)
        t = torch.from_numpy(a).to(dev, non_blocking=False)
        host = True
    if dtype is not None and t.dtype != dtype:
        t = t.to(dtype)
    return t.contiguous(), host


def _to_host(t: torch.Tensor) -> np.ndarray:
    """Device tensor -> numpy through page-locked memory (torch caches the pinned block, so repeated calls neither
    page-fault a fresh pageable array nor re-register memory); the array keeps the pinned storage alive."""
    if not t.is_cuda:
        return t.numpy()
    t = t.contiguous()
    h = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
    h.copy_(t, non_blocking=True)
    torch.cuda.current_stream().synchronize()
    return h.numpy()


def _pinned_result_cap() -> int:
    gb = os.environ.get("TF_PINNED_RESULT_MAX_GB")
    if gb is not None:
        return int(float(gb) * (1 << 30))
    try:
        return os.sysconf("SC_PAGE_SIZE") * os.sysconf("SC_PHYS_PAGES") // 4
    except (ValueError, OSError):
        return 32 << 30


_HOST_CHUNK_BYTES = 192 << 20     # result bytes per pipelined chunk of the host path
_HOST_PAIR_BATCH = 8              # pairs per launch batch while a host operand is still being uploaded
_SIDE_STREAMS = {}


def _side_streams(dev):
    """(upload, download) copy streams of a device, created once."""
    key = (dev.type, dev.index)
    if key not in _SIDE_STREAMS:
        _SIDE_STREAMS[key] = (torch.cuda.Stream(dev), torch.cuda.Stream(dev))
    return _SIDE_STREAMS[key]


_OP_STREAMS = {}


def _operator_stream(dev):
    """High-priority compute stream of a device: the operator kernels of a host call run here while the flow kernels of
    the ``create_flow`` just before are still queued on the current stream (see ``Flow._ready``)."""
    key = (dev.type, dev.index)
    if key not in _OP_STREAMS:
        _OP_STREAMS[key] = torch.cuda.Stream(dev, priority=-1)
    return _OP_STREAMS[key]


def _host_batch_plan(n_pairs: int, big: int):
    """Pair batches of the host path: small first (the upload has only just started and the operators can begin on the
    first frames), doubling up to the device path's batch size (full kernel efficiency once the data is there)."""
    plan, b, left = [], _HOST_PAIR_BATCH, n_pairs
    while left > 0:
        n = min(b, left, big)
        plan.append(n)
        left -= n
        b = min(2 * b, big)
    return plan


class _OperandCache:
    """Device copies of host operands, so that ``create_flow(bt)`` followed by ``flow.diff(bt)``, ``flow.sobel(bt)``,
    ``flow.convolve(bt)`` uploads ``bt`` once instead of four times.

    Key = (buffer address, shape, strides, dtype) of the host array.  Guards against stale hits: the entry dies with the
    array object it was made from (weak reference), and a fingerprint of ~4 k sampled elements plus both ends of the
    buffer is re-taken on every lookup, so an array that was modified in place is uploaded again (a write that misses
    every sampled element is not detected: ``TF_OPERAND_CACHE=0`` or :func:`operand_cache_clear` switch the cache off /
    empty it).  Bounded by ``TF_OPERAND_CACHE_MB`` (default 16 GiB, at most a quarter of the device memory), LRU.
    """

    def __init__(self):
        self.entries = {}          # key -> [tensor, fingerprint, weakref, bytes]
        self.order = []
        self.bytes = 0

    @staticmethod
    def enabled():
        return os.environ.get("TF_OPERAND_CACHE", "1") != "0"

    @staticmethod
    def _key(a: np.ndarray):
        return (a.__array_interface__["data"][0], a.shape, a.strides, a.dtype.str)

    @staticmethod
    def _fingerprint(a: np.ndarray):
        flat = a.reshape(-1)
        n = flat.shape[0]
        if n == 0:
            return 0
        step = max(1, n // 4096)
        sample = np.concatenate([flat[::step], flat[:64], flat[-64:]])
        return hash(sample.tobytes())

    def _limit(self):
        mb = os.environ.get("TF_OPERAND_CACHE_MB")
        if mb is not None:
            return int(mb) << 20
        total = torch.cuda.get_device_properties(torch.cuda.current_device()).total_memory
        return min(16 << 30, total // 4)

    def _drop(self, key):
        e = self.entries.pop(key, None)
        if e is not None:
            self.bytes -= e[3]
            if key in self.order:
                self.order.remove(key)

    def get(self, a: np.ndarray, dev):
        if not self.enabled() or not a.flags.c_contiguous:
            return None
        key = self._key(a)
        e = self.entries.get(key)
        if e is None:
            return None
        if e[2]() is None or e[0].device != dev or e[1] != self._fingerprint(a):
            self._drop(key)
            return None
        self.order.remove(key)
        self.order.append(key)
        return e[0]

    def put(self, a: np.ndarray, t: torch.Tensor):
        if not self.enabled() or not a.flags.c_contiguous:
            return
        import weakref
        nbytes = t.numel() * t.element_size()
        limit = self._limit()
        if nbytes > limit:
            return
        key = self._key(a)
        self._drop(key)
        while self.order and self.bytes + nbytes > limit:
            self._drop(self.order[0])
        try:
            ref = weakref.ref(a, lambda _r, k=key: self._drop(k))
        except TypeError:
            return
        self.entries[key] = [t, self._fingerprint(a), ref, nbytes]
        self.order.append(key)
        self.bytes += nbytes

    def clear(self):
        self.entries.clear()
        self.order.clear()
        self.bytes = 0


_OPERANDS = _OperandCache()


def operand_cache_clear():
    """Forget every cached device copy of a host operand (see ``_OperandCache``)."""
    _OPERANDS.clear()


def _dtype_code(np_dtype):
    """``dtype=`` of the reference (a numpy dtype or None -> float64, np.full semantics) -> (torch dtype, code)."""
    dt = np.dtype(np.float64 if np_dtype is None else np_dtype)
    if dt == np.float32:
        return torch.float32, _lib.TF_F32
    if dt == np.float64:
        return torch.float64, _lib.TF_F64
    if dt == np.int32:
        return torch.int32, _lib.TF_I32
    raise NotImplementedError(f"dtype {dt} is not built in tobac_flow_b200 (float32, float64, int32 are)")


# ------------------------------------------------------------------------------------------------------------------
# reducer recognition
# ------------------------------------------------------------------------------------------------------------------
def diff_func(x):
    """The reducer of ``Flow.diff`` (tobac_flow/flow.py:182-186)."""
    return np.nansum([x[2] - x[1], x[1] - x[0]], axis=0) * 1 / np.maximum(
        np.sum([np.isfinite(x[2]), np.isfinite(x[0])], 0), 1)


def _sobel_ref(direction):
    w = np.array([1, 2, 1])
    d = np.array([-1, 0, 1])
    S = w[:, None, None] * w[None, :, None] * d[None, None, :]
    ks = [k.ravel()[:, None, None] for k in (S, S.transpose(1, 2, 0), S.transpose(2, 0, 1))]

    def f(x):
        if direction == "uphill":
            x = np.fmax(x - x[13], 0)
        elif direction == "downhill":
            x = np.fmin(x - x[13], 0)
        else:
            x = x - x[13]
        return sum(np.nansum(x * k, 0) ** 2 for k in ks) ** 0.5
    return f


_CANDIDATES = [
    (_lib.TF_RED_NANMEAN, None, lambda x: np.nanmean(x, 0)),
    (_lib.TF_RED_NANMAX, None, lambda x: np.nanmax(x, 0)),
    (_lib.TF_RED_NANMIN, None, lambda x: np.nanmin(x, 0)),
    (_lib.TF_RED_ANY, None, lambda x: np.any(x, 0)),
    (_lib.TF_RED_DIFF, 3, diff_func),
    (_lib.TF_RED_SOBEL, 27, _sobel_ref(None)),
    (_lib.TF_RED_SOBEL_UPHILL, 27, _sobel_ref("uphill")),
    (_lib.TF_RED_SOBEL_DOWNHILL, 27, _sobel_ref("downhill")),
]


def recognise_reducer(func: Callable, n_taps: int, stack_dtype) -> int | None:
    """Map a Python ``func=`` to a fused kernel reducer, or None if it is not one the library implements.

    Callers of the reference pass anonymous lambdas (``lambda x: np.nanmean(x, 0)``, detection.py:53-55), so
    identity checks are not enough: the callable is probed on two small seeded tap stacks containing NaNs and
    matched, bit for bit, against the numpy definition of each built reducer.
    """
    if func is None:
        return _lib.TF_RED_NONE
    tagged = getattr(func, "_tf_reducer", None)
    if tagged is not None:
        return tagged
    if isinstance(func, partial) and func.func is np.any and func.keywords == {"axis": 0} and not func.args:
        return _lib.TF_RED_ANY
    # Anything else is an anonymous callable: it is identified by behaviour.  TF_RECOGNISE_REDUCERS=0 switches this off
    # (every untagged callable then takes the Python path); a substitution is announced once per reducer.
    if os.environ.get("TF_RECOGNISE_REDUCERS", "1") == "0":
        return None
    import warnings
    rng = np.random.default_rng(20240229)
    dt = np.dtype(np.float64 if stack_dtype is None else stack_dtype)
    probes = []
    # magnitudes from unit scale to physical values with sentinels (a callable that clips at 150..350 K or masks
    # values above 1000 before reducing differs from the plain reducer on these), infinities, NaNs and zeros
    for scale, offset in ((10.0, 0.0), (40.0, 250.0), (3000.0, 0.0)):
        x = rng.standard_normal((n_taps, 3, 4)) * scale + offset
        x[rng.random(x.shape) < 0.25] = np.nan
        x[:, 0, 0] = np.nan
        x[rng.random(x.shape) < 0.1] = 0
        x[rng.random(x.shape) < 0.05] = 1.0e4
        x[rng.random(x.shape) < 0.03] = -np.inf
        x[rng.random(x.shape) < 0.03] = np.inf
        if dt.kind in "iub":
            x = np.nan_to_num(x, posinf=30000, neginf=-30000).astype(dt)
        else:
            x = x.astype(dt)
        probes.append(x)
    matched = None
    with warnings.catch_warnings(), np.errstate(all="ignore"):
        warnings.simplefilter("ignore")
        try:
            got = [np.asarray(func(p.copy())) for p in probes]
        except Exception:
            return None
        for code, need, ref in _CANDIDATES:
            if need is not None and need != n_taps:
                continue
            try:
                want = [np.asarray(ref(p.copy())) for p in probes]
            except Exception:
                continue
            if all(g.shape == w.shape and np.array_equal(g.astype(np.float64), w.astype(np.float64), equal_nan=True)
                   for g, w in zip(got, want)):
                matched = code
                break
    if matched is not None and matched not in _ANNOUNCED:
        _ANNOUNCED.add(matched)
        warnings.warn(f"tobac_flow_b200: func={getattr(func, '__name__', func)!r} behaves like the built-in reducer "
                      f"#{matched} on the probe stacks and runs as a fused CUDA reducer (TF_RECOGNISE_REDUCERS=0 keeps "
                      "the Python callable)", stacklevel=3)
    return matched


_ANNOUNCED = set()


def _tag(code):
    def deco(f):
        f._tf_reducer = code
        return f
    return deco


# ------------------------------------------------------------------------------------------------------------------
# the stencil operator
# ------------------------------------------------------------------------------------------------------------------
def convolve_device(data: torch.Tensor, fwd: torch.Tensor, bwd: torch.Tensor, structure, method, fill_value,
                    dtype, reducer: int, has_prev: bool = False, has_next: bool = False,
                    out: torch.Tensor | None = None) -> torch.Tensor:
    """Launch tf_sl_convolve on device tensors.

    ``data`` is (T, H, W).  With ``has_prev`` / ``has_next`` the first / last frame of ``data`` is a halo frame
    (time sharding): it is only read, and the flows/outputs then cover the T-1 / T-2 interior frames.
    """
    lib = _lib.load()
    interp = _interp_code(method)
    structure = np.asarray(structure)
    assert structure.shape == (3, 3, 3), "Structure input must be a 3x3x3 array"  # convolve.py:290
    n_taps = int(np.count_nonzero(structure))
    out_t, stack_code = _dtype_code(dtype)
    if data.dtype not in _TORCH_DT:
        if data.dtype in (torch.int64, torch.int16, torch.int8, torch.uint8, torch.bool):
            data = data.to(torch.int32)  # cv2's binding narrows wider integers the same way
        elif data.dtype in (torch.float16, torch.bfloat16):
            data = data.to(torch.float32)
        else:
            raise NotImplementedError(f"operand dtype {data.dtype} is not supported")
    data = data.contiguous()
    T_all, H, W = data.shape
    n_frames = T_all - int(bool(has_prev)) - int(bool(has_next))
    if tuple(fwd.shape) != (n_frames, H, W, 2) or tuple(bwd.shape) != (n_frames, H, W, 2):
        raise AssertionError("Data input must have the same shape as the Flow object")
    fwd = fwd.contiguous()
    bwd = bwd.contiguous()
    shape = (n_frames, H, W) if reducer != _lib.TF_RED_NONE else (n_taps, n_frames, H, W)
    if out is None:
        out = torch.empty(shape, dtype=out_t, device=data.device)
    else:
        assert tuple(out.shape) == shape and out.dtype == out_t and out.is_contiguous()
    if n_frames == 0:
        return out
    cur0 = data.data_ptr() + (data.element_size() * H * W if has_prev else 0)
    rc = lib.tf_sl_convolve(cur0, n_frames, int(bool(has_prev)), int(bool(has_next)), fwd.data_ptr(), bwd.data_ptr(),
                            out.data_ptr(), n_frames * H * W, H, W, _TORCH_DT[data.dtype], stack_code, interp,
                            reducer, _lib.structure_bytes(structure), float(fill_value), _stream())
    _lib.check(rc, "tf_sl_convolve")
    return out


class Flow:
    """Semi-Lagrangian operators on optical-flow vectors (drop-in for ``tobac_flow.flow.Flow``)."""

    def __init__(self, forward_flow, backward_flow) -> None:
        if tuple(forward_flow.shape) != tuple(backward_flow.shape):
            raise ValueError("Forward and backward flow vector arrays must have the same shape")
        if forward_flow.shape[-1] != 2:
            raise ValueError("Flow vectors must have a size of 2 in the trailing dimension")
        self.shape = tuple(forward_flow.shape[:-1])
        # [(frames_ready, event)]: set by create_flow on a host array.  The flow kernels are queued batch by batch on the
        # current stream and create_flow returns without waiting for them; event k fires when flow vectors [0, frames_ready_k)
        # are final.  Work queued on the current stream is ordered behind all of them anyway; the host operators use the
        # events to start on the first frames (on the operator stream) while the later pairs are still being computed.
        self._ready = None
        self._ready_frames = None      # data_ptr of the device copy of the frames those batches were computed from
        self._fwd_np = forward_flow if isinstance(forward_flow, np.ndarray) else None
        self._bwd_np = backward_flow if isinstance(backward_flow, np.ndarray) else None
        self._fwd_t = forward_flow if isinstance(forward_flow, torch.Tensor) else None
        self._bwd_t = backward_flow if isinstance(backward_flow, torch.Tensor) else None
        if self._fwd_np is None and self._fwd_t is None:
            self._fwd_np = np.asarray(forward_flow)
        if self._bwd_np is None and self._bwd_t is None:
            self._bwd_np = np.asarray(backward_flow)

    # -- flow vectors ------------------------------------------------------------------------------
    @property
    def forward_flow(self) -> np.ndarray:
        if self._fwd_np is None:
            self._fwd_np = _to_host(self._fwd_t.detach())
        return self._fwd_np

    @property
    def backward_flow(self) -> np.ndarray:
        if self._bwd_np is None:
            self._bwd_np = _to_host(self._bwd_t.detach())
        return self._bwd_np

    @property
    def forward_flow_device(self) -> torch.Tensor:
        if self._fwd_t is None or not self._fwd_t.is_cuda:
            src = self._fwd_t if self._fwd_t is not None else self._fwd_np
            self._fwd_t = _to_device(src, torch.float32)[0]
        return self._fwd_t

    @property
    def backward_flow_device(self) -> torch.Tensor:
        if self._bwd_t is None or not self._bwd_t.is_cuda:
            src = self._bwd_t if self._bwd_t is not None else self._bwd_np
            self._bwd_t = _to_device(src, torch.float32)[0]
        return self._bwd_t

    @property
    def flow(self):
        return self.forward_flow, self.backward_flow

    def __getitem__(self, items) -> "Flow":
        f = self._fwd_t[items] if self._fwd_t is not None else self._fwd_np[items]
        b = self._bwd_t[items] if self._bwd_t is not None else self._bwd_np[items]
        return Flow(f, b)

    # -- operators ---------------------------------------------------------------------------------
    def convolve(self, data, structure=None, method: str = "linear", fill_value: float = np.nan,
                 dtype: type = np.float32, func: Callable | None = None):
        """``Flow.convolve`` (tobac_flow/flow.py:105-157 -> tobac_flow/convolve.py:248-348)."""
        if structure is None:
            structure = _default_structure()
        assert tuple(data.shape) == self.shape, "Data input must have the same shape as the Flow object"
        structure = np.asarray(structure)
        assert structure.shape == (3, 3, 3), "Structure input must be a 3x3x3 array"
        _interp_code(method)
        n_taps = int(np.count_nonzero(structure))
        reducer = recognise_reducer(func, n_taps, dtype)
        if reducer is not None and not isinstance(data, torch.Tensor):
            return self._convolve_host_pipelined(_as_numpy(data), structure, method, fill_value, dtype, reducer, n_taps)
        t, from_host = _to_device(data)
        if reducer is None:
            res = self._convolve_python_func(t, structure, method, fill_value, dtype, func)
        else:
            res = convolve_device(t, self.forward_flow_device, self.backward_flow_device, structure, method,
                                  fill_value, dtype, reducer)
        return _to_host(res) if from_host else res

    def _convolve_host_pipelined(self, a: np.ndarray, structure, method, fill_value, dtype, reducer, n_taps):
        """Host operand -> host result with the PCIe copies overlapped with the kernels: the operand is uploaded in
        time chunks on one side stream, each chunk is computed as soon as its one-frame halo has arrived, and its
        result is copied into page-locked host memory on a second side stream while the next chunk computes."""
        dev = _device()
        a = np.ascontiguousarray(a)
        if a.dtype == np.bool_ or (a.dtype.kind in "iu" and a.dtype != np.int32):
            a = a.astype(np.int32)          # cv2's binding narrows wider integers the same way
        elif a.dtype == np.float16:
            a = a.astype(np.float32)
        elif a.dtype not in (np.float32, np.float64, np.int32):
            raise NotImplementedError(f"operand dtype {a.dtype} is not supported")
        resident = _OPERANDS.get(a, dev)       # the device copy a previous create_flow / operator call left behind
        src = torch.from_numpy(a)
        T, H, W = src.shape
        out_t, _ = _dtype_code(dtype)
        stack = reducer == _lib.TF_RED_NONE
        # Results land in page-locked memory (a pageable target halves the PCIe rate).  torch's pinned allocator never
        # returns blocks to the OS, so results beyond the cap (TF_PINNED_RESULT_MAX_GB, default a quarter of the host RAM)
        # go to an ordinary numpy array through two pinned staging chunks instead.
        shape_all = (n_taps, T, H, W) if stack else (T, H, W)
        nbytes_all = int(np.prod(shape_all)) * out_t.itemsize
        pinned = nbytes_all <= _pinned_result_cap()
        host = torch.empty(shape_all, dtype=out_t, pin_memory=pinned)
        if T == 0:
            return host.numpy()
        stage, ev_stage, pending = [None, None], [None, None], [None, None]
        fwd, bwd = self.forward_flow_device, self.backward_flow_device
        per_frame = H * W * out_t.itemsize * (n_taps if stack else 1)
        # chunks of at most _HOST_CHUNK_BYTES of result, and at least four of them so that upload, kernels and download
        # of neighbouring chunks overlap even for the small results (diff)
        Tc = max(1, min(T, _HOST_CHUNK_BYTES // max(per_frame, 1), -(-T // 4)))
        chunks = [(a0, min(a0 + Tc, T)) for a0 in range(0, T, Tc)]
        cur = torch.cuda.current_stream()
        s_in, s_out = _side_streams(dev)
        # Flow vectors still being computed (create_flow on a host array returned without waiting): the operator kernels go
        # to the high-priority operator stream, each chunk behind the event of the pair batch that completes its frames,
        # so results start to flow back over PCIe while the later pairs are in the iteration kernels.  Only taken when the
        # operand is the resident copy that create_flow uploaded (its upload events are behind the same batch events).
        ready = self._ready
        if ready is not None and (resident is None or resident.data_ptr() != self._ready_frames or ready[-1][1].query()):
            ready = None               # (another operand's upload is ordered on the current stream, not behind these events)
        s_k = _operator_stream(dev) if ready is not None else cur

        def wait_flow(b0):
            if ready is not None:
                for upto, ev in ready:
                    if upto >= b0:
                        s_k.wait_event(ev)
                        return
                s_k.wait_event(ready[-1][1])
        # the operand buffer belongs to the upload stream's pool, so the copies need not wait for the work already queued
        # on the current stream (typically the flow kernels of the create_flow call just before): they run underneath it
        if ready is None:
            s_out.wait_stream(cur)
        ev_in = []
        if resident is not None:
            d_in = resident
        else:
            with torch.cuda.stream(s_in):
                d_in = torch.empty((T, H, W), dtype=src.dtype, device=dev)
            d_in.record_stream(cur)
            with torch.cuda.stream(s_in):
                for a0, b0 in chunks:
                    d_in[a0:b0].copy_(src[a0:b0], non_blocking=True)
                    ev_in.append(torch.cuda.Event())
                    ev_in[-1].record(s_in)
        bufs, ev_free = [None, None], [None, None]
        for k, (a0, b0) in enumerate(chunks):
            if ev_in:
                s_k.wait_event(ev_in[min(k + 1, len(chunks) - 1)])  # this chunk and its right halo frame are here
            wait_flow(b0)           # vectors of [a0, b0) final (the batch that made them also waited for frame b0's upload)
            slot = k & 1
            if ev_free[slot] is not None:
                s_k.wait_event(ev_free[slot])                       # the buffer's previous contents are on the host
            n = b0 - a0
            shape = (n_taps, n, H, W) if stack else (n, H, W)
            with torch.cuda.stream(s_k):
                if bufs[slot] is None or tuple(bufs[slot].shape) != shape:
                    bufs[slot] = torch.empty(shape, dtype=out_t, device=dev)
                convolve_device(d_in[max(a0 - 1, 0):min(b0 + 1, T)], fwd[a0:b0], bwd[a0:b0], structure, method, fill_value,
                                dtype, reducer, has_prev=a0 > 0, has_next=b0 < T, out=bufs[slot])
            ev_c = torch.cuda.Event()
            ev_c.record(s_k)
            s_out.wait_event(ev_c)
            if not pinned:
                # flush the staging chunk this slot used two chunks ago into the pageable result (host-side copy)
                if pending[slot] is not None:
                    ev_stage[slot].synchronize()
                    pa, pb = pending[slot]
                    host[(slice(None), slice(pa, pb)) if stack else slice(pa, pb)] = stage[slot][(slice(None), slice(0, pb - pa)) if stack else slice(0, pb - pa)]
                if stage[slot] is None or stage[slot].shape[1 if stack else 0] < n:
                    stage[slot] = torch.empty((n_taps, Tc, H, W) if stack else (Tc, H, W), dtype=out_t, pin_memory=True)
            with torch.cuda.stream(s_out):
                tgt = host if pinned else stage[slot]
                off = a0 if pinned else 0
                if stack:
                    for tap in range(n_taps):
                        tgt[tap, off:off + n].copy_(bufs[slot][tap], non_blocking=True)
                else:
                    tgt[off:off + n].copy_(bufs[slot], non_blocking=True)
                ev_free[slot] = torch.cuda.Event()
                ev_free[slot].record(s_out)
                if not pinned:
                    ev_stage[slot] = ev_free[slot]
                    pending[slot] = (a0, b0)
        s_out.synchronize()
        if not pinned:
            for slot in (0, 1):
                if pending[slot] is not None:
                    pa, pb = pending[slot]
                    host[(slice(None), slice(pa, pb)) if stack else slice(pa, pb)] = stage[slot][(slice(None), slice(0, pb - pa)) if stack else slice(0, pb - pa)]
        cur.wait_stream(s_in)
        if ready is not None:
            cur.wait_stream(s_k)           # (the chunk buffers go back to the operator stream's pool behind its kernels)
        if resident is None:
            _OPERANDS.put(a, d_in)
        return host.numpy()

    def _convolve_python_func(self, t, structure, method, fill_value, dtype, func):
        """Compatibility path for arbitrary Python reducers: the tap stack of each step is gathered by the
        CUDA kernel and ``func`` is applied to it on the host (convolve.py:316-331, 346-347)."""
        T = t.shape[0]
        out_t, _ = _dtype_code(dtype)
        res = torch.full(tuple(t.shape), float(fill_value) if out_t.is_floating_point else int(fill_value),
                         dtype=out_t, device=t.device)
        fwd, bwd = self.forward_flow_device, self.backward_flow_device
        for i in range(T):
            lo, hi = max(i - 1, 0), min(i + 2, T)
            stack = convolve_device(t[lo:hi], fwd[i:i + 1], bwd[i:i + 1], structure, method, fill_value, dtype,
                                    _lib.TF_RED_NONE, has_prev=i > 0, has_next=i < T - 1)
            r = np.asarray(func(stack[:, 0].cpu().numpy()))
            res[i] = torch.from_numpy(np.ascontiguousarray(r)).to(device=t.device, dtype=out_t)
        if t.dtype.is_floating_point:
            res[torch.isnan(t)] = float(fill_value) if out_t.is_floating_point else int(fill_value)
        return res

    def diff(self, data, method: str = "linear", dtype: type = np.float32):
        """``Flow.diff`` (tobac_flow/flow.py:159-191)."""
        diff_struct = np.zeros([3, 3, 3])
        diff_struct[:, 1, 1] = 1
        return self.convolve(data, structure=diff_struct, func=_DIFF, method=method, dtype=dtype)

    def sobel(self, data, method: str = "linear", dtype: type = None, fill_value: float = np.nan,
              direction: str | None = None):
        """``Flow.sobel`` (tobac_flow/flow.py:193-234 -> tobac_flow/sobel.py:89-143); dtype=None -> float64."""
        from .sobel import sobel_reducer
        return self.convolve(data, structure=np.ones((3, 3, 3), bool), method=method, fill_value=fill_value,
                             dtype=dtype, func=sobel_reducer(direction))

    # -- downstream consumers ---------------------------------------------------------------------------------------
    # watershed (and label with sub-segmentation) stay the reference's own code; label / link_overlap are native
    def _delegate(self, name, *args, **kwargs):
        try:
            import tobac_flow.flow as ref  # the reference package, when installed next to this one
        except Exception as e:  # pragma: no cover
            raise NotImplementedError(
                f"Flow.{name} is outside the dense-flow hot path; it delegates to the reference's tobac_flow.{name} "
                "which is not importable here") from e
        return getattr(ref.Flow, name)(self, *args, **kwargs)

    def watershed(self, field, markers, mask=None, connectivity=1):
        """``Flow.watershed`` (tobac_flow/flow.py:236-279 -> tobac_flow/watershed.py:17-168): the offset fields are
        prepared on the device, the (value, age) priority flood runs in the native library on the host."""
        from .watershed import watershed
        return watershed(self.forward_flow_device, self.backward_flow_device, _as_numpy(field) if not isinstance(field, torch.Tensor) else field.cpu().numpy(),
                         _as_numpy(markers) if not isinstance(markers, torch.Tensor) else markers.cpu().numpy(),
                         mask=None if mask is None else (_as_numpy(mask) if not isinstance(mask, torch.Tensor) else mask.cpu().numpy()),
                         connectivity=connectivity)

    def label(self, data, structure=None, dtype: type = np.int32, overlap: float = 0, absolute_overlap: int = 1,
              subsegment_shrink: float = 0, peak_min_distance: int = 5):
        """``Flow.label`` (tobac_flow/flow.py:281-330 -> tobac_flow/label.py:84-175)."""
        if structure is None:
            structure = _default_structure()
        if subsegment_shrink != 0:   # skimage sub-segmentation: not on the path, the reference's own code handles it
            return self._delegate("label", data, structure=structure, dtype=dtype, overlap=overlap,
                                  absolute_overlap=absolute_overlap, subsegment_shrink=subsegment_shrink,
                                  peak_min_distance=peak_min_distance)
        from .label import flow_label
        return flow_label(self, data, structure=structure, dtype=dtype, overlap=overlap,
                          absolute_overlap=absolute_overlap)

    def link_overlap(self, data, structure=None, dtype: type = np.int32, overlap: float = 0,
                     absolute_overlap: int = 1):
        """``Flow.link_overlap`` (tobac_flow/flow.py:332-355 -> tobac_flow/label.py:249-321)."""
        if structure is None:
            structure = _default_structure()
        from .label import flow_link_overlap
        return flow_link_overlap(self, data, structure=structure, dtype=dtype, overlap=overlap,
                                 absolute_overlap=absolute_overlap)


_DIFF = _tag(_lib.TF_RED_DIFF)(diff_func)

try:  # register against the reference ABC when the reference is importable (it is optional)
    from tobac_flow.core import AbstractFlow as _AbstractFlow  # type: ignore

    _AbstractFlow.register(Flow)
except Exception:  # pragma: no cover
    pass


# ------------------------------------------------------------------------------------------------------------------
# flow construction
# ------------------------------------------------------------------------------------------------------------------
def _is_dis(model) -> bool:
    from .dis import DISOpticalFlow
    return isinstance(model, DISOpticalFlow)


def _check_model(model, vr_steps: int):
    """``model``: the reference's model name, or a :class:`tobac_flow_b200.DISOpticalFlow` instance."""
    if _is_dis(model):
        return
    if model not in _REFERENCE_MODELS:
        raise ValueError(  # utils/flow_utils.py:72-75
            "'model' parameter must be one of: 'Farneback', 'DeepFlow', 'PCA', 'SimpleFlow', 'SparseToDense', "
            "'DIS', 'DenseRLOF', 'DualTVL1'")
    if model != "Farneback":
        raise NotImplementedError(f"optical-flow model '{model}' is not built in tobac_flow_b200 (only 'Farneback')")


def _pair_batch(n_pairs: int, H: int, W: int, params, vr: bool = False, model=None) -> int:
    """Pairs per launch batch: as many as fit comfortably in free HBM, at most 512 Mpx (larger batches amortise the wave
    quantisation and the latency-bound launches of the small pyramid levels: 28.4 vs 30.5 ms per 96 CONUS frames for
    the coarse levels at 512 vs 256 Mpx), in equally sized batches (a small last batch would run at a fraction of the
    efficiency)."""
    # (the answer for a shape is remembered: `cudaMemGetInfo` is a driver call that can wait milliseconds behind a
    # monitoring query -- nvidia-smi -- and it sits in front of a call's first kernel launch; a shape whose workspace
    # allocation fails later drops its entry, see calculate_flow_device)
    dis = _is_dis(model)
    key = (torch.cuda.current_device(), n_pairs, H, W, bool(vr), model.key() if dis else params.num_levels,
           os.environ.get("TF_PAIR_BATCH_MPX"))
    if key in _PAIR_BATCH_CACHE:
        return _PAIR_BATCH_CACHE[key]
    per_pair = (model.workspace_bytes(1, H, W) if dis else _lib.workspace_bytes(1, H, W, params)) + 2 * H * W
    if vr:
        per_pair += int(_lib.load().tf_vr_workspace_bytes(1, H, W))
    free, _ = torch.cuda.mem_get_info()
    free += max(0, torch.cuda.memory_reserved() - torch.cuda.memory_allocated())   # blocks torch holds but can reuse
    by_mem = max(1, int(free * 0.6) // per_pair)
    by_px = max(1, (int(os.environ.get("TF_PAIR_BATCH_MPX", "512")) << 20) // (H * W))
    nb = max(1, min(n_pairs, by_mem, by_px))
    n_batches = -(-n_pairs // nb)
    _PAIR_BATCH_CACHE[key] = -(-n_pairs // n_batches)
    return _PAIR_BATCH_CACHE[key]


_PAIR_BATCH_CACHE = {}


def calculate_flow_device(frames: torch.Tensor, fwd: torch.Tensor, bwd: torch.Tensor, smoothing_passes: int = 0,
                          interp_method: str = "linear", max_value: float | None = None,
                          next_frames: torch.Tensor | None = None, batch: int | None = None, vr_steps: int = 0,
                          frames_ready: Callable | None = None, batch_plan=None, batch_done: Callable | None = None,
                          model=None) -> None:
    """Fill ``fwd[i]`` and ``bwd[i + 1]`` for every consecutive pair of ``frames`` (device tensors, in place).

    ``frames`` (T, H, W) float32 or float64; ``fwd``/``bwd`` (>= T, H, W, 2) float32.  With ``next_frames`` the pairs are
    (frames[i], next_frames[i]) and results go to fwd[i], bwd[i + 1] for every i (``calculate_flow_2``).
    ``max_value`` fuses the clamp of ``create_flow`` into the last kernel when no smoothing follows.
    ``model``: None (Farneback) or a :class:`tobac_flow_b200.DISOpticalFlow`.
    """
    lib = _lib.load()
    T, H, W = frames.shape
    n_pairs = T - 1 if next_frames is None else T
    if n_pairs <= 0:
        return
    interp = _interp_code(interp_method)
    use_vr = bool(vr_steps) and vr_steps > 0   # flow.py:513-519: one refinement whenever vr_steps > 0
    fuse_clamp = (max_value is not None) and smoothing_passes == 0 and not use_vr
    dis = _is_dis(model)
    params = _lib.default_params(max_value if fuse_clamp else 0.0)
    if dis:
        dis_params = model.params(max_value if fuse_clamp else 0.0)
    nb = batch or _pair_batch(n_pairs, H, W, params, use_vr, model)
    if batch_plan is None:
        batch_plan = [min(nb, n_pairs - p0) for p0 in range(0, n_pairs, nb)]
    nb = max(batch_plan)
    # (measured: alternating consecutive pair batches between two streams, to fill the half-empty grids of the small
    # pyramid levels and the tail waves, gains nothing: 458-475 vs 460 ms per CONUS day)
    dev = frames.device
    q0 = torch.empty((nb, H, W), dtype=torch.uint8, device=dev)
    q1 = torch.empty((nb, H, W), dtype=torch.uint8, device=dev)
    f64 = frames.dtype == torch.float64        # float64 frames are normalised in float64, as numpy does for the reference
    mm = torch.empty((2 * nb,), dtype=frames.dtype, device=dev)
    normalise = lib.tf_pair_normalise_u8_f64 if f64 else lib.tf_pair_normalise_u8
    ws_bytes = model.workspace_bytes(nb, H, W) if dis else _lib.workspace_bytes(nb, H, W, params)
    try:
        ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
    except torch.cuda.OutOfMemoryError:
        _PAIR_BATCH_CACHE.clear()          # the remembered batch size no longer fits: the next call asks the driver again
        raise
    vr_params = vr_ws = None
    vr_bytes = 0
    if use_vr:
        vr_params = _lib.default_vr_params()
        vr_bytes = int(lib.tf_vr_workspace_bytes(nb, H, W))
        vr_ws = torch.empty((vr_bytes,), dtype=torch.uint8, device=dev)
    tmp_f = tmp_b = None
    if smoothing_passes > 0:
        tmp_f = torch.empty((nb, H, W, 2), dtype=torch.float32, device=dev)
        tmp_b = torch.empty((nb, H, W, 2), dtype=torch.float32, device=dev)
    hw = H * W
    es = frames.element_size()
    st = _stream()
    for bi, n in enumerate(batch_plan):
        p0 = sum(batch_plan[:bi])
        if frames_ready is not None:
            frames_ready(p0 + n)          # make the stream wait until frames [0, p0 + n] have been uploaded
        f0 = frames.data_ptr() + p0 * hw * es
        f1 = (frames.data_ptr() + (p0 + 1) * hw * es) if next_frames is None else (next_frames.data_ptr() + p0 * hw * es)
        _lib.check(normalise(f0, f1, hw, q0.data_ptr(), q1.data_ptr(), n, H, W, mm.data_ptr(), st),
                   "tf_pair_normalise_u8")
        fo = fwd.data_ptr() + p0 * hw * 2 * 4
        bo = bwd.data_ptr() + (p0 + 1) * hw * 2 * 4
        if dis:
            _lib.check(lib.tf_dis_pairs(q0.data_ptr(), q1.data_ptr(), fo, hw * 2, bo, hw * 2, n, H, W,
                                        ctypes.byref(dis_params), ws.data_ptr(), ws_bytes, st), "tf_dis_pairs")
        else:
            _lib.check(lib.tf_farneback_pairs(q0.data_ptr(), q1.data_ptr(), fo, hw * 2, bo, hw * 2, n, H, W,
                                              ctypes.byref(params), ws.data_ptr(), ws_bytes, st), "tf_farneback_pairs")
        if use_vr:
            _lib.check(lib.tf_variational_refinement(q0.data_ptr(), q1.data_ptr(), fo, hw * 2, bo, hw * 2, n, H, W,
                                                     ctypes.byref(vr_params), vr_ws.data_ptr(), vr_bytes, st),
                       "tf_variational_refinement")
        for _ in range(smoothing_passes):
            _lib.check(lib.tf_smooth_flow_step(fo, bo, tmp_f.data_ptr(), tmp_b.data_ptr(), hw * 2, n, H, W, interp, st),
                       "tf_smooth_flow_step")
            fwd[p0:p0 + n].copy_(tmp_f[:n])
            bwd[p0 + 1:p0 + 1 + n].copy_(tmp_b[:n])
        if batch_done is not None:
            batch_done(p0, n)


def finalise_flow_device(fwd: torch.Tensor, bwd: torch.Tensor, max_value: float | None, clamp_all: bool,
                         mirror_first: bool = True, mirror_last: bool = True) -> None:
    T, H, W, _ = fwd.shape
    _lib.check(_lib.load().tf_flow_finalise(fwd.data_ptr(), bwd.data_ptr(), T, H, W,
                                            float(max_value) if max_value is not None else 0.0, int(clamp_all),
                                            int(mirror_first), int(mirror_last), _stream()), "tf_flow_finalise")


def _select_normalisation(method: str):
    if method not in _NORMALISATIONS:  # normalisation_utils.py:130-133
        raise ValueError(f"{method} not an acceptable normalisation method, method must be one of {_NORMALISATIONS}")
    if method != "linear":
        raise NotImplementedError(f"normalisation '{method}' is not built in tobac_flow_b200 (only 'linear')")


def _calculate_flow_tensors(data, model, vr_steps, smoothing_passes, interp_method, normalisation_method,
                            max_value, data_b=None):
    _check_model(model, vr_steps)
    _select_normalisation(normalisation_method)
    _interp_code(interp_method)
    frames_ready = batch = None
    host_plan = False
    ready = None
    host_a = None if isinstance(data, torch.Tensor) else _as_numpy(data)
    if host_a is not None and data_b is None and host_a.ndim == 3 and host_a.dtype == np.float32 and host_a.shape[0] > 2 * _HOST_PAIR_BATCH:
        # host input: upload in chunks on a side stream and start on the first pairs while the rest is in flight
        dev = _device()
        src = torch.from_numpy(np.ascontiguousarray(host_a))
        frames = torch.empty(tuple(src.shape), dtype=torch.float32, device=dev)
        s_in, _ = _side_streams(dev)
        s_in.wait_stream(torch.cuda.current_stream())
        events = []
        with torch.cuda.stream(s_in):
            for a0 in range(0, src.shape[0], _HOST_PAIR_BATCH):
                frames[a0:a0 + _HOST_PAIR_BATCH].copy_(src[a0:a0 + _HOST_PAIR_BATCH], non_blocking=True)
                events.append(torch.cuda.Event())
                events[-1].record(s_in)

        def frames_ready(last_frame):
            torch.cuda.current_stream().wait_event(events[min(last_frame // _HOST_PAIR_BATCH, len(events) - 1)])
        host_plan = True
        frames.record_stream(s_in)
        _OPERANDS.put(host_a if host_a.flags.c_contiguous else src.numpy(), frames)   # the operators reuse this copy
    else:
        frames, _ = _to_device(data)
        if frames.dtype not in (torch.float32, torch.float64):
            frames = frames.to(torch.float64)      # integer data: numpy promotes (array - vmin) * factor to float64
    if frames.dim() != 3:
        raise ValueError("data must have shape (t, y, x)")
    frames_b = None
    if data_b is not None:
        frames_b, _ = _to_device(data_b, frames.dtype)
    T, H, W = frames.shape
    # the reference pre-fills with NaN (flow.py:408-409); for T > 1 every element is overwritten (pairs + end
    # rules), so the fill is only materialised for the degenerate single-frame case
    if T > 1:
        fwd = torch.empty((T, H, W, 2), dtype=torch.float32, device=frames.device)
        bwd = torch.empty((T, H, W, 2), dtype=torch.float32, device=frames.device)
    else:
        fwd = torch.full((T, H, W, 2), float("nan"), dtype=torch.float32, device=frames.device)
        bwd = torch.full((T, H, W, 2), float("nan"), dtype=torch.float32, device=frames.device)
    early_final = False
    if frames_b is None:
        plan = batch_done = None
        if host_plan:
            use_vr = bool(vr_steps) and vr_steps > 0
            plan = _host_batch_plan(T - 1, _pair_batch(T - 1, H, W, _lib.default_params(0.0), use_vr, model))
            if max_value is not None and max_value != 0 and smoothing_passes == 0 and not use_vr:
                # the clamp is fused into the last iteration kernel, so a batch's vectors are final once the end rules of
                # the first / last frame (flow.py:425-426) are applied: do that with the batch that computes them and mark
                # every batch with an event (Flow._ready)
                early_final, ready = True, []
                fe = H * W * 2 * 4

                def batch_done(p0, n):
                    if p0 == 0:
                        _lib.check(_lib.load().tf_flow_finalise(fwd.data_ptr(), bwd.data_ptr(), 1, H, W, 0.0, 0, 1, 0,
                                                                _stream()), "tf_flow_finalise")
                    last = p0 + n == T - 1
                    if last:
                        _lib.check(_lib.load().tf_flow_finalise(fwd.data_ptr() + (T - 1) * fe, bwd.data_ptr() + (T - 1) * fe, 1,
                                                                H, W, 0.0, 0, 0, 1, _stream()), "tf_flow_finalise")
                    ev = torch.cuda.Event()
                    ev.record(torch.cuda.current_stream())
                    # vectors of frames [0, p0 + n) are final: fwd[i] comes from pair i, bwd[i] from pair i - 1
                    ready.append((T if last else p0 + n, ev))
        calculate_flow_device(frames, fwd, bwd, smoothing_passes, interp_method, max_value, vr_steps=vr_steps,
                              batch=batch, frames_ready=frames_ready, batch_plan=plan, batch_done=batch_done,
                              model=model)
    else:
        # calculate_flow_2 (flow.py:431-496): pairs (a[i], b[i]) for i < T-1
        calculate_flow_device(frames[:T - 1], fwd, bwd, smoothing_passes, interp_method, max_value,
                              next_frames=frames_b[:T - 1], vr_steps=vr_steps, model=model)
    clamp_all = max_value is not None and (smoothing_passes > 0 or (bool(vr_steps) and vr_steps > 0))
    if not early_final:
        finalise_flow_device(fwd, bwd, max_value, clamp_all)
    if max_value is not None and max_value == 0:
        # np.minimum(np.maximum(f, -0), 0) (flow.py:60-61): every finite vector becomes 0 (the kernels read a zero clamp
        # as "no clamp")
        fwd = torch.where(torch.isnan(fwd), fwd, torch.zeros_like(fwd))
        bwd = torch.where(torch.isnan(bwd), bwd, torch.zeros_like(bwd))
    return fwd, bwd, (ready, frames.data_ptr()) if ready is not None else None


def calculate_flow(data, model: str = "Farneback", vr_steps: int = 0, smoothing_passes: int = 0,
                   interp_method: str = "linear", normalisation_method: str = "linear", **normalisation_kwargs):
    """``calculate_flow`` (tobac_flow/flow.py:362-428): returns (forward_flow, backward_flow) numpy arrays."""
    if normalisation_kwargs:
        raise NotImplementedError("normalisation keyword arguments are not supported by the 'linear' method here")
    fwd, bwd, _ = _calculate_flow_tensors(data, model, vr_steps, smoothing_passes, interp_method,
                                          normalisation_method, None)
    return fwd.cpu().numpy(), bwd.cpu().numpy()


def calculate_flow_2(a, b, model: str = "Farneback", vr_steps: int = 0, smoothing_passes: int = 0,
                     normalisation_method: str = "linear", **normalisation_kwargs):
    """``calculate_flow_2`` (tobac_flow/flow.py:431-496)."""
    if normalisation_kwargs:
        raise NotImplementedError("normalisation keyword arguments are not supported by the 'linear' method here")
    fwd, bwd, _ = _calculate_flow_tensors(a, model, vr_steps, smoothing_passes, "linear", normalisation_method, None,
                                          data_b=b)
    return fwd.cpu().numpy(), bwd.cpu().numpy()


def create_flow(data, model: str = "Farneback", vr_steps: int = 0, smoothing_passes: int = 0,
                interp_method: str = "linear", max_value=20) -> Flow:
    """``create_flow`` (tobac_flow/flow.py:23-65): flow vectors for ``data`` (t, y, x), clamped to +-max_value.

    ``model`` is "Farneback" or a :class:`tobac_flow_b200.DISOpticalFlow` (as for ``calculate_flow`` /
    ``calculate_flow_2``).

    The returned ``Flow`` keeps the vectors on the GPU.
    """
    fwd, bwd, ready = _calculate_flow_tensors(data, model, vr_steps, smoothing_passes, interp_method, "linear", max_value)
    flow = Flow(fwd, bwd)
    if ready is not None:
        flow._ready, flow._ready_frames = ready
    return flow


def smooth_flow_step(forward_flow, backward_flow, method: str = "linear"):
    """``smooth_flow_step`` (tobac_flow/flow.py:530-568) for one (H, W, 2) pair of fields."""
    interp = _interp_code(method)
    f, host = _to_device(forward_flow, torch.float32)
    b, _ = _to_device(backward_flow, torch.float32)
    H, W, _two = f.shape
    fo, bo = torch.empty_like(f), torch.empty_like(b)
    _lib.check(_lib.load().tf_smooth_flow_step(f.data_ptr(), b.data_ptr(), fo.data_ptr(), bo.data_ptr(), H * W * 2, 1,
                                               H, W, interp, _stream()), "tf_smooth_flow_step")
    return (fo.cpu().numpy(), bo.cpu().numpy()) if host else (fo, bo)


def pair_to_8bit(frame0, frame1):
    """``to_8bit(linear_norm(stack), 0, 1)`` for one pair (normalisation_utils.py:59-72, 10-33); float64 frames are
    normalised in float64, as numpy does."""
    a, host = _to_device(np.stack([_as_numpy(frame0), _as_numpy(frame1)]) if not isinstance(frame0, torch.Tensor)
                         else torch.stack([frame0, frame1]))
    if a.dtype not in (torch.float32, torch.float64):
        a = a.to(torch.float64)
    _, H, W = a.shape
    q = torch.empty((2, H, W), dtype=torch.uint8, device=a.device)
    mm = torch.empty((2,), dtype=a.dtype, device=a.device)
    fn = _lib.load().tf_pair_normalise_u8_f64 if a.dtype == torch.float64 else _lib.load().tf_pair_normalise_u8
    _lib.check(fn(a.data_ptr(), a.data_ptr() + H * W * a.element_size(), H * W, q.data_ptr(), q.data_ptr() + H * W, 1, H,
                  W, mm.data_ptr(), _stream()), "tf_pair_normalise_u8")
    return (q[0].cpu().numpy(), q[1].cpu().numpy()) if host else (q[0], q[1])


# ----------------------------------------------------------------------------------------------------------------
# stage-level entry points (parity tests against the oracle's per-stage restatement of OpenCV's Farneback)
# ----------------------------------------------------------------------------------------------------------------
def fb_pyramid_level(q0, q1, level, two_pass=False):
    """Level image ``level`` (index into ``_lib.level_plan``, coarsest first) of the quantised pair ``q0``, ``q1``
    ((H, W) uint8 each): convertTo -> GaussianBlur -> resize from the full-resolution image, as
    ``FarnebackOpticalFlow::calc`` builds it.  Returns (2, h, w) float32 (numpy)."""
    q = torch.from_numpy(np.ascontiguousarray(np.stack([q0, q1]), dtype=np.uint8)).to(_device())
    _, H, W = q.shape
    params = _lib.default_params()
    h, w = _lib.level_plan(H, W, params)[level]
    nbytes = _lib.workspace_bytes(1, H, W, params)
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=q.device)
    out = torch.empty((2, h, w), dtype=torch.float32, device=q.device)
    _lib.check(_lib.load().tf_fb_pyramid_level(q.data_ptr(), q.data_ptr() + H * W, 1, H, W, ctypes.byref(params),
                                               int(level), out.data_ptr(), ws.data_ptr(), nbytes, int(bool(two_pass)),
                                               _stream()), "tf_fb_pyramid_level")
    return out.cpu().numpy()


def fb_polyexp(images):
    """FarnebackPolyExp of (n, h, w) float32 level images -> (n, h, w, 5) float32 (numpy), channels in OpenCV's order."""
    I = torch.from_numpy(np.ascontiguousarray(images, dtype=np.float32)).to(_device())
    n, h, w = I.shape
    params = _lib.default_params()
    rs = int(_lib.load().tf_fb_r_stride(h, w))
    R = torch.empty((n, rs), dtype=torch.float32, device=I.device)
    _lib.check(_lib.load().tf_fb_polyexp(I.data_ptr(), n, h, w, ctypes.byref(params), R.data_ptr(), _stream()),
               "tf_fb_polyexp")
    out = torch.empty((n, h, w, 5), dtype=torch.float32, device=I.device)
    out[..., :4] = R[:, :4 * h * w].reshape(n, h, w, 4)
    out[..., 4] = R[:, 4 * h * w:5 * h * w].reshape(n, h, w)
    return out.cpu().numpy()
