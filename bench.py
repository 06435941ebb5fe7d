#!/usr/bin/env python
"""Benchmark of the dense-flow hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

A *step* is one pass of the hot path over one rank's batch of synthetic input: the 288-frame, 1500 x 2500
GOES-CONUS-shaped brightness-temperature day of BASELINE.json configs[1] — forward+backward Farneback flow for
every consecutive pair (normalise, quantise, 6-level pyramid, 10 iterations per level, clamp, end rules) plus
``Flow.diff``, ``Flow.sobel`` (linear) and ``Flow.convolve`` (7-tap stack) on every frame.  With N GPUs the series
is 288*N frames, time-sharded one day per rank with NCCL point-to-point halo exchange (weak scaling).

``value``   frames/s with the inputs resident in HBM (CUDA events, max over ranks).
``e2e``     the same unit of work through the public numpy API (create_flow / Flow.diff / sobel / convolve) with the
            input in pinned host memory and every result copied back to the host inside the timed region, on a
            bounded number of frames of the same shape.
``roofline`` the dominant kernel (the fused Farneback iteration at the full-resolution level): algorithmic bytes
            (56 B per pixel-iteration; the level's first iteration also forms its initial flow from the previous level's
            result and carries the 10 B per pixel SURVEY 8d counts for that up-sampling) / its CUDA-event time measured
            live during the timed steps.
``cpu_baseline`` the reference's CPU implementation of the same unit of work (OpenCV Farneback + cv2.remap through
            the oracle's restatement of the reference's Python) timed on this box's host cores on a bounded sample.

``--impl reference`` times only that CPU implementation, with all host cores (a process pool over independent
frames of work), and prints the same JSON line with "impl": "reference".

``--dump-outputs DIR`` writes what the last timed step returned (rank 0's shard with N GPUs) to ``DIR/<name>.npy``:
``forward_flow``, ``backward_flow``, ``diff``, ``convolve`` in float32 and ``sobel`` in float64.  An array of more than
2**20 elements is stored as the 2**20 elements at fixed, seeded flat positions (sorted).  The operator results are NaN
where an input pixel is NaN or a tap falls outside the series; such elements are written as 0 in ``<name>.npy`` and as 1
in ``<name>_nan.npy`` (0 elsewhere, same dtype and shape), so every file is finite.  The files (48 MiB at most) of two
builds run with the same arguments can be compared element for element: the synthetic input is seeded.
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "frames/s (fwd+bwd flow + flow-convolve), GOES CONUS 1500x2500"
UNIT = "frames/s"


# BASELINE.json configs: (frames, H, W, how the frames map to ranks, name)
#   "per_rank": every rank gets `frames` frames (weak scaling: the series is frames * N long)
#   "split":    the `frames`-frame series is split over the ranks (the 144-frame full-disk day does not fit one GPU
#               together with all three operator outputs; at N = 1 the first `single` frames are run)
CONFIGS = {
    "c1": dict(frames=10, H=100, W=100, mode="per_rank", name="tests/test_flow.py-style synthetic stack 10x100x100"),
    "c2": dict(frames=288, H=1500, W=2500, mode="per_rank", name="GOES-16 ABI CONUS-shaped synthetic BT 288 frames x 1500x2500 (1 day, 5-min)"),
    "c3": dict(frames=1440, H=500, W=500, mode="per_rank", name="ABI mesoscale-shaped 1440 frames x 500x500 (1-min cadence)"),
    "c4": dict(frames=96, H=3712, W=3712, mode="per_rank", name="SEVIRI full-disk-shaped 96 frames x 3712x3712 (15-min)"),
    "c5": dict(frames=144, H=5424, W=5424, mode="split", single=48, name="GOES ABI full-disk-shaped 144 frames x 5424x5424 (10-min), time-sharded"),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS),
                    help="BASELINE.json configs[i-1]; c2 (the metric's GOES-CONUS day) is the default")
    ap.add_argument("--frames", type=int, default=None, help="frames per rank (overrides the config's)")
    ap.add_argument("--height", type=int, default=None)
    ap.add_argument("--width", type=int, default=None)
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling sub-record at N > 1")
    ap.add_argument("--e2e-frames", type=int, default=288, help="frames per end-to-end step (bounded by host memory)")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-detection", action="store_true", help="skip the detect_growth_markers extra (not the metric)")
    ap.add_argument("--detection-frames", type=int, default=48)
    ap.add_argument("--ref-workers", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step to DIR/<name>.npy (sampled when large)")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the CUDA path; --impl reference has none")
    cfg = CONFIGS[a.config]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if a.frames is None:
        a.frames = cfg["frames"] if cfg["mode"] == "per_rank" else (cfg["single"] if world == 1 else cfg["frames"] // world)
    a.height = a.height or cfg["H"]
    a.width = a.width or cfg["W"]
    a.config_name = cfg["name"]
    a.config_mode = cfg["mode"]
    return a


def level_sizes(H, W):
    """OpenCV's level plan (coarsest first) — host arithmetic only."""
    k, scale = 0, 1.0
    while k < 5:
        scale *= 0.5
        if W * scale < 32 or H * scale < 32:
            break
        k += 1
    out = []
    for kk in range(k, -1, -1):
        s = 0.5 ** kk
        out.append((int(np.rint(H * s)), int(np.rint(W * s))))
    return out


def algorithmic_bytes_per_frame(H, W):
    """SURVEY.md §8(d): B_frame = (140 + 2L) N + 1196 S."""
    lv = level_sizes(H, W)
    N = H * W
    S = sum(h * w for h, w in lv)
    return (140 + 2 * len(lv)) * N + 1196 * S, len(lv), S


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


DUMP_ELEMENTS = 1 << 20


def dump_outputs(out_dir, arrays):
    """Write each device tensor to out_dir/<name>.npy: whole when it has at most DUMP_ELEMENTS elements, otherwise the
    DUMP_ELEMENTS elements at flat positions drawn without replacement by a generator seeded with 0.  NaN elements are
    written as 0 there and marked with 1 in out_dir/<name>_nan.npy."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        if t.numel() > DUMP_ELEMENTS:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), DUMP_ELEMENTS, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        a = t.cpu().numpy()
        nan = np.isnan(a)
        np.save(os.path.join(out_dir, name + ".npy"), np.where(nan, a.dtype.type(0), a))
        np.save(os.path.join(out_dir, name + "_nan.npy"), nan.astype(a.dtype))


# ----------------------------------------------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------------------------------------------
class ClockSampler:
    # One looping nvidia-smi, started BEFORE the warm-up steps: a fresh NVML client attaching to the device stalls kernel
    # launches for some milliseconds, which showed up as 6-30 ms idle gaps inside the timed region when it was started
    # there.  Only the samples taken between mark_begin() and mark_end() (the timed region) are reported.
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.path = tempfile.mktemp(suffix=".csv")
        self.proc = None
        self.gpu_index = gpu_index
        self.t0 = self.t1 = None

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def start(self):
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.gpu_index)], stdout=self.f,
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        import datetime
        for line in open(self.path):
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 9:
                continue
            if self.t0 is not None and self.t1 is not None:
                try:
                    ts = datetime.datetime.strptime(parts[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                    if ts < self.t0 - 0.05 or ts > self.t1 + 0.05:
                        continue
                except ValueError:
                    pass
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for n, v in zip(names, parts[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        try:
            os.unlink(self.path)
        except OSError:
            pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------------------
# CPU reference arm (the only place outside tests/smoke where oracle/ is executed)
# ----------------------------------------------------------------------------------------------------------------
_CPU_FRAME_CACHE = {}


def _cpu_frames(H, W, t_centre, seed=1234):
    """Three consecutive synthetic frames (cached per worker process so input generation is not timed twice)."""
    key = (H, W, t_centre, seed)
    if key not in _CPU_FRAME_CACHE:
        from tobac_flow_b200 import synthetic
        base = synthetic.base_field(H, W, seed)
        T = 288
        cores = synthetic.core_table(T, H, W, seed)
        plan = synthetic.nan_plan(T, H, W, seed)
        _CPU_FRAME_CACHE.clear()
        _CPU_FRAME_CACHE[key] = np.stack([synthetic.bt_frame(base, t, cores, plan, T)
                                          for t in (t_centre - 1, t_centre, t_centre + 1)])
    return _CPU_FRAME_CACHE[key]


def _cpu_prime(args):
    H, W, t_centre, _ = args
    _cpu_frames(H, W, t_centre)
    time.sleep(0.2)   # keep this worker busy so every worker of the pool receives one priming job
    return 0


def _cpu_frame_of_work(args):
    """One frame of work on the CPU exactly as the reference computes it: one pair flow (fwd+bwd) + the three
    stencils on the middle frame of a 3-frame window."""
    H, W, t_centre, threads = args
    from oracle import flow_ops as ops
    backend = "cv2" if ops.have_cv2() else "numpy"
    if backend == "cv2":
        import cv2
        cv2.setNumThreads(threads)
    bt = _cpu_frames(H, W, t_centre)
    t0 = time.perf_counter()
    fwd, bwd = ops.create_flow(bt[:2], backend=backend)              # one pair, both directions
    t1 = time.perf_counter()
    # the three stencils on the middle frame only (convolve.py's per-step body), fed with the pair's fields
    ff, bf = fwd[1], bwd[1]
    s_diff = np.zeros((3, 3, 3)); s_diff[:, 1, 1] = 1
    s_cross = np.zeros((3, 3, 3)); s_cross[1, 1, :] = s_cross[1, :, 1] = s_cross[:, 1, 1] = 1
    d = ops.diff_reducer(ops.tap_stack(bt[0], bt[1], bt[2], ff, bf, s_diff, "linear", np.float32, np.nan, backend))
    s = ops.sobel_reducer(None)(ops.tap_stack(bt[0], bt[1], bt[2], ff, bf, np.ones((3, 3, 3)), "linear", np.float64,
                                              np.nan, backend))
    c = ops.tap_stack(bt[0], bt[1], bt[2], ff, bf, s_cross, "linear", np.float32, np.nan, backend)
    t2 = time.perf_counter()
    return (t1 - t0), (t2 - t1), float(np.nansum(d) + np.nansum(s) + np.nansum(c))


def cpu_baseline_single(H, W):
    from oracle import flow_ops as ops
    import multiprocessing as mp
    threads = os.cpu_count() or 1
    t_pair, t_stencil, _ = _cpu_frame_of_work((H, W, 10, -1))
    backend = "cv2" if ops.have_cv2() else "numpy"
    cores = 1
    if backend == "cv2":
        import cv2
        cores = cv2.getNumThreads()
    return {
        "value": 1.0 / (t_pair + t_stencil), "unit": UNIT, "cores": cores, "kind": "port",
        "sample": (f"1 pair (fwd+bwd Farneback) + diff/sobel/convolve on 1 frame of {H}x{W}; reference Python "
                   f"restated in oracle/flow_ops.py calling {'OpenCV ' + __import__('cv2').__version__ if backend == 'cv2' else 'the numpy restatement'}"
                   f"; single process as the reference runs it; pair {t_pair:.2f} s + stencils {t_stencil:.2f} s per frame"),
        "host_cpus": threads,
    }


def run_reference(args):
    """--impl reference: the CPU implementation with all host cores; each step = one frame of work per worker."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    from oracle import flow_ops as ops
    H, W = args.height, args.width
    ncpu = os.cpu_count() or 1
    try:
        import psutil
        avail = psutil.virtual_memory().available
    except Exception:
        avail = 64 << 30
    per_worker = 40 * H * W * 8 + (1 << 30)      # tap stacks + temporaries of the 27-tap float64 sobel
    workers = args.ref_workers or max(1, min(ncpu, int(avail * 0.6 // per_worker), 64))
    ctx = mp.get_context("spawn")
    times = []
    with ctx.Pool(workers) as pool:
        jobs = [(H, W, 10, 1) for i in range(workers)]
        pool.map(_cpu_prime, jobs, chunksize=1)     # untimed: synthesize (and cache) the input frames in every worker
        for step in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            pool.map(_cpu_frame_of_work, jobs)
            dt = time.perf_counter() - t0
            if step >= args.warmup:
                times.append(dt)
    ms = 1e3 * float(np.mean(times))
    value = workers / (ms / 1e3)
    backend = "cv2" if ops.have_cv2() else "numpy"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"GOES CONUS-shaped synthetic BT {H}x{W}: per step, {workers} independent frames of work "
                               "(1 pair fwd+bwd Farneback + diff + sobel + 7-tap convolve each) on the host CPU"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": workers, "kind": "port",
                         "sample": f"{workers} worker processes x 1 frame of work per step, cv2 threads = 1 per worker, "
                                   f"backend {backend}"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------------------------
# the B200 arm
# ----------------------------------------------------------------------------------------------------------------
def _parse_cpulist(text):
    cpus = set()
    for part in text.strip().split(","):
        if not part:
            continue
        a, _, b = part.partition("-")
        cpus.update(range(int(a), int(b or a) + 1))
    return cpus


def pin_to_numa(local_rank, n_local):
    """Pin this rank's host threads to cores of its GPU's NUMA node (the end-to-end path is host-memory / PCIe bound);
    ranks that share a core set split it.  Returns a short description for the bench line."""
    try:
        import torch
        allowed = os.sched_getaffinity(0)
        pr = torch.cuda.get_device_properties(local_rank)
        node = -1
        bus = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        path = f"/sys/bus/pci/devices/{bus}/numa_node"
        if os.path.exists(path):
            node = int(open(path).read().strip())
        local = set(allowed)
        if node >= 0 and os.path.exists(f"/sys/devices/system/node/node{node}/cpulist"):
            cand = _parse_cpulist(open(f"/sys/devices/system/node/node{node}/cpulist").read()) & allowed
            if cand:
                local = cand
        cpus = sorted(local)
        # ranks with the same candidate set take disjoint slices of it
        share = max(1, n_local)
        if len(cpus) >= 2 * share:
            per = len(cpus) // share
            cpus = cpus[local_rank % share * per:(local_rank % share + 1) * per]
        os.sched_setaffinity(0, cpus)
        return {"numa_node": node, "cpus": len(cpus), "allowed": len(allowed)}
    except Exception as e:  # pragma: no cover
        return {"numa_node": None, "error": str(e)[:80]}


def run_b200(args):
    import torch
    import torch.distributed as dist
    from tobac_flow_b200 import _lib, synthetic
    from tobac_flow_b200 import distributed as D
    import tobac_flow_b200 as tfb

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.load()
    affinity0 = os.sched_getaffinity(0)
    pinned = pin_to_numa(local_rank, int(os.environ.get("LOCAL_WORLD_SIZE", str(world))))

    T, H, W = args.frames, args.height, args.width
    N = H * W
    # ---- synthetic input, resident in HBM: this rank's frames of the (T * world)-frame series ----------------------
    base = synthetic.base_field(H, W, 1234)
    base_t = torch.as_tensor(base, device=dev)

    def series(T_total):
        return synthetic.core_table(T_total, H, W, 1234), synthetic.nan_plan(T_total, H, W, 1234)

    def fill_shard(sh, T_loc, t0, T_total, cores_, plan_):
        for i in range(T_loc):
            sh.buf[1 + i] = synthetic.bt_frame(base_t, t0 + i, cores_, plan_, T_total)
        sh.buf[0] = float("nan")
        sh.buf[-1] = float("nan")

    cores, plan = series(T * world)
    shard = D.Shard(torch.empty((T + 2, H, W), dtype=torch.float32, device=dev), rank, world)
    fill_shard(shard, T, rank * T, T * world, cores, plan)

    fwd = torch.empty((T, H, W, 2), dtype=torch.float32, device=dev)
    bwd = torch.empty((T + 1, H, W, 2), dtype=torch.float32, device=dev)
    out_diff = torch.empty((T, H, W), dtype=torch.float32, device=dev)
    out_sobel = torch.empty((T, H, W), dtype=torch.float64, device=dev)
    out_conv = torch.empty((7, T, H, W), dtype=torch.float32, device=dev)
    s_diff = np.zeros((3, 3, 3)); s_diff[:, 1, 1] = 1
    s_full = np.ones((3, 3, 3))
    s_cross = np.zeros((3, 3, 3)); s_cross[1, 1, :] = s_cross[1, :, 1] = s_cross[:, 1, 1] = 1

    def run_step(sh, fwd_, bwd_, od, os_, oc):
        fl = D.create_flow_sharded(sh, max_value=20, fwd=fwd_, bwd=bwd_)           # halo exchange inside (side stream)
        fl.convolve(sh, s_diff, reducer=_lib.TF_RED_DIFF, exchange=False, out=od)
        fl.convolve(sh, s_full, dtype=None, reducer=_lib.TF_RED_SOBEL, exchange=False, out=os_)
        fl.convolve(sh, s_cross, reducer=_lib.TF_RED_NONE, exchange=False, out=oc)
        return fl

    def step():
        return run_step(shard, fwd, bwd, out_diff, out_sobel, out_conv)

    def same(a, b):
        return bool(((a == b) | (torch.isnan(a) & torch.isnan(b))).all().item())

    def sharded_parity(sh, fwd_, bwd_, od, os_, oc, t0, T_loc, T_total, cores_, plan_):
        """Every rank recomputes, unsharded and locally, the 4-frame window around each of its shard edges (the inputs
        are synthetic, so the neighbour's frames can be generated here) and compares the flow fields and the three
        operator results of its edge frame bit for bit with what the sharded run (NCCL halos) produced."""
        ok = True
        edges = []
        if sh.has_prev and t0 >= 2 and T_loc >= 2:
            edges.append((t0, [t0 - 2, t0 - 1, t0, t0 + 1], 2))
        if sh.has_next and t0 + T_loc + 1 < T_total and T_loc >= 2:
            tg = t0 + T_loc - 1
            edges.append((tg, [tg - 1, tg, tg + 1, tg + 2], 1))
        for tg, win, k in edges:
            fr = torch.stack([synthetic.bt_frame(base_t, t, cores_, plan_, T_total) for t in win])
            fl = tfb.create_flow(fr)
            d, sb, cv = fl.diff(fr), fl.sobel(fr), fl.convolve(fr)
            li = tg - t0
            ok = (ok and same(fl.forward_flow_device[k], fwd_[li]) and same(fl.backward_flow_device[k], bwd_[li])
                  and same(d[k], od[li]) and same(sb[k], os_[li]) and same(cv[:, k], oc[:, li]))
        if world > 1:
            t = torch.tensor([1 if ok else 0], device=dev, dtype=torch.int32)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            ok = bool(t.item())
        return ok

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        step()
    barrier()
    _lib.profile_reset()
    _lib.profile_enable(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # The timed region starts with an empty launch queue, so a host pause before the first launches is fully exposed
    # (6-50 ms gaps showed up in some runs): no cyclic garbage collection inside the region.
    gc.collect()
    gc.disable()
    barrier()
    sampler.mark_begin()
    e0.record()
    for _ in range(args.steps):
        fl = step()
    e1.record()
    barrier()
    sampler.mark_end()
    gc.enable()
    elapsed_ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None
    prof = _lib.profile_read()
    _lib.profile_enable(False)
    if world > 1:
        t = torch.tensor([elapsed_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms = float(t.item())
    ms_per_step = elapsed_ms / args.steps
    value = T * world / (ms_per_step / 1e3)
    if args.dump_outputs and rank == 0:
        # before the strong-scaling run below reuses the buffers
        dump_outputs(args.dump_outputs, {"forward_flow": fl.fwd, "backward_flow": fl.bwd, "diff": out_diff,
                                         "sobel": out_sobel, "convolve": out_conv})

    # ---- multi-GPU evidence: the sharded result equals a local unsharded recomputation at the shard edges; the same
    # day split over the ranks (strong scaling) ------------------------------------------------------------------------
    parity_ok = strong = None
    if world > 1:
        parity_ok = sharded_parity(shard, fwd, bwd, out_diff, out_sobel, out_conv, rank * T, T, T * world, cores, plan)
        if not args.no_strong and args.config_mode == "per_rank" and T % world == 0 and T // world >= 2:
            Ts = T // world
            cores_s, plan_s = series(T)
            sh_s = D.Shard(shard.buf[:Ts + 2], rank, world)
            fill_shard(sh_s, Ts, rank * Ts, T, cores_s, plan_s)
            oc_s = out_conv.view(-1)[:7 * Ts * N].view(7, Ts, H, W)
            bufs = (sh_s, fwd[:Ts], bwd[:Ts + 1], out_diff[:Ts], out_sobel[:Ts], oc_s)
            for _ in range(max(1, args.warmup)):
                run_step(*bufs)
            barrier()
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s0.record()
            for _ in range(args.steps):
                run_step(*bufs)
            s1.record()
            barrier()
            t = torch.tensor([s0.elapsed_time(s1)], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            s_ms = float(t.item()) / args.steps
            s_ok = sharded_parity(*bufs, rank * Ts, Ts, T, cores_s, plan_s)
            strong = {"scaling": "strong", "frames": T, "frames_per_gpu": Ts, "ms_per_step": s_ms,
                      "value": T / (s_ms / 1e3), "unit": UNIT, "sharded_parity": s_ok,
                      "note": f"the single {T}-frame series time-sharded over {world} GPUs (NCCL p2p halos on a side stream)"}
            # restore this rank's frames of the weak-scaling series for the end-to-end / detection extras below
            fill_shard(shard, T, rank * T, T * world, cores, plan)

    # ---- roofline of the dominant kernel ---------------------------------------------------------------------------
    peak, peak_src = measured_peak()
    dom = prof["fb_iter_fullres"]
    achieved = dom["bytes"] / 1e9 / (dom["ms"] / 1e3) if dom["ms"] > 0 else 0.0
    # measured DRAM bytes per launch of that kernel from the committed ncu capture (profiles/traffic.json), scaled to
    # this run's average launch size; only meaningful at the captured frame size
    traffic = None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    bytes_per_launch = dom["bytes"] / max(dom["launches"], 1)
    if os.path.exists(tp) and (H, W) == (1500, 2500):
        try:
            tj = json.load(open(tp))
            traffic = tj["fb_iter_fullres_dram_bytes_per_launch"] * bytes_per_launch / tj["algorithmic_bytes_of_captured_launch"]
        except Exception:
            traffic = None
    b_frame, L, S = algorithmic_bytes_per_frame(H, W)
    total_kernel_ms = sum(v["ms"] for v in prof.values())
    launches = int(sum(v["launches"] for v in prof.values()))
    roofline = {
        "bound": "hbm", "kernel": "fb_iter_v3_kernel (fused Farneback iteration: TMA-staged, tensor-memory ring, packed fp32) at the full-resolution level", "achieved": achieved, "peak": peak,
        "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
        "bytes_per_launch": bytes_per_launch, "avg_launch_ms": dom["ms"] / max(dom["launches"], 1),
        "share_of_step_kernel_time": dom["ms"] / total_kernel_ms if total_kernel_ms else None,
        "whole_step": {"algorithmic_bytes_per_frame": b_frame, "achieved": value / world * b_frame / 1e9,
                       "frac": value / world * b_frame / 1e9 / peak},
        "per_class": {k: {"ms_per_step": v["ms"] / args.steps, "GBps": (v["bytes"] / 1e9 / (v["ms"] / 1e3)) if v["ms"] > 0 else None,
                          "launches_per_step": v["launches"] / args.steps} for k, v in prof.items() if v["launches"]},
    }

    # ---- end to end through the public numpy API with host buffers ---------------------------------------------------
    e2e = None
    if not args.no_e2e:
        # every result of a step lands in page-locked host memory (164 MB per CONUS frame): keep all ranks of the box
        # together within half of the available RAM
        try:
            import psutil
            avail = psutil.virtual_memory().available
        except Exception:
            avail = 64 << 30
        n_local = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
        per_frame = N * (4 + 4 + 8 + 28) + 1
        Te = max(4, min(args.e2e_frames, T, int(avail * 0.5 / n_local / per_frame)))
        host_in = torch.empty((Te, H, W), dtype=torch.float32, pin_memory=True)
        host_in.copy_(shard.buf[1:1 + Te])
        torch.cuda.synchronize()
        host_np = host_in.numpy()

        def e2e_step(stack_first=True):
            fl = tfb.create_flow(host_np)                  # H2D inside; returns with the flow kernels queued
            if stack_first:
                c = fl.convolve(host_np)                   # D2H inside; the largest result first: it streams back while
                s = fl.sobel(host_np)                      # the later pairs are still in the iteration kernels
                d = fl.diff(host_np)
            else:
                d = fl.diff(host_np)
                s = fl.sobel(host_np)
                c = fl.convolve(host_np)
            return float(d[0, 0, 0]) + float(s[0, 0, 0]) + float(c[0, 0, 0, 0])

        def e2e_time(stack_first):
            e2e_step(stack_first)
            barrier()
            t0 = time.perf_counter()
            for _ in range(args.e2e_steps):
                e2e_step(stack_first)
            barrier()
            dt = (time.perf_counter() - t0) / args.e2e_steps
            if world > 1:
                t = torch.tensor([dt], device=dev, dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                dt = float(t.item())
            return dt

        dt_alt = e2e_time(False)
        dt = e2e_time(True)
        e2e = {"value": Te * world / dt, "unit": UNIT, "h2d_bytes_per_step": Te * N * 4,
               "d2h_bytes_per_step": Te * N * (4 + 8 + 28), "frames_per_step": Te,
               "order": "create_flow, convolve, sobel, diff",
               "value_diff_sobel_convolve_order": Te * world / dt_alt,
               "note": "create_flow + convolve + sobel + diff via the numpy API; input pinned; create_flow uploads the "
                       "frames once per step, queues the flow kernels batch by batch and returns; the three operators "
                       "reuse the device copy of the frames (operand cache keyed on the host buffer) and start on the "
                       "first frames while later pairs are still being computed (per-batch events, operator kernels on a "
                       "high-priority stream); every operator result is copied back to a host array inside the timed "
                       "region, and every call returns only when its result is complete on the host; flows stay on the "
                       "device (Flow keeps them resident).  PCIe-bound: 150 MB of results per frame.  Calling the "
                       "operator with the largest result first hides the flow computation behind its download; "
                       "value_diff_sobel_convolve_order is the same step with the small results first"}

    # ---- extra (not the metric): the device-resident growth-marker detection on this rank's first frames ---------------
    detection = None
    if not args.no_detection and rank == 0:
        from tobac_flow_b200.detection import growth_markers_device
        Td = min(args.detection_frames, T)
        wvd = synthetic.wvd_from_bt(shard.buf[1:1 + Td]).float().contiguous()
        fl_d = tfb.Flow(fwd[:Td], bwd[:Td])
        dtm = np.full(Td, 5.0)
        growth_markers_device(fl_d, wvd, dtm)
        torch.cuda.synchronize()
        d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        d0.record()
        for _ in range(3):
            r = growth_markers_device(fl_d, wvd, dtm)
        d1.record()
        torch.cuda.synchronize()
        dms = d0.elapsed_time(d1) / 3
        detection = {"what": "detect_growth_markers on device tensors (diff, /dt, 3-frame nanmean, grey opening x "
                             "curvature filter, thresholds, opening, flow_label, label filters), flow given",
                     "frames": Td, "ms": dms, "frames_per_s": Td / (dms / 1e3),
                     "flat_labels": int(r["flat"].max()), "linked_labels": int(r["linked"].max())}
        del wvd, r

    # ---- CPU baseline (rank 0, N = 1 only) --------------------------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            os.sched_setaffinity(0, affinity0)      # the CPU baseline gets every host core the process may use
            cpu = cpu_baseline_single(H, W)
        except Exception as e:  # pragma: no cover
            cpu = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": f"failed: {e}"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{args.config}: {args.config_name}; {T} frames x {H}x{W} per GPU "
                                   f"({T * world} frames time-sharded over {world} GPU(s), NCCL p2p halos): fwd+bwd "
                                   "Farneback per pair + Flow.diff + Flow.sobel(linear, f64) + Flow.convolve(7-tap stack)",
                       "baseline_config": args.config, "frames_per_gpu": T, "height": H, "width": W, "pyramid_levels": L,
                       "l2": f"inputs ({T * N * 4 / 1e9:.2f} GB of frames per GPU) "
                             + ("are far larger than the 126 MB L2; no explicit flush" if T * N * 4 > 4 * (126 << 20)
                                else "and working set are L2-sized: see roofline note"),
                       "host_pinning": pinned},
            "clocks": clocks, "e2e": e2e, "detection": detection, "gpu_launches": launches // max(args.steps, 1) * args.steps,
            "roofline": roofline, "cpu_baseline": cpu,
        }
        if world > 1:
            line["sharded_parity"] = parity_ok
            line["strong"] = strong
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
