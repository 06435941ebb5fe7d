"""Frames/s of create_flow with FarnebackOpticalFlow settings, the general iteration kernel's time, and cv2 on the host.

usage: python profiles/tools/fb_config_time.py [T] [H] [W] [out.json]      (default 288 1500 2500)

Prints one JSON line.  Per setting: frames/s of create_flow on device input (frames already in HBM, timed with a device
synchronise) and on numpy input end to end (upload, flow, and the vectors back on the host); the full-resolution
iterations' device time from the library's CUDA events (tf_profile_*, class fb_iter_fullres) against its 56 B per
pixel-iteration model at 7.7 TB/s; cv2.FarnebackOpticalFlow with the same settings on the host cores (both directions
of a few pairs); and the card's name and power limit.
"""
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import tobac_flow_b200 as tfb  # noqa: E402
from oracle import flow_ops  # noqa: E402
from tobac_flow_b200 import _lib, synthetic  # noqa: E402

HBM_BYTES_PER_S = 7.7e12
SETTINGS = {
    "default": dict(),
    "legacy_gauss16_iters3": dict(flags=256, win_size=16, num_iters=3),
    "box21": dict(win_size=21),
    "poly_n7": dict(poly_n=7, poly_sigma=1.5),
    "pyr_scale07": dict(pyr_scale=0.7),
}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
        return dict(name=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:  # pragma: no cover
        return dict(name=torch.cuda.get_device_name(0), power_limit=f"unknown ({e})")


def timed(fn, reps=2):
    fn()                          # warm-up of every shape the timed calls use
    torch.cuda.synchronize()
    best = None
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return best


def main():
    T = int(sys.argv[1]) if len(sys.argv) > 1 else 288
    H = int(sys.argv[2]) if len(sys.argv) > 2 else 1500
    W = int(sys.argv[3]) if len(sys.argv) > 3 else 2500
    out_path = sys.argv[4] if len(sys.argv) > 4 else None
    assert torch.cuda.is_available(), "fb_config_time.py measures the GPU: no CUDA device"
    bt_dev = synthetic.bt_sequence(T, H, W, seed=1234, nans=True, device="cuda")
    bt_host = bt_dev.cpu().numpy()
    res = dict(T=T, H=H, W=W, card=card())
    import cv2
    n_cv = 2
    qs = [flow_ops.pair_to_u8(bt_host[i], bt_host[i + 1]) for i in range(n_cv)]
    for name, kw in SETTINGS.items():
        model = tfb.FarnebackOpticalFlow(**kw)
        t_dev = timed(lambda: tfb.create_flow(bt_dev, model=model))
        t_np = timed(lambda: tfb.create_flow(bt_host, model=model).forward_flow)
        _lib.profile_reset()
        _lib.profile_enable(True)
        tfb.create_flow(bt_dev, model=model)
        torch.cuda.synchronize()
        prof = _lib.profile_read()["fb_iter_fullres"]
        _lib.profile_enable(False)
        t0 = time.perf_counter()
        for q0, q1 in qs:
            for a, b in ((q0, q1), (q1, q0)):
                cv2.FarnebackOpticalFlow_create(model.num_levels, model.pyr_scale, False, model.win_size,
                                                model.num_iters, model.poly_n, model.poly_sigma,
                                                model.flags).calc(a, b, None)
        t_cv = (time.perf_counter() - t0) / n_cv
        res[name] = dict(settings=repr(model), device_frames_per_s=T / t_dev, numpy_e2e_frames_per_s=T / t_np,
                         device_ms=1e3 * t_dev,
                         fullres_iter_ms=prof["ms"], fullres_iter_launches=prof["launches"],
                         fullres_iter_model_bytes=prof["bytes"],
                         fullres_iter_model_fraction=(prof["bytes"] / HBM_BYTES_PER_S) / (prof["ms"] * 1e-3)
                         if prof["ms"] > 0 else None,
                         cv2_host_frames_per_s=1.0 / t_cv, cv2_threads=cv2.getNumThreads(), cpus=os.cpu_count())
    line = json.dumps(res)
    print(line)
    if out_path:
        with open(out_path, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
