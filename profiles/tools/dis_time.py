"""Frames/s of create_flow with the DIS model (FAST, MEDIUM) next to Farneback and cv2 DIS on the host cores.

usage: python profiles/tools/dis_time.py [T] [H] [W] [out.json]      (default 288 1500 2500)

Prints one JSON line: per configuration the frames/s of create_flow on device input (frames already in HBM, timed
with a device synchronise) and on numpy input end to end (upload, flow, and the vectors back on the host), the
fraction of the byte floor (u8 pair in plus 2 x 8 N bytes of flow out per pair at 7.7 TB/s) the device-input time
reaches, cv2.DISOpticalFlow on the host cores (both directions of a few pairs), and the card name and power limit.
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
from tobac_flow_b200 import synthetic  # noqa: E402

HBM_BYTES_PER_S = 7.7e12


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
    assert torch.cuda.is_available(), "dis_time.py measures the GPU: no CUDA device"
    bt_dev = synthetic.bt_sequence(T, H, W, seed=1234, nans=True, device="cuda")
    bt_host = bt_dev.cpu().numpy()
    floor_s = (T - 1) * (2 * H * W + 2 * 8 * H * W) / HBM_BYTES_PER_S
    res = dict(T=T, H=H, W=W, card=card(), byte_floor_ms=1e3 * floor_s)
    models = {"dis_fast": tfb.DISOpticalFlow(1), "dis_medium": tfb.DISOpticalFlow(2), "farneback": "Farneback"}
    for name, model in models.items():
        t_dev = timed(lambda: tfb.create_flow(bt_dev, model=model))
        t_np = timed(lambda: tfb.create_flow(bt_host, model=model).forward_flow)
        res[name] = dict(device_frames_per_s=T / t_dev, numpy_e2e_frames_per_s=T / t_np, device_ms=1e3 * t_dev,
                         byte_floor_fraction=floor_s / t_dev)
    import cv2
    n = 3
    for preset, name in ((1, "cv2_dis_fast"), (2, "cv2_dis_medium")):
        m = cv2.DISOpticalFlow_create(preset)
        qs = [flow_ops.pair_to_u8(bt_host[i], bt_host[i + 1]) for i in range(n)]
        t0 = time.perf_counter()
        for q0, q1 in qs:
            cv2.DISOpticalFlow_create(preset).calc(q0, q1, None)
            cv2.DISOpticalFlow_create(preset).calc(q1, q0, None)
        dt = (time.perf_counter() - t0) / n
        res[name] = dict(frames_per_s=1.0 / dt, threads=cv2.getNumThreads(), cpus=os.cpu_count())
        del m
    line = json.dumps(res)
    print(line)
    if out_path:
        with open(out_path, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
