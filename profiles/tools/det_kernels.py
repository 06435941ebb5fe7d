"""Device activities (kernels, copies, memsets) and their counts for one ``growth_markers_device`` call, one
single-rank ``ShardedFlow.detect_growth_markers`` call and numpy-input calls of ``detect_growth_markers``, ``flow_label``
and ``filter_labels_by_length_and_mask`` on the ``growth_multi`` golden case (torch.profiler, CUDA); the bytes of each
kind of copy are listed with the copies.

    python profiles/tools/det_kernels.py [OUT.json]

Run from the root of a checkout; the package and the golden case are taken from the working directory, so running this
file from the roots of two checkouts shows whether they launch the same work."""
import collections
import json
import os
import sys
import tempfile

import numpy as np
import torch
from torch.autograd import DeviceType
from torch.profiler import ProfilerActivity, profile

ROOT = os.getcwd()
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests", "golden")]
import make_golden as mg  # noqa: E402
import pandas as pd  # noqa: E402
import refshim  # noqa: E402
import tobac_flow_b200 as tfb  # noqa: E402
from tobac_flow_b200 import analysis  # noqa: E402
from tobac_flow_b200 import distributed as D  # noqa: E402
from tobac_flow_b200.detection import detect_growth_markers, growth_markers_device  # noqa: E402
from tobac_flow_b200.label import flow_label  # noqa: E402

g = np.load(os.path.join(ROOT, "tests", "golden", "growth_multi.npz"))
wvd = torch.from_numpy(mg.growth_multi_case()).cuda()
fwd = torch.from_numpy(g["fwd_q256"].astype(np.float32) / 256).cuda()
bwd = torch.from_numpy(g["bwd_q256"].astype(np.float32) / 256).cuda()
dt = np.full(wvd.shape[0], 5.0)
flow = tfb.Flow(fwd, bwd)
wvd_np = mg.growth_multi_case()
t = pd.date_range("2020-01-01", periods=wvd_np.shape[0], freq="5min")
wvd_da = refshim.DataArray(wvd_np, coords={"t": t}, dims=("t", "y", "x"), t=t)
linked = g["linked"].astype(np.int32)
calls = {
    "growth_markers_device": lambda: growth_markers_device(flow, wvd, dt),
    "ShardedFlow.detect_growth_markers":
        lambda: D.ShardedFlow(fwd, bwd, 0, 1).detect_growth_markers(D.make_shard(wvd, 0, 1), dt, 0),
    "detect_growth_markers(numpy)": lambda: detect_growth_markers(flow, wvd_da),
    "flow_label(numpy float32 mask)": lambda: flow_label(flow, (wvd_np > -10).astype(np.float32)),
    "filter_labels_by_length_and_mask(numpy, bool mask)":
        lambda: analysis.filter_labels_by_length_and_mask(linked, wvd_np > -10, 3),
    "filter_labels_by_length_and_mask(numpy, float32 mask)":
        lambda: analysis.filter_labels_by_length_and_mask(linked, (wvd_np > -10).astype(np.float32), 3),
}
result = {}
for name, call in calls.items():
    call()                                   # module loading and allocator warm-up stay out of the trace
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        call()
        torch.cuda.synchronize()
    counts = collections.Counter(e.name for e in prof.events() if e.device_type == DeviceType.CUDA)
    copy_bytes = collections.Counter()
    with tempfile.TemporaryDirectory() as tmp:
        prof.export_chrome_trace(os.path.join(tmp, "trace.json"))
        with open(os.path.join(tmp, "trace.json")) as f:
            for ev in json.load(f)["traceEvents"]:
                if ev.get("cat") == "gpu_memcpy":
                    copy_bytes[ev["name"]] += int(ev.get("args", {}).get("bytes", 0))
    result[name] = dict(sorted(counts.items()))
    result[name + " copy bytes"] = dict(sorted(copy_bytes.items()))
    print(f"{name}: {sum(counts.values())} device activities")
    for k, v in result[name].items():
        print(f"  {v:4d}  {k}" + (f"  ({copy_bytes[k]} bytes)" if k in copy_bytes else ""))
result["device"] = torch.cuda.get_device_name()
if len(sys.argv) > 1:
    with open(sys.argv[1], "w") as f:
        json.dump(result, f, indent=1)
