"""Device activities (kernels, copies, memsets) and their counts for one ``growth_markers_device`` call and one
single-rank ``ShardedFlow.detect_growth_markers`` call on the ``growth_multi`` golden case (torch.profiler, CUDA).

    python profiles/tools/det_kernels.py [OUT.json]

Run from the root of a checkout; the package and the golden case are taken from the working directory, so running this
file from the roots of two checkouts shows whether they launch the same work."""
import collections
import json
import os
import sys

import numpy as np
import torch
from torch.autograd import DeviceType
from torch.profiler import ProfilerActivity, profile

ROOT = os.getcwd()
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests", "golden")]
import make_golden as mg  # noqa: E402
import tobac_flow_b200 as tfb  # noqa: E402
from tobac_flow_b200 import distributed as D  # noqa: E402
from tobac_flow_b200.detection import growth_markers_device  # noqa: E402

g = np.load(os.path.join(ROOT, "tests", "golden", "growth_multi.npz"))
wvd = torch.from_numpy(mg.growth_multi_case()).cuda()
fwd = torch.from_numpy(g["fwd_q256"].astype(np.float32) / 256).cuda()
bwd = torch.from_numpy(g["bwd_q256"].astype(np.float32) / 256).cuda()
dt = np.full(wvd.shape[0], 5.0)
flow = tfb.Flow(fwd, bwd)
calls = {
    "growth_markers_device": lambda: growth_markers_device(flow, wvd, dt),
    "ShardedFlow.detect_growth_markers":
        lambda: D.ShardedFlow(fwd, bwd, 0, 1).detect_growth_markers(D.make_shard(wvd, 0, 1), dt, 0),
}
result = {}
for name, call in calls.items():
    call()                                   # module loading and allocator warm-up stay out of the trace
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        call()
        torch.cuda.synchronize()
    counts = collections.Counter(e.name for e in prof.events() if e.device_type == DeviceType.CUDA)
    result[name] = dict(sorted(counts.items()))
    print(f"{name}: {sum(counts.values())} device activities")
    for k, v in result[name].items():
        print(f"  {v:4d}  {k}")
result["device"] = torch.cuda.get_device_name()
if len(sys.argv) > 1:
    with open(sys.argv[1], "w") as f:
        json.dump(result, f, indent=1)
