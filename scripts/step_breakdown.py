"""Where the time of one C2 resident step goes: event-timed step, the device time of its kernels and memory operations
(torch.profiler with CUDA activities), and the host time of the call (bmo_trace_rays inside solver.trace_rays, plus the
Python wrapper around it).  The step is bench.py's `value` leg: 2^20 rays resident in HBM, segment table not kept.

    python scripts/step_breakdown.py --out DIR [--steps 20]

Writes DIR/step_breakdown.json and DIR/step_breakdown.pt.trace.json.  Run once with BMO_HOST_PROFILE=1 for libbmo's own
host timeline on stderr.  The profiled steps are slower than bench.py's (tracing costs host time); the event-timed steps
come from a separate loop with the profiler off."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rays", type=int, default=1 << 20)
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    import torch
    from torch.profiler import ProfilerActivity, profile
    import __graft_entry__ as ge
    ge.build_libbmo()
    m = ge.load_package()
    from bmo_b200 import _lib as L
    from tests import scenes
    n = args.rays
    stream = torch.cuda.current_stream()
    L.set_stream(stream.cuda_stream, 0)
    dsys = m.upload_system(scenes.doublet_spot(m)["system"], [707e-9], device=0)
    pos, d = scenes.fibonacci_disc(n)
    pos_d, dir_d = torch.from_numpy(pos).cuda(), torch.from_numpy(d).cuda()
    lam_d = torch.zeros(n, dtype=torch.int32, device="cuda")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def step():
        res = m.trace_rays(dsys, (pos_d.data_ptr(), n), dir_d.data_ptr(), lam_d.data_ptr(), None, None, 100,
                           keep_segments=False, device_inputs=True)
        res.free()

    for _ in range(5):
        step()
    torch.cuda.synchronize()
    ev_ms, host_ms, lib_ms = [], [], []
    for _ in range(args.steps):
        flush.fill_(1)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        t0 = time.perf_counter()
        step()
        host_ms.append((time.perf_counter() - t0) * 1e3)
        e1.record(stream)
        torch.cuda.synchronize()
        ev_ms.append(e0.elapsed_time(e1))
        lib_ms.append(L.counters(0)["trace_ms"])     # libbmo's own event bracket of the call (bmo_trace_rays)
    L.counters_reset(0)
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for _ in range(args.steps):
            flush.fill_(1)
            torch.cuda.synchronize()
            step()
            torch.cuda.synchronize()
    prof.export_chrome_trace(os.path.join(args.out, "step_breakdown.pt.trace.json"))
    kernels = {}
    for e in prof.events():
        if e.device_type.name == "CUDA" and "fill" not in e.name.lower() and "elementwise" not in e.name.lower():
            k = kernels.setdefault(e.name, [0, 0.0])
            k[0] += 1
            k[1] += e.device_time_total / 1e3 if hasattr(e, "device_time_total") else e.cuda_time_total / 1e3
    per_step = {k: {"calls_per_step": v[0] / args.steps, "ms_per_step": v[1] / args.steps} for k, v in kernels.items()}
    dev_ms = sum(v["ms_per_step"] for v in per_step.values())
    c = L.counters(0)
    out = {"rays": n, "steps": args.steps, "gpu": torch.cuda.get_device_name(0),
           "event_ms_per_step_median": float(np.median(ev_ms)), "event_ms_per_step_min": float(np.min(ev_ms)),
           "lib_event_ms_per_step_median": float(np.median(lib_ms)),
           "host_ms_per_call_median": float(np.median(host_ms)),
           "device_ms_per_step_profiled": dev_ms, "device_ops": per_step,
           "launches_per_step": c["kernel_launches"] / args.steps,
           "note": "device_ops: kernels and memory operations of the library per step under the profiler (the L2 flush excluded)"}
    with open(os.path.join(args.out, "step_breakdown.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
