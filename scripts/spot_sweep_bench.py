"""Through-focus spot-diagram sweep of C2 on one GPU: P one-pose solves against one pose sweep.

The Spotdetector of the C2 doublet (AC254-150-AB, 707 nm, UniformDiscSource 20 mm) is swept along the optical axis over
+-2 mm around its C2 position.  Both legs move it with the device kinematics (KinProgram.translate3d_), so pose p of the
two legs is the same table to the bit:

  (a) P one-pose solves: bmo_source_create; then per pose bmo_system_apply_poses (1 pose) -> bmo_trace_rays(BMO_INPUT_DEVICE)
      -> bmo_spot_stats with a histogram.  One pose per trace, so the tables are staged and the persistent kernel can run.
  (b) one sweep: bmo_source_create_poses (P tiles) -> bmo_system_apply_poses (P poses) -> one bmo_trace_rays with the
      source's pose ids -> bmo_spot_stats_poses.

A step is one whole sweep, timed with CUDA events ending in a synchronise; the legs alternate step by step and the L2 is
flushed (256 MiB write) before every step.  Reported per leg: ms per pose (median, min, max over the steps), bytes over the
bus per sweep, the kernels the trace launched (1 = solve_rays_persistent, more = the wave kernels), and whether (a) and (b)
give the same bits pose by pose.  A separate profiled run of each leg splits the device time into source_*, kinematics,
trace and spot_* kernels.

    python scripts/spot_sweep_bench.py --out FILE.json [--steps 5] [--warmup 1] [--shapes 1048576x64,65536x256]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
LAMBDA = 707e-9
BINS = 64
HALF = 0.25e-3          # histogram window: +-0.25 mm around the detector origin


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                             timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out = f"unavailable ({e})"
    return dict(zip(q.split(","), [s.strip() for s in out.split(",")])) if out.count(",") == 3 else {"query": out}


def kind_of(name):
    if "source_" in name:
        return "source"
    if "spot_" in name or "Radix" in name or "iota32" in name:
        return "spot"
    if "apply_poses" in name:
        return "kinematics"
    return "trace"


def run_shape(m, L, torch, n, P, steps, warmup, dev=0):
    from torch.profiler import ProfilerActivity, profile
    from tests import scenes
    lib = L.lib()
    ctx = L.context(dev)
    stream = torch.cuda.current_stream()
    sc = scenes.doublet_spot(m)
    dsys_a = m.upload_system(sc["system"], [LAMBDA], device=dev)
    dsys_b = m.upload_system(sc["system"], [LAMBDA], device=dev)
    det = next(i for i, o in enumerate(dsys_a.flat.objects) if o is sc["spot"])
    src = m.UniformDiscSource((0.0, -0.05, 0.0), (0.0, 1.0, 0.0), 20e-3, LAMBDA, num_rays=n, e1=(1.0, 0.0, 0.0), on_device=True)
    focus = np.linspace(-2e-3, 2e-3, P)
    offs = np.stack([np.zeros(P), focus, np.zeros(P)], axis=1)
    progs_a = []
    for p in range(P):
        q = m.KinProgram(dsys_a.flat, 1)
        q.translate3d_(sc["spot"], offs[p:p + 1])
        progs_a.append(q)
    prog_b = m.KinProgram(dsys_b.flat, P)
    prog_b.translate3d_(sc["spot"], offs)
    window = np.array([-HALF, HALF, -HALF, HALF])
    info_a, counts_a = (L.bmo_spot_info * P)(), np.zeros((P, BINS, BINS), np.int64)
    info_b, counts_b = (L.bmo_spot_info * P)(), np.zeros((P, BINS, BINS), np.int64)
    trace_launches = {}

    def counted(key, fn):
        """the trace's kernel launches, read once (during the warm-up) so that the timed steps do not query counters"""
        if key in trace_launches:
            return fn()
        c0 = L.counters(dev)["kernel_launches"]
        fn()
        trace_launches[key] = L.counters(dev)["kernel_launches"] - c0

    def leg_a():
        s = C.c_void_p()
        L.check(lib.bmo_source_create(ctx, C.byref(src.desc), C.byref(s)))
        nn, pp, dd, u = C.c_int64(), C.c_void_p(), C.c_void_p(), C.c_int32()
        L.check(lib.bmo_source_device(s, C.byref(nn), C.byref(pp), C.byref(dd), C.byref(u)))
        flags = L.INPUT_DEVICE | (L.UNIFORM_DIR if u.value else 0)
        for p in range(P):
            progs_a[p].apply(dsys_a)
            h = C.c_void_p()
            counted("a", lambda: L.check(lib.bmo_trace_rays(dsys_a.h, nn.value, pp, dd, None, None, None, 100, flags, C.byref(h))))
            L.check(lib.bmo_spot_stats(h, det, L.ptr(window), BINS, BINS, C.byref(info_a[p]), L.ptr(counts_a[p]), 0))
            lib.bmo_result_free(h)
        lib.bmo_source_free(s)

    def leg_b():
        s = C.c_void_p()
        L.check(lib.bmo_source_create_poses(ctx, C.byref(src.desc), P, C.byref(s)))
        nn, pp, dd, u = C.c_int64(), C.c_void_p(), C.c_void_p(), C.c_int32()
        L.check(lib.bmo_source_device(s, C.byref(nn), C.byref(pp), C.byref(dd), C.byref(u)))
        npo, pid = C.c_int32(), C.c_void_p()
        L.check(lib.bmo_source_pose_ids(s, C.byref(npo), C.byref(pid)))
        prog_b.apply(dsys_b)
        h = C.c_void_p()
        flags = L.INPUT_DEVICE | (L.UNIFORM_DIR if u.value else 0)
        counted("b", lambda: L.check(lib.bmo_trace_rays(dsys_b.h, nn.value, pp, dd, None, None, pid, 100, flags, C.byref(h))))
        L.check(lib.bmo_spot_stats_poses(h, det, P, L.ptr(window), BINS, BINS, info_b, L.ptr(counts_b), 0))
        lib.bmo_result_free(h)
        lib.bmo_source_free(s)

    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def timed(fn):
        flush.fill_(1)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        fn()
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    for _ in range(warmup):
        leg_a(); leg_b()
    ta, tb = [], []
    for _ in range(steps):
        ta.append(timed(leg_a) / P)
        tb.append(timed(leg_b) / P)
    same = [bytes(info_a[p]) == bytes(info_b[p]) and bool(np.array_equal(counts_a[p], counts_b[p])) for p in range(P)]

    def kernel_ms(fn):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            flush.fill_(1)
            torch.cuda.synchronize()
            fn()
            torch.cuda.synchronize()
        acc = {}
        for e in prof.events():
            if e.device_type.name != "CUDA" or "fill" in e.name or "elementwise" in e.name.lower() or e.name.startswith(("Memcpy", "Memset")):
                continue
            t = e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
            k = kind_of(e.name)
            acc[k] = acc.get(k, 0.0) + t / 1e3
            if k == "spot":
                name = e.name.split("(")[0].split("<")[0].replace("void ", "").replace("bmo::", "")
                acc.setdefault("spot_kernels", {})
                acc["spot_kernels"][name] = acc["spot_kernels"].get(name, 0.0) + t / 1e3
        return acc

    ka, kb = kernel_ms(leg_a), kernel_ms(leg_b)
    n_params = len(prog_b.params)
    kin_bytes = lambda poses: len(prog_b.ops) * C.sizeof(L.bmo_kin_op) + poses * n_params * 9 * 8
    info_sz, counts_sz = C.sizeof(L.bmo_spot_info), BINS * BINS * 8
    med = lambda t: float(np.median(t))
    rms_a = np.array([info_a[p].rms for p in range(P)])
    return {
        "rays": n, "poses": P, "rays_per_sweep": n * P, "steps": steps, "warmup": warmup,
        "leg_a_one_pose_solves": {
            "ms_per_pose_median": med(ta), "ms_per_pose_min": float(np.min(ta)), "ms_per_pose_max": float(np.max(ta)),
            "h2d_bytes_per_sweep": P * (kin_bytes(1) + 4 * 8), "d2h_bytes_per_sweep": P * (info_sz + counts_sz + 48),
            "bytes_note": "per pose: the kinematic program and its parameters (+ the 32-byte window) in; bmo_spot_info, the "
                          f"{BINS}x{BINS} int64 histogram and the 48-byte device counters out; no per-ray data",
            "trace_kernel_launches": trace_launches.get("a"),
            "trace_path": "solve_rays_persistent" if trace_launches.get("a") == 1 else "waves",
            "device_ms_per_sweep_profiled": ka},
        "leg_b_pose_sweep": {
            "ms_per_pose_median": med(tb), "ms_per_pose_min": float(np.min(tb)), "ms_per_pose_max": float(np.max(tb)),
            "h2d_bytes_per_sweep": kin_bytes(P) + 4 * 8 + (2 * P + 1) * 8 + (P + 1) * 4,
            "d2h_bytes_per_sweep": P * (info_sz + counts_sz) + 48 + (P + 1) * 8,
            "bytes_note": "the kinematic program and P parameter sets, the window and the per-pose slice table in; P x "
                          "(bmo_spot_info + histogram), the device counters and the per-pose beam counts out; no per-ray data",
            "trace_kernel_launches": trace_launches.get("b"),
            "trace_path": "solve_rays_persistent" if trace_launches.get("b") == 1 else "waves",
            "device_ms_per_sweep_profiled": kb},
        "speedup_a_over_b": med(ta) / med(tb),
        "bit_identical_poses": int(sum(same)), "bit_identical_all": bool(all(same)),
        "rms_min_pose": int(np.nanargmin(rms_a)), "rms_min_m": float(np.nanmin(rms_a)),
        "hits_min": int(min(info_b[p].hits for p in range(P))),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--shapes", default="1048576x64,65536x256", help="rays x poses, comma separated")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("spot_sweep_bench.py: no CUDA device")
    import __graft_entry__ as ge
    ge.build_libbmo()
    m = ge.load_package()
    from bmo_b200 import _lib as L
    L.set_stream(torch.cuda.current_stream().cuda_stream, 0)
    card_before = card()
    shapes = [tuple(int(v) for v in s.split("x")) for s in args.shapes.split(",")]
    res = [run_shape(m, L, torch, n, P, args.steps, args.warmup) for n, P in shapes]
    out = {
        "workload": "C2 through focus: AC254-150-AB doublet + Spotdetector swept +-2 mm along the axis, UniformDiscSource 20 mm, "
                    "707 nm, r_max 100, one GPU",
        "card_before": card_before, "card_after": card(), "torch_device_name": torch.cuda.get_device_name(0),
        "l2": "flushed with a 256 MiB write before every timed step",
        "histogram": f"{BINS}x{BINS} over +-{HALF * 1e3} mm",
        "shapes": res,
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
