"""C2 spot diagram end to end on one GPU: host rays and host spots against a source generated on the device and spots reduced
there.  The two arms alternate step by step in one run, each step timed with CUDA events ending in a synchronise, the L2
flushed between steps (a 256 MiB write, as bench.py does).

  (a) host leg: pinned host positions [n][3] + one direction (BMO_UNIFORM_DIR) -> bmo_trace_rays_spots -> spots [n][2] on
      the host (bench.py's end-to-end leg).
  (b) device leg: bmo_source_create (UniformDiscSource descriptor) -> bmo_trace_rays(BMO_INPUT_DEVICE | BMO_UNIFORM_DIR) ->
      bmo_spot_stats with a 256 x 256 histogram over the detector face -> statistics and histogram on the host.

Both arms trace the same rays: (a)'s host buffer is the download of (b)'s source.  The statistics numpy computes from (a)'s
spots are checked against (b)'s.  A second, profiled run of (b) gives the device time of the generation and reduction
kernels on their own, and CollimatedSource at the same size is timed twice: the host constructor (CPU) and bmo_source_create
(device, serial ring recurrence).

    python scripts/source_spot_bench.py --out FILE.json [--steps 20] [--rays 1048576]
"""
import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
LAMBDA = 707e-9
BINS = 256


def card():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                             timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out = f"unavailable ({e})"
    return dict(zip(q.split(","), [s.strip() for s in out.split(",")])) if out.count(",") == 2 else {"query": out}


def np_stats(xz, window, nx, nz):
    """What bmo_spot_stats computes, from host spots (NaN = no Spotdetector reached; C2 has one)."""
    x, z = xz[:, 0], xz[:, 1]
    hit = ~np.isnan(x)
    x, z = x[hit], z[hit]
    cx, cz = x.mean(), z.mean()
    xl, xh, zl, zh = window
    inside = (x >= xl) & (x <= xh) & (z >= zl) & (z <= zh)
    i = np.minimum(np.floor((x[inside] - xl) / (xh - xl) * nx), nx - 1).astype(np.int64)
    j = np.minimum(np.floor((z[inside] - zl) / (zh - zl) * nz), nz - 1).astype(np.int64)
    counts = np.zeros((nz, nx), np.int64)
    np.add.at(counts, (j, i), 1)
    return dict(hits=int(hit.sum()), centroid=(float(cx), float(cz)), rms=math.sqrt(((x - cx) ** 2 + (z - cz) ** 2).sum() / len(x)),
                max_r=float(np.sqrt(x * x + z * z).max()), lo=(float(x.min()), float(z.min())), hi=(float(x.max()), float(z.max())),
                outside=int((~inside).sum())), counts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rays", type=int, default=1 << 20)
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile
    if not torch.cuda.is_available():
        raise SystemExit("source_spot_bench.py: no CUDA device")
    import __graft_entry__ as ge
    ge.build_libbmo()
    m = ge.load_package()
    from bmo_b200 import _lib as L
    from tests import scenes
    card_before = card()
    n, dev = args.rays, 0
    lib = L.lib()
    stream = torch.cuda.current_stream()
    L.set_stream(stream.cuda_stream, dev)
    ctx = L.context(dev)
    sc = scenes.doublet_spot(m)
    dsys = m.upload_system(sc["system"], [LAMBDA], device=dev)
    det = next(i for i, o in enumerate(dsys.flat.objects) if o is sc["spot"])
    hw = sc["spot"].hw
    window = np.array([-hw, hw, -hw, hw])
    src = m.UniformDiscSource((0.0, -0.05, 0.0), (0.0, 1.0, 0.0), 20e-3, LAMBDA, num_rays=n, e1=(1.0, 0.0, 0.0), on_device=True)
    pos_h, dir_h = src.rays(dev)
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    pos_p, dir1_p = pin(pos_h), pin(dir_h[0])
    xz_p = torch.empty((n, 2), dtype=torch.float64).pin_memory()
    counts_p = torch.zeros((BINS, BINS), dtype=torch.int64).pin_memory()
    info = L.bmo_spot_info()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()

    def step_a():
        h = C.c_void_p()
        L.check(lib.bmo_trace_rays_spots(dsys.h, n, C.c_void_p(pos_p.data_ptr()), C.c_void_p(dir1_p.data_ptr()), None, None, None, 100,
                                         L.UNIFORM_DIR, None, C.c_void_p(xz_p.data_ptr()), C.byref(h)))
        lib.bmo_result_free(h)

    def step_b():
        s, h = C.c_void_p(), C.c_void_p()
        L.check(lib.bmo_source_create(ctx, C.byref(src.desc), C.byref(s)))
        nn, p, d, u = C.c_int64(), C.c_void_p(), C.c_void_p(), C.c_int32()
        L.check(lib.bmo_source_device(s, C.byref(nn), C.byref(p), C.byref(d), C.byref(u)))
        L.check(lib.bmo_trace_rays(dsys.h, nn.value, p, d, None, None, None, 100, L.INPUT_DEVICE | (L.UNIFORM_DIR if u.value else 0), C.byref(h)))
        L.check(lib.bmo_spot_stats(h, det, L.ptr(window), BINS, BINS, C.byref(info), C.c_void_p(counts_p.data_ptr()), 0))
        lib.bmo_result_free(h)
        lib.bmo_source_free(s)

    def timed(fn):
        flush.fill_(1)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        fn()
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    for _ in range(args.warmup):
        step_a(); step_b()
    ta, tb = [], []
    for _ in range(args.steps):     # alternate the arms
        ta.append(timed(step_a))
        tb.append(timed(step_b))

    # agreement: numpy on (a)'s spots against (b)'s reduction of the same rays
    ref, ref_counts = np_stats(xz_p.numpy(), window, BINS, BINS)
    got = dict(hits=int(info.hits), centroid=(info.centroid[0], info.centroid[1]), rms=info.rms, max_r=info.max_r,
               lo=(info.lo[0], info.lo[1]), hi=(info.hi[0], info.hi[1]), outside=int(info.outside))
    rel = lambda g, r, s: abs(g - r) / s
    agree = {
        "exact_hits_outside_max_r_lo_hi": got["hits"] == ref["hits"] and got["outside"] == ref["outside"] and got["max_r"] == ref["max_r"]
                                          and got["lo"] == ref["lo"] and got["hi"] == ref["hi"],
        "histogram_equal": bool(np.array_equal(counts_p.numpy(), ref_counts)),
        "centroid_rel_to_max_r": max(rel(g, r, ref["max_r"]) for g, r in zip(got["centroid"], ref["centroid"])),
        "rms_rel": rel(got["rms"], ref["rms"], ref["rms"]),
    }
    agree["ok"] = bool(agree["exact_hits_outside_max_r_lo_hi"] and agree["histogram_equal"] and agree["centroid_rel_to_max_r"] <= 1e-12
                       and agree["rms_rel"] <= 1e-12)

    # device time of the generation and reduction kernels on their own (profiled run of arm (b))
    kern = ("source_disc", "source_rings", "spot_sums", "spot_spread", "solve_rays_persistent")

    def kernel_ms(fn, steps):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(steps):
                flush.fill_(1)
                torch.cuda.synchronize()
                fn()
                torch.cuda.synchronize()
        acc = {}
        for e in prof.events():
            if e.device_type.name != "CUDA":
                continue
            for k in kern:
                if k in e.name:
                    t = e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
                    acc[k] = acc.get(k, 0.0) + t / 1e3 / steps
        return acc

    kb = kernel_ms(step_b, 10)

    # CollimatedSource at the same size: host constructor (CPU) against bmo_source_create (device)
    t0 = time.perf_counter()
    host_col = m.CollimatedSource((0.0, -0.05, 0.0), (0.0, 1.0, 0.0), 20e-3, LAMBDA, num_rings=10, num_rays=n, b1=(1.0, 0.0, 0.0))
    host_col_s = time.perf_counter() - t0
    col = m.CollimatedSource((0.0, -0.05, 0.0), (0.0, 1.0, 0.0), 20e-3, LAMBDA, num_rings=10, num_rays=n, b1=(1.0, 0.0, 0.0), on_device=True)

    def make_col():
        s = C.c_void_p()
        L.check(lib.bmo_source_create(ctx, C.byref(col.desc), C.byref(s)))
        torch.cuda.synchronize()
        lib.bmo_source_free(s)

    make_col()
    col_ms = [timed(make_col) for _ in range(5)]
    kc = kernel_ms(make_col, 3)
    cpos, cdir = col.rays(dev)
    col_equal = bool(np.array_equal(cpos.view(np.int64), host_col.pos.view(np.int64)) and np.array_equal(cdir.view(np.int64), host_col.dir.view(np.int64)))

    med = lambda t: float(np.median(t))
    ring_bytes = int(col.desc.n_rings) * C.sizeof(L.bmo_source_ring)
    out = {
        "workload": "C2: AC254-150-AB doublet + Spotdetector, UniformDiscSource 20 mm, r_max 100, one GPU",
        "rays": n, "steps_per_arm": args.steps, "warmup": args.warmup,
        "card_before": card_before, "card_after": card(), "torch_device_name": torch.cuda.get_device_name(0),
        "l2": "flushed with a 256 MiB write before every timed step",
        "arm_a_host_rays_host_spots": {
            "step_ms_median": med(ta), "step_ms_min": float(np.min(ta)), "step_ms_max": float(np.max(ta)),
            "h2d_bytes": int(n * 24 + 24), "d2h_bytes": int(n * 16 + 48),
            "bytes_note": "positions [n][3] f64 + one direction in; spots (x, z) [n][2] f64 + the 48-byte device counters out"},
        "arm_b_device_source_device_stats": {
            "step_ms_median": med(tb), "step_ms_min": float(np.min(tb)), "step_ms_max": float(np.max(tb)),
            "h2d_bytes": 0, "d2h_bytes": int(C.sizeof(L.bmo_spot_info) + BINS * BINS * 8 + 48),
            "bytes_note": "a disc descriptor has no ring table: its fields travel as kernel parameters; out: bmo_spot_info (80 B), "
                          "the 256 x 256 int64 histogram and the 48-byte device counters"},
        "arm_b_kernel_ms_profiled": kb,
        "speedup_a_over_b": med(ta) / med(tb),
        "agreement_numpy_on_a_vs_b": agree,
        "stats_b": got,
        "collimated_source_2p20": {
            "num_rings": 10, "host_constructor_cpu_s": host_col_s, "bmo_source_create_ms_median": med(col_ms),
            "kernel_ms_profiled": kc, "ring_table_h2d_bytes": ring_bytes, "device_equals_host_bitwise": col_equal},
    }
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
