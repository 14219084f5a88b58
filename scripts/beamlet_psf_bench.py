"""PSFDetector records of GaussianBeamlet solves: bench.py's Airy-disc PSF scene (test/runtests.jl:2765-2802) with 2^16 beamlets on a
512 x 512 map, crop_factor 5, :bbox window.  Every beamlet ends on the detector and pushes three records (chief, waist, divergence):
196 608 records.

    python scripts/beamlet_psf_bench.py --out FILE.json [--steps 5] [--warmup 1] [--beamlets 65536] [--px 512]

Two legs alternate step by step after the warm-up, each timed with CUDA events ending in a synchronise; the L2 is flushed (a 256 MiB
write) before every step.
  beamlets:  bmo_trace_beamlets (host arrays) -> bmo_psf_collect -> bmo_psf_lims -> bmo_psf_intensity (map to device memory), split
             by events into trace, collect, lims and the intensity call; K6's own time is libbmo's event bracket of the kernel (psf_ms).
  rays:      the same steps for a ray bundle with as many records (3 x 2^16 rays of a 15 mm disc, bmo_trace_rays).  K6 does not know
             where its records came from, so its pixel-hit pairs per second should be those of the beamlet leg: this checks it.
Card name, power limit and SM clock are read in the same run, before and after.
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
LAMBDA = 1e-6


def card(index):
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", str(index)], capture_output=True, text=True,
                             timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out = f"unavailable ({e})"
    parts = [s.strip() for s in out.split(",")]
    return dict(zip(q.split(","), parts)) if len(parts) == 4 else {"query": out}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--beamlets", type=int, default=1 << 16)
    ap.add_argument("--px", type=int, default=512)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("beamlet_psf_bench.py: no CUDA device")
    import __graft_entry__ as ge
    m = ge.load_package()
    from bmo_b200 import _lib as L
    from tests import scenes
    dev = 0
    card_before = card(dev)
    lib = L.lib()
    stream = torch.cuda.current_stream()
    L.set_stream(stream.cuda_stream, dev)

    lens = m.SphericalLens(100e-3, np.inf, 1e-3, 25.4e-3, 1.5)
    psfd = m.PSFDetector(10e-3)
    psfd.translate3d_([0.0, 200e-3 + 0.13e-3, 0.0])
    system = m.System([lens, psfd])
    dsys = m.upload_system(system, [LAMBDA], device=dev)
    oi = next(i for i, o in enumerate(dsys.flat.objects) if o is psfd)
    nb, n = args.beamlets, args.px
    pos, _ = scenes.fibonacci_disc(nb, diameter=15e-3, y0=-10e-3)
    bundle = m.BeamletBundle.from_params(pos, (0.0, 1.0, 0.0), LAMBDA, w0=0.2e-3, support=(1.0, 0.0, 0.0))
    g_rays = np.ascontiguousarray(bundle.rays.reshape(-1, 18))
    g_lam = np.zeros(nb, np.int32)
    g_e0 = np.ascontiguousarray(np.stack([bundle.E0.real, bundle.E0.imag], axis=-1))
    n_rays = 3 * nb
    r_pos, _ = scenes.fibonacci_disc(n_rays, diameter=15e-3, y0=-10e-3)
    r_dir = np.array([0.0, 1.0, 0.0])
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    out = torch.zeros(n * n, dtype=torch.float64, device="cuda")
    lims = np.zeros(4)
    records = {}

    def ev():
        e = torch.cuda.Event(enable_timing=True)
        e.record(stream)
        return e

    def step(leg):
        e0 = ev()
        marks = {}
        h, psf = C.c_void_p(), C.c_void_p()
        if leg == "beamlets":
            L.check(lib.bmo_trace_beamlets(dsys.h, nb, L.ptr(g_rays), L.ptr(g_lam), L.ptr(bundle.w0), L.ptr(g_e0), None, 100, 0, C.byref(h)))
        else:
            L.check(lib.bmo_trace_rays(dsys.h, n_rays, L.ptr(r_pos), L.ptr(r_dir), None, None, None, 100, L.KEEP_SEGMENTS | L.UNIFORM_DIR,
                                       C.byref(h)))
        marks["trace"] = ev()
        cnt = C.c_int64()
        L.check(lib.bmo_psf_collect(dsys.h, h, oi, C.byref(psf), C.byref(cnt)))
        records[leg] = int(cnt.value)
        marks["collect"] = ev()
        L.check(lib.bmo_psf_lims(dsys.h, psf, oi, 0, 5.0, 1, L.ptr(lims)))
        marks["lims"] = ev()
        L.check(lib.bmo_psf_intensity(dsys.h, psf, oi, 0, n, L.ptr(lims), 0.0, 0.0, C.c_void_p(out.data_ptr()), L.INPUT_DEVICE))
        marks["intensity"] = ev()
        k6 = L.counters(dev)["psf_ms"]
        lib.bmo_psf_free(psf)
        lib.bmo_result_free(h)
        torch.cuda.synchronize()
        parts, prev = {}, e0
        for k, e in marks.items():
            parts[k] = prev.elapsed_time(e)
            prev = e
        parts["k6"] = k6
        return e0.elapsed_time(prev), parts

    legs = ("beamlets", "rays")
    for _ in range(args.warmup):
        for leg in legs:
            step(leg)
    times = {leg: [] for leg in legs}
    parts = {leg: [] for leg in legs}
    for _ in range(args.steps):        # alternate the legs
        for leg in legs:
            flush.fill_(1)
            torch.cuda.synchronize()
            t, p = step(leg)
            times[leg].append(t)
            parts[leg].append(p)
    card_after = card(dev)

    out_legs = {}
    for leg in legs:
        split = {k: float(np.median([p[k] for p in parts[leg]])) for k in parts[leg][0]}
        pairs = float(records[leg]) * n * n
        out_legs[leg] = {
            "records": records[leg], "step_ms_median": float(np.median(times[leg])), "step_ms_min": float(np.min(times[leg])),
            "step_ms_max": float(np.max(times[leg])), "split_ms_median": split,
            "k6_ms_min": float(np.min([p["k6"] for p in parts[leg]])), "k6_ms_max": float(np.max([p["k6"] for p in parts[leg]])),
            "k6_px_hits_per_s": pairs / (split["k6"] * 1e-3),
        }
    result = {
        "workload": f"Airy-disc PSF scene (bench.py's PSF leg): {nb} GaussianBeamlets (w0 0.2 mm, Fibonacci disc of 15 mm) against "
                    f"{n_rays} rays, {n} x {n} map, crop_factor 5, :bbox window",
        "steps_per_leg": args.steps, "warmup": args.warmup, "card_before": card_before, "card_after": card_after,
        "torch_device_name": torch.cuda.get_device_name(dev),
        "l2": "flushed with a 256 MiB write before every timed step",
        "timing": "CUDA events ending in a synchronise; K6 from libbmo's event bracket of psf_intensity_kernel",
        "check": {"beamlet_records_equal_3x_beamlets": records["beamlets"] == 3 * nb, "same_record_count": records["beamlets"] == records["rays"],
                  "k6_rate_beamlets_over_rays": out_legs["beamlets"]["k6_px_hits_per_s"] / out_legs["rays"]["k6_px_hits_per_s"]},
        "legs": out_legs,
    }
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()
