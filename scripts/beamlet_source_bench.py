"""GaussianBeamlet bundles built on the host against beamlet sources generated on the device, through the Photodetector.

    python scripts/beamlet_source_bench.py --out FILE.json [--steps 5] [--warmup 1]

Workloads (collimated sources, lambda = 1 um, support = x):
  c3_64k:   2^16 beamlets of an 8 mm source (256 rings), w0 = 1.5 * 8 mm / 256, through the C3 expander onto 512 x 512.
  c3_1m:    2^20 beamlets of the same source (1024 rings) onto 64 x 64.
  mzi_4k:   4096 beamlets of a 1 mm source (64 rings), w0 = 1.5 * 1 mm / 64, x 64 poses of the C5 Mach-Zehnder (m1 moved along
            its normal over 2 lambda by a KinProgram on the device), bmo_pd_accumulate_poses into 64 fields of 64 x 64.
Legs, alternated step by step after the warm-up, the L2 flushed (a 256 MiB write) before every step, each step timed with CUDA
events ending in a synchronise:
  host:    bmo_trace_beamlets from host arrays built beforehand by CollimatedSource + BeamletBundle.from_params (and np.tile with pose
           ids for the sweep), then bmo_pd_accumulate(_poses) into a zeroed device field.  The host construction is timed once
           with the host clock and reported apart.
  device:  bmo_source_create_beamlets (n_poses tiles), bmo_trace_beamlets(BMO_INPUT_DEVICE), the same accumulate.  The source is
           part of the step; its host-side construction (descriptor and create call, synchronised) is reported apart too.
A separate torch.profiler run of one step per leg gives the per-kernel device times and the host<->device bytes from the memcpy
records.  Both legs' fields must be equal bit for bit.  Card name, power limit and SM clock are read in the same run.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
LAM = 1e-6
HBM_BYTES_PER_S = 7.7e12     # HGX B200 data sheet, one GPU


def card(index):
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", str(index)], capture_output=True, text=True,
                             timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out = f"unavailable ({e})"
    parts = [s.strip() for s in out.split(",")]
    return dict(zip(q.split(","), parts)) if len(parts) == 4 else {"query": out}


def workloads(m, s2):
    """name -> (system builder, source kwargs, beamlet kwargs, n_poses, pd pixels)"""
    c3 = dict(pos=(0.0, -0.05, 0.0), dir=(0.0, 1.0, 0.0), diameter=8e-3, b1=(1.0, 0.0, 0.0))
    mz = dict(pos=(0.0, -0.1, 0.0), dir=(0.0, 1.0, 0.0), diameter=1e-3, b1=(1.0, 0.0, 0.0))
    bl = lambda w0, n: dict(w0=w0, M2=1.0, P0=1e-3 / n, z0=0.0, support=(1.0, 0.0, 0.0))
    return {
        "c3_64k": (lambda: s2.expander(m, 512), dict(c3, num_rings=256, num_rays=1 << 16), bl(1.5 * 8e-3 / 256, 1 << 16), 1),
        "c3_1m": (lambda: s2.expander(m, 64), dict(c3, num_rings=1024, num_rays=1 << 20), bl(1.5 * 8e-3 / 256, 1 << 20), 1),
        "mzi_4k": (lambda: s2.mzi(m, pd_n=64), dict(mz, num_rings=64, num_rays=4096), bl(1.5 * 1e-3 / 64, 4096), 64),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--only", default=None, help="comma-separated workload names")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("beamlet_source_bench.py: no CUDA device")
    import __graft_entry__ as ge
    m = ge.load_package()
    from bmo_b200 import _lib as L
    from bmo_b200 import beams
    from tests import scenes2 as s2
    dev = 0
    card_before = card(dev)
    lib = L.lib()
    stream = torch.cuda.current_stream()
    L.set_stream(stream.cuda_stream, dev)
    ctx = L.context(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    result = {"workloads": {}}

    for name, (build, skw, bkw, P) in workloads(m, s2).items():
        if args.only and name not in args.only.split(","):
            continue
        sc = build()
        npx = sc["pd"].n
        dsys = m.upload_system(sc["system"], [LAM], device=dev)
        oi = next(i for i, o in enumerate(dsys.flat.objects) if o is sc["pd"])
        if P > 1:
            prog = m.KinProgram(dsys.flat, P)
            prog.translate3d_(sc["m1"], np.array([s2.mzi_shift(k, P) for k in range(P)]))
            prog.apply(dsys)
        # host leg inputs: the host constructors, then tiled per pose
        t0 = time.perf_counter()
        hsrc = m.CollimatedSource(skw["pos"], skw["dir"], skw["diameter"], LAM, num_rings=skw["num_rings"], num_rays=skw["num_rays"], b1=skw["b1"])
        bundle = m.BeamletBundle.from_params(hsrc.pos, skw["dir"], LAM, **bkw)
        nb = len(bundle)
        g_rays = np.ascontiguousarray(np.tile(bundle.rays.reshape(nb, 18), (P, 1)))
        g_w0 = np.ascontiguousarray(np.tile(bundle.w0, P))
        E0 = np.tile(bundle.E0, P)
        g_e0 = np.ascontiguousarray(np.stack([E0.real, E0.imag], axis=-1))
        g_lam = np.zeros(nb * P, np.int32)
        g_pid = np.ascontiguousarray(np.repeat(np.arange(P, dtype=np.int32), nb)) if P > 1 else None
        host_build_s = time.perf_counter() - t0
        # device leg: the descriptor of the same beamlets
        t0 = time.perf_counter()
        dsrc = m.CollimatedSource(skw["pos"], skw["dir"], skw["diameter"], LAM, num_rings=skw["num_rings"], num_rays=skw["num_rays"], b1=skw["b1"],
                                  on_device=True)
        bdesc = beams.beamlet_desc(dsrc.direction, LAM, **bkw)
        h = C.c_void_p()
        L.check(lib.bmo_source_create_beamlets(ctx, C.byref(dsrc.desc), C.byref(bdesc), P, 0, nb, C.byref(h)))
        torch.cuda.synchronize()
        lib.bmo_source_free(h)
        device_build_s = time.perf_counter() - t0
        field = torch.zeros(P * npx * npx * 2, dtype=torch.float64, device="cuda")
        fields = {}

        def ev():
            e = torch.cuda.Event(enable_timing=True)
            e.record(stream)
            return e

        def accumulate(res):
            if P > 1:
                L.check(lib.bmo_pd_accumulate_poses(dsys.h, res, oi, P, C.c_void_p(field.data_ptr()), L.INPUT_DEVICE))
            else:
                L.check(lib.bmo_pd_accumulate(dsys.h, res, oi, 0, C.c_void_p(field.data_ptr()), L.INPUT_DEVICE))

        def step(leg):
            field.zero_()
            flush.fill_(1)
            torch.cuda.synchronize()
            e0 = ev()
            res, src = C.c_void_p(), C.c_void_p()
            if leg == "host":
                L.check(lib.bmo_trace_beamlets(dsys.h, nb * P, L.ptr(g_rays), L.ptr(g_lam), L.ptr(g_w0), L.ptr(g_e0), L.ptr(g_pid), 100, 0,
                                               C.byref(res)))
                e1 = e0
            else:
                L.check(lib.bmo_source_create_beamlets(ctx, C.byref(dsrc.desc), C.byref(bdesc), P, 0, nb, C.byref(src)))
                e1 = ev()
                n, r, w, e, pid = C.c_int64(), C.c_void_p(), C.c_void_p(), C.c_void_p(), C.c_void_p()
                L.check(lib.bmo_source_beamlets_device(src, C.byref(n), C.byref(r), C.byref(w), C.byref(e)))
                L.check(lib.bmo_source_pose_ids(src, None, C.byref(pid)))
                L.check(lib.bmo_trace_beamlets(dsys.h, n.value, r, None, w, e, pid, 100, L.INPUT_DEVICE, C.byref(res)))
            e2 = ev()
            accumulate(res)
            e3 = ev()
            torch.cuda.synchronize()
            lib.bmo_result_free(res)
            if src:
                lib.bmo_source_free(src)
            fields[leg] = field.cpu().numpy().copy()
            return e0.elapsed_time(e3), {"source": e0.elapsed_time(e1), "trace": e1.elapsed_time(e2), "accumulate": e2.elapsed_time(e3)}

        legs = ("host", "device")
        for _ in range(args.warmup):
            for leg in legs:
                step(leg)
        times, parts = {leg: [] for leg in legs}, {leg: [] for leg in legs}
        for _ in range(args.steps):
            for leg in legs:
                t, p = step(leg)
                times[leg].append(t)
                parts[leg].append(p)
        same = fields["host"].tobytes() == fields["device"].tobytes()

        # one profiled step per leg: kernel times and copied bytes
        prof = {}
        for leg in legs:
            with tempfile.TemporaryDirectory() as tmp:
                from torch.profiler import ProfilerActivity, profile
                with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as pr:
                    step(leg)
                path = os.path.join(tmp, "trace.json")
                pr.export_chrome_trace(path)
                with open(path) as f:
                    evs = json.load(f)["traceEvents"]
            kern, copies = {}, {"HtoD": 0, "DtoH": 0, "DtoD": 0}
            for e in evs:
                cat = e.get("cat", "")
                if cat == "kernel":
                    k = e["name"].split("(")[0].replace("void ", "")
                    kern.setdefault(k, [0.0, 0])
                    kern[k][0] += e.get("dur", 0) * 1e-3
                    kern[k][1] += 1
                elif cat == "gpu_memcpy":
                    for d in copies:
                        if d in e["name"]:
                            copies[d] += int(e.get("args", {}).get("bytes", 0))
            prof[leg] = {"kernels_ms": {k: {"ms": round(v[0], 6), "launches": v[1]} for k, v in sorted(kern.items(), key=lambda kv: -kv[1][0])},
                         "memcpy_bytes": copies}
        # source_beamlets: writes rays, w0, E0 (and pose ids), reads one tile's positions
        total = nb * P
        kb = total * (18 + 1 + 2) * 8 + (total * 4 if P > 1 else 0) + nb * 24
        kt = next((v["ms"] for k, v in prof["device"]["kernels_ms"].items() if "source_beamlets" in k), None)
        result["workloads"][name] = {
            "beamlets": nb, "poses": P, "pixels": npx,
            "host_construction_s": host_build_s, "device_construction_s": device_build_s,
            "fields_equal_bit_for_bit": same,
            "legs": {leg: {"step_ms_median": float(np.median(times[leg])), "step_ms_min": float(np.min(times[leg])),
                           "step_ms_max": float(np.max(times[leg])),
                           "split_ms_median": {k: float(np.median([p[k] for p in parts[leg]])) for k in parts[leg][0]},
                           "profiled_step": prof[leg]} for leg in legs},
            "source_beamlets": {"bytes": kb, "ms": kt, "bytes_per_s": (kb / (kt * 1e-3)) if kt else None,
                                "share_of_7.7TB_s": (kb / (kt * 1e-3) / HBM_BYTES_PER_S) if kt else None},
        }
        print(name, json.dumps({k: v for k, v in result["workloads"][name].items() if k != "legs"}), flush=True)
        dsys.free()
    result.update({
        "steps_per_leg": args.steps, "warmup": args.warmup, "card_before": card_before, "card_after": card(dev),
        "torch_device_name": torch.cuda.get_device_name(dev),
        "l2": "flushed with a 256 MiB write before every timed step",
        "timing": "CUDA events ending in a synchronise; kernel times and memcpy bytes from a separate torch.profiler step per leg",
    })
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()
