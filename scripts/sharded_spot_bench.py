"""C2 spot diagram sharded over GPUs: each rank generates its slice of one UniformDiscSource on its GPU, traces it and joins
bmo_spot_stats_sharded, so every rank ends with the spot statistics and the 256 x 256 histogram of the whole bundle while
no ray or hit crosses the bus.

    torchrun --nproc_per_node=N scripts/sharded_spot_bench.py --out FILE.json [--steps 20] [--warmup 3] [--baseline ONE_GPU.json]
    python scripts/sharded_spot_bench.py --out FILE.json            (N = 1)

A step is bmo_source_create_slice (the rank's spot_shard_slice of the source) -> bmo_trace_rays(BMO_INPUT_DEVICE |
BMO_UNIFORM_DIR) -> bmo_spot_stats_sharded, timed per rank with CUDA events ending in a synchronise; the step time is the
largest over the ranks.  The L2 is flushed (a 256 MiB write) before every step.  Two legs alternate step by step after the
warm-up: weak (2^20 rays per rank) and strong (2^20 rays in all).  Efficiency against N = 1 needs --baseline, the JSON of a
one-GPU run: weak t1 / tN, strong t1 / (N tN).  A second, profiled run of each leg gives the NCCL kernels' share of the
device time of a step and the bytes the step copies each way (the profiler's memcpy records).  Every rank checks its statistics against bmo_spot_stats of one unsharded trace of the same rays on
its own GPU, bit for bit.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
LAMBDA = 707e-9
BINS = 256
RAYS = 1 << 20


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
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--baseline", default=None)
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile
    if not torch.cuda.is_available():
        raise SystemExit("sharded_spot_bench.py: no CUDA device")
    import __graft_entry__ as ge
    m = ge.load_package()
    from bmo_b200 import _lib as L
    from bmo_b200 import parallel as par
    from tests import scenes
    rank, ws, dev = par.world()
    torch.cuda.set_device(dev)
    dist = None
    if ws > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", dev))
    card_before = card(dev)
    lib = L.lib()
    stream = torch.cuda.current_stream()
    L.set_stream(stream.cuda_stream, dev)
    ctx = L.context(dev)
    comm = par.FieldComm.from_torch(device=dev) if ws > 1 else par.FieldComm(0, 1, par.FieldComm.unique_id(), dev)
    sc = scenes.doublet_spot(m)
    dsys = m.upload_system(sc["system"], [LAMBDA], device=dev)
    det = next(i for i, o in enumerate(dsys.flat.objects) if o is sc["spot"])
    hw = sc["spot"].hw
    window = np.array([-hw, hw, -hw, hw])
    counts = torch.zeros((BINS, BINS), dtype=torch.int64).pin_memory()
    info = L.bmo_spot_info()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    legs = {"weak": RAYS * ws, "strong": RAYS}
    srcs = {k: m.UniformDiscSource((0.0, -0.05, 0.0), (0.0, 1.0, 0.0), 20e-3, LAMBDA, num_rays=n, e1=(1.0, 0.0, 0.0), on_device=True)
            for k, n in legs.items()}
    cut = {k: par.spot_shard_slice(n, rank, ws) for k, n in legs.items()}

    def step(leg):
        s, h = C.c_void_p(), C.c_void_p()
        first, count = cut[leg]
        L.check(lib.bmo_source_create_slice(ctx, C.byref(srcs[leg].desc), first, count, C.byref(s)))
        nn, p, d, u = C.c_int64(), C.c_void_p(), C.c_void_p(), C.c_int32()
        L.check(lib.bmo_source_device(s, C.byref(nn), C.byref(p), C.byref(d), C.byref(u)))
        L.check(lib.bmo_trace_rays(dsys.h, nn.value, p, d, None, None, None, 100, L.INPUT_DEVICE | L.UNIFORM_DIR, C.byref(h)))
        L.check(lib.bmo_spot_stats_sharded(comm.h, h, det, L.ptr(window), BINS, BINS, C.byref(info), C.c_void_p(counts.data_ptr()), 0))
        lib.bmo_result_free(h)
        lib.bmo_source_free(s)

    def sync_ranks():
        torch.cuda.synchronize()
        if dist:
            dist.barrier()

    def timed(leg):
        flush.fill_(1)
        sync_ranks()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        step(leg)
        e1.record(stream)
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        if dist:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for _ in range(args.warmup):
        for leg in legs:
            step(leg)
    times = {leg: [] for leg in legs}
    for _ in range(args.steps):        # alternate the legs
        for leg in legs:
            times[leg].append(timed(leg))

    # bit for bit against one unsharded trace of the same rays on this GPU, and the same bits on every rank
    checks = {}
    for leg in legs:
        step(leg)
        got = bytes(info) + counts.numpy().tobytes()
        res = m.solve_system_(sc["system"], srcs[leg], retrace=False, device=dev, keep_segments=False, collect_spots=False)
        one = m.spot_stats(res, sc["spot"], bins=BINS, window=tuple(window))
        ref = L.bmo_spot_info()
        ref.hits, ref.outside = one["hits"], one["outside"]
        ref.centroid[:], ref.rms, ref.max_r, ref.lo[:], ref.hi[:] = one["centroid"], one["rms"], one["max_r"], one["lo"], one["hi"]
        same = got == bytes(ref) + one["counts"].tobytes()
        res.free()
        if dist:
            box = [None] * ws
            dist.all_gather_object(box, (same, got))
            same = all(b[0] for b in box) and all(b[1] == box[0][1] for b in box)
        checks[leg] = dict(bit_identical_to_one_gpu_trace_on_every_rank=bool(same), hits=int(info.hits), rms=info.rms)

    # NCCL share of the device time of a step and the bytes the step copies over the bus (separate, profiled run).  The bytes
    # are the profiler's own memcpy records (the trace's gpu_memcpy events carry their size), read from a trace written to a
    # temporary directory.
    def profiled(leg, steps=5):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(steps):
                flush.fill_(1)
                sync_ranks()
                step(leg)
                torch.cuda.synchronize()
        acc = {}
        for e in prof.events():
            if e.device_type.name != "CUDA" or "Memcpy" in e.name or "Memset" in e.name:
                continue
            if "elementwise" in e.name or "fill" in e.name.lower():
                continue                # the L2 flush
            t = (e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total) / 1e3 / steps
            key = "nccl" if "nccl" in e.name.lower() else e.name.split("(")[0].split("<")[0]
            acc[key] = acc.get(key, 0.0) + t
        with tempfile.TemporaryDirectory() as tmp:
            path = os.path.join(tmp, "trace.json")
            prof.export_chrome_trace(path)
            with open(path) as f:
                trace = json.load(f)
        copies = {}
        for ev in trace.get("traceEvents", []):
            if ev.get("cat") != "gpu_memcpy":
                continue
            kind = ev.get("name", "").split("(")[0].replace("Memcpy", "").strip()     # HtoD, DtoH, DtoD
            c = copies.setdefault(kind, {"copies": 0, "bytes": 0})
            c["copies"] += 1
            c["bytes"] += int(ev.get("args", {}).get("bytes", 0))
        copies = {k: {"copies_per_step": v["copies"] / steps, "bytes_per_step": v["bytes"] / steps} for k, v in copies.items()}
        total = sum(acc.values())
        return dict(device_ms_per_step=acc, nccl_share=acc.get("nccl", 0.0) / total if total else None, memcpy=copies)

    prof = {leg: profiled(leg) for leg in legs}
    card_after = card(dev)

    base = None
    if args.baseline and os.path.exists(args.baseline):
        with open(args.baseline) as f:
            base = json.load(f)
    out_legs = {}
    for leg, n in legs.items():
        t = times[leg]
        med = float(np.median(t))
        eff = None
        if base is not None:
            t1 = base["legs"][leg]["step_ms_median"]
            eff = t1 / med if leg == "weak" else t1 / (ws * med)
        out_legs[leg] = {
            "rays_total": n, "rays_this_rank": cut[leg][1], "step_ms_median": med, "step_ms_min": float(np.min(t)), "step_ms_max": float(np.max(t)),
            "efficiency_vs_1gpu": eff,
            # what crosses the bus per step and rank, measured (profiled run); the statistics and the histogram are
            # these many bytes of the device -> host total
            "h2d_bytes_measured": prof[leg]["memcpy"].get("HtoD", {}).get("bytes_per_step", 0),
            "d2h_bytes_measured": prof[leg]["memcpy"].get("DtoH", {}).get("bytes_per_step", 0),
            "stats_and_histogram_bytes": C.sizeof(L.bmo_spot_info) + BINS * BINS * 8,
            "profiled": prof[leg], "check": checks[leg],
        }
    result = {
        "workload": "C2: AC254-150-AB doublet + Spotdetector, UniformDiscSource 20 mm, r_max 100, 256 x 256 histogram over the detector face",
        "gpus": ws, "steps_per_leg": args.steps, "warmup": args.warmup, "nccl_version": comm.nccl_version(),
        "card_before": card_before, "card_after": card_after, "torch_device_name": torch.cuda.get_device_name(dev),
        "l2": "flushed with a 256 MiB write before every timed step", "timing": "CUDA events per rank ending in a synchronise; max over ranks",
        "baseline": args.baseline if base is not None else None, "legs": out_legs,
    }
    if rank == 0:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
        print(json.dumps(result, indent=1))
    comm.free()
    if dist:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
