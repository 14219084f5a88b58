"""PSFDetector map sharded over GPUs by pixel columns: bench.py's Airy-disc PSF scene (test/runtests.jl:2765-2802), strong-scaled,
at a size a user would run: one UniformDiscSource of 2^18 rays on a 1024 x 1024 map, crop_factor 5, :bbox window.

    torchrun --nproc_per_node=N scripts/sharded_psf_bench.py --out FILE.json [--steps 5] [--warmup 1] [--rays 262144] [--px 1024]
    python scripts/sharded_psf_bench.py --out FILE.json            (N = 1)

Two legs alternate step by step after the warm-up, each timed per rank with CUDA events ending in a synchronise; a step's time is
the largest over the ranks.  The L2 is flushed (a 256 MiB write) before every step.
  sharded:   bmo_source_create_slice (the rank's shard_slice) -> bmo_trace_rays -> bmo_psf_collect -> bmo_psf_allgather ->
             bmo_psf_lims -> bmo_psf_intensity_sharded (map to device memory), split by events into trace, collect, record
             gather, lims and the intensity call; the band kernel's own time is libbmo's event bracket of K6 (psf_ms), the rest of
             the call is the argument agreement and the map gather.
  one_gpu:   the same workload unsharded on this rank's GPU: whole source -> trace -> collect -> lims -> bmo_psf_intensity.  This is
             the 1-GPU run the efficiency is measured against: t_one_gpu / (N t_sharded).
Every rank checks its sharded map against the one_gpu map bit for bit.  The bytes exchanged per rank and step are computed from
shapes.  Card name, power limit and SM clock are read in the same run, before and after.
"""
import argparse
import ctypes as C
import hashlib
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
    ap.add_argument("--rays", type=int, default=1 << 18)
    ap.add_argument("--px", type=int, default=1024)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("sharded_psf_bench.py: no CUDA device")
    import __graft_entry__ as ge
    m = ge.load_package()
    from bmo_b200 import _lib as L
    from bmo_b200 import parallel as par
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

    lens = m.SphericalLens(100e-3, np.inf, 1e-3, 25.4e-3, 1.5)
    psfd = m.PSFDetector(10e-3)
    psfd.translate3d_([0.0, 200e-3 + 0.13e-3, 0.0])
    system = m.System([lens, psfd])
    dsys = m.upload_system(system, [LAMBDA], device=dev)
    oi = next(i for i, o in enumerate(dsys.flat.objects) if o is psfd)
    n_rays, n = args.rays, args.px
    src = m.UniformDiscSource((0.0, -10e-3, 0.0), (0.0, 1.0, 0.0), 15e-3, LAMBDA, num_rays=n_rays, e1=(1.0, 0.0, 0.0), on_device=True)
    first, stop = par.shard_slice(n_rays, rank, ws)
    j0, j1 = par.psf_shard_band(n, rank, ws)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    maps = {leg: torch.zeros(n * n, dtype=torch.float64, device="cuda") for leg in ("sharded", "one_gpu")}
    lims = np.zeros(4)
    counts = {}

    def ev():
        e = torch.cuda.Event(enable_timing=True)
        e.record(stream)
        return e

    def trace(first, count):
        """-> (bmo_psf handle or NULL, events after trace and after collect)"""
        s, h, psf = C.c_void_p(), C.c_void_p(), C.c_void_p()
        if count:
            L.check(lib.bmo_source_create_slice(ctx, C.byref(src.desc), first, count, C.byref(s)))
            nn, p, d, u = C.c_int64(), C.c_void_p(), C.c_void_p(), C.c_int32()
            L.check(lib.bmo_source_device(s, C.byref(nn), C.byref(p), C.byref(d), C.byref(u)))
            L.check(lib.bmo_trace_rays(dsys.h, nn.value, p, d, None, None, None, 100, L.KEEP_SEGMENTS | L.INPUT_DEVICE | L.UNIFORM_DIR, C.byref(h)))
        e_trace = ev()
        if count:
            L.check(lib.bmo_psf_collect(dsys.h, h, oi, C.byref(psf), None))
            lib.bmo_result_free(h)
            lib.bmo_source_free(s)
        return psf, e_trace, ev()

    def step(leg):
        e0 = ev()
        marks = {}
        if leg == "sharded":
            psf, marks["trace"], marks["collect"] = trace(first, stop - first)
            a = C.c_void_p()
            L.check(lib.bmo_psf_allgather(comm.h, psf, C.byref(a)))
            marks["record_gather"] = ev()
            L.check(lib.bmo_psf_lims(dsys.h, a, oi, 0, 5.0, 1, L.ptr(lims)))
            marks["lims"] = ev()
            L.check(lib.bmo_psf_intensity_sharded(comm.h, dsys.h, a, oi, 0, n, L.ptr(lims), 0.0, 0.0, C.c_void_p(maps[leg].data_ptr()),
                                                  L.INPUT_DEVICE))
            marks["band_kernel_and_map_gather"] = ev()
            band_ms = L.counters(dev)["psf_ms"] if j1 > j0 else 0.0
            cnt = C.c_int64()
            L.check(lib.bmo_psf_count(a, C.byref(cnt)))
            counts["records_total"] = int(cnt.value)
            if psf:
                L.check(lib.bmo_psf_count(psf, C.byref(cnt)))
                counts["records_this_rank"] = int(cnt.value)
            else:
                counts["records_this_rank"] = 0
            lib.bmo_psf_free(a)
        else:
            psf, marks["trace"], marks["collect"] = trace(0, n_rays)
            L.check(lib.bmo_psf_lims(dsys.h, psf, oi, 0, 5.0, 1, L.ptr(lims)))
            marks["lims"] = ev()
            L.check(lib.bmo_psf_intensity(dsys.h, psf, oi, 0, n, L.ptr(lims), 0.0, 0.0, C.c_void_p(maps[leg].data_ptr()), L.INPUT_DEVICE))
            marks["intensity"] = ev()
            band_ms = L.counters(dev)["psf_ms"]
        lib.bmo_psf_free(psf)
        torch.cuda.synchronize()
        parts, prev = {}, e0
        for k, e in marks.items():
            parts[k] = prev.elapsed_time(e)
            prev = e
        if leg == "sharded":
            parts["band_kernel"] = band_ms
            parts["agreement_and_map_gather"] = parts["band_kernel_and_map_gather"] - band_ms
        else:
            parts["kernel"] = band_ms
        return e0.elapsed_time(prev), parts

    def sync_ranks():
        torch.cuda.synchronize()
        if dist:
            dist.barrier()

    def timed(leg):
        flush.fill_(1)
        sync_ranks()
        t, parts = step(leg)
        if dist:
            x = torch.tensor([t], dtype=torch.float64, device="cuda")
            dist.all_reduce(x, op=dist.ReduceOp.MAX)
            t = float(x.item())
        return t, parts

    legs = ("sharded", "one_gpu")
    for _ in range(args.warmup):
        for leg in legs:
            step(leg)
            sync_ranks()
    times = {leg: [] for leg in legs}
    parts = {leg: [] for leg in legs}
    for _ in range(args.steps):        # alternate the legs
        for leg in legs:
            t, p = timed(leg)
            times[leg].append(t)
            parts[leg].append(p)
    same = maps["sharded"].cpu().numpy().tobytes() == maps["one_gpu"].cpu().numpy().tobytes()
    digest = hashlib.sha256(maps["sharded"].cpu().numpy().tobytes()).hexdigest()
    if dist:
        box = [None] * ws
        dist.all_gather_object(box, (same, digest))
        same = all(b[0] for b in box) and all(b[1] == box[0][1] for b in box)
    card_after = card(dev)

    pairs = float(counts["records_total"]) * n * n
    med = {leg: float(np.median(times[leg])) for leg in legs}
    most = counts["records_this_rank"]
    if dist:
        box = [None] * ws
        dist.all_gather_object(box, counts["records_this_rank"])
        most = max(box)
    B = -(-n // ws)
    out_legs = {}
    for leg in legs:
        t = times[leg]
        out_legs[leg] = {
            "step_ms_median": med[leg], "step_ms_min": float(np.min(t)), "step_ms_max": float(np.max(t)),
            "px_hits_per_s": pairs / (med[leg] * 1e-3),
            "split_ms_median_this_rank": {k: float(np.median([p[k] for p in parts[leg]])) for k in parts[leg][0]},
        }
    out_legs["sharded"]["efficiency_vs_1gpu"] = med["one_gpu"] / (ws * med["sharded"])
    out_legs["sharded"]["speedup_vs_1gpu"] = med["one_gpu"] / med["sharded"]
    other = (ws - 1) / ws          # the share of a gathered buffer that comes from other ranks (none with one rank: device copies)
    out_legs["sharded"]["bytes_from_other_ranks_per_rank_from_shapes"] = {
        "argument_words": int(other * 8 * ws * (2 + 11)),          # the two agreement all-gathers
        "records": int(other * 8 * ws * most * (9 + 5)),           # [most][9] records + [most][5] fast words per rank, padded
        "map_bands": int(other * 8 * ws * n * B),                  # n * B doubles per rank's band
        "map_to_host": 0,                                          # the map stays in device memory (BMO_INPUT_DEVICE)
    }
    result = {
        "workload": f"Airy-disc PSF scene (bench.py's PSF leg): UniformDiscSource 15 mm, {n_rays} rays, {counts['records_total']} PSF records, "
                    f"{n} x {n} map, crop_factor 5, :bbox window",
        "gpus": ws, "rank_columns": [j0, j1], "rank_rays": [first, stop], "steps_per_leg": args.steps, "warmup": args.warmup,
        "nccl_version": comm.nccl_version(), "card_before": card_before, "card_after": card_after,
        "torch_device_name": torch.cuda.get_device_name(dev),
        "l2": "flushed with a 256 MiB write before every timed step",
        "timing": "CUDA events per rank ending in a synchronise; step time is the max over ranks; split is rank 0's",
        "check": {"sharded_map_bit_identical_to_one_gpu_map_on_every_rank": bool(same)},
        "legs": out_legs,
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
