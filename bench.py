#!/usr/bin/env python
"""bench.py -- headline benchmark of the trace hot path (BASELINE.json configs[1], "C2"):
AC254-150-AB doublet spot diagram, 2^20 collimated rays (Fibonacci disc, 20 mm), sequential SDF
lens-surface path, Spotdetector at the vendor back focus.  Metric: ray-surface interactions/s.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

One "step" = one full solve_system! of the ray bundle (all waves).  `value` is measured with the rays
resident in HBM (device pointers into the C ABI, spot output left on the device); `e2e` goes through
the same C ABI with pinned HOST buffers, host->device and device->host copies inside the timed
region.  Rank r of an N-GPU run traces its own 2^20-ray shard (weak scaling, no data-path
collective: rays are independent, outputs are disjoint slices).

--dump-outputs DIR writes what the last timed step of each leg returned to its caller as DIR/<name>.npy
(rank 0's shard), so that two builds can be compared output for output; the inputs are fixed, so the same
arguments give the same inputs on every run:
    spot_xz, spot_object, nseg, interactions   resident leg: Spotdetector (x, z) per ray (NaN: no detector
                                               reached), detector object id (-1: none), segments per ray
    e2e_spot_xz, e2e_interactions              the same from the host-buffer leg
    detector_field, detector_pixel_index       C3 Photodetector field (re, im) at a fixed seeded sample of
                                               its pixels (column-major pixel index)
    ray_index                                  only with --rays above 2^20: the fixed seeded sample of rays
                                               the per-ray arrays hold
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_RAYS = 1 << 20
LAMBDA = 707e-9
WORKLOAD = "C2: AC254-150-AB doublet spot diagram, 2^20 collimated rays, Fibonacci disc d=20mm, Spotdetector at BFL"
CPU_SAMPLE = 1 << 14
# algorithmic FP64 work per unit (SURVEY 8(d) cost table): primitive SDF eval 45, triangle test 40, interaction 60
FLOP_SDF, FLOP_TRI, FLOP_INT = 45.0, 40.0, 60.0
# intersect_wave (lean build), 2^20 rays per launch: dram__bytes_read.sum + dram__bytes_write.sum, mean over the 4 waves of one C2
# solve (ncu --set full, profiles/r02l_ncu_k1_lean.txt).  Round 1 read 68.1 MB and wrote 89.0 MB (spill lines evicted from L1).
K1_DRAM_BYTES_PER_LAUNCH = 91.1e6
K1_TRAFFIC_SOURCE = ("profiles/r02l_ncu_k1_lean.txt (mean of the 4 waves, 2^20 rays per launch: 67.2 MB read + 23.9 MB written; algorithmic = 64 B ray "
                     "state read + 36 B hit record written per ray -- part of the hit records is still in the 126 MB L2 when the kernel ends)")
# --dump-outputs: at most this many bytes in all; per-ray arrays keep at most DUMP_RAYS rows, the detector field DUMP_PIXELS pixels
DUMP_BYTES, DUMP_RAYS, DUMP_PIXELS = 64 << 20, 1 << 20, 1 << 18


def rays_for_rank(rank, n=N_RAYS):
    """Fibonacci disc of this rank's shard; ranks get discs rotated by the golden angle so shards differ."""
    from tests import scenes
    pos, d = scenes.fibonacci_disc(n)
    if rank:
        a = rank * 0.1
        c, s = math.cos(a), math.sin(a)
        x, z = pos[:, 0].copy(), pos[:, 2].copy()
        pos[:, 0], pos[:, 2] = c * x - s * z, s * x + c * z
    return np.ascontiguousarray(pos), np.ascontiguousarray(d)


def sample_index(n, cap, seed):
    """Rows kept by --dump-outputs: all n, or a fixed seeded sample of `cap` of them in ascending order."""
    if n <= cap:
        return np.arange(n)
    return np.sort(np.random.default_rng(seed).choice(n, cap, replace=False))


def dump_outputs(path, arrays):
    """Writes each array as <path>/<name>.npy; all are float32 / float64 and DUMP_BYTES at most together."""
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BYTES:
        raise SystemExit(f"bench.py: --dump-outputs would write {total} bytes, more than {DUMP_BYTES}")
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(path, name + ".npy"), a)


def bind_to_gpu_numa(local_rank):
    """Pin this process (and the threads it starts later) to the CPUs of the NUMA node the rank's GPU hangs off, before
    anything allocates pinned host memory: Linux places the pages of cudaHostAlloc on the node of the allocating CPU, and
    a rank whose staging buffers sit on the other socket pays the inter-socket link on every host<->device copy.
    Returns a description for the JSON line (None: topology unknown, nothing changed)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:          # NVML prints an 8-digit PCI domain, sysfs a 4-digit one
            bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0)
        use = cpus & allowed
        if not use:
            return {"numa_node": node, "bound": False, "why": "no allowed CPU on the GPU's node"}
        os.sched_setaffinity(0, use)
        return {"numa_node": node, "bound": True, "cpus": len(use)}
    except Exception as e:      # no NVML / no sysfs topology: leave the affinity alone
        return {"bound": False, "why": type(e).__name__}


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons of the rank's GPU, sampled through NVML every 5 ms for as long as the bench runs
    (nvidia-smi, one process per sample, is the fallback)."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag, self.sm_max = index, [], False, None
        self.marks = {}          # name -> (first sample, one past the last sample) of a timed region

    def mark(self, name, begin):
        lo, hi = self.marks.get(name, (len(self.samples), len(self.samples)))
        self.marks[name] = (len(self.samples), hi) if begin else (lo, len(self.samples))

    def run(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            bits = [getattr(pynvml, n, 0) for n in ("nvmlClocksEventReasonHwSlowdown", "nvmlClocksEventReasonHwThermalSlowdown",
                                                    "nvmlClocksEventReasonSwThermalSlowdown", "nvmlClocksEventReasonSwPowerCap")]
            fallback = [0x8, 0x40, 0x20, 0x4]
            bits = [b or f for b, f in zip(bits, fallback)]
            get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
            while not self.stop_flag:
                mhz = float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                r = int(get_reasons(h))
                self.samples.append((mhz, [bool(r & b) for b in bits]))
                time.sleep(0.005)
            return
        except Exception:
            pass
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    f = [x.strip() for x in out.split(",")]
                    self.sm_max = float(f[1])
                    self.samples.append((float(f[0]), [x.lower().startswith("active") for x in f[2:6]]))
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        def part(lo, hi):
            sel = self.samples[lo:hi] or self.samples
            mhz = sorted(x[0] for x in sel)
            return {"sm_mhz": mhz[len(mhz) // 2], "sm_mhz_min": mhz[0], "samples": len(sel),
                    "reasons": [n for k, n in enumerate(self.NAMES) if any(x[1][k] for x in sel)]}
        out = part(0, len(self.samples))
        out["sm_max_mhz"] = self.sm_max
        out["how"] = "NVML every 5 ms over the whole run; per-leg medians under `legs`"
        out["legs"] = {k: part(lo, hi) for k, (lo, hi) in self.marks.items() if hi > lo}
        return out


def run_reference(args, rank):
    """Reference arm: the reference's CPU algorithm for this path (oracle port: Julia is not installed
    and the reference has no compiled component) on all host cores, bounded sample per step."""
    if rank != 0:
        return
    import __graft_entry__ as ge
    ge.build_oracle()
    from oracle import oracle as orc
    from tests import scenes
    cores = os.cpu_count() or 1
    osc = scenes.doublet_spot_oracle()
    pos, d = rays_for_rank(0, N_RAYS)
    sel = np.linspace(0, N_RAYS - 1, CPU_SAMPLE).astype(np.int64)   # evenly spread over the pupil
    pos, d = np.ascontiguousarray(pos[sel]), np.ascontiguousarray(d[sel])
    times, inter = [], 0
    for it in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        r = orc.bulk_trace_rays(osc["system"], pos, d, LAMBDA, r_max=100, nthreads=cores, want_segments=False, spot=osc["spot"])
        dt = time.perf_counter() - t0
        if it >= args.warmup:
            times.append(dt)
            inter = r["interactions"]
    total = sum(times)
    value = inter * len(times) / total
    sample = f"{CPU_SAMPLE} of {N_RAYS} rays per step (evenly spaced over the pupil), threaded driver over rays (BASELINE.md B2/B3)"
    print(json.dumps({
        "impl": "reference", "metric": "ray-surface interactions/s", "value": value, "unit": "interactions/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "rays_per_gpu": N_RAYS, "r_max": 100},
        "cpu_baseline": {"value": value, "unit": "interactions/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "interactions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rays", type=int, default=N_RAYS)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-detector", action="store_true", help="skip the secondary Photodetector (C3) measurement")
    ap.add_argument("--c3-side", type=int, default=256, help="beamlets per side of the C3 lattice (256 = the full 65536-beamlet config), split over the ranks")
    ap.add_argument("--c3-pixels", type=int, default=2048)
    ap.add_argument("--no-extras", action="store_true", help="skip the secondary retrace (a4) and PSFDetector (N2) measurements")
    ap.add_argument("--no-numa", action="store_true", help="leave the CPU affinity of the rank alone")
    ap.add_argument("--full-inputs", action="store_true", help="e2e ships a direction and a wavelength id per ray (52 B/ray) instead of one of each per bundle")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step of each leg as DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    # stdout carries exactly one JSON line: native libraries that print to fd 1 (NCCL's version banner) go to stderr
    sys.stdout.flush()
    json_out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    numa = None if args.no_numa else bind_to_gpu_numa(local_rank)     # before torch starts threads / pins memory
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    import __graft_entry__ as ge
    if rank == 0:
        ge.build_libbmo()
    if world > 1:
        dist.barrier()
    m = ge.load_package()
    from bmo_b200 import _lib as L
    from tests import scenes
    dev = local_rank
    n = args.rays
    stream = torch.cuda.current_stream()
    L.set_stream(stream.cuda_stream, dev)
    comm = m.parallel.FieldComm.from_torch(device=dev) if world > 1 else None     # NCCL behind the C ABI (bmo_comm_init)

    sc = scenes.doublet_spot(m)
    dsys = m.upload_system(sc["system"], [LAMBDA], device=dev)       # system upload: outside the timed region
    pos_h, dir_h = rays_for_rank(rank, n)
    lam_h = np.zeros(n, dtype=np.int32)
    # pinned host buffers (e2e) and resident device copies (value)
    pin = lambda a: torch.from_numpy(a).pin_memory()
    pos_p, dir_p, lam_p = pin(pos_h), pin(dir_h), pin(lam_h)
    dir1_p = pin(np.ascontiguousarray(dir_h[0]))                      # the one direction of the collimated bundle
    pos_d, dir_d, lam_d = pos_p.cuda(non_blocking=True), dir_p.cuda(non_blocking=True), lam_p.cuda(non_blocking=True)
    spot_obj_p = torch.empty(n, dtype=torch.int32).pin_memory()
    spot_xz_p = torch.empty((n, 2), dtype=torch.float64).pin_memory()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")   # > 126 MB L2
    torch.cuda.synchronize()

    kept = []      # the newest resident result: freed when the next step starts, so the last one is still there for --dump-outputs

    def step_device():
        while kept:
            kept.pop().free()
        res = m.trace_rays(dsys, (pos_d.data_ptr(), n), dir_d.data_ptr(), lam_d.data_ptr(), None, None, 100,
                           keep_segments=False, device_inputs=True)
        kept.append(res)
        return res.interactions

    import ctypes as C
    if args.full_inputs:
        e2e_args = (C.c_void_p(dir_p.data_ptr()), C.c_void_p(lam_p.data_ptr()), 0, C.c_void_p(spot_obj_p.data_ptr()))
        h2d, d2h = int(pos_h.nbytes + dir_h.nbytes + lam_h.nbytes), int(n * 4 + n * 16)
        e2e_inputs = "pos, dir [n][3] f64 + lambda id [n] i32 in; detector id [n] i32 + spot (x,z) [n][2] f64 out"
    else:
        # a collimated bundle: one direction and one wavelength for all rays (BMO_UNIFORM_DIR, lambda_id = NULL); the spot of a
        # ray that reached no detector comes back as NaN, so the per-ray detector id is not requested
        e2e_args = (C.c_void_p(dir1_p.data_ptr()), None, L.UNIFORM_DIR, None)
        h2d, d2h = int(pos_h.nbytes + 24), int(n * 16)
        e2e_inputs = "pos [n][3] f64 + one direction [3] (BMO_UNIFORM_DIR) in; spot (x,z) [n][2] f64 out (NaN = no detector reached)"

    def step_e2e():
        h = C.c_void_p()
        # solve_system! + Spotdetector.data in one C-ABI call: host buffers in, host buffers out
        L.check(L.lib().bmo_trace_rays_spots(dsys.h, n, C.c_void_p(pos_p.data_ptr()), e2e_args[0], e2e_args[1],
                                             None, None, 100, e2e_args[2], e2e_args[3], C.c_void_p(spot_xz_p.data_ptr()), C.byref(h)))
        info = L.bmo_result_info()
        L.check(L.lib().bmo_result_get_info(h, C.byref(info)))
        L.lib().bmo_result_free(h)
        return info.interactions

    sampler = ClockSampler(dev)

    def timed(fn, steps, warmup, leg, together=True):
        for _ in range(warmup):
            fn()
        L.counters_reset(dev)                    # per-kernel counters cover the timed steps only
        times, inter = [], 0
        sampler.mark(leg, True)
        for _ in range(steps):
            flush.fill_(1)                       # evict inputs from L2 between timed iterations
            torch.cuda.synchronize()
            if world > 1 and together:
                dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            inter = fn()
            e1.record(stream)
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1))
        sampler.mark(leg, False)
        return times, inter

    if rank == 0:
        sampler.start()
    times, inter = timed(step_device, args.steps, args.warmup, "trace_resident")
    c = L.counters(dev)
    dump = {} if args.dump_outputs and rank == 0 else None
    last = kept.pop()
    if dump is not None:
        rows = sample_index(n, DUMP_RAYS, seed=1)
        obj, xz = last.spots()
        dump.update(spot_xz=xz[rows], spot_object=obj[rows].astype(np.float32),
                    nseg=last.beams()["nseg"][rows].astype(np.float32), interactions=np.array([last.interactions], np.float64))
        if len(rows) < n:
            dump["ray_index"] = rows.astype(np.float64)
    last.free()
    n_total_steps = args.steps
    solo_ms = None
    if world > 1:
        # the same end-to-end step on rank 0 alone, the other ranks idle: the denominator of the weak-scaling efficiency of e2e
        if rank == 0:
            t_solo, _ = timed(step_e2e, args.steps, args.warmup, "trace_e2e_solo", together=False)
            solo_ms = sum(t_solo) / len(t_solo)
        dist.barrier()
    times_e, inter_e = timed(step_e2e, args.steps, args.warmup, "trace_e2e")
    if dump is not None:
        dump.update(e2e_spot_xz=spot_xz_p.numpy()[rows], e2e_interactions=np.array([inter_e], np.float64))

    def agg(times):
        t = torch.tensor([sum(times)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)    # max over ranks
        return float(t.item())
    tot_ms, tot_ms_e = agg(times), agg(times_e)
    it = torch.tensor([float(inter), float(inter_e)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(it, op=dist.ReduceOp.SUM)
    inter_all, inter_all_e = float(it[0].item()), float(it[1].item())

    peak = L.measure_fp64_peak(dev)
    parity = multi_gpu_parity(m, L, dev, comm, rank, world) if world > 1 else None
    # the retrace leg runs before the detector leg: after the detector's 64 MiB fields have gone through the stream-ordered pool
    # the retrace's wave buffers (4 x 100 MB per call) hit a fragmented pool and its timings scatter between 6 and 30 ms
    extras = None
    if rank == 0 and not args.no_extras:
        extras = {"retrace": bench_retrace(m, L, dev, stream, dsys, sc, pos_d, dir_d, lam_d, n, flush)}
    det = None
    if not args.no_detector:
        sampler.mark("detector", True)
        det = bench_detector(m, L, dev, stream, args.c3_side, args.c3_pixels, 2, 1, flush, peak, rank, world, comm, dump)
        sampler.mark("detector", False)
    if extras is not None:
        extras["psf"] = bench_psf(m, L, dev, stream, flush, peak)
    if rank == 0:
        value = inter_all * args.steps / (tot_ms * 1e-3)
        e2e = inter_all_e * args.steps / (tot_ms_e * 1e-3)
        # roofline of the dominant kernel (trace_step, FP64-pipe bound): algorithmic flops per launch / mean launch time
        flops = (FLOP_SDF * c["sdf_evals"] + FLOP_TRI * c["tri_tests"] + FLOP_INT * c["interactions"])
        k1_ms, k1_n = c["trace_step_ms"], max(c["trace_step_launches"], 1)
        achieved = flops / (k1_ms * 1e-3) / 1e12 if k1_ms > 0 else None
        hbm_peak = None
        try:
            hbm_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
        except Exception:
            hbm_peak = 6650.0
        comp = bench_compaction(m, L, dev, dsys, n, hbm_peak)
        sampler.stop_flag = True
        e2e_ms = tot_ms_e / args.steps
        out = {
            "metric": "ray-surface interactions/s", "value": value, "unit": "interactions/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": tot_ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "rays_per_gpu": n, "r_max": 100, "l2": "flushed with a 256 MiB write between timed iterations",
                       "outputs": "spot (x,z) per ray; segment table not kept"},
            "e2e": {"value": e2e, "unit": "interactions/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "buffers": e2e_inputs,
                    "solo_ms_per_step": solo_ms,
                    "weak_scaling_efficiency": (solo_ms / e2e_ms) if solo_ms else None,
                    "efficiency_note": "rank 0's e2e step alone on the box / the same step with all ranks running (max over ranks)" if solo_ms else None},
            "gpu_launches": int(c["kernel_launches"] * args.steps / n_total_steps),
            "roofline": {"bound": "fp64", "kernel": "intersect_wave", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                         "frac": (achieved / peak) if achieved else None,
                         # dram__bytes_read.sum + dram__bytes_write.sum per launch, mean of the 4 waves of one solve, from the
                         # ncu --set full capture named in traffic_source
                         "traffic": K1_DRAM_BYTES_PER_LAUNCH * n / N_RAYS, "traffic_algorithmic": 100.0 * n,
                         "traffic_source": K1_TRAFFIC_SOURCE,
                         "peak_source": "measured here: DFMA probe (bmo_measure_fp64_peak); MEASURED_PEAKS.json has no FP64 entry",
                         "flops_per_launch": flops / k1_n, "ms_per_launch": k1_ms / k1_n,
                         "share_of_step": k1_ms / n_total_steps / (tot_ms / args.steps) if tot_ms else None,
                         "counted": {"sdf_evals_per_step": c["sdf_evals"] / n_total_steps, "interactions_per_step": c["interactions"] / n_total_steps}},
            "roofline_compaction": comp,
            "clocks": sampler.summary(),
            "numa": numa,
        }
        if parity is not None:
            out.update(parity)
        if det is not None:
            out["detector"] = det
        if extras is not None:
            out.update(extras)
        if not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline()
        if dump is not None:
            dump_outputs(args.dump_outputs, dump)
        print(json.dumps(out), file=json_out)
        json_out.flush()
    if comm is not None:
        comm.free()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def multi_gpu_parity(m, L, dev, comm, rank, world, k=16, pd_n=256):
    """N > 1: the field of a small C3 lattice (k^2 beamlets, pd_n^2 pixels) sharded over the ranks and summed with
    bmo_pd_allreduce, against the same lattice traced and accumulated by rank 0 alone.  Relative L2 of the difference."""
    import ctypes as C
    import torch
    import torch.distributed as dist
    from tests import scenes2 as s2
    sc = s2.expander(m, pd_n)
    lat = s2.beamlet_lattice(k, aperture=8e-3 * k / 256)
    bundle = m.BeamletBundle.from_params(lat["pos"], lat["dir"], lat["lam"], lat["w0"], M2=lat["M2"], P0=1e-3 / 65536, support=lat["support"])
    dsys = m.upload_system(sc["system"], [lat["lam"]], device=dev)
    pd_index = dsys.flat.object_index(sc["pd"])
    nb = k * k

    def field_of(idx):
        f = torch.zeros(pd_n * pd_n * 2, dtype=torch.float64, device="cuda")
        if len(idx):
            res = m.trace_beamlets(dsys, np.ascontiguousarray(bundle.rays[idx]), np.zeros(len(idx), np.int32), np.ascontiguousarray(bundle.w0[idx]),
                                   np.ascontiguousarray(bundle.E0[idx]))
            L.check(L.lib().bmo_pd_accumulate(dsys.h, res.h, pd_index, 0, C.c_void_p(f.data_ptr()), L.INPUT_DEVICE))
            res.free()
        torch.cuda.synchronize()
        return f
    mine = np.arange(rank, nb, world)                 # interleaved shards
    f = field_of(mine)
    comm.allreduce(int(f.data_ptr()), pd_n * pd_n, sync=True)
    rel = torch.zeros(1, dtype=torch.float64, device="cuda")
    if rank == 0:
        ref = field_of(np.arange(nb))
        rel[0] = torch.linalg.norm(f - ref) / torch.linalg.norm(ref)
    dist.all_reduce(rel, op=dist.ReduceOp.MAX)
    return {"multi_gpu_parity_rel_l2": float(rel.item()),
            "multi_gpu_parity": f"{nb}-beamlet C3 lattice on a {pd_n}^2 Photodetector: field of the interleaved shards summed by bmo_pd_allreduce (NCCL {comm.nccl_version()} inside libbmo.so) "
                                f"vs the whole lattice on rank 0 alone; tolerance 1e-8 (addition order across ranks differs)"}


FLOP_PAIR_REF = 760.0   # flop-equivalents per pixel-beamlet pair in the reference's operation sequence (SURVEY 8(d))
FLOP_PAIR = 226.0       # the same weights (add/mul 1, sqrt/div 8, transcendental 40) over the strength-reduced sequence of
                        # pd_field_fast, counted op by op in DESIGN.md "K4" -- the work the kernel actually has to do


def bench_detector(m, L, dev, stream, k_side, pd_n, steps, warmup, flush, peak_tflops, rank=0, world=1, comm=None, dump=None):
    """Metric 2 (Photodetector px-beamlets/s) on the C3 workload: Keplerian expander + Photodetector(40 mm, pd_n), the
    k_side x k_side beamlet lattice (pitch 8 mm / 256, w0 = 1.5 pitch, lambda = 1 um; k_side = 256 is BASELINE's 65536-beamlet
    config).  STRONG scaling: the lattice is cut into `world` bands of rows, rank r traces and accumulates band r onto a full
    partial field, and the partial fields are summed by bmo_pd_allreduce (NCCL inside libbmo.so) inside the timed region.
    `dump` (a dict, --dump-outputs) receives a fixed sample of the field the last timed step left on the device."""
    import ctypes as C
    import torch
    from tests import scenes2 as s2
    sc = s2.expander(m, pd_n)
    import torch.distributed as dist
    lat = s2.beamlet_lattice(k_side, aperture=8e-3 * k_side / 256)
    nb_all = k_side * k_side
    lo, hi = rank * nb_all // world, (rank + 1) * nb_all // world
    nb = hi - lo
    sel = slice(lo, hi)
    bundle = m.BeamletBundle.from_params(lat["pos"][sel], lat["dir"], lat["lam"], lat["w0"], M2=lat["M2"], P0=1e-3 / 65536, support=lat["support"])
    dsys = m.upload_system(sc["system"], [lat["lam"]], device=dev)
    res = m.trace_beamlets(dsys, bundle.rays, np.zeros(nb, np.int32), bundle.w0, bundle.E0)
    pd_index = dsys.flat.object_index(sc["pd"])
    field_d = torch.zeros(pd_n * pd_n * 2, dtype=torch.float64, device="cuda")
    field_h = torch.zeros(pd_n * pd_n * 2, dtype=torch.float64).pin_memory()

    def run_device():
        field_d.zero_()                      # partial field of this rank
        L.check(L.lib().bmo_pd_accumulate(dsys.h, res.h, pd_index, 0, C.c_void_p(field_d.data_ptr()), L.INPUT_DEVICE))
        if world > 1:
            stream.synchronize()             # the library reduces on its context stream (= this stream); keep the order explicit
            comm.allreduce(int(field_d.data_ptr()), pd_n * pd_n, sync=False)

    def run_e2e():
        if world == 1:
            # pd.field (host) += field of the bundle: the C-ABI call with a host field copies it in, accumulates, copies it out
            L.check(L.lib().bmo_pd_accumulate(dsys.h, res.h, pd_index, 0, C.c_void_p(field_h.data_ptr()), 0))
        else:
            run_device()
            field_h.copy_(field_d, non_blocking=True)   # every rank ends with the whole field in host memory

    out = {}
    for name, fn in (("device", run_device), ("e2e", run_e2e)):
        for _ in range(warmup):
            fn()
        L.counters_reset(dev)
        times = []
        for _ in range(steps):
            flush.fill_(1)
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            fn()
            e1.record(stream)
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1))
        c = L.counters(dev)
        tot = torch.tensor([sum(times) / steps], dtype=torch.float64, device="cuda")
        pr = torch.tensor([c["px_beamlets"] / steps], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tot, op=dist.ReduceOp.MAX)       # max over ranks
            dist.all_reduce(pr, op=dist.ReduceOp.SUM)        # whole-job pairs
        out[name] = dict(ms=float(tot.item()), pairs=float(pr.item()), k4_ms=c["pd_field_ms"] / steps, launches=c["kernel_launches"] / steps,
                         pairs_rank=c["px_beamlets"] / steps)
    pairs = out["device"]["pairs"]
    ach = FLOP_PAIR * out["device"]["pairs_rank"] / (out["device"]["k4_ms"] * 1e-3) / 1e12
    res.free()
    if dump is not None:
        px = sample_index(pd_n * pd_n, DUMP_PIXELS, seed=2)
        dump.update(detector_field=field_d.view(-1, 2).cpu().numpy()[px], detector_pixel_index=px.astype(np.float64))
    nbytes = int(field_h.numel() * 8)
    return {
        "metric": "Photodetector px-beamlets/s", "unit": "px-beamlets/s",
        "value": pairs / (out["device"]["ms"] * 1e-3), "ms_per_step": out["device"]["ms"],
        "e2e": {"value": out["e2e"]["pairs"] / (out["e2e"]["ms"] * 1e-3), "ms_per_step": out["e2e"]["ms"],
                "h2d_bytes_per_step": nbytes if world == 1 else 0, "d2h_bytes_per_step": nbytes,
                "what": "bmo_pd_accumulate onto a pinned host field (copied in, accumulated, copied out)" if world == 1 else
                        "partial field on the device, bmo_pd_allreduce, whole field copied to pinned host memory on every rank"},
        "config": {"workload": f"C3: Keplerian beam expander, {nb_all} GaussianBeamlets ({k_side}x{k_side} lattice) onto a {pd_n}^2 Photodetector, coherent field sum"
                               + (f"; {nb} beamlets per GPU, all-reduce of the {pd_n}^2 complex128 field over {world} GPUs inside the timed region" if world > 1 else ""),
                   "beamlets": nb_all, "beamlets_per_gpu": nb, "pixels": pd_n * pd_n, "pairs_per_step": pairs},
        "n_gpus": world, "scaling": "strong",
        "gpu_launches": out["device"]["launches"],
        "roofline": {"bound": "fp64", "kernel": "pd_field_fast", "achieved": ach, "peak": peak_tflops, "unit": "TFLOP/s (FP64 flop-equivalents)",
                     "frac": ach / peak_tflops if peak_tflops else None, "ms_per_launch": out["device"]["k4_ms"],
                     "flop_equiv_per_pair": FLOP_PAIR, "reference_sequence_flop_equiv_per_pair": FLOP_PAIR_REF,
                     "achieved_in_reference_sequence_units": ach * FLOP_PAIR_REF / FLOP_PAIR,
                     "share_of_step": out["device"]["k4_ms"] / out["device"]["ms"]},
    }


def _time_ms(fn, stream, flush, steps=5, warmup=2):
    import torch
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(steps):
        flush.fill_(1)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        fn()
        e1.record(stream)
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    print(f"[bench] {getattr(fn, '__name__', 'step')}: ms per step {['%.3f' % t for t in ts]}", file=sys.stderr)
    return sorted(ts)[len(ts) // 2]      # median of the timed steps


def bench_retrace(m, L, dev, stream, dsys, sc, pos_d, dir_d, lam_d, n, flush):
    """SURVEY 8(a) row a4: solve_system!(...; retrace=true) of the solved C2 bundle (bmo_retrace: every stored ray
    re-validated against the object it hit before) next to a fresh non-sequential solve that keeps the same outputs
    (segment table kept in both: the retrace needs the stored path)."""
    prev = m.trace_rays(dsys, (pos_d.data_ptr(), n), dir_d.data_ptr(), lam_d.data_ptr(), None, None, 100, keep_segments=True, device_inputs=True)
    prev.keep = True
    inter = {}

    def fresh():
        r = m.trace_rays(dsys, (pos_d.data_ptr(), n), dir_d.data_ptr(), lam_d.data_ptr(), None, None, 100, keep_segments=True, device_inputs=True)
        inter["fresh"] = r.interactions
        r.free()

    def again():
        r = m.retrace(dsys, prev, 100, keep_segments=True)
        inter["retrace"] = r.interactions
        r.free()
    ms_f = _time_ms(fresh, stream, flush)
    L.counters_reset(dev)
    ms_r = _time_ms(again, stream, flush, steps=5, warmup=2)
    c = L.counters(dev)
    prev.free()
    return {"workload": "C2 bundle, 2^20 rays already solved, same poses: bmo_retrace vs a fresh bmo_trace_rays, segment table kept by both, rays resident in HBM",
            "fresh_ms": ms_f, "retrace_ms": ms_r, "interactions": inter.get("retrace"), "interactions_fresh": inter.get("fresh"),
            "retrace_interactions_per_s": inter.get("retrace", 0) / (ms_r * 1e-3),
            "sdf_evals_per_retrace": c["sdf_evals"] / 7.0}


FLOP_PSF_PAIR = 48.0    # per pixel-hit pair: 3 FMA phase, sincos as 40 (the transcendental weight of SURVEY 8(d)), 2 FMA accumulate


def bench_psf(m, L, dev, stream, flush, peak_tflops, n_rays=1 << 16, n_px=512):
    """N2: PSFDetector intensity map (PSFDetector.jl:190-237) of the reference's Airy-disc scene (test/runtests.jl:2765-2802)
    with 2^16 rays on a 512^2 grid: pixel-hit pairs/s of psf_intensity_kernel."""
    import ctypes as C
    import torch
    from tests import scenes
    lens = m.SphericalLens(100e-3, math.inf, 1e-3, 25.4e-3, 1.5)
    psfd = m.PSFDetector(10e-3)
    psfd.translate3d_([0.0, 200e-3 + 0.13e-3, 0.0])
    system = m.System([lens, psfd])
    pos, d = scenes.fibonacci_disc(n_rays, diameter=15e-3, y0=-10e-3)
    res = m.solve_system_(system, m.RayBundle(pos, d, 1e-6))
    hits = len(psfd)
    dsys, oi = psfd._dsys, psfd._index
    lims = np.array(psfd.calc_local_lims(5.0, "bbox"))
    out_d = torch.zeros(n_px * n_px, dtype=torch.float64, device="cuda")
    out_h = torch.zeros(n_px * n_px, dtype=torch.float64).pin_memory()

    def run(ptr, flags):
        L.check(L.lib().bmo_psf_intensity(dsys.h, C.c_void_p(psfd._psf), oi, 0, n_px, L.ptr(lims), 0.0, 0.0, C.c_void_p(ptr), flags))
    ms_d = _time_ms(lambda: run(out_d.data_ptr(), L.INPUT_DEVICE), stream, flush, steps=3, warmup=1)
    k_ms = L.counters(dev)["psf_ms"]
    ms_h = _time_ms(lambda: run(out_h.data_ptr(), 0), stream, flush, steps=3, warmup=1)
    pairs = float(hits) * n_px * n_px
    ach = FLOP_PSF_PAIR * pairs / (k_ms * 1e-3) / 1e12
    psfd.empty_()
    res.free()
    return {"metric": "PSFDetector px-hits/s", "value": pairs / (ms_d * 1e-3), "ms_per_step": ms_d,
            "e2e": {"value": pairs / (ms_h * 1e-3), "ms_per_step": ms_h, "h2d_bytes_per_step": 32, "d2h_bytes_per_step": n_px * n_px * 8},
            "config": {"workload": f"Airy-disc scene of test/runtests.jl:2765-2802, {hits} ray hits, {n_px}^2 pixels, crop_factor 5, :bbox window"},
            "roofline": {"bound": "fp64", "kernel": "psf_intensity_kernel", "achieved": ach, "peak": peak_tflops, "unit": "TFLOP/s (FP64 flop-equivalents)",
                         "frac": ach / peak_tflops if peak_tflops else None, "ms_per_launch": k_ms, "flop_equiv_per_pair": FLOP_PSF_PAIR}}


def bench_compaction(m, L, dev, dsys, n, hbm_peak):
    """K3 (queue compaction, HBM-bound) does not run in C2 proper -- every ray lives for all 4 waves.  Overfilling the pupil
    (disc of 40 mm on the 25.4 mm doublet: 60 % of the rays miss everything on the first wave) makes the dead slots the
    majority, which triggers one compaction of the queue; achieved GB/s = algorithmic bytes / CUDA-event time.  Measured on
    the 2^20-slot queue of the headline bundle (75 MB: launch + grid-barrier latency is a third of the time) and on a
    2^23-slot queue (604 MB), where the bytes are what bounds it."""
    import torch
    from tests import scenes

    def one(nq):
        pos, d = scenes.fibonacci_disc(nq, diameter=40e-3)
        pos_d, dir_d = torch.from_numpy(pos).cuda(), torch.from_numpy(d).cuda()
        lam_d = torch.zeros(nq, dtype=torch.int32, device="cuda")
        best = None
        for it in range(4):
            L.counters_reset(dev)
            res = m.trace_rays(dsys, (pos_d.data_ptr(), nq), dir_d.data_ptr(), lam_d.data_ptr(), None, None, 100, keep_segments=False, device_inputs=True)
            res.free()
            c = L.counters(dev)
            if it and c["scatter_ms"] > 0:
                gbs = c["scatter_bytes"] / (c["scatter_ms"] * 1e-3) / 1e9
                best = gbs if best is None else max(best, gbs)
        return best

    best, big = one(n), one(8 * n)
    return {"bound": "hbm", "kernel": "compact_fused (one cooperative launch: count, grid barrier, offsets, scatter)", "achieved": best, "peak": hbm_peak,
            "unit": "GB/s", "frac": (best / hbm_peak) if best else None, "peak_source": "MEASURED_PEAKS.json hbm_gbs",
            "workload": f"C2 doublet with an overfilled pupil (40 mm disc): one compaction of the {n}-slot queue to the ~40 % live rays",
            "large_queue": {"slots": 8 * n, "achieved": big, "frac": (big / hbm_peak) if big else None}}


def cpu_baseline():
    """The oracle port on the host cores over a bounded sample of the same workload (~10-30 s of CPU work)."""
    import __graft_entry__ as ge
    ge.build_oracle()
    from oracle import oracle as orc
    from tests import scenes
    cores = os.cpu_count() or 1
    osc = scenes.doublet_spot_oracle()
    pos, d = rays_for_rank(0, N_RAYS)
    sel = np.linspace(0, N_RAYS - 1, CPU_SAMPLE).astype(np.int64)
    pos, d = np.ascontiguousarray(pos[sel]), np.ascontiguousarray(d[sel])
    t0 = time.perf_counter()
    reps, inter = 0, 0
    while reps < 2 or time.perf_counter() - t0 < 10.0:
        inter += orc.bulk_trace_rays(osc["system"], pos, d, LAMBDA, r_max=100, nthreads=cores, want_segments=False, spot=osc["spot"])["interactions"]
        reps += 1
        if reps >= 8:
            break
    dt = time.perf_counter() - t0
    return {"value": inter / dt, "unit": "interactions/s", "cores": cores, "kind": "port",
            "sample": f"{reps} x {CPU_SAMPLE} of {N_RAYS} rays (evenly spaced over the pupil), OpenMP threaded driver over rays; "
                      "restatement of the Julia reference (Julia is not installed), not the reference itself"}


if __name__ == "__main__":
    main()
