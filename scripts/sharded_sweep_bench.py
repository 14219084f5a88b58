"""Photodetector pose sweep (BASELINE C5) sharded over GPUs by pose range, strong-scaled.

    torchrun --nproc_per_node=N scripts/sharded_sweep_bench.py --out FILE.json [--steps 5] [--warmup 1] [--only c5,c5_large]
    python scripts/sharded_sweep_bench.py --out FILE.json            (N = 1)

Workloads (the Mach-Zehnder of scripts/bench_configs.py, m1 moved along its normal over [0, 2 lambda] by a KinProgram on the
device, power only):
  c5:        one GaussianBeamlet (BASELINE C5's beam), 4096 poses, 256 x 256 Photodetector.
  c5_large:  16 beamlets of a 1 mm DeviceBeamletSource, 4096 poses, 512 x 512: 17.2 GB of fields on one GPU, the leg that shows
             what a rank holds.
Two legs alternate step by step after the warm-up, each timed per rank with CUDA events ending in a synchronise; a step's time is
the largest over the ranks.  The L2 is flushed (a 256 MiB write) before every step.
  sharded:   KinProgram.apply of the rank's shard_slice of the poses -> the beam tiled once per local pose -> trace ->
             bmo_pd_sweep_sharded (powers gathered on every rank, fields not requested).
  one_gpu:   what solve_pose_sweep_device does on the device for all poses on this rank's GPU: apply -> tiles -> trace ->
             bmo_pd_sweep.  The flattening and upload of the system are done once, outside both legs.  This is the 1-GPU run the
             efficiency is measured against: t_one_gpu / (N t_sharded).
Every rank checks its gathered powers against its one_gpu powers bit for bit.  Device memory per rank: the library keeps the blocks
a step freed (stream-ordered pool, parked large blocks), so the device memory in use after one step of a leg, started from a
trimmed pool, minus what was in use before it, is the most that step held at once (rounded up to the pool's size classes).  Card
name, power limit and SM clock are read in the same run, before and after.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
LAM = 1e-6


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
    ap.add_argument("--poses", type=int, default=4096)
    ap.add_argument("--only", default="c5,c5_large")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("sharded_sweep_bench.py: no CUDA device")
    import __graft_entry__ as ge
    m = ge.load_package()
    from bmo_b200 import _lib as L
    from bmo_b200 import parallel as par
    from bmo_b200 import sweep as sw
    from bmo_b200.flatten import FlatSystem
    from bmo_b200.solver import DeviceSystem
    from tests import scenes2 as s2
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
    comm = par.FieldComm.from_torch(device=dev) if ws > 1 else par.FieldComm(0, 1, par.FieldComm.unique_id(), dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    P = args.poses
    first, stop = par.shard_slice(P, rank, ws)
    count = stop - first

    def sync_ranks():
        torch.cuda.synchronize()
        if dist:
            dist.barrier()

    def gather(x, op):
        if not dist:
            return x
        t = torch.tensor([float(x)], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=op)
        return float(t.item())

    def used():
        free, total = torch.cuda.mem_get_info(dev)
        return total - free

    B = s2.MZI_BEAM
    results = {}
    for name in args.only.split(","):
        n = 256 if name == "c5" else 512
        sc = s2.mzi(m, pd_n=n)
        if name == "c5":
            beam = m.GaussianBeamlet(B["pos"], B["dir"], B["lam"], B["w0"], M2=B["M2"], P0=B["P0"], support=B["support"])
        else:
            src = m.UniformDiscSource(B["pos"], B["dir"], 1e-3, LAM, num_rays=16, e1=(1.0, 0.0, 0.0), on_device=True)
            beam = src.beamlets(w0=B["w0"], M2=1.0, P0=B["P0"] / 16, z0=0.0, support=B["support"])
        lams, lam_id, beam = sw._beamlet_lambdas(beam)
        shifts = np.array([s2.mzi_shift(p, P) for p in range(P)])
        f0 = FlatSystem(sc["system"], lams)
        dsys = {leg: DeviceSystem(f0, dev) for leg in ("sharded", "one_gpu")}
        prog = sw.KinProgram(f0, P)
        prog.translate3d_(sc["m1"], shifts)
        oi = f0.object_index(sc["pd"])
        power = {"sharded": np.zeros(P), "one_gpu": np.zeros(P)}

        def step(leg):
            e0 = torch.cuda.Event(enable_timing=True)
            e1 = torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            d = dsys[leg]
            if leg == "sharded":
                res = None
                if count:
                    prog.apply(d, first, count)
                    res = sw._trace_beamlet_sweep(d, beam, lam_id, count, 100)
                power[leg][:] = comm.pd_sweep(d, res, oi, P, first, count, want_fields=False)[0]
            else:
                prog.apply(d)
                res = sw._trace_beamlet_sweep(d, beam, lam_id, P, 100)
                L.check(lib.bmo_pd_sweep(d.h, res.h, oi, P, None, L.ptr(power[leg]), 0))
            e1.record(stream)
            torch.cuda.synchronize()
            if res is not None:
                res.free()
            return e0.elapsed_time(e1)

        legs = ("sharded", "one_gpu")
        mem = {}
        for leg in legs:               # first step of each leg from a trimmed pool: the device memory it holds
            sync_ranks()
            L.trim(dev)
            torch.cuda.synchronize()
            u0 = used()
            step(leg)
            mem[leg] = used() - u0
        for _ in range(args.warmup):
            for leg in legs:
                step(leg)
                sync_ranks()
        times = {leg: [] for leg in legs}
        for _ in range(args.steps):    # alternate the legs
            for leg in legs:
                flush.fill_(1)
                sync_ranks()
                times[leg].append(gather(step(leg), dist.ReduceOp.MAX if dist else None))
        same = power["sharded"].tobytes() == power["one_gpu"].tobytes()
        same = bool(gather(1.0 if same else 0.0, dist.ReduceOp.MIN if dist else None))
        med = {leg: float(np.median(times[leg])) for leg in legs}
        mem_most = {leg: int(gather(mem[leg], dist.ReduceOp.MAX if dist else None)) for leg in legs}
        out = {leg: {"step_ms_median": med[leg], "step_ms_min": float(np.min(times[leg])), "step_ms_max": float(np.max(times[leg])),
                     "device_bytes_held_by_one_step_max_over_ranks": mem_most[leg]} for leg in legs}
        out["sharded"]["efficiency_vs_1gpu"] = med["one_gpu"] / (ws * med["sharded"])
        out["sharded"]["speedup_vs_1gpu"] = med["one_gpu"] / med["sharded"]
        most = -(-P // ws)
        results[name] = {
            "workload": (f"C5 Mach-Zehnder, m1 over [0, 2 lambda] by a KinProgram, {P} poses, "
                         + ("one GaussianBeamlet" if name == "c5" else "16 beamlets of a 1 mm DeviceBeamletSource")
                         + f", {n} x {n} Photodetector, power only"),
            "rank_poses": [first, stop],
            "fields_bytes_from_shapes": {"one_gpu": P * n * n * 16, "sharded_largest_rank": most * n * n * 16},
            "power_bytes_gathered_per_rank_from_shapes": 8 * most * ws,
            "check": {"sharded_powers_bit_identical_to_one_gpu_on_every_rank": same},
            "legs": out,
        }
        del dsys, prog
        L.trim(dev)
    result = {
        "gpus": ws, "steps_per_leg": args.steps, "warmup": args.warmup, "nccl_version": comm.nccl_version(),
        "card_before": card_before, "card_after": card(dev), "torch_device_name": torch.cuda.get_device_name(dev),
        "l2": "flushed with a 256 MiB write before every timed step",
        "timing": "CUDA events per rank ending in a synchronise; step time is the max over ranks",
        "scaling_2_4_8_gpus": "see the files of runs with torchrun --nproc_per_node=N" if ws > 1 else "not measured",
        "workloads": results,
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
