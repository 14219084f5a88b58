"""Spot-diagram pose sweep sharded over GPUs by pose range, strong-scaled.

    torchrun --nproc_per_node=N scripts/sharded_spot_sweep_bench.py --out FILE.json [--steps 5] [--warmup 1]
    python scripts/sharded_spot_sweep_bench.py --out FILE.json            (N = 1)

Workloads (DESIGN §10's): the Spotdetector of the C2 doublet (AC254-150-AB, 707 nm, UniformDiscSource 20 mm on the device) swept
+-2 mm along the axis by a KinProgram, a 64 x 64 histogram over +-0.25 mm on every pose:
  65536x256:   2^16 rays x 256 poses.
  1048576x64:  2^20 rays x 64 poses.
Two legs alternate step by step after the warm-up (sharded first in even steps, one_gpu first in odd ones), each timed per rank with CUDA events ending in a synchronise; a step's time is
the largest over the ranks.  The L2 is flushed (a 256 MiB write) before every step.  Both legs are the public calls, so a step
includes flattening the system and uploading it; the source's pose tiles are built in the warm-up and kept by the source.
  sharded:   parallel.solve_spot_sweep_sharded: KinProgram.apply of the rank's shard_slice of the poses -> trace ->
             bmo_spot_stats_poses_sharded (every pose's statistics and histogram gathered on every rank).
  one_gpu:   solve_spot_sweep_device of all poses on this rank's GPU.  This is the 1-GPU run the efficiency is measured against:
             t_one_gpu / (N t_sharded).
Every rank checks that the two legs give statistics and histograms with the same sha256.  Card name, power limit and SM clock are
read in the same run, before and after.
"""
import argparse
import hashlib
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
KEYS = ("hits", "outside", "centroid", "rms", "max_r", "lo", "hi", "counts")


def card(index):
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", str(index)], capture_output=True, text=True,
                             timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out = f"unavailable ({e})"
    parts = [s.strip() for s in out.split(",")]
    return dict(zip(q.split(","), parts)) if len(parts) == 4 else {"query": out}


def sha256(stats):
    h = hashlib.sha256()
    for k in KEYS:
        h.update(np.ascontiguousarray(stats[k]).tobytes())
    return h.hexdigest()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--shapes", default="65536x256,1048576x64", help="rays x poses, comma separated")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("sharded_spot_sweep_bench.py: no CUDA device")
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
    stream = torch.cuda.current_stream()
    L.set_stream(stream.cuda_stream, dev)
    comm = par.FieldComm.from_torch(device=dev) if ws > 1 else par.FieldComm(0, 1, par.FieldComm.unique_id(), dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    window = (-HALF, HALF, -HALF, HALF)

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

    results = {}
    for shape in args.shapes.split(","):
        n, P = (int(v) for v in shape.split("x"))
        first, stop = par.shard_slice(P, rank, ws)
        sc = scenes.doublet_spot(m)
        src = m.UniformDiscSource((0.0, -0.05, 0.0), (0.0, 1.0, 0.0), 20e-3, LAMBDA, num_rays=n, e1=(1.0, 0.0, 0.0), on_device=True)
        offs = np.stack([np.zeros(P), np.linspace(-2e-3, 2e-3, P), np.zeros(P)], axis=1)

        def program(prog):
            prog.translate3d_(sc["spot"], offs)
        stats = {}

        def step(leg):
            e0 = torch.cuda.Event(enable_timing=True)
            e1 = torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            if leg == "sharded":
                out = par.solve_spot_sweep_sharded(sc["system"], src, P, sc["spot"], program=program, bins=BINS, window=window, comm=comm)
            else:
                out = m.solve_spot_sweep_device(sc["system"], src, P, program, sc["spot"], bins=BINS, window=window, device=dev)
            e1.record(stream)
            torch.cuda.synchronize()
            stats[leg] = out["stats"]
            del out
            return e0.elapsed_time(e1)

        legs = ("sharded", "one_gpu")
        for _ in range(args.warmup):
            for leg in legs:
                step(leg)
                sync_ranks()
        times = {leg: [] for leg in legs}
        for i in range(args.steps):    # alternate the legs, the first leg of a pair swapping from step to step
            for leg in (legs if i % 2 == 0 else legs[::-1]):
                flush.fill_(1)
                sync_ranks()
                times[leg].append(gather(step(leg), dist.ReduceOp.MAX if dist else None))
        digest = {leg: sha256(stats[leg]) for leg in legs}
        same = bool(gather(1.0 if digest["sharded"] == digest["one_gpu"] else 0.0, dist.ReduceOp.MIN if dist else None))
        med = {leg: float(np.median(times[leg])) for leg in legs}
        out = {leg: {"step_ms_median": med[leg], "step_ms_min": float(np.min(times[leg])), "step_ms_max": float(np.max(times[leg])),
                     "ms_per_pose_median": med[leg] / P, "stats_sha256": digest[leg]} for leg in legs}
        out["sharded"]["efficiency_vs_1gpu"] = med["one_gpu"] / (ws * med["sharded"])
        out["sharded"]["speedup_vs_1gpu"] = med["one_gpu"] / med["sharded"]
        most = -(-P // ws)
        results[shape] = {
            "workload": f"C2 through focus, Spotdetector swept +-2 mm by a KinProgram, {n} rays x {P} poses, {BINS}x{BINS} histogram over "
                        f"+-{HALF * 1e3} mm",
            "rank_poses": [first, stop],
            "source_bytes_from_shapes": {"one_gpu": 28 * n * P, "sharded_largest_rank": 28 * n * most},
            "gathered_bytes_per_rank_from_shapes": most * ws * (80 + 8 * BINS * BINS),
            "check": {"sharded_stats_sha256_equal_to_one_gpu_on_every_rank": same},
            "hits_min": int(stats["sharded"]["hits"].min()),
            "legs": out,
        }
        src.free()
        L.trim(dev)
    result = {
        "gpus": ws, "steps_per_leg": args.steps, "warmup": args.warmup, "nccl_version": comm.nccl_version(),
        "card_before": card_before, "card_after": card(dev), "torch_device_name": torch.cuda.get_device_name(dev),
        "l2": "flushed with a 256 MiB write before every timed step",
        "timing": "CUDA events per rank ending in a synchronise; step time is the max over ranks",
        "baseline_design_s10": "0.074 ms per pose at 65536x256 (bmo_spot_stats_poses sweep, measured with an earlier build)",
        "scaling_2_4_8_gpus": "see the files of runs with torchrun --nproc_per_node=N" if ws > 1 else "not measured",
        "workloads": results,
    }
    if rank == 0:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
        print(json.dumps(result, indent=1))
    comm.free()
    if dist:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
