"""The detector call of a Photodetector pose sweep (bmo_pd_sweep) of one build, for an A/B against another build's tree.

    python scripts/pd_sweep_ab.py [--root TREE] [--beamlets 256] [--poses 1024] [--px 64] [--steps 10] [--warmup 2]

TREE (default: this script's tree) is the repository whose package and libbmo.so are loaded; only calls every build since DESIGN §13
has are used, so the same file times an older tree.  Workload: the C5 Mach-Zehnder, m1 moved along its normal over [0, 2 lambda]
by a KinProgram on the device, a 1 mm disc of Gaussian beamlets tiled once per pose on the device, traced once; then bmo_pd_sweep
(power only) is timed alone, the L2 flushed (a 256 MiB write) before every call, with CUDA events ending in a synchronise.  The
records of the sweep (m, from libbmo's pixel-beamlet counter) and the bytes of one PdRec (272) give the record bytes a host
round trip would move.  Prints one JSON line with the card name, power limit and SM clock read in the same run.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys

import numpy as np


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--root", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    ap.add_argument("--beamlets", type=int, default=256)
    ap.add_argument("--poses", type=int, default=1024)
    ap.add_argument("--px", type=int, default=64)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("pd_sweep_ab.py: no CUDA device")
    sys.path.insert(0, os.path.abspath(args.root))
    import __graft_entry__ as ge
    m = ge.load_package()
    from bmo_b200 import _lib as L
    from bmo_b200 import sweep as sw
    from bmo_b200.flatten import FlatSystem
    from bmo_b200.solver import DeviceSystem
    from tests import scenes2 as s2
    P, n = args.poses, args.px
    sc = s2.mzi(m, pd_n=n)
    src = m.UniformDiscSource((0.0, -0.1, 0.0), (0.0, 1.0, 0.0), 1e-3, 1e-6, num_rays=args.beamlets, e1=(1.0, 0.0, 0.0), on_device=True)
    beam = src.beamlets(w0=5e-4, M2=1.0, P0=1e-3 / args.beamlets, z0=0.0, support=(1.0, 0.0, 0.0))
    lams, lam_id, beam = sw._beamlet_lambdas(beam)
    f0 = FlatSystem(sc["system"], lams)
    dsys = DeviceSystem(f0, 0)
    prog = sw.KinProgram(f0, P)
    prog.translate3d_(sc["m1"], np.array([s2.mzi_shift(p, P) for p in range(P)]))
    prog.apply(dsys)
    res = sw._trace_beamlet_sweep(dsys, beam, lam_id, P, 100)
    oi = f0.object_index(sc["pd"])
    power = np.zeros(P)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream()
    L.set_stream(stream.cuda_stream, 0)
    times = []
    for k in range(args.warmup + args.steps):
        flush.fill_(1)
        torch.cuda.synchronize()
        L.counters_reset()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        L.check(L.lib().bmo_pd_sweep(dsys.h, res.h, oi, P, None, L.ptr(power), 0))
        e1.record(stream)
        torch.cuda.synchronize()
        if k >= args.warmup:
            times.append(e0.elapsed_time(e1))
    c = L.counters()
    recs = c["px_beamlets"] // (n * n)
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    card = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                          timeout=30).stdout.strip()
    print(json.dumps({"root": os.path.abspath(args.root), "card": card, "beamlets": args.beamlets, "poses": P, "pixels": n,
                      "beams_traced": int(res.n_beams), "records": int(recs), "record_bytes_272_each": int(recs) * 272,
                      "pd_sweep_ms_median": float(np.median(times)), "pd_sweep_ms_min": float(np.min(times)),
                      "pd_sweep_ms_max": float(np.max(times)), "k4_ms_last_call": c["pd_field_ms"],
                      "power_sha256": hashlib.sha256(power.tobytes()).hexdigest()}), flush=True)


if __name__ == "__main__":
    main()
