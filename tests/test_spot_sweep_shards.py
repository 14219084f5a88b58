"""Spot-diagram pose sweeps sharded over GPUs by pose range: bmo_spot_stats_poses_sharded, FieldComm.spot_sweep and
parallel.solve_spot_sweep_sharded.

The promise under test: every rank receives the statistics and histograms of all poses, each pose with the bits of one sweep of
all poses on one GPU.  It rests on one premise checked here on one GPU: a sweep of a range of poses lists every pose's spot entries
as the whole sweep does, so bmo_spot_stats_poses, which reduces each pose from its own entries alone, gives it the same bits
(checked by joining ranges, on the C2 through-focus scan and on a beamsplitter scene).  CPU: the prototype and the argument checks.
GPU: the premise, a one-rank communicator, refusals and, with two or more GPUs, NCCL ranks."""
import ctypes as C
import math
import os
import sys
import time

import numpy as np
import pytest

from tests.test_device_sources import _same, splitter_scene
from tests.test_spot_sweep import FOCUS, LAM, WIN, _det, _disc, _header_params

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BINS = (24, 16)


def _same_stats(a, b):
    """two spot_stats_poses dicts hold the same keys with the same bits"""
    assert sorted(a) == sorted(b)
    for k in a:
        assert _same(a[k], b[k]), k


# ---- CPU ---------------------------------------------------------------------------------------------------------------------
def test_new_prototype(bmo):
    from bmo_b200 import _lib as L
    lib = L.lib()
    name = "bmo_spot_stats_poses_sharded"
    assert name in L.EXPORTS
    params = _header_params(name)
    assert len(lib.bmo_spot_stats_poses_sharded.argtypes) == len(params)
    assert params[:2] == ["bmo_comm* comm", "bmo_result* r"]
    assert params[3:6] == ["int32_t n_poses", "int32_t first", "int32_t count"]
    # bmo_spot_stats_poses with a communicator in front and the pose range after n_poses
    a, b = lib.bmo_spot_stats_poses_sharded.argtypes, lib.bmo_spot_stats_poses.argtypes
    assert a[1:4] == b[:3] and a[6:] == b[3:] and a[4:6] == [C.c_int32, C.c_int32]
    types = [q.rsplit(" ", 1)[0] for q in params]
    ref = [q.rsplit(" ", 1)[0] for q in _header_params("bmo_spot_stats_poses")]
    assert types[1:4] == ref[:3] and types[6:] == ref[3:]


def test_sharded_spot_sweep_argument_checks(bmo, monkeypatch):
    """Refused before any library call: the library is replaced by one that fails on use."""
    from bmo_b200 import _lib as L
    from bmo_b200 import parallel as par
    from tests import scenes
    sc = scenes.doublet_spot(bmo)
    rb = bmo.RayBundle(np.array([[0.0, -0.05, 0.0]]), np.array([0.0, 1.0, 0.0]), LAM)

    def no_library():
        raise AssertionError("the library was called")
    monkeypatch.setattr(L, "lib", no_library)

    def prog(p):
        p.translate3d_(sc["spot"], np.zeros((4, 3)))

    def apply_pose(p):
        pass
    with pytest.raises(ValueError, match="exactly one"):
        par.solve_spot_sweep_sharded(sc["system"], rb, 4, sc["spot"])
    with pytest.raises(ValueError, match="exactly one"):
        par.solve_spot_sweep_sharded(sc["system"], rb, 4, sc["spot"], program=prog, apply_pose=apply_pose)
    for P in (0, -3):
        with pytest.raises(ValueError, match="n_poses"):
            par.solve_spot_sweep_sharded(sc["system"], rb, P, sc["spot"], program=prog)


# ---- GPU helpers ---------------------------------------------------------------------------------------------------------------
def _focus(bmo):
    """C2's through-focus scan (test_spot_sweep's focus_sweep): the Spotdetector moved along the axis over FOCUS.  Returns
    (scene, program, apply_pose); apply_pose(p) puts a fresh scene moved into pose p into the system, so that host poses do not
    depend on the poses before them."""
    from tests import scenes
    sc = scenes.doublet_spot(bmo)
    offs = np.stack([np.zeros_like(FOCUS), FOCUS, np.zeros_like(FOCUS)], axis=1)

    def apply_pose(p):
        fresh = scenes.doublet_spot(bmo)
        fresh["spot"].translate3d_(tuple(float(v) for v in offs[p]))
        sc["system"].objects[:] = fresh["system"].objects
    return sc, (lambda prog: prog.translate3d_(sc["spot"], offs)), apply_pose


def _splitter(bmo, P):
    """test_spot_sweep's beamsplitter scene: the transmitted beam's Spotdetector moved along the axis."""
    system, sds = splitter_scene(bmo)
    offs = np.stack([np.zeros(P), np.linspace(-0.02, 0.02, P), np.zeros(P)], axis=1)
    return dict(system=system, spot=sds[0]), (lambda prog: prog.translate3d_(sds[0], offs))


def _beam(bmo, kind, n=1 << 16):
    src = _disc(bmo, n)
    if kind == "device":
        return src
    pos, dirs = src.rays()
    return bmo.RayBundle(pos, dirs, LAM, normalize=False)


def _one_rank():
    import torch  # noqa: F401  (libnccl.so.2 comes with torch)
    from bmo_b200 import parallel as par
    return par.FieldComm(0, 1, par.FieldComm.unique_id(), 0)


def _range_stats(bmo, sc, beam, P, first, count, det, program=None, apply_pose=None, bins=BINS, window=WIN):
    """What one rank of solve_spot_sweep_sharded reduces for poses [first, first + count), through bmo_spot_stats_poses."""
    from bmo_b200 import parallel as par
    from bmo_b200 import sweep as sw
    lams, lam_id = sw._beam_lambdas(beam)
    _, dsys = par._pose_range_system(sc["system"], lams, P, first, count, program, apply_pose, 0)
    res = sw._trace_spot_sweep(dsys, beam, lam_id, count, 100)
    return bmo.spot_stats_poses(res, det, count, bins=bins, window=window)


def _join(parts):
    return {k: np.concatenate([p[k] for p in parts]) for k in parts[0]}


# ---- 1. ranges of poses join to the whole sweep ------------------------------------------------------------------------------
EDGES = [0, 1, 6, 7, len(FOCUS)]      # cuts at 1 and at an odd position, and the one-pose ranges [0, 1) and [6, 7)


@pytest.mark.gpu
@pytest.mark.parametrize("beam_kind", ["device", "bundle"])
@pytest.mark.parametrize("poses", ["device", "host"])
def test_pose_ranges_join_to_the_whole_sweep(bmo, beam_kind, poses):
    P = len(FOCUS)
    sc, program, apply_pose = _focus(bmo)
    beam = _beam(bmo, beam_kind)
    ref = bmo.solve_spot_sweep_device(sc["system"], beam, P, program, sc["spot"], bins=BINS, window=WIN)
    det = _det(ref["result"], sc["spot"])
    if poses == "host":
        ref = bmo.solve_spot_sweep(sc["system"], beam, P, apply_pose, det, bins=BINS, window=WIN)
    stats = ref["stats"]
    assert (stats["hits"] > 0.9 * (1 << 16)).all() and len(set(stats["rms"].tolist())) > 1 and stats["counts"].sum() > 0
    kw = dict(program=program) if poses == "device" else dict(apply_pose=apply_pose)
    parts = [_range_stats(bmo, sc, beam, P, a, b - a, det, **kw) for a, b in zip(EDGES[:-1], EDGES[1:])]
    _same_stats(_join(parts), stats)


@pytest.mark.gpu
def test_splitter_ranges_join_to_the_whole_sweep(bmo):
    """Beamsplitter children follow all roots, so the sweep and the many-pose ranges take bmo_spot_stats_poses' sort branch."""
    P, n = 8, 1 << 12
    win = (-5e-3, 4e-3, -3e-3, 6e-3)
    sc, program = _splitter(bmo, P)
    src = bmo.PointSource((0.0, 0.0, 0.0), (0.0, 1.0, 0.0), 0.05, LAM, num_rings=12, num_rays=n, b1=(1.0, 0.0, 0.0), on_device=True)
    ref = bmo.solve_spot_sweep_device(sc["system"], src, P, program, sc["spot"], bins=(16, 12), window=win)
    assert ref["result"].n_beams > ref["result"].n_roots == n * P
    assert (ref["stats"]["hits"] > 0).all() and len(set(ref["stats"]["rms"].tolist())) > 1
    det = _det(ref["result"], sc["spot"])
    edges = [0, 1, 3, 4, P]
    parts = [_range_stats(bmo, sc, src, P, a, b - a, det, program=program, bins=(16, 12), window=win) for a, b in zip(edges[:-1], edges[1:])]
    _same_stats(_join(parts), ref["stats"])


# ---- 2. one rank ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("bins", [None, BINS])
@pytest.mark.parametrize("poses", ["device", "host"])
def test_one_rank_equals_the_one_gpu_sweep(bmo, poses, bins):
    from bmo_b200 import parallel as par
    P = len(FOCUS)
    sc, program, apply_pose = _focus(bmo)
    src = _beam(bmo, "device", 1 << 14)
    ref = bmo.solve_spot_sweep_device(sc["system"], src, P, program, sc["spot"], bins=bins, window=WIN)
    det = _det(ref["result"], sc["spot"])
    if poses == "host":
        ref = bmo.solve_spot_sweep(sc["system"], src, P, apply_pose, det, bins=bins, window=WIN)
    comm = _one_rank()
    try:
        kw = dict(program=program) if poses == "device" else dict(apply_pose=apply_pose)
        got = par.solve_spot_sweep_sharded(sc["system"], src, P, det, bins=bins, window=WIN, comm=comm, **kw)
    finally:
        comm.free()
    assert got["first"] == 0 and got["result"] is not None and got["result"].n_beams == len(src) * P
    assert ("counts" in got["stats"]) == (bins is not None)
    _same_stats(got["stats"], ref["stats"])


@pytest.mark.gpu
def test_one_rank_device_counts(bmo):
    """BMO_INPUT_DEVICE histograms, and a sweep of one pose."""
    import torch
    from bmo_b200 import _lib as L
    from bmo_b200 import parallel as par
    from bmo_b200.solver import _spot_pose_dict
    P = len(FOCUS)
    nx, nz = BINS
    sc, program, _ = _focus(bmo)
    src = _beam(bmo, "device", 1 << 14)
    ref = bmo.solve_spot_sweep_device(sc["system"], src, P, program, sc["spot"], bins=BINS, window=WIN)
    res = ref["result"]
    det = _det(res, sc["spot"])
    win = np.array(WIN)
    comm = _one_rank()
    try:
        info = (L.bmo_spot_info * P)()
        d = torch.full((P * nz * nx,), -1, dtype=torch.int64, device="cuda:0")
        torch.cuda.synchronize()
        L.check(L.lib().bmo_spot_stats_poses_sharded(comm.h, res.h, det, P, 0, P, L.ptr(win), nx, nz, info, C.c_void_p(d.data_ptr()),
                                                     L.INPUT_DEVICE))
        _same_stats(_spot_pose_dict(info, P, d.cpu().numpy().reshape(P, nz, nx)), ref["stats"])
        # a sweep of one pose: bmo_spot_stats_poses' one-pose path
        def one_pose(prog):
            prog.translate3d_(sc["spot"], [[0.0, 1e-3, 0.0]])
        got = par.solve_spot_sweep_sharded(sc["system"], src, 1, sc["spot"], program=one_pose, bins=BINS, window=WIN, comm=comm)
        one = bmo.solve_spot_sweep_device(sc["system"], src, 1, one_pose, sc["spot"], bins=BINS, window=WIN)
        assert one["stats"]["hits"][0] > 0
        _same_stats(got["stats"], one["stats"])
    finally:
        comm.free()


@pytest.mark.gpu
def test_one_rank_refusals_leave_the_context_usable(bmo):
    from bmo_b200 import _lib as L
    from bmo_b200 import parallel as par
    from bmo_b200 import sweep as sw
    from bmo_b200.solver import _spot_pose_dict
    P = len(FOCUS)
    nx, nz = BINS
    sc, program, _ = _focus(bmo)
    src = _beam(bmo, "device", 1 << 14)
    ref = bmo.solve_spot_sweep_device(sc["system"], src, P, program, sc["spot"], bins=BINS, window=WIN)
    res = ref["result"]
    det, lens = _det(res, sc["spot"]), _det(res, sc["doublet"])
    lib = L.lib()
    # a trace of poses [1, P), which one rank alone cannot tile the sweep with
    _, dsys = par._pose_range_system(sc["system"], [LAM], P, 1, P - 1, program, None, 0)
    short = sw._trace_spot_sweep(dsys, src, 0, P - 1, 100)
    good = np.array(WIN)
    comm = _one_rank()
    try:
        def call(r=res.h, obj=det, n_poses=P, first=0, count=P, win=good, bins=BINS):
            info = (L.bmo_spot_info * (P + 2))()
            counts = np.zeros(((P + 2) * nz * nx,), np.int64)
            rc = lib.bmo_spot_stats_poses_sharded(comm.h, r, obj, n_poses, first, count, L.ptr(win), bins[0], bins[1], info, L.ptr(counts), 0)
            return rc, info, counts

        def usable():
            rc, info, counts = call()
            assert rc == 0
            _same_stats(_spot_pose_dict(info, P, counts[:P * nz * nx].reshape(P, nz, nx)), ref["stats"])
        for kw, why in [
            (dict(r=short.h, first=1, count=P - 1), "sweeps from pose 1, not 0"),   # the range does not start the sweep
            (dict(r=short.h, count=P - 1), "sweep 32 of 33 poses"),               # poses missing
            (dict(first=1, count=P - 1), "poses the result was traced with"),     # not the result's pose count
            (dict(n_poses=P - 1), "outside [0, n_poses)"),                        # count > n_poses
            (dict(n_poses=P + 1, count=P + 1), "poses the result was traced with"),   # not the result's pose count
            (dict(n_poses=0, count=0), "outside [0, n_poses)"),                   # an empty sweep
            (dict(obj=lens), "is not a Spotdetector"),
            (dict(obj=99), "is not a Spotdetector"),
            (dict(win=np.array([1e-3, -1e-3, -1e-3, 1e-3])), "x_hi > x_lo"),
            (dict(win=np.array([-1e-3, 1e-3, math.inf, 1e-3])), "not finite"),
            (dict(win=None), "needs a window"),
            (dict(bins=(0, nz)), "nx and nz"),
            (dict(r=None), "NULL result on a rank with poses"),
        ]:
            rc, info, counts = call(**kw)
            assert rc == -1, kw
            assert why in lib.bmo_last_error().decode(), (kw, lib.bmo_last_error())
            assert bytes(info) == bytes(len(info) * C.sizeof(L.bmo_spot_info)) and not counts.any(), kw
            usable()
        assert lib.bmo_spot_stats_poses_sharded(comm.h, res.h, det, P, 0, P, None, 0, 0, None, None, 0) == -1    # no out
        usable()
    finally:
        comm.free()


# ---- 3. several GPUs -------------------------------------------------------------------------------------------------------------
P_RANKS = 13           # not a multiple of 2, 4 or 8


def _rank_scene(m, P):
    """A P-pose through-focus scan of C2: (scene, host system, program, apply_pose, the Spotdetector's object index)."""
    from tests import scenes
    from bmo_b200.flatten import FlatSystem
    sc = scenes.doublet_spot(m)
    offs = np.stack([np.zeros(P), np.linspace(-2e-3, 2e-3, P), np.zeros(P)], axis=1)
    hsys = m.System(list(sc["system"].objects))

    def apply_pose(p):
        fresh = scenes.doublet_spot(m)
        fresh["spot"].translate3d_(tuple(float(v) for v in offs[p]))
        hsys.objects[:] = fresh["system"].objects
    det = FlatSystem(sc["system"], [LAM]).object_index(sc["spot"])
    return sc, hsys, (lambda prog: prog.translate3d_(sc["spot"], offs)), apply_pose, det


def _rank_main(rank, world_size, uid, tmp, mode, P):
    sys.path.insert(0, ROOT)
    import torch
    torch.cuda.set_device(rank)
    import __graft_entry__ as ge
    m = ge.load_package()
    from bmo_b200 import _lib as L
    from bmo_b200 import parallel as par
    comm = par.FieldComm(rank, world_size, uid, device=rank)
    sc, hsys, program, apply_pose, det = _rank_scene(m, P)
    src = _disc(m, 1 << 14)
    out = {}
    if mode in ("device", "host"):
        if mode == "device":
            got = par.solve_spot_sweep_sharded(sc["system"], src, P, sc["spot"], program=program, bins=BINS, window=WIN, comm=comm)
        else:
            got = par.solve_spot_sweep_sharded(hsys, src, P, det, apply_pose=apply_pose, bins=BINS, window=WIN, comm=comm)
        out = dict(stats=got["stats"], first=got["first"])
    else:               # the last rank disagrees: an overlapping range, another n_poses, another object or other window bits
        first, stop = par.shard_slice(P, rank, world_size)
        count = stop - first
        got = par.solve_spot_sweep_sharded(sc["system"], src, P, sc["spot"], program=program, comm=comm)
        res = got["result"]
        n_poses, win = P, np.array(WIN)
        if rank == world_size - 1:
            if mode == "overlap":
                first -= 1
            elif mode == "n_poses":
                n_poses += 1
            elif mode == "object":
                det = got["dsys"].flat.object_index(sc["doublet"])
            elif mode == "window":
                win[1] = np.nextafter(win[1], 1.0)
        info = (L.bmo_spot_info * n_poses)()
        counts = np.zeros(n_poses * BINS[0] * BINS[1], np.int64)
        t0 = time.perf_counter()
        out["rc"] = int(L.lib().bmo_spot_stats_poses_sharded(comm.h, None if res is None else res.h, det, n_poses, first, count, L.ptr(win),
                                                             BINS[0], BINS[1], info, L.ptr(counts), 0))
        out["seconds"] = time.perf_counter() - t0
        out["msg"] = L.lib().bmo_last_error().decode()
    comm.free()
    np.save(os.path.join(tmp, f"rank{rank}.npy"), out, allow_pickle=True)


def _spawn(world_size, tmp, mode, P, timeout=300):
    import torch.multiprocessing as mp
    from bmo_b200 import parallel as par
    uid = par.FieldComm.unique_id()
    ctx = mp.spawn(_rank_main, args=(world_size, uid, str(tmp), mode, P), nprocs=world_size, join=False)
    deadline = time.monotonic() + timeout
    while not ctx.join(timeout=5):
        if time.monotonic() > deadline:
            for p in ctx.processes:
                if p.is_alive():
                    p.kill()
            for p in ctx.processes:
                p.join()
            pytest.fail(f"{world_size} ranks did not finish within {timeout} s")
    return [np.load(os.path.join(tmp, f"rank{r}.npy"), allow_pickle=True).item() for r in range(world_size)]


def _gpus():
    import torch
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


@pytest.mark.gpu
@pytest.mark.parametrize("poses", ["device", "host"])
def test_ranks_equal_the_one_gpu_sweep(bmo, tmp_path, poses):
    if _gpus() < 2:
        pytest.skip(f"needs >= 2 GPUs, this box has {_gpus()}")
    from bmo_b200 import parallel as par
    for w in sorted({2, _gpus()}):
        for P in (P_RANKS, w - 1 if w > 2 else 1):      # P < w: some ranks have no poses
            sc, hsys, program, apply_pose, det = _rank_scene(bmo, P)
            src = _disc(bmo, 1 << 14)
            if poses == "device":
                ref = bmo.solve_spot_sweep_device(sc["system"], src, P, program, sc["spot"], bins=BINS, window=WIN)
            else:
                ref = bmo.solve_spot_sweep(hsys, src, P, apply_pose, det, bins=BINS, window=WIN)
            for r, got in enumerate(_spawn(w, tmp_path, poses, P)):
                assert got["first"] == par.shard_slice(P, r, w)[0]
                _same_stats(got["stats"], ref["stats"])


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["overlap", "n_poses", "object", "window"])
def test_disagreeing_rank_refuses_on_every_rank(bmo, tmp_path, mode):
    if _gpus() < 2:
        pytest.skip(f"needs >= 2 GPUs, this box has {_gpus()}")
    outs = _spawn(min(4, _gpus()), tmp_path, mode, P_RANKS, timeout=240)
    for o in outs:
        assert o["rc"] == -1, o
        assert o["seconds"] < 30, o
