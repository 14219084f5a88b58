"""Photodetector pose sweeps sharded over GPUs by pose range: the device grouping of a sweep's records by pose (bmo_pd_sweep,
bmo_pd_accumulate_poses), KinProgram.apply of a range of poses, bmo_pd_sweep_sharded and parallel.solve_pose_sweep_sharded.

The promise under test: every rank's powers of all poses and its own poses' fields have the bits of one sweep of all poses on one
GPU.  It rests on two premises checked here on one GPU: the records of a sweep are grouped by pose in trace order (checked against
bmo_pd_accumulate's pose filter, which never groups), and a sweep of a range of poses leaves every pose the records of the whole
sweep in the same order (checked by joining ranges).  CPU: the prototype, the parameter rows of a range, argument checks.  GPU: the
premises, a one-rank communicator, refusals and, with two or more GPUs, NCCL ranks."""
import ctypes as C
import math
import os
import sys
import time

import numpy as np
import pytest

from tests import scenes
from tests import scenes2 as s2
from tests.scenes import INCH
from tests.test_spot_sweep import _header_params

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BEAMLETS = dict(w0=5e-4, M2=1.0, P0=1e-3 / 16, z0=0.0, support=(1.0, 0.0, 0.0))


def _same(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and a.tobytes() == b.tobytes()


# ---- CPU ---------------------------------------------------------------------------------------------------------------------
def test_new_prototype(bmo):
    from bmo_b200 import _lib as L
    lib = L.lib()
    name = "bmo_pd_sweep_sharded"
    assert name in L.EXPORTS
    params = _header_params(name)
    assert len(lib.bmo_pd_sweep_sharded.argtypes) == len(params)
    assert params[:3] == ["bmo_comm* comm", "bmo_sys* sys", "bmo_result* r"]
    assert params[5:7] == ["int32_t first", "int32_t count"]
    # bmo_pd_sweep with a communicator in front and the pose range after n_poses
    a, b = lib.bmo_pd_sweep_sharded.argtypes, lib.bmo_pd_sweep.argtypes
    assert a[1:5] == b[:4] and a[7:] == b[4:] and a[5:7] == [C.c_int32, C.c_int32]
    types = [q.rsplit(" ", 1)[0] for q in params]
    ref = [q.rsplit(" ", 1)[0] for q in _header_params("bmo_pd_sweep")]
    assert types[1:5] == ref[:4] and types[7:] == ref[4:]


class _FakeLib:
    """Records what KinProgram.apply hands to bmo_system_apply_poses."""

    def __init__(self):
        self.calls = []

    def bmo_system_set_kinematics(self, *a):
        return 0

    def bmo_system_apply_poses(self, h, n_poses, n_ops, ops, n_params, params):
        arr = np.ctypeslib.as_array(C.cast(params, C.POINTER(C.c_double)), shape=(n_poses * max(n_params, 1) * 9,))
        self.calls.append((n_poses, n_ops, n_params, arr[:n_poses * n_params * 9].reshape(n_poses, n_params, 9).copy()))
        return 0


class _FakeSys:
    h = None


@pytest.mark.parametrize("kind", ["translate", "translate_to", "rotate", "mixed"])
def test_kin_program_range_applies_its_rows(bmo, monkeypatch, kind):
    from bmo_b200 import _lib as L
    from bmo_b200 import sweep as sw
    from bmo_b200.flatten import FlatSystem
    P = 11
    sc = s2.mzi(bmo)
    prog = sw.KinProgram(FlatSystem(sc["system"], [1e-6]), P)
    offs = np.array([s2.mzi_shift(k, P) for k in range(P)])
    thetas = np.linspace(-0.01, 0.02, P)
    if kind in ("translate", "mixed"):
        prog.translate3d_(sc["m1"], offs)
    if kind in ("translate_to", "mixed"):
        prog.translate_to3d_(sc["pd"], np.asarray(sc["pd"].position()) + offs[::-1])
    if kind in ("rotate", "mixed"):
        prog.rotate3d_(sc["b2"], (0.0, 0.0, 1.0), thetas)
    whole = prog.param_table()
    assert whole.shape == (P, len(prog.params), 9)
    fake = _FakeLib()
    monkeypatch.setattr(L, "lib", lambda: fake)
    ranges = [(0, P), (0, 1), (1, 5), (6, 1), (7, 4), (P - 1, 1)]
    for first, count in ranges:
        prog.apply(_FakeSys(), first, count)
        n_poses, n_ops, n_params, rows = fake.calls[-1]
        assert (n_poses, n_ops, n_params) == (count, len(prog.ops), len(prog.params))
        assert _same(rows, whole[first:first + count]), (first, count)
    prog.apply(_FakeSys())
    assert fake.calls[-1][0] == P and _same(fake.calls[-1][3], whole)
    for first, count in [(-1, 2), (0, 0), (3, P - 2), (P, 1)]:
        with pytest.raises(ValueError):
            prog.apply(_FakeSys(), first, count)
    assert len(fake.calls) == len(ranges) + 1


def test_sharded_sweep_argument_checks(bmo):
    from bmo_b200 import parallel as par
    sc = s2.mzi(bmo)
    g = bmo.GaussianBeamlet((0.0, -0.1, 0.0), (0.0, 1.0, 0.0), 1e-6, 5e-4)

    def prog(p):
        p.translate3d_(sc["m1"], np.zeros((4, 3)))

    def apply_pose(p):
        pass
    with pytest.raises(ValueError, match="exactly one"):
        par.solve_pose_sweep_sharded(sc["system"], g, 4, sc["pd"])
    with pytest.raises(ValueError, match="exactly one"):
        par.solve_pose_sweep_sharded(sc["system"], g, 4, sc["pd"], program=prog, apply_pose=apply_pose)
    for P in (0, -3):
        with pytest.raises(ValueError, match="n_poses"):
            par.solve_pose_sweep_sharded(sc["system"], g, P, sc["pd"], program=prog)


# ---- GPU helpers ---------------------------------------------------------------------------------------------------------------
def _source(bmo, n=16):
    return bmo.UniformDiscSource((0.0, -0.1, 0.0), (0.0, 1.0, 0.0), 1e-3, 1e-6, num_rays=n, e1=(1.0, 0.0, 0.0), on_device=True)


def _beam(bmo, kind, n=16):
    src = _source(bmo, n)
    if kind == "device":
        return src.beamlets(**BEAMLETS)
    pos, _ = src.rays(0)
    return bmo.BeamletBundle.from_params(pos, src.direction, src.lam, **BEAMLETS)


def _mzi_sweep(bmo, P):
    """The Mach-Zehnder scene with m1 moved along its normal over [0, 2 lambda]: (scene, program, apply_pose)."""
    sc = s2.mzi(bmo)
    offs = np.array([s2.mzi_shift(k, P) for k in range(P)])
    base = sc["m1"].position()

    def apply_pose(k):
        sc["m1"].translate_to3d_(base)
        sc["m1"].translate3d_(offs[k])
    return sc, (lambda prog: prog.translate3d_(sc["m1"], offs)), apply_pose


def _lens_sweep(bmo, P):
    """A splitter-free scene: a lens moved along the beam in front of a Photodetector."""
    F = scenes._ProductFactory(bmo)
    lens = F.SphericalLens(0.1, math.inf, 2e-3, INCH, 1.5); lens.translate3d_([0.0, 0.03, 0.0])
    pd = F.Photodetector(5e-3, 48); pd.translate3d_([0.0, 0.15, 0.0])
    sc = dict(system=F.System([lens, pd]), lens=lens, pd=pd)
    offs = np.zeros((P, 3)); offs[:, 1] = np.linspace(0.0, 2e-3, P)
    return sc, (lambda prog: prog.translate3d_(lens, offs)), None


def _one_rank():
    import torch  # noqa: F401  (libnccl.so.2 comes with torch)
    from bmo_b200 import parallel as par
    return par.FieldComm(0, 1, par.FieldComm.unique_id(), 0)


def _range_sweep(bmo, sc, beam, P, first, count, program=None, apply_pose=None):
    """What one rank of solve_pose_sweep_sharded computes for poses [first, first + count), through bmo_pd_sweep."""
    from bmo_b200 import _lib as L
    from bmo_b200 import sweep as sw
    from bmo_b200.flatten import FlatSystem
    from bmo_b200.solver import DeviceSystem
    lams, lam_id, beam = sw._beamlet_lambdas(beam)
    if apply_pose is not None:
        f0, t = sw.flatten_poses(sc["system"], lams, count, lambda k: apply_pose(first + k))
        dsys = DeviceSystem(f0, 0)
        L.check(L.lib().bmo_system_set_poses(dsys.h, count, *[L.ptr(x) for x in t]))
    else:
        f0 = FlatSystem(sc["system"], lams)
        dsys = DeviceSystem(f0, 0)
        prog = sw.KinProgram(f0, P)
        program(prog)
        prog.apply(dsys, first, count)
    res = sw._trace_beamlet_sweep(dsys, beam, lam_id, count, 100)
    n = sc["pd"].n
    fields, power = np.zeros((count, n * n * 2)), np.zeros(count)
    L.check(L.lib().bmo_pd_sweep(dsys.h, res.h, f0.object_index(sc["pd"]), count, L.ptr(fields), L.ptr(power), 0))
    z = fields[:, 0::2] + 1j * fields[:, 1::2]
    return power, z.reshape(count, n, n).transpose(0, 2, 1)


# ---- 1. device grouping by pose ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("scene", ["mzi", "splitter_free"])
def test_sweep_fields_equal_the_pose_filter(bmo, scene):
    """bmo_pd_accumulate(pose=p) builds only pose p's records, in trace order, and never groups: the grouped sweep must match it."""
    from bmo_b200 import _lib as L
    P = 64
    sc, program, _ = (_mzi_sweep if scene == "mzi" else _lens_sweep)(bmo, P)
    out = bmo.solve_pose_sweep_device(sc["system"], _beam(bmo, "device"), P, program, sc["pd"])
    res, dsys = out["result"], out["dsys"]
    # the roots are pose-major and splitter children follow all of them, so pose ids decrease exactly when there are children:
    # the MZI takes the sort branch, the lens scene the no-sort branch
    assert (res.n_beams > res.n_roots) == (scene == "mzi")
    assert np.ptp(out["power"]) > 0
    n = sc["pd"].n
    oi = dsys.flat.object_index(sc["pd"])
    for p in range(P):
        f = np.zeros(n * n * 2)
        L.check(L.lib().bmo_pd_accumulate(dsys.h, res.h, oi, p, L.ptr(f), 0))
        z = (f[0::2] + 1j * f[1::2]).reshape(n, n).T
        assert _same(z, out["fields"][p]), p
    # the batched accumulation groups the same way
    fields = np.zeros((P, n * n * 2))
    L.check(L.lib().bmo_pd_accumulate_poses(dsys.h, res.h, oi, P, L.ptr(fields), 0))
    z = (fields[:, 0::2] + 1j * fields[:, 1::2]).reshape(P, n, n).transpose(0, 2, 1)
    assert _same(z, out["fields"])


# ---- 2. ranges of poses join to the whole sweep ------------------------------------------------------------------------------
EDGES = [0, 1, 6, 7, 13]        # cuts at 1 and at an odd position, and the one-pose ranges [0, 1) and [6, 7)


@pytest.mark.gpu
@pytest.mark.parametrize("beam_kind", ["device", "bundle"])
@pytest.mark.parametrize("poses", ["device", "host"])
def test_pose_ranges_join_to_the_whole_sweep(bmo, beam_kind, poses):
    P = EDGES[-1]
    sc, program, apply_pose = _mzi_sweep(bmo, P)
    beam = _beam(bmo, beam_kind)
    if poses == "device":
        ref = bmo.solve_pose_sweep_device(sc["system"], beam, P, program, sc["pd"])
    else:
        ref = bmo.solve_pose_sweep(sc["system"], beam, P, apply_pose, sc["pd"])
    assert np.ptp(ref["power"]) > 0
    parts = [_range_sweep(bmo, sc, beam, P, a, b - a, *((program, None) if poses == "device" else (None, apply_pose)))
             for a, b in zip(EDGES[:-1], EDGES[1:])]
    assert _same(np.concatenate([p for p, _ in parts]), ref["power"])
    assert _same(np.concatenate([f for _, f in parts]), ref["fields"])


# ---- 3. one rank ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("want_fields", [True, False])
@pytest.mark.parametrize("poses", ["device", "host"])
def test_one_rank_equals_the_one_gpu_sweep(bmo, poses, want_fields):
    from bmo_b200 import parallel as par
    P = 24
    sc, program, apply_pose = _mzi_sweep(bmo, P)
    beam = _beam(bmo, "device")
    if poses == "device":
        ref = bmo.solve_pose_sweep_device(sc["system"], beam, P, program, sc["pd"], want_fields=want_fields)
    else:
        ref = bmo.solve_pose_sweep(sc["system"], beam, P, apply_pose, sc["pd"], want_fields=want_fields)
    comm = _one_rank()
    try:
        kw = dict(program=program) if poses == "device" else dict(apply_pose=apply_pose)
        got = par.solve_pose_sweep_sharded(sc["system"], beam, P, sc["pd"], comm=comm, want_fields=want_fields, **kw)
    finally:
        comm.free()
    assert got["first"] == 0 and got["result"] is not None
    assert _same(got["power"], ref["power"])
    if want_fields:
        assert _same(got["fields"], ref["fields"])
    else:
        assert got["fields"] is None


@pytest.mark.gpu
def test_one_rank_gaussian_beamlet_and_device_pointers(bmo):
    """A single GaussianBeamlet (tiled count times) and BMO_INPUT_DEVICE fields and powers."""
    import torch
    from bmo_b200 import _lib as L
    from bmo_b200 import parallel as par
    P = 9
    sc, program, _ = _mzi_sweep(bmo, P)
    g = bmo.GaussianBeamlet((0.0, -0.1, 0.0), (0.0, 1.0, 0.0), 1e-6, 5e-4, M2=1.0, P0=1e-3, support=(1.0, 0.0, 0.0))
    ref = bmo.solve_pose_sweep_device(sc["system"], g, P, program, sc["pd"])
    comm = _one_rank()
    try:
        got = par.solve_pose_sweep_sharded(sc["system"], g, P, sc["pd"], program=program, comm=comm)
        assert _same(got["power"], ref["power"]) and _same(got["fields"], ref["fields"])
        n = sc["pd"].n
        f = torch.full((P * n * n * 2,), -1.0, dtype=torch.float64, device="cuda:0")
        pw = torch.full((P,), -1.0, dtype=torch.float64, device="cuda:0")
        torch.cuda.synchronize()
        dsys, res = got["dsys"], got["result"]
        L.check(L.lib().bmo_pd_sweep_sharded(comm.h, dsys.h, res.h, dsys.flat.object_index(sc["pd"]), P, 0, P, C.c_void_p(f.data_ptr()),
                                             C.c_void_p(pw.data_ptr()), L.INPUT_DEVICE))
        assert _same(pw.cpu().numpy(), ref["power"])
        fh = f.cpu().numpy().reshape(P, n * n * 2)
        assert _same((fh[:, 0::2] + 1j * fh[:, 1::2]).reshape(P, n, n).transpose(0, 2, 1), ref["fields"])
    finally:
        comm.free()


@pytest.mark.gpu
def test_one_rank_refusals_leave_the_context_usable(bmo):
    from bmo_b200 import _lib as L
    from bmo_b200.solver import trace_rays
    P = 8
    sc, program, _ = _mzi_sweep(bmo, P)
    ref = bmo.solve_pose_sweep_device(sc["system"], _beam(bmo, "device"), P, program, sc["pd"])
    dsys, res = ref["dsys"], ref["result"]
    oi, mirror = dsys.flat.object_index(sc["pd"]), dsys.flat.object_index(sc["m1"])
    rays = trace_rays(dsys, np.array([[0.0, -0.1, 0.0]]), np.array([[0.0, 1.0, 0.0]]), None)
    lib = L.lib()
    n = sc["pd"].n
    fields, power = np.zeros((P, n * n * 2)), np.zeros(P)
    comm = _one_rank()
    try:
        def call(r, obj, n_poses, first, count, pw=power):
            return lib.bmo_pd_sweep_sharded(comm.h, dsys.h, r, obj, n_poses, first, count, L.ptr(fields), L.ptr(pw), 0)
        assert call(res.h, oi, P, 1, P - 1) == -1                 # first != 0: the range does not start the sweep
        assert call(res.h, oi, P, 0, P - 1) == -1                 # count != P: poses missing
        assert call(res.h, oi, P - 1, 0, P) == -1                 # count > n_poses
        assert call(res.h, oi, P + 1, 0, P + 1) == -1             # the system holds P poses
        assert call(rays.h, oi, P, 0, P) == -1                    # a ray result
        assert "Gaussian beamlets" in lib.bmo_last_error().decode()
        assert call(res.h, mirror, P, 0, P) == -1                 # not a Photodetector
        assert call(None, oi, P, 0, P) == -1                      # no result for P poses
        assert call(res.h, oi, P, 0, P, pw=None) == -1            # no power
        assert call(res.h, oi, 0, 0, 0) == -1                     # an empty sweep
        assert not fields.any() and not power.any()
        L.check(call(res.h, oi, P, 0, P))
    finally:
        comm.free()
    assert _same(power, ref["power"])
    z = (fields[:, 0::2] + 1j * fields[:, 1::2]).reshape(P, n, n).transpose(0, 2, 1)
    assert _same(z, ref["fields"])


# ---- 4. several GPUs -------------------------------------------------------------------------------------------------------------
P_RANKS = 13           # not a multiple of 2, 4 or 8


def _rank_main(rank, world_size, uid, tmp, mode, P):
    sys.path.insert(0, ROOT)
    import torch
    torch.cuda.set_device(rank)
    import __graft_entry__ as ge
    m = ge.load_package()
    from bmo_b200 import _lib as L
    from bmo_b200 import parallel as par
    comm = par.FieldComm(rank, world_size, uid, device=rank)
    sc, program, apply_pose = _mzi_sweep(m, P)
    beam = _beam(m, "device")
    out = {}
    if mode in ("device", "host"):
        kw = dict(program=program) if mode == "device" else dict(apply_pose=apply_pose)
        got = par.solve_pose_sweep_sharded(sc["system"], beam, P, sc["pd"], comm=comm, **kw)
        out = dict(power=got["power"], fields=got["fields"], first=got["first"])
    else:               # the last rank disagrees: an overlapping range, another n_poses or another object
        first, stop = par.shard_slice(P, rank, world_size)
        count = stop - first
        got = par.solve_pose_sweep_sharded(sc["system"], beam, P, sc["pd"], comm=comm, program=program, want_fields=False)
        dsys, res = got["dsys"], got["result"]
        oi, n_poses = dsys.flat.object_index(sc["pd"]), P
        if rank == world_size - 1:
            if mode == "overlap":
                first -= 1
            elif mode == "n_poses":
                n_poses += 1
            elif mode == "object":
                oi = dsys.flat.object_index(sc["m1"])
        power = np.zeros(n_poses)
        t0 = time.perf_counter()
        out["rc"] = int(L.lib().bmo_pd_sweep_sharded(comm.h, dsys.h, None if res is None else res.h, oi, n_poses, first, count, None,
                                                     L.ptr(power), 0))
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
            sc, program, apply_pose = _mzi_sweep(bmo, P)
            if poses == "device":
                ref = bmo.solve_pose_sweep_device(sc["system"], _beam(bmo, "device"), P, program, sc["pd"])
            else:
                ref = bmo.solve_pose_sweep(sc["system"], _beam(bmo, "device"), P, apply_pose, sc["pd"])
            for r, got in enumerate(_spawn(w, tmp_path, poses, P)):
                first, stop = par.shard_slice(P, r, w)
                assert got["first"] == first
                assert _same(got["power"], ref["power"]), (w, P, r)
                assert _same(got["fields"], ref["fields"][first:stop]), (w, P, r)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["overlap", "n_poses", "object"])
def test_disagreeing_rank_refuses_on_every_rank(bmo, tmp_path, mode):
    if _gpus() < 2:
        pytest.skip(f"needs >= 2 GPUs, this box has {_gpus()}")
    outs = _spawn(min(4, _gpus()), tmp_path, mode, P_RANKS, timeout=240)
    for o in outs:
        assert o["rc"] == -1, o
        assert o["seconds"] < 30, o
