"""Spot diagrams over kinematic poses: pose-tiled device sources (bmo_source_create_poses) and per-pose spot statistics
(bmo_spot_stats_poses), with the Python sweeps solve_spot_sweep / solve_spot_sweep_device on top.

The promise under test: the statistics of pose p of a sweep are bit-identical to bmo_spot_stats of a one-pose solve of the
same source at pose p.  CPU: host tiling of a RayBundle and the ctypes prototypes.  GPU: tiled sources against the
untiled ones, a through-focus scan of the C2 doublet against one-pose solves, numpy and the oracle, a tolerance sweep with
host- and device-made poses, a beamsplitter system, a beamlet result, edge cases and refused arguments."""
import copy
import ctypes as C
import math
import os
import re

import numpy as np
import pytest

from tests.test_device_sources import _check_stats, _same, np_stats, splitter_scene

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LAM = 707e-9
FIELDS = ("hits", "outside", "centroid", "rms", "max_r", "lo", "hi")


# ---- CPU ---------------------------------------------------------------------------------------------------------------
def test_tile_ray_bundle_is_pose_major(bmo):
    rng = np.random.default_rng(5)
    n, P = 37, 5
    b = bmo.RayBundle(rng.normal(size=(n, 3)), rng.normal(size=(n, 3)), rng.uniform(500e-9, 900e-9, n))
    pos, dir, lam, pose_id = bmo.tile_ray_bundle(b, P)
    i = np.arange(n * P)
    assert _same(pos, b.pos[i % n]) and _same(dir, b.dir[i % n]) and _same(lam, b.lam[i % n])
    assert pose_id.dtype == np.int32 and np.array_equal(pose_id, i // n)
    # a collimated bundle keeps its one direction
    u = bmo.RayBundle(rng.normal(size=(n, 3)), np.array([0.0, 1.0, 0.0]), LAM)
    pos, dir, lam, pose_id = bmo.tile_ray_bundle(u, P)
    assert dir.shape == (3,) and _same(dir, u.dir[0]) and _same(pos, u.pos[i % n])


def _header_params(name):
    txt = open(os.path.join(ROOT, "include", "bmo.h")).read()
    m = re.search(r"int32_t\s+" + name + r"\s*\(([^)]*)\)", txt)
    assert m, name
    return [p.strip() for p in re.sub(r"/\*.*?\*/", "", m.group(1), flags=re.S).split(",")]


def test_new_prototypes(bmo):
    from bmo_b200 import _lib as L
    lib = L.lib()
    for name in ("bmo_source_create_poses", "bmo_source_pose_ids", "bmo_spot_stats_poses"):
        assert name in L.EXPORTS
        assert len(getattr(lib, name).argtypes) == len(_header_params(name)), name
    assert lib.bmo_source_create_poses.argtypes[2] is C.c_int32
    assert lib.bmo_spot_stats_poses.argtypes[1:3] == [C.c_int32, C.c_int32]
    assert lib.bmo_spot_stats_poses.argtypes[6] is C.POINTER(L.bmo_spot_info)
    assert _header_params("bmo_spot_stats_poses")[2] == "int32_t n_poses"


# ---- GPU helpers -------------------------------------------------------------------------------------------------------
def _device_int32(ptr, n):
    """Host copy of a device int32 array (through torch's __cuda_array_interface__ import)."""
    import torch

    class _View:
        def __init__(self):
            self.__cuda_array_interface__ = dict(shape=(n,), typestr="<i4", data=(ptr, False), version=2)
    torch.cuda.synchronize()
    return torch.as_tensor(_View(), device="cuda").cpu().numpy().copy()


def _pose_stats(stats, p):
    """Pose p of a spot_stats_poses dict in spot_stats's form."""
    out = dict(hits=int(stats["hits"][p]), outside=int(stats["outside"][p]), centroid=tuple(float(v) for v in stats["centroid"][p]),
               rms=float(stats["rms"][p]), max_r=float(stats["max_r"][p]), lo=tuple(float(v) for v in stats["lo"][p]),
               hi=tuple(float(v) for v in stats["hi"][p]))
    if "counts" in stats:
        out["counts"] = stats["counts"][p]
    return out


def _same_pose(stats, p, one):
    """pose p of a sweep has exactly the bits of a one-pose spot_stats dict"""
    got = _pose_stats(stats, p)
    for k in one:
        assert _same(np.asarray(got[k], dtype=np.float64 if k != "counts" else np.int64),
                     np.asarray(one[k], dtype=np.float64 if k != "counts" else np.int64)), (p, k, got[k], one[k])


def _det(res, obj):
    return next(i for i, o in enumerate(res.dsys.flat.objects) if o is obj)


def _disc(bmo, n, on_device=True):
    return bmo.UniformDiscSource((0.0, -0.05, 0.0), (0.0, 1.0, 0.0), 20e-3, LAM, num_rays=n, e1=(1.0, 0.0, 0.0), on_device=on_device)


FOCUS = np.linspace(-2e-3, 2e-3, 33)            # detector offsets along the axis around the C2 position
WIN = (-0.15e-3, 0.15e-3, -0.15e-3, 0.15e-3)


# ---- 1. sources --------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("P", [1, 3, 64])
@pytest.mark.parametrize("kind", ["disc", "collimated", "point"])
def test_tiled_sources_equal_untiled(bmo, kind, P):
    if kind == "disc":
        src = _disc(bmo, 5000)
    elif kind == "collimated":
        src = bmo.CollimatedSource((0.0, -0.05, 0.0), (0.1, 1.0, 0.0), 20e-3, LAM, num_rings=9, num_rays=4001, b1=(1.0, 0.0, 0.0), on_device=True)
    else:
        src = bmo.PointSource((0.0, 0.0, 0.0), (0.0, 1.0, 0.1), 0.4, LAM, num_rings=11, num_rays=3003, b1=(1.0, 0.0, 0.0), on_device=True)
    n = len(src)
    pos1, dir1 = src.rays()
    posP, dirP = src.rays(n_poses=P)
    i = np.arange(n * P)
    assert _same(posP, pos1[i % n]) and _same(dirP, dir1[i % n])
    m, p, d, u, pid = src.device_arrays(0, P)
    assert m == n * P and u == src.uniform_dir
    if P == 1:
        assert pid is None
    else:
        assert np.array_equal(_device_int32(pid, n * P), i // n)
    src.free()
    assert src._handles == {}


# ---- 2. through focus, bit-identical to one-pose solves -----------------------------------------------------------------
@pytest.fixture(scope="module")
def focus_sweep(bmo):
    from tests import scenes
    sc = scenes.doublet_spot(bmo)
    src = _disc(bmo, 1 << 16)
    offs = np.stack([np.zeros_like(FOCUS), FOCUS, np.zeros_like(FOCUS)], axis=1)
    out = bmo.solve_spot_sweep_device(sc["system"], src, len(FOCUS), lambda prog: prog.translate3d_(sc["spot"], offs), sc["spot"],
                                      bins=32, window=WIN)
    return sc, src, out


@pytest.mark.gpu
def test_through_focus_equals_one_pose_solves(bmo, focus_sweep):
    from tests import scenes
    _, src, out = focus_sweep
    stats = out["stats"]
    assert stats["counts"].shape == (len(FOCUS), 32, 32) and out["result"].n_beams == len(src) * len(FOCUS)
    for p, dy in enumerate(FOCUS):
        sc = scenes.doublet_spot(bmo)
        sc["spot"].translate3d_((0.0, float(dy), 0.0))
        res = bmo.solve_system_(sc["system"], src, keep_segments=False, collect_spots=False)
        _same_pose(stats, p, bmo.spot_stats(res, sc["spot"], bins=32, window=WIN))
    rms = stats["rms"]
    assert stats["hits"].min() > 0.9 * len(src)
    assert 0 < int(np.argmin(rms)) < len(FOCUS) - 1          # the focus lies inside the scan


@pytest.mark.gpu
def test_through_focus_against_numpy(bmo, focus_sweep):
    sc, src, out = focus_sweep
    res, stats = out["result"], out["stats"]
    obj, xz = res.spots()
    n, det = len(src), _det(res, sc["spot"])
    for p in range(len(FOCUS)):
        s = slice(p * n, (p + 1) * n)
        _check_stats(_pose_stats(stats, p), np_stats(obj[s], xz[s], det, WIN, 32, 32))


# ---- 3. against the oracle -----------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_through_focus_against_oracle(bmo, orc):
    from tests import scenes
    sc = scenes.doublet_spot(bmo)
    kw = dict(num_rings=10, num_rays=1000, b1=(1.0, 0.0, 0.0))
    src = bmo.CollimatedSource((0.0, -0.05, 0.0), (0.0, 1.0, 0.0), 20e-3, LAM, on_device=True, **kw)
    host = bmo.CollimatedSource((0.0, -0.05, 0.0), (0.0, 1.0, 0.0), 20e-3, LAM, **kw)
    offs = np.stack([np.zeros_like(FOCUS), FOCUS, np.zeros_like(FOCUS)], axis=1)
    out = bmo.solve_spot_sweep_device(sc["system"], src, len(FOCUS), lambda prog: prog.translate3d_(sc["spot"], offs), sc["spot"])
    stats = out["stats"]
    ref_rms = []
    for p, dy in enumerate(FOCUS):
        osc = scenes.doublet_spot_oracle()
        osc["spot"].translate3d_([0.0, float(dy), 0.0])
        ref = orc.bulk_trace_rays(osc["system"], host.pos, np.tile(host.dir[0], (len(host), 1)), LAM, max_seg=8, spot=osc["spot"], want_segments=False)
        hit = ~np.isnan(ref["spot"][:, 0])
        r = np_stats(np.where(hit, 1, -1), np.where(hit[:, None], ref["spot"], 0.0), 1)
        _check_stats(_pose_stats(stats, p), r)
        ref_rms.append(r["rms"])
    assert int(np.argmin(stats["rms"])) == int(np.argmin(ref_rms))


# ---- 4. tolerance sweep: host-made poses, device-made poses, one-pose solves ----------------------------------------------
@pytest.mark.gpu
def test_tolerance_sweep_host_device_and_one_pose(bmo):
    from tests import scenes
    P = 16
    th = np.radians(np.linspace(-2.0, 2.0, P))
    offs = np.stack([np.linspace(-0.5e-3, 0.5e-3, P), np.zeros(P), np.linspace(0.3e-3, -0.3e-3, P)], axis=1)
    src = bmo.PointSource((0.0, -0.3, 0.0), (0.0, 1.0, 0.0), 0.03, LAM, num_rings=8, num_rays=4096, b1=(1.0, 0.0, 0.0), on_device=True)
    pristine = scenes.doublet_spot(bmo)

    def moved(p):
        sc = copy.deepcopy(pristine)
        sc["doublet"].rotate3d_((0.0, 0.0, 1.0), float(th[p]))
        sc["doublet"].translate3d_(tuple(float(v) for v in offs[p]))
        return sc

    sc = copy.deepcopy(pristine)

    def program(prog):
        prog.rotate3d_(sc["doublet"], (0.0, 0.0, 1.0), th)
        prog.translate3d_(sc["doublet"], offs)
    dev = bmo.solve_spot_sweep_device(sc["system"], src, P, program, sc["spot"], bins=(24, 16), window=(-2e-3, 2e-3, -1e-3, 1e-3))

    hsys = bmo.System(list(pristine["system"].objects))

    def apply_pose(p):
        hsys.objects[:] = moved(p)["system"].objects
    det = _det(dev["result"], sc["spot"])
    host = bmo.solve_spot_sweep(hsys, src, P, apply_pose, det, bins=(24, 16), window=(-2e-3, 2e-3, -1e-3, 1e-3))
    for k in FIELDS + ("counts",):
        assert _same(dev["stats"][k], host["stats"][k]), k
    assert (dev["stats"]["hits"] > 0).all()
    for p in range(P):
        m = moved(p)
        res = bmo.solve_system_(m["system"], src, keep_segments=False, collect_spots=False)
        _same_pose(dev["stats"], p, bmo.spot_stats(res, m["spot"], bins=(24, 16), window=(-2e-3, 2e-3, -1e-3, 1e-3)))
    # a RayBundle is tiled on the host: the same bits
    pos, dirs = src.rays()
    rb = bmo.RayBundle(pos, dirs, LAM, normalize=False)
    hb = bmo.solve_spot_sweep_device(sc["system"], rb, P, program, sc["spot"], bins=(24, 16), window=(-2e-3, 2e-3, -1e-3, 1e-3))
    for k in FIELDS + ("counts",):
        assert _same(dev["stats"][k], hb["stats"][k]), k


# ---- 5. beamsplitter system ----------------------------------------------------------------------------------------------
def _beam_pose(res, n_per_pose):
    b = res.beams()
    pose = np.empty(res.n_beams, np.int64)
    pose[:res.n_roots] = np.arange(res.n_roots) // n_per_pose
    for i in range(res.n_roots, res.n_beams):         # children have larger ids than their parents
        pose[i] = pose[b["parent"][i]]
    return pose


@pytest.mark.gpu
def test_splitter_system_per_pose_against_numpy(bmo):
    P, n = 8, 1 << 12
    system, sds = splitter_scene(bmo)
    src = bmo.PointSource((0.0, 0.0, 0.0), (0.0, 1.0, 0.0), 0.05, LAM, num_rings=12, num_rays=n, b1=(1.0, 0.0, 0.0), on_device=True)
    offs = np.stack([np.zeros(P), np.linspace(-0.02, 0.02, P), np.zeros(P)], axis=1)
    win = (-5e-3, 4e-3, -3e-3, 6e-3)
    out = bmo.solve_spot_sweep_device(system, src, P, lambda prog: prog.translate3d_(sds[0], offs), sds[0], bins=(16, 12), window=win)
    res = out["result"]
    assert res.n_beams > res.n_roots == n * P
    obj, xz = res.spots()
    pose = _beam_pose(res, n)
    seen = 0
    for sd in sds:
        det = _det(res, sd)
        st = out["stats"] if sd is sds[0] else bmo.spot_stats_poses(res, sd, P, bins=(16, 12), window=win)
        for p in range(P):
            sel = pose == p
            ref = np_stats(obj[sel], xz[sel], det, win, 16, 12)
            _check_stats(_pose_stats(st, p), ref)
            seen += ref["hits"]
    assert seen == int((obj >= 0).sum())
    # the moved detector is hit in every pose, and its spot changes with the pose
    assert (out["stats"]["hits"] > 0).all() and len(set(out["stats"]["rms"].tolist())) > 1


# ---- 6. beamlet result ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_beamlet_result_per_pose(bmo):
    from tests import scenes
    P, n = 4, 1024
    sc = scenes.doublet_spot(bmo)
    pos, _ = scenes.fibonacci_disc(n, diameter=15e-3)
    bb = bmo.BeamletBundle.from_params(pos, (0.0, 1.0, 0.0), LAM, w0=0.2e-3)
    dsys = bmo.upload_system(sc["system"], [LAM])
    prog = bmo.KinProgram(dsys.flat, P)
    prog.translate3d_(sc["spot"], np.stack([np.zeros(P), np.linspace(-1e-3, 1e-3, P), np.zeros(P)], axis=1))
    prog.apply(dsys)
    res = bmo.trace_beamlets(dsys, np.tile(bb.rays.reshape(n, 18), (P, 1)), np.zeros(n * P, np.int32), np.tile(bb.w0, P), np.tile(bb.E0, P),
                             pose_id=np.repeat(np.arange(P, dtype=np.int32), n))
    assert res.R == 3
    win = (-1e-3, 1e-3, -1e-3, 1e-3)
    st = bmo.spot_stats_poses(res, sc["spot"], P, bins=50, window=win)
    obj, xz = res.spots()
    det = _det(res, sc["spot"])
    for p in range(P):
        s = slice(3 * n * p, 3 * n * (p + 1))
        ref = np_stats(obj[s], xz[s], det, win, 50, 50)
        assert ref["hits"] > n
        _check_stats(_pose_stats(st, p), ref)


# ---- 7. one pose and edge cases ------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_one_pose_equals_spot_stats_c2_2p20(bmo):
    from tests import scenes
    from bmo_b200 import _lib as L
    sc = scenes.doublet_spot(bmo)
    res = bmo.solve_system_(sc["system"], _disc(bmo, 1 << 20), keep_segments=False, collect_spots=False)
    det = _det(res, sc["spot"])
    h = 0.5 * bmo.spot_stats(res, sc["spot"])["max_r"]
    w = np.array([-h, 0.7 * h, -0.8 * h, h])              # smaller than the spot: some hits fall outside
    a, b = L.bmo_spot_info(), (L.bmo_spot_info * 1)()
    ca, cb = np.zeros((64, 48), np.int64), np.zeros((1, 64, 48), np.int64)
    L.check(L.lib().bmo_spot_stats(res.h, det, L.ptr(w), 48, 64, C.byref(a), L.ptr(ca), 0))
    L.check(L.lib().bmo_spot_stats_poses(res.h, det, 1, L.ptr(w), 48, 64, b, L.ptr(cb), 0))
    assert bytes(a) == bytes(b[0]) and np.array_equal(ca, cb[0])
    assert a.hits > 0.9 * (1 << 20) and a.outside > 0


@pytest.mark.gpu
def test_pose_out_of_the_beam_and_repeatability(bmo):
    from tests import scenes
    P = 3
    sc = scenes.doublet_spot(bmo)
    src = _disc(bmo, 1 << 14)
    offs = np.array([[0.0, 0.0, 0.0], [0.05, 0.0, 0.0], [0.0, 0.5e-3, 0.0]])   # pose 1: the detector is 50 mm off the axis
    out = bmo.solve_spot_sweep_device(sc["system"], src, P, lambda prog: prog.translate3d_(sc["spot"], offs), sc["spot"], bins=16, window=WIN)
    st = out["stats"]
    assert st["hits"][1] == 0 and st["outside"][1] == 0 and not st["counts"][1].any()
    assert all(np.isnan(st[k][1]).all() for k in ("centroid", "rms", "max_r", "lo", "hi"))
    assert st["hits"][0] > 0 and st["hits"][2] > 0 and st["counts"][0].sum() > 0
    again = bmo.spot_stats_poses(out["result"], sc["spot"], P, bins=16, window=WIN)
    for k in FIELDS + ("counts",):
        assert _same(st[k], again[k]), k


# ---- 8. refusals -----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_refused_arguments_leave_the_context_usable(bmo, focus_sweep):
    from bmo_b200 import _lib as L
    lib = L.lib()
    sc, src, out = focus_sweep
    res = out["result"]
    P = len(FOCUS)
    det = _det(res, sc["spot"])
    info = (L.bmo_spot_info * (P + 1))()
    counts = np.zeros((P + 1) * 16, np.int64)
    good = np.array(WIN)
    for n_poses, d_obj, win, nx, nz, cnt in [
        (P - 1, det, None, 0, 0, None),              # not the result's pose count
        (1, det, None, 0, 0, None),
        (P + 1, det, None, 0, 0, None),
        (0, det, None, 0, 0, None),
        (P, 0, None, 0, 0, None),                    # the doublet is not a Spotdetector
        (P, 99, None, 0, 0, None),
        (P, det, np.array([1e-3, -1e-3, -1e-3, 1e-3]), 4, 4, counts),
        (P, det, np.array([-1e-3, 1e-3, math.inf, 1e-3]), 4, 4, counts),
        (P, det, None, 4, 4, counts),                # bins without a window
        (P, det, good, 0, 4, counts),
    ]:
        assert lib.bmo_spot_stats_poses(res.h, d_obj, n_poses, L.ptr(win), nx, nz, info, L.ptr(cnt), 0) == -1
    ctx = L.context(0)
    h = C.c_void_p()
    for n_poses in (0, -3):
        assert lib.bmo_source_create_poses(ctx, C.byref(src.desc), n_poses, C.byref(h)) == -1
    d = L.bmo_source_desc.from_buffer_copy(src.desc)
    d.n_rays = 1 << 62
    assert lib.bmo_source_create_poses(ctx, C.byref(d), 4, C.byref(h)) == -1        # n_rays * n_poses overflows int64
    # the context still traces and reduces
    r2 = bmo.solve_system_(sc["system"], src, keep_segments=False, collect_spots=False)
    assert r2.n_beams == len(src) and bmo.spot_stats(r2, sc["spot"])["hits"] > 0
    again = bmo.spot_stats_poses(res, sc["spot"], P, bins=32, window=WIN)
    for k in FIELDS + ("counts",):
        assert _same(again[k], out["stats"][k]), k
