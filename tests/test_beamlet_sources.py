"""GaussianBeamlet sources generated on the device (DeviceSource.beamlets -> bmo_source_create_beamlets).

Definition: tile t, beamlet i of a beamlet source has exactly the bits of BeamletBundle.from_params(P, direction, lam, w0, M2,
P0, z0, support) row i, P the positions DeviceSource.rays() gives the underlying one-pose source and `direction` the direction
the source was built with.  CPU: the descriptor's constants are from_params' and bad input is refused before any library call.
GPU: the generated beamlets, tiles and slices bit for bit; refusals; Photodetector fields, PSF records and maps, spot statistics
and a Mach-Zehnder pose sweep bit for bit with a host BeamletBundle of the same beamlets; one collimated case against the oracle."""
import ctypes as C
import math
import os
import sys
import time

import numpy as np
import pytest

from tests import scenes
from tests import scenes2 as s2
from tests.test_psf import D_BEAM, LAM, _airy
from tests.test_spot_sweep import _device_int32

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELD_TOL = 1e-8
# z0 != 0, M2 != 1 and a support vector of length != 1
PARAMS = dict(w0=0.3e-3, M2=1.3, P0=2e-3, z0=0.05, support=(2.0, 0.0, 1.0))


def _same(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and a.tobytes() == b.tobytes()


def _rel_l2(a, b):
    return float(np.linalg.norm((a - b).ravel()) / np.linalg.norm(b.ravel()))


def _host_bundle(bmo, src, **p):
    """from_params over the positions the device source generates (the definition of the beamlet source's bits)."""
    pos, _ = src.rays(0)
    return bmo.BeamletBundle.from_params(pos, src.direction, src.lam, **p)


# ---- CPU -------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("direction,p", [((0.0, 1.0, 0.0), PARAMS),
                                         ((0.1, 2.0, -0.3), dict(w0=1e-3, M2=2.0, P0=1e-3, z0=-0.2, support=(0.0, 0.0, 3.0))),
                                         ((0.0, 1.0, 0.0), dict(w0=5e-4, M2=1.0, P0=1e-3, z0=0.0, support=(1.0, 0.0, 0.0)))])
def test_descriptor_constants_equal_from_params(bmo, direction, p):
    from bmo_b200 import beams
    lam = 632.8e-9
    b = beams.beamlet_desc(direction, lam, **p)
    P = np.array([[1e-3, -2e-3, 3e-3]])
    ref = bmo.BeamletBundle.from_params(P, direction, lam, **p)
    s, dv, dd = np.array(b.s), np.array(b.dv), np.array(b.dd)
    assert _same(ref.rays[0, 0, :3], P[0]) and _same(ref.rays[0, 0, 3:], dv)
    assert _same(ref.rays[0, 1, :3], P[0] + s * b.w0) and _same(ref.rays[0, 1, 3:], dv)
    assert _same(ref.rays[0, 2, :3], P[0] + s * b.div_offset) and _same(ref.rays[0, 2, 3:], dd)
    assert ref.w0[0] == b.w0 and ref.E0[0] == complex(b.E0[0], b.E0[1]) and b.E0[1] == 0.0
    assert (b.div_offset != 0.0) == (p["z0"] != 0.0)


def test_bad_input_refused_before_any_library_call(bmo, monkeypatch):
    from bmo_b200 import _lib

    def no_lib():
        raise AssertionError("the library was called")
    monkeypatch.setattr(_lib, "lib", no_lib)
    point = bmo.PointSource((0.0, 0.0, 0.0), (0.0, 1.0, 0.0), 0.1, num_rings=3, num_rays=60, b1=(1.0, 0.0, 0.0), on_device=True)
    with pytest.raises(ValueError, match="point source"):
        point.beamlets(1e-3)
    disc = bmo.UniformDiscSource((0.0, 0.0, 0.0), (0.0, 1.0, 0.0), 1e-3, num_rays=50, e1=(1.0, 0.0, 0.0), on_device=True)
    for kw in (dict(w0=0.0), dict(w0=-1e-3), dict(w0=math.nan), dict(w0=1e-3, z0=math.inf), dict(w0=1e-3, P0=math.nan),
               dict(w0=1e-3, M2=math.inf), dict(w0=1e-3, support=(math.nan, 0.0, 0.0)), dict(w0=1e-3, support=(0.0, 0.0, 0.0))):
        with pytest.raises(ValueError):
            disc.beamlets(**kw)


# ---- GPU: the bits -------------------------------------------------------------------------------------------------------
def _source(bmo, kind, n):
    if kind == "disc":
        return bmo.UniformDiscSource((1e-3, -0.05, 2e-3), (0.0, 1.0, 0.1), 8e-3, 1e-6, num_rays=n, e1=(1.0, 0.0, 0.0), on_device=True)
    return bmo.CollimatedSource((1e-3, -0.05, 2e-3), (0.0, 1.0, 0.1), 8e-3, 1e-6, num_rings=max(10, n // 10000), num_rays=n,
                                b1=(1.0, 0.0, 0.0), on_device=True)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,n", [("disc", 1000), ("disc", 1 << 16), ("collimated", 2000)])
def test_gpu_tiles_equal_from_params(bmo, kind, n):
    src = _source(bmo, kind, n)
    bs = src.beamlets(**PARAMS)
    ref = _host_bundle(bmo, src, **PARAMS)
    for P in (1, 3, 64):
        rays, w0, E0 = bs.beamlets(0, P)
        for t in range(P):
            sl = slice(t * n, (t + 1) * n)
            assert _same(rays[sl], ref.rays) and _same(w0[sl], ref.w0) and _same(E0[sl], ref.E0), (P, t)
        m, *_, pid = bs.device_beamlets(0, P)
        assert m == n * P
        if P == 1:
            assert pid is None
        else:
            assert np.array_equal(_device_int32(pid, n * P), np.arange(n * P) // n)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,n,cuts", [("collimated", 2000, [(37, 500), (1234, 1), (0, 1), (1999, 1), (150, 1300)]),
                                         ("disc", 1 << 20, [(12345, 333333), ((1 << 20) - 7, 7), (1, (1 << 20) - 2)]),
                                         ("collimated", 1 << 20, [(12345, 333333), ((1 << 20) - 7, 7), (777, 1)])])
def test_gpu_slices_equal_rows_of_the_whole_source(bmo, kind, n, cuts):
    bs = _source(bmo, kind, n).beamlets(**PARAMS)
    rays, w0, E0 = bs.beamlets(0)
    for first, count in cuts:
        part = bs.shard(first, count)
        r, w, e = part.beamlets(0)
        sl = slice(first, first + count)
        assert _same(r, rays[sl]) and _same(w, w0[sl]) and _same(e, E0[sl]), (first, count)


@pytest.mark.gpu
def test_gpu_refusals_leave_the_context_usable(bmo):
    from bmo_b200 import _lib as L
    lib, ctx = L.lib(), L.context(0)
    src = _source(bmo, "collimated", 2000)
    bd = src.beamlets(**PARAMS).bdesc
    h = C.c_void_p()

    def create(desc, b, P=1, first=0, count=None):
        return lib.bmo_source_create_beamlets(ctx, C.byref(desc), C.byref(b), P, first, src.n if count is None else count, C.byref(h))
    point = bmo.PointSource((0.0, 0.0, 0.0), (0.0, 1.0, 0.0), 0.1, num_rings=3, num_rays=60, b1=(1.0, 0.0, 0.0), on_device=True)
    assert lib.bmo_source_create_beamlets(ctx, C.byref(point.desc), C.byref(bd), 1, 0, 60, C.byref(h)) == -1
    for field, v in (("w0", math.nan), ("w0", 0.0), ("w0", -1.0), ("div_offset", math.inf)):
        b = L.bmo_beamlet_desc.from_buffer_copy(bd)
        setattr(b, field, v)
        assert create(src.desc, b) == -1, field
    for arr in ("dv", "dd", "s", "E0"):
        b = L.bmo_beamlet_desc.from_buffer_copy(bd)
        getattr(b, arr)[0] = math.nan
        assert create(src.desc, b) == -1, arr
    assert create(src.desc, bd, P=0) == -1
    assert create(src.desc, bd, P=2, first=1, count=10) == -1              # several poses only for the whole source
    assert create(src.desc, bd, first=1999, count=2) == -1
    assert create(src.desc, bd, first=-1, count=1) == -1
    assert create(src.desc, bd, count=0) == -1
    huge = L.bmo_source_desc.from_buffer_copy(_source(bmo, "disc", 10).desc)
    huge.n_rays = (1 << 62) + 1
    assert create(huge, bd, P=2, count=huge.n_rays) == -1                  # count * n_poses overflows int64
    # calls that do not match the source's kind
    bs = src.beamlets(**PARAMS)
    hb, hr = bs.handle(0), src.handle(0)
    n, p, q, u = C.c_int64(), C.c_void_p(), C.c_void_p(), C.c_int32()
    assert lib.bmo_source_device(hb, C.byref(n), C.byref(p), C.byref(q), C.byref(u)) == -1
    assert lib.bmo_source_rays(hb, None, None) == -1
    assert lib.bmo_source_beamlets_device(hr, C.byref(n), C.byref(p), C.byref(q), C.byref(q)) == -1
    assert lib.bmo_source_beamlets(hr, None, None, None) == -1
    # the context still traces
    sc = s2.expander(bmo, 32)
    bmo.solve_system_(sc["system"], bs.shard(0, 100))
    assert np.abs(sc["pd"].field).max() > 0


# ---- GPU: Photodetector --------------------------------------------------------------------------------------------------
def _c3_source(bmo, n=4096, rings=32, diameter=8e-3):
    return bmo.CollimatedSource((0.0, -0.05, 0.0), (0.0, 1.0, 0.0), diameter, 1e-6, num_rings=rings, num_rays=n, b1=(1.0, 0.0, 0.0),
                                on_device=True)


@pytest.mark.gpu
@pytest.mark.parametrize("scene", ["c3", "michelson"])
def test_gpu_photodetector_equals_host_bundle(bmo, scene, monkeypatch):
    from bmo_b200 import solver
    if scene == "c3":
        src = _c3_source(bmo)
        p = dict(w0=1.5 * 8e-3 / 64, M2=1.0, P0=1e-3 / 4096, z0=0.0, support=(1.0, 0.0, 0.0))
        dev, host = s2.expander(bmo, 256), s2.expander(bmo, 256)
        move = (dev["l2"], host["l2"])
    else:
        src = bmo.UniformDiscSource((0.0, 0.0, 0.0), (0.0, 1.0, 0.0), 1e-3, 632.8e-9, num_rays=200, e1=(1.0, 0.0, 0.0), on_device=True)
        p = dict(w0=1e-4, M2=2.0, P0=1e-3 / 200, z0=0.01, support=(1.0, 0.0, 0.0))
        dev, host = scenes.michelson(bmo, pd_n=64), scenes.michelson(bmo, pd_n=64)
        move = (dev["m1"], host["m1"]) if "m1" in dev else (None, None)
    bs, bundle = src.beamlets(**p), _host_bundle(bmo, src, **p)
    rd = bmo.solve_system_(dev["system"], bs)
    rh = bmo.solve_system_(host["system"], bundle)
    assert rd.n_beams == rh.n_beams and np.abs(host["pd"].field).max() > 0
    assert _same(dev["pd"].field, host["pd"].field)
    assert dev["pd"].optical_power() == host["pd"].optical_power()
    # a second solve after a small move retraces the stored solution, from the device source as from the host bundle
    calls, orig = [], solver.retrace
    monkeypatch.setattr(solver, "retrace", lambda *a, **k: calls.append(1) or orig(*a, **k))
    for sc, obj in zip((dev, host), move):
        sc["pd"].empty_()
        if obj is not None:
            obj.translate3d_([0.0, 1e-7, 0.0])
    bmo.solve_system_(dev["system"], bs)
    bmo.solve_system_(host["system"], bundle)
    assert len(calls) == 2
    assert _same(dev["pd"].field, host["pd"].field) and np.abs(dev["pd"].field).max() > 0
    assert dev["pd"].optical_power() == host["pd"].optical_power()


@pytest.mark.gpu
def test_gpu_collimated_beamlet_source_against_oracle(bmo, orc):
    n = 96
    src = _c3_source(bmo, n=100, rings=5, diameter=4e-3)
    p = dict(w0=1.5 * 4e-3 / 10, M2=1.0, P0=1e-5, z0=0.0, support=(1.0, 0.0, 0.0))
    sc, osc = s2.expander(bmo, n), s2.expander_oracle(n)
    bmo.solve_system_(sc["system"], src.beamlets(**p))
    for q in src.rays(0)[0]:
        orc.solve_system_(osc["system"], orc.gaussian_beamlet(q, src.direction, src.lam, p["w0"], M2=p["M2"], P0=p["P0"], support=p["support"]))
    ref = osc["pd"].pd_field(n)
    assert np.abs(ref).max() > 0
    assert _rel_l2(sc["pd"].field, ref) <= FIELD_TOL


# ---- GPU: PSF records, maps and spots ------------------------------------------------------------------------------------
def _airy_source(bmo, n=1500):
    return bmo.UniformDiscSource((0.0, -10e-3, 0.0), (0.0, 1.0, 0.0), D_BEAM, LAM, num_rays=n, e1=(1.0, 0.0, 0.0), on_device=True)


MAP_KW = dict(n=64, crop_factor=3.0, center="bbox")
AIRY_P = dict(w0=0.2e-3, M2=1.0, P0=1e-3, z0=0.0, support=(1.0, 0.0, 0.0))


def _one_rank():
    import torch  # noqa: F401  (libnccl.so.2 comes with torch)
    from bmo_b200 import parallel as par
    return par.FieldComm(0, 1, par.FieldComm.unique_id(), 0)


@pytest.mark.gpu
def test_gpu_psf_records_maps_and_shards(bmo):
    from bmo_b200 import parallel as par
    src = _airy_source(bmo)
    bs = src.beamlets(**AIRY_P)
    dev, host = _airy(scenes._ProductFactory(bmo)), _airy(scenes._ProductFactory(bmo))
    bmo.solve_system_(dev["system"], bs, retrace=False)
    bmo.solve_system_(host["system"], _host_bundle(bmo, src, **AIRY_P), retrace=False)
    assert len(host["psf"]) >= 3 * src.n // 2
    assert _same(dev["psf"].data, host["psf"].data)
    ref = host["psf"].intensity(**MAP_KW)
    for a, b in zip(dev["psf"].intensity(**MAP_KW), ref):
        assert _same(a, b)
    # one rank: the map of the unsharded solve
    sc = _airy(scenes._ProductFactory(bmo))
    comm = _one_rank()
    try:
        got = par.solve_psf_sharded(sc["system"], bs, sc["psf"], comm=comm, **MAP_KW)
    finally:
        comm.free()
    for a, b in zip(got, ref):
        assert _same(a, b)
    # three shards solved one after another: the whole source's records in order
    sc = _airy(scenes._ProductFactory(bmo))
    for r in range(3):
        first, stop = par.shard_slice(src.n, r, 3)
        bmo.solve_system_(sc["system"], bs.shard(first, stop - first), retrace=False)
    assert _same(sc["psf"].data, host["psf"].data)


@pytest.mark.gpu
def test_gpu_spot_stats_equal_host_bundle(bmo):
    src = bmo.UniformDiscSource((0.0, -0.05, 0.0), (0.0, 1.0, 0.0), 20e-3, 707e-9, num_rays=3000, e1=(1.0, 0.0, 0.0), on_device=True)
    p = dict(w0=1e-3, M2=1.0, P0=1e-3, z0=0.0, support=(1.0, 0.0, 0.0))
    dev, host = scenes.doublet_spot(bmo), scenes.doublet_spot(bmo)
    rd = bmo.solve_system_(dev["system"], src.beamlets(**p), collect_spots=False)
    rh = bmo.solve_system_(host["system"], _host_bundle(bmo, src, **p), collect_spots=False)
    a = bmo.spot_stats(rd, dev["spot"], bins=32)
    b = bmo.spot_stats(rh, host["spot"], bins=32)
    assert a["hits"] > 0
    for k in b:
        assert _same(a[k], b[k]), k


# ---- GPU: Mach-Zehnder pose sweep ----------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_gpu_mzi_sweep_tiled_on_the_device(bmo):
    P = 64
    src = bmo.UniformDiscSource((0.0, -0.1, 0.0), (0.0, 1.0, 0.0), 1e-3, 1e-6, num_rays=16, e1=(1.0, 0.0, 0.0), on_device=True)
    p = dict(w0=5e-4, M2=1.0, P0=1e-3 / 16, z0=0.0, support=(1.0, 0.0, 0.0))
    out = []
    for beam in (src.beamlets(**p), _host_bundle(bmo, src, **p)):
        sc = s2.mzi(bmo)
        offs = np.array([s2.mzi_shift(k, P) for k in range(P)])
        out.append(bmo.solve_pose_sweep_device(sc["system"], beam, P, lambda prog: prog.translate3d_(sc["m1"], offs), sc["pd"]))
    d, h = out
    assert np.ptp(h["power"]) > 0                                        # the fringes move through the sweep
    assert _same(d["power"], h["power"]) and _same(d["fields"], h["fields"])


@pytest.mark.gpu
def test_gpu_host_posed_sweep_tiled_on_the_device(bmo):
    P = 8
    src = bmo.UniformDiscSource((0.0, -0.1, 0.0), (0.0, 1.0, 0.0), 1e-3, 1e-6, num_rays=16, e1=(1.0, 0.0, 0.0), on_device=True)
    p = dict(w0=5e-4, M2=1.0, P0=1e-3 / 16, z0=0.0, support=(1.0, 0.0, 0.0))
    out = []
    for beam in (src.beamlets(**p), _host_bundle(bmo, src, **p)):
        sc = s2.mzi(bmo)
        base = sc["m1"].position()

        def apply_pose(k, sc=sc, base=base):
            sc["m1"].translate_to3d_([b + o for b, o in zip(base, s2.mzi_shift(k, P))])
        out.append(bmo.solve_pose_sweep(sc["system"], beam, P, apply_pose, sc["pd"]))
    d, h = out
    assert _same(d["power"], h["power"]) and _same(d["fields"], h["fields"])


# ---- two or more GPUs ----------------------------------------------------------------------------------------------------
def _rank_main(rank, world_size, uid, tmp):
    sys.path.insert(0, ROOT)
    import torch
    torch.cuda.set_device(rank)
    import __graft_entry__ as ge
    m = ge.load_package()
    from bmo_b200 import parallel as par
    comm = par.FieldComm(rank, world_size, uid, device=rank)
    sc = _airy(scenes._ProductFactory(m))
    xs, zs, I = par.solve_psf_sharded(sc["system"], _airy_source(m).beamlets(**AIRY_P), sc["psf"], comm=comm, **MAP_KW)
    comm.free()
    np.save(os.path.join(tmp, f"rank{rank}.npy"), dict(xs=xs, zs=zs, I=I), allow_pickle=True)


def _gpus():
    import torch
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


@pytest.mark.gpu
def test_ranks_beamlet_source_equal_one_gpu_map(bmo, tmp_path):
    if _gpus() < 2:
        pytest.skip(f"needs >= 2 GPUs, this box has {_gpus()}")
    import torch.multiprocessing as mp
    from bmo_b200 import parallel as par
    sc = _airy(scenes._ProductFactory(bmo))
    bmo.solve_system_(sc["system"], _airy_source(bmo).beamlets(**AIRY_P), retrace=False)
    ref = sc["psf"].intensity(**MAP_KW)
    w = 2
    ctx = mp.spawn(_rank_main, args=(w, par.FieldComm.unique_id(), str(tmp_path)), nprocs=w, join=False)
    deadline = time.monotonic() + 300
    while not ctx.join(timeout=5):
        if time.monotonic() > deadline:
            for p in ctx.processes:
                if p.is_alive():
                    p.kill()
            for p in ctx.processes:
                p.join()
            pytest.fail(f"{w} ranks did not finish within 300 s")
    for r in range(w):
        got = np.load(os.path.join(tmp_path, f"rank{r}.npy"), allow_pickle=True).item()
        for k, v in zip(("xs", "zs", "I"), ref):
            assert _same(got[k], v), (r, k)
