"""PSFDetector maps sharded over GPUs by pixel columns: bmo_psf_intensity_cols (a band of columns of bmo_psf_intensity's map),
bmo_psf_allgather (every rank's hit records in rank order) and bmo_psf_intensity_sharded (each rank's band, all-gathered), with
parallel.FieldComm.psf_intensity / solve_psf_sharded on top.

The promise under test: for a splitter-free system the map of a source traced in contiguous slices, on one GPU or on several, has
the bits of one trace's map.  It rests on two premises checked here on one GPU: slices of a DeviceSource leave the records of one
trace, and bands of columns concatenate to the whole map.  CPU: the band arithmetic and the ctypes prototypes.  GPU: the two
premises, a one-rank communicator, the beamsplitter scene against the CPU checker, refused arguments and, with two or more GPUs,
NCCL ranks."""
import ctypes as C
import math
import os
import sys
import time

import numpy as np
import pytest

from tests import scenes
from tests.scenes import INCH
from tests.test_psf import D_BEAM, LAM, _airy, _OF
from tests.test_spot_sweep import _header_params

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- CPU ---------------------------------------------------------------------------------------------------------------
def test_band_arithmetic(bmo):
    from bmo_b200 import parallel as par
    for n in (1, 2, 7, 33, 100, 101, 1024):
        for w in (1, 2, 3, 4, 7, 8, 9, 200):
            B = -(-n // w)
            bands = [par.psf_shard_band(n, r, w) for r in range(w)]
            assert bands[0][0] == 0 and bands[-1][1] == n, (n, w, bands)
            assert all(bands[r][1] == bands[r + 1][0] for r in range(w - 1))
            assert all(j0 <= j1 and j1 - j0 <= B for j0, j1 in bands)
            assert all(j0 == min(n, r * B) and j1 == min(n, (r + 1) * B) for r, (j0, j1) in enumerate(bands))
            # column-major bands of n * B doubles land at n * (r * B): the first n * n doubles are the map
            assert all(n * B * r == n * (r * B) for r in range(w))
            empty = sum(1 for j0, j1 in bands if j0 == j1)
            assert empty == w - (-(-n // B)), (n, w, bands)
    assert par.psf_shard_band(1, 0, 4) == (0, 1) and par.psf_shard_band(1, 3, 4) == (1, 1)


def test_new_prototypes(bmo):
    from bmo_b200 import _lib as L
    lib = L.lib()
    for name in ("bmo_psf_intensity_cols", "bmo_psf_allgather", "bmo_psf_intensity_sharded"):
        assert name in L.EXPORTS
        assert len(getattr(lib, name).argtypes) == len(_header_params(name)), name
    assert _header_params("bmo_psf_intensity_cols")[8:10] == ["int32_t j0", "int32_t j1"]
    assert lib.bmo_psf_intensity_cols.argtypes[8:10] == [C.c_int32, C.c_int32]
    assert _header_params("bmo_psf_allgather") == ["bmo_comm* comm", "bmo_psf* local", "bmo_psf** all"]
    assert _header_params("bmo_psf_intensity_sharded")[:3] == ["bmo_comm* comm", "bmo_sys* sys", "bmo_psf* all"]
    # the sharded call is bmo_psf_intensity with a communicator in front
    assert lib.bmo_psf_intensity_sharded.argtypes[1:] == lib.bmo_psf_intensity.argtypes
    types = [[q.rsplit(" ", 1)[0] for q in _header_params(name)] for name in ("bmo_psf_intensity_sharded", "bmo_psf_intensity")]
    assert types[0][1:] == types[1]


# ---- GPU helpers -------------------------------------------------------------------------------------------------------
def _disc_source(bmo, n):
    return bmo.UniformDiscSource((0.0, -10e-3, 0.0), (0.0, 1.0, 0.0), D_BEAM, LAM, num_rays=n, e1=(1.0, 0.0, 0.0), on_device=True)


def _solve(bmo, sc, src):
    return bmo.solve_system_(sc["system"], src, retrace=False)


def _same(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and a.tobytes() == b.tobytes()


def _splitter(F):
    """The beamsplitter scene of tests/test_psf.py: children reach the detector after all roots, so records come in another order."""
    bs = F.ThinBeamsplitter(INCH, reflectance=0.5); bs.zrotate3d_(math.radians(45))
    m = F.SquarePlanoMirror2D(INCH); m.zrotate3d_(math.radians(90)); m.translate3d_([-0.05, 0.0, 0.0])
    lens = F.SphericalLens(0.1, math.inf, 2e-3, INCH, 1.5); lens.translate3d_([0.0, 0.03, 0.0])
    psfd = F.PSFDetector(10e-3); psfd.translate3d_([0.0, 0.2, 0.0])
    return dict(system=F.System([bs, m, lens, psfd]), psf=psfd)


def _splitter_rays(n=50):
    rng = np.random.default_rng(1)
    pos = np.zeros((n, 3)); pos[:, 0] = rng.uniform(-2e-3, 2e-3, n); pos[:, 2] = rng.uniform(-2e-3, 2e-3, n); pos[:, 1] = -0.1
    return pos


def _rel_l2(a, b):
    return np.linalg.norm((a - b).ravel()) / np.linalg.norm(b.ravel())


@pytest.fixture(scope="module")
def airy(bmo):
    """The Airy-disc scene with 4000 records of one trace of a DeviceSource disc."""
    sc = _airy(scenes._ProductFactory(bmo))
    src = _disc_source(bmo, 4000)
    _solve(bmo, sc, src)
    assert len(sc["psf"]) == 4000
    return sc, src


def _one_rank(bmo):
    import torch  # noqa: F401  (libnccl.so.2 comes with torch)
    from bmo_b200 import parallel as par
    return par.FieldComm(0, 1, par.FieldComm.unique_id(), 0)


# ---- 1. the premises -----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("cut", ["2", "3", "random"])
def test_slices_collect_the_records_of_one_trace(bmo, cut):
    from bmo_b200 import parallel as par
    n = 1 << 14
    src = _disc_source(bmo, n)
    whole = _airy(scenes._ProductFactory(bmo))
    _solve(bmo, whole, src)
    ref = whole["psf"].data
    assert ref.shape == (n, 9)
    if cut == "random":
        edges = [0] + sorted(np.random.default_rng(5).choice(np.arange(1, n), 5, replace=False).tolist()) + [n]
    else:
        w = int(cut)
        edges = [par.shard_slice(n, r, w)[0] for r in range(w)] + [n]
    pieces = _airy(scenes._ProductFactory(bmo))
    for a, b in zip(edges[:-1], edges[1:]):
        _solve(bmo, pieces, src.shard(a, b - a))
    got = pieces["psf"].data
    assert _same(got, ref), np.abs(got - ref).max(axis=0)


def _map(L, sc, n, lims, xs=0.0, zs=0.0):
    I = np.zeros((n, n), order="F")
    L.check(L.lib().bmo_psf_intensity(sc["psf"]._dsys.h, C.c_void_p(sc["psf"]._psf), sc["psf"]._index, 0, n, L.ptr(lims), xs, zs, L.ptr(I), 0))
    return I


def _cols(L, sc, n, lims, j0, j1, xs=0.0, zs=0.0):
    out = np.zeros((n, j1 - j0), order="F")
    L.check(L.lib().bmo_psf_intensity_cols(sc["psf"]._dsys.h, C.c_void_p(sc["psf"]._psf), sc["psf"]._index, 0, n, L.ptr(lims), xs, zs,
                                           j0, j1, L.ptr(out), 0))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 7, 33, 160])
def test_column_bands_concatenate_to_the_map(bmo, airy, n):
    from bmo_b200 import _lib as L
    sc, _ = airy
    rng = np.random.default_rng(n)
    windows = [(np.array(sc["psf"].calc_local_lims(5.0, c)), 0.0, 0.0) for c in ("centroid", "bbox")]
    windows.append((np.array([-2e-5, 3e-5, -1e-5, 1e-5]), 2e-6, -1e-6))       # explicit window and shifts
    for lims, xs, zs in windows:
        whole = _map(L, sc, n, lims, xs, zs)
        assert whole.max() > 0
        for _ in range(3):
            inner = sorted(rng.integers(0, n + 1, 3).tolist())       # repeated edges: empty bands
            edges = [0] + inner + [n]
            got = np.concatenate([_cols(L, sc, n, lims, a, b, xs, zs) for a, b in zip(edges[:-1], edges[1:])], axis=1)
            assert _same(got, whole), (n, edges)
        assert _cols(L, sc, n, lims, n, n).shape == (n, 0)


@pytest.mark.gpu
def test_column_band_to_device_memory(bmo, airy):
    import torch
    from bmo_b200 import _lib as L
    sc, _ = airy
    n, j0, j1 = 160, 37, 101
    lims = np.array(sc["psf"].calc_local_lims(5.0, "bbox"))
    whole = _map(L, sc, n, lims)
    out = torch.full(((j1 - j0) * n,), -1.0, dtype=torch.float64, device="cuda:0")
    torch.cuda.synchronize()
    p = sc["psf"]
    L.check(L.lib().bmo_psf_intensity_cols(p._dsys.h, C.c_void_p(p._psf), p._index, 0, n, L.ptr(lims), 0.0, 0.0, j0, j1,
                                           C.c_void_p(out.data_ptr()), L.INPUT_DEVICE))
    assert _same(out.cpu().numpy().reshape(j1 - j0, n).T, whole[:, j0:j1])


# ---- 2. one rank ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_one_rank_allgather_and_sharded_intensity(bmo, airy):
    import torch
    from bmo_b200 import _lib as L
    sc, _ = airy
    lib = L.lib()
    p = sc["psf"]
    comm = _one_rank(bmo)
    try:
        h = C.c_void_p()
        L.check(lib.bmo_psf_allgather(comm.h, C.c_void_p(p._psf), C.byref(h)))
        n_all = C.c_int64()
        L.check(lib.bmo_psf_count(h, C.byref(n_all)))
        rec = np.zeros((n_all.value, 9))
        L.check(lib.bmo_psf_data(h, L.ptr(rec)))
        assert _same(rec, p.data)
        n = 101
        for center in (0, 1):
            lims = np.zeros(4)
            L.check(lib.bmo_psf_lims(p._dsys.h, h, p._index, 0, 5.0, center, L.ptr(lims)))
            assert _same(lims, np.array(p.calc_local_lims(5.0, "centroid" if center == 0 else "bbox")))
            I = np.zeros((n, n), order="F")
            L.check(lib.bmo_psf_intensity_sharded(comm.h, p._dsys.h, h, p._index, 0, n, L.ptr(lims), 1e-6, 0.0, L.ptr(I), 0))
            assert _same(I, _map(L, sc, n, lims, 1e-6, 0.0))
        out = torch.zeros(n * n, dtype=torch.float64, device="cuda:0")
        torch.cuda.synchronize()
        L.check(lib.bmo_psf_intensity_sharded(comm.h, p._dsys.h, h, p._index, 0, n, L.ptr(lims), 1e-6, 0.0, C.c_void_p(out.data_ptr()),
                                              L.INPUT_DEVICE))
        assert _same(out.cpu().numpy().reshape(n, n).T, I)
        lib.bmo_psf_free(h)
        # a rank without hits passes NULL and receives an empty handle
        e = C.c_void_p()
        L.check(lib.bmo_psf_allgather(comm.h, None, C.byref(e)))
        L.check(lib.bmo_psf_count(e, C.byref(n_all)))
        assert n_all.value == 0
        lib.bmo_psf_free(e)
        # FieldComm.psf_intensity of the detector is PSFDetector.intensity
        kw = dict(n=48, crop_factor=3.0, center="bbox")
        for got, ref in zip(comm.psf_intensity(p, **kw), p.intensity(**kw)):
            assert _same(got, ref)
        kw = dict(n=33, x_min=-2e-5, x_max=3e-5, z_min=-1e-5, z_max=1e-5, x0_shift=2e-6, z0_shift=-1e-6)
        for got, ref in zip(comm.psf_intensity(p, **kw), p.intensity(**kw)):
            assert _same(got, ref)
    finally:
        comm.free()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["device", "bundle"])
def test_one_rank_solve_psf_sharded_equals_solve_and_intensity(bmo, kind):
    from bmo_b200 import parallel as par
    n_rays = 3001
    if kind == "device":
        src = _disc_source(bmo, n_rays)
    else:
        pos, d = scenes.fibonacci_disc(n_rays, diameter=D_BEAM, y0=-10e-3)
        src = bmo.RayBundle(pos, d, LAM)
    ref_sc, sc = _airy(scenes._ProductFactory(bmo)), _airy(scenes._ProductFactory(bmo))
    bmo.solve_system_(ref_sc["system"], src, retrace=False)
    kw = dict(n=64, crop_factor=5.0, center="bbox")
    ref = ref_sc["psf"].intensity(**kw)
    comm = _one_rank(bmo)
    try:
        got = par.solve_psf_sharded(sc["system"], src, sc["psf"], comm=comm, **kw)
    finally:
        comm.free()
    assert len(sc["psf"]) == n_rays
    for a, b in zip(got, ref):
        assert _same(a, b)


@pytest.mark.gpu
def test_one_rank_beamsplitter_scene_against_the_checker(bmo, orc):
    from bmo_b200 import parallel as par
    sc, osc = _splitter(scenes._ProductFactory(bmo)), _splitter(_OF())
    pos = _splitter_rays()
    for p in pos:
        orc.solve_system_(osc["system"], orc.beam(p, [0.0, 1.0, 0.0], LAM))
    _, _, Io = osc["psf"].psf_intensity(n=48, crop_factor=2)
    comm = _one_rank(bmo)
    try:
        _, _, I = par.solve_psf_sharded(sc["system"], bmo.RayBundle(pos, np.array([0.0, 1.0, 0.0]), LAM), sc["psf"], n=48, crop_factor=2,
                                        comm=comm)
    finally:
        comm.free()
    assert len(sc["psf"]) >= len(pos)
    assert _rel_l2(I, Io) <= 1e-8


# ---- 3. refusals -----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_refused_arguments_leave_the_context_usable(bmo, airy):
    from bmo_b200 import _lib as L
    sc, _ = airy
    lib = L.lib()
    p = sc["psf"]
    dsys, oi, h = p._dsys.h, p._index, C.c_void_p(p._psf)
    n = 16
    lims = np.array(p.calc_local_lims(5.0, "bbox"))
    whole = _map(L, sc, n, lims)
    out = np.zeros((n, n), order="F")
    for j0, j1 in [(-1, 2), (3, 2), (0, n + 1), (n + 1, n + 1)]:
        assert lib.bmo_psf_intensity_cols(dsys, h, oi, 0, n, L.ptr(lims), 0.0, 0.0, j0, j1, L.ptr(out), 0) == -1, (j0, j1)
    assert lib.bmo_psf_intensity_cols(dsys, h, oi, 0, n, L.ptr(lims), 0.0, 0.0, 0, n, None, 0) == -1
    assert lib.bmo_psf_intensity_cols(dsys, h, oi - 1, 0, n, L.ptr(lims), 0.0, 0.0, 0, n, L.ptr(out), 0) == -1      # the lens
    assert lib.bmo_psf_intensity_cols(dsys, h, oi, 0, 0, L.ptr(lims), 0.0, 0.0, 0, 0, L.ptr(out), 0) == -1
    assert not out.any()
    comm = _one_rank(bmo)
    try:
        a = C.c_void_p()
        assert lib.bmo_psf_allgather(comm.h, h, None) == -1
        L.check(lib.bmo_psf_allgather(comm.h, h, C.byref(a)))
        assert lib.bmo_psf_intensity_sharded(comm.h, dsys, a, oi, 0, 0, L.ptr(lims), 0.0, 0.0, L.ptr(out), 0) == -1
        assert lib.bmo_psf_intensity_sharded(comm.h, dsys, a, oi, 0, n, L.ptr(lims), 0.0, 0.0, None, 0) == -1
        assert lib.bmo_psf_intensity_sharded(comm.h, dsys, a, oi - 1, 0, n, L.ptr(lims), 0.0, 0.0, L.ptr(out), 0) == -1
        assert lib.bmo_psf_intensity_sharded(comm.h, dsys, None, oi, 0, n, L.ptr(lims), 0.0, 0.0, L.ptr(out), 0) == -1
        assert not out.any()
        L.check(lib.bmo_psf_intensity_sharded(comm.h, dsys, a, oi, 0, n, L.ptr(lims), 0.0, 0.0, L.ptr(out), 0))
        assert _same(out, whole)
        lib.bmo_psf_free(a)
    finally:
        comm.free()
    assert _same(_cols(L, sc, n, lims, 0, n), whole)


# ---- 4. several GPUs ---------------------------------------------------------------------------------------------------------
N_RAYS = 1 << 16
N_PX = 101          # not a multiple of the rank count: the last band is short


def _rank_main(rank, world_size, uid, tmp, mode):
    sys.path.insert(0, ROOT)
    import torch
    torch.cuda.set_device(rank)
    import __graft_entry__ as ge
    m = ge.load_package()
    from bmo_b200 import _lib as L
    from bmo_b200 import parallel as par
    comm = par.FieldComm(rank, world_size, uid, device=rank)
    out = {}
    if mode == "splitter":
        sc = _splitter(scenes._ProductFactory(m))
        xs, zs, I = par.solve_psf_sharded(sc["system"], m.RayBundle(_splitter_rays(), np.array([0.0, 1.0, 0.0]), LAM), sc["psf"], n=48,
                                          crop_factor=2, comm=comm)
        out = dict(xs=xs, zs=zs, I=I)
    elif mode is None:
        sc = _airy(scenes._ProductFactory(m))
        xs, zs, I = par.solve_psf_sharded(sc["system"], _disc_source(m, N_RAYS), sc["psf"], n=N_PX, crop_factor=5.0, center="bbox", comm=comm)
        out = dict(xs=xs, zs=zs, I=I)
    else:               # one rank disagrees: another n, other lims bits, or its own records instead of the gathered ones
        sc = _airy(scenes._ProductFactory(m))
        src = _disc_source(m, N_RAYS)
        first, stop = par.shard_slice(N_RAYS, rank, world_size)
        m.solve_system_(sc["system"], src.shard(first, stop - first), retrace=False, device=rank)
        p = sc["psf"]
        lib = L.lib()
        a = C.c_void_p()
        L.check(lib.bmo_psf_allgather(comm.h, C.c_void_p(p._psf), C.byref(a)))
        lims = np.zeros(4)
        L.check(lib.bmo_psf_lims(p._dsys.h, a, p._index, 0, 5.0, 1, L.ptr(lims)))
        n, h = N_PX, a
        odd = rank == world_size - 1
        if odd and mode == "n":
            n += 1
        if odd and mode == "lims":
            lims[1] = np.nextafter(lims[1], np.inf)
        if odd and mode == "local":
            h = C.c_void_p(p._psf)
        I = np.zeros((n, n), order="F")
        t0 = time.perf_counter()
        out["rc"] = int(lib.bmo_psf_intensity_sharded(comm.h, p._dsys.h, h, p._index, 0, n, L.ptr(lims), 0.0, 0.0, L.ptr(I), 0))
        out["seconds"] = time.perf_counter() - t0
        out["msg"] = lib.bmo_last_error().decode()
        lib.bmo_psf_free(a)
    comm.free()
    np.save(os.path.join(tmp, f"rank{rank}.npy"), out, allow_pickle=True)


def _spawn(world_size, tmp, mode, timeout=300):
    import torch.multiprocessing as mp
    from bmo_b200 import parallel as par
    uid = par.FieldComm.unique_id()
    ctx = mp.spawn(_rank_main, args=(world_size, uid, str(tmp), mode), nprocs=world_size, join=False)
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
def test_ranks_equal_one_gpu_map(bmo, tmp_path):
    if _gpus() < 2:
        pytest.skip(f"needs >= 2 GPUs, this box has {_gpus()}")
    sc = _airy(scenes._ProductFactory(bmo))
    _solve(bmo, sc, _disc_source(bmo, N_RAYS))
    ref = sc["psf"].intensity(n=N_PX, crop_factor=5.0, center="bbox")
    for w in sorted({2, min(4, _gpus())}):
        for got in _spawn(w, tmp_path, None):
            for k, r in zip(("xs", "zs", "I"), ref):
                assert _same(got[k], r), (w, k)


@pytest.mark.gpu
def test_ranks_beamsplitter_scene_against_the_checker(bmo, orc, tmp_path):
    if _gpus() < 2:
        pytest.skip(f"needs >= 2 GPUs, this box has {_gpus()}")
    osc = _splitter(_OF())
    for p in _splitter_rays():
        orc.solve_system_(osc["system"], orc.beam(p, [0.0, 1.0, 0.0], LAM))
    _, _, Io = osc["psf"].psf_intensity(n=48, crop_factor=2)
    for got in _spawn(2, tmp_path, "splitter"):
        assert _rel_l2(got["I"], Io) <= 1e-8


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["n", "lims", "local"])
def test_disagreeing_rank_refuses_on_every_rank(bmo, tmp_path, mode):
    """The last rank passes another n, lims one ulp off, or its ungathered records: every rank returns BMO_EINVAL promptly."""
    if _gpus() < 2:
        pytest.skip(f"needs >= 2 GPUs, this box has {_gpus()}")
    outs = _spawn(min(4, _gpus()), tmp_path, mode, timeout=240)
    for o in outs:
        assert o["rc"] == -1, o
        assert o["seconds"] < 30, o
        assert "than rank 0" in o["msg"], o
