"""Sharded device sources and spot statistics across several traces and ranks: source slices (bmo_source_create_slice),
the statistics of several results on one device (bmo_spot_stats_results) and across ranks (bmo_spot_stats_sharded), with
parallel.spot_shard_slice / solve_spot_sharded on top.

The promise under test: a splitter-free bundle traced in pieces, on one GPU or on several, has the spot statistics of one
trace of the whole bundle bit for bit, histogram included.  CPU: the shard cut and the ctypes prototypes.  GPU: slices
against the unsliced sources, C2 cut into aligned and unaligned pieces, a beamsplitter system and a ray result mixed with a
beamlet result against numpy, refused arguments, a one-rank communicator and, with two or more GPUs, NCCL ranks."""
import ctypes as C
import math
import os
import sys
import time

import numpy as np
import pytest

from tests.test_device_sources import _check_stats, _same, np_stats, splitter_scene
from tests.test_spot_sweep import _header_params

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LAM = 707e-9
FIELDS = ("hits", "outside", "centroid", "rms", "max_r", "lo", "hi", "counts")


# ---- CPU ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("R", [1, 3])
def test_spot_shard_slice_partitions_in_whole_blocks(bmo, R):
    from bmo_b200 import parallel as par
    from bmo_b200 import _lib as L
    for n in (1, 4095, 4096, 1 << 20, (1 << 20) + 1, 10 ** 7):
        per = L.spot_per(n * R)
        for w in (1, 2, 3, 8):
            sl = [par.spot_shard_slice(n, r, w, R) for r in range(w)]
            assert sl[0][0] == 0 and sum(c for _, c in sl) == n
            assert all(sl[r][0] + sl[r][1] == sl[r + 1][0] for r in range(w - 1))
            assert all(c * R % per == 0 for _, c in sl[:-1]), (n, w, sl)
            sizes = [c for _, c in sl]
            assert max(sizes) - min(sizes) <= per, (n, w, sizes)


def test_spot_per_is_the_header_formula(bmo):
    from bmo_b200 import _lib as L
    for m in (0, 1, 4096, 4096 * 1024, 4096 * 1024 + 1, 8 << 20, 10 ** 7, 3 * 10 ** 7):
        assert L.spot_per(m) == 4096 * max(1, math.ceil(m / (4096 * 1024))), m
    assert L.spot_per(8 << 20) == 8192 and L.spot_per(1 << 20) == 4096


def test_new_prototypes(bmo):
    from bmo_b200 import _lib as L
    lib = L.lib()
    for name in ("bmo_source_create_slice", "bmo_spot_stats_results", "bmo_spot_stats_sharded"):
        assert name in L.EXPORTS
        assert len(getattr(lib, name).argtypes) == len(_header_params(name)), name
    assert lib.bmo_source_create_slice.argtypes[2:4] == [C.c_int64, C.c_int64]
    assert _header_params("bmo_source_create_slice")[2:4] == ["int64_t first", "int64_t count"]
    assert lib.bmo_spot_stats_results.argtypes[0] is C.c_int32 and lib.bmo_spot_stats_results.argtypes[6] is C.POINTER(L.bmo_spot_info)
    assert _header_params("bmo_spot_stats_results")[:2] == ["int32_t n_results", "bmo_result* const* results"]
    assert lib.bmo_spot_stats_sharded.argtypes[6] is C.POINTER(L.bmo_spot_info)
    assert _header_params("bmo_spot_stats_sharded")[0] == "bmo_comm* comm"


# ---- GPU helpers -------------------------------------------------------------------------------------------------------
def _disc(bmo, n):
    return bmo.UniformDiscSource((0.0, -0.05, 0.0), (0.0, 1.0, 0.0), 20e-3, LAM, num_rays=n, e1=(1.0, 0.0, 0.0), on_device=True)


def _source(bmo, kind):
    if kind == "disc":
        return _disc(bmo, 5000)
    if kind == "collimated":
        return bmo.CollimatedSource((0.0, -0.05, 0.0), (0.1, 1.0, 0.0), 20e-3, LAM, num_rings=9, num_rays=4001, b1=(1.0, 0.0, 0.0), on_device=True)
    return bmo.PointSource((0.0, 0.0, 0.0), (0.0, 1.0, 0.1), 0.4, LAM, num_rings=11, num_rays=3003, b1=(1.0, 0.0, 0.0), on_device=True)


def _same_stats(a, b):
    for k in FIELDS:
        if k in a or k in b:
            assert _same(np.asarray(a[k], dtype=np.int64 if k == "counts" else np.float64),
                         np.asarray(b[k], dtype=np.int64 if k == "counts" else np.float64)), (k, a[k], b[k])


def _trace(bmo, system, src):
    return bmo.solve_system_(system, src, retrace=False, keep_segments=False, collect_spots=False)


# ---- 1. slices ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["disc", "collimated", "point"])
def test_slices_equal_the_rays_of_the_whole_source(bmo, kind):
    from bmo_b200 import _lib as L
    src = _source(bmo, kind)
    n = len(src)
    pos, dirs = src.rays()
    cuts = [(0, n), (0, 1), (n - 1, 1), (0, 17), (1, n - 1), (n // 2, 1)]
    rings = [src.desc.rings[i] for i in range(src.desc.n_rings)]
    if rings:
        g, h = rings[3], rings[4]
        cuts += [(g.first + g.count // 2, g.count // 2 + h.count // 3),     # starts and ends mid-ring
                 (g.first + 1, g.count - 2),                                # inside one ring
                 (g.first, g.count),                                        # one whole ring
                 (g.first - 1, 2)]                                          # the last ray of a ring and the first of the next
    for first, count in cuts:
        sh = src.shard(first, count)
        m, p, d, u = sh.device_arrays()
        assert m == count == len(sh) and u == src.uniform_dir
        npo, pid = C.c_int32(), C.c_void_p()
        L.check(L.lib().bmo_source_pose_ids(sh.handle(), C.byref(npo), C.byref(pid)))
        assert npo.value == 1 and pid.value is None
        sp, sd = sh.rays()
        assert _same(sp, pos[first:first + count]) and _same(sd, dirs[first:first + count]), (kind, first, count)
        assert sh.signature() != src.signature()
        sh.free()


@pytest.mark.gpu
def test_disc_2p20_cut_at_unaligned_offsets(bmo):
    src = _disc(bmo, 1 << 20)
    pos, dirs = src.rays()
    edges = [0, 12345, 700001, 700002, (1 << 20) - 3, 1 << 20]
    got = np.concatenate([src.shard(a, b - a).rays()[0] for a, b in zip(edges[:-1], edges[1:])])
    assert _same(got, pos)
    # a shard of a shard counts from its parent's first ray
    assert _same(src.shard(1000, 5000).shard(10, 20).rays()[0], pos[1010:1030])


# ---- 2. C2 in pieces on one device ---------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def c2_whole(bmo):
    from tests import scenes
    sc = scenes.doublet_spot(bmo)
    src = _disc(bmo, 1 << 20)
    res = _trace(bmo, sc["system"], src)
    h = 0.5 * bmo.spot_stats(res, sc["spot"])["max_r"]
    win = (-h, 0.7 * h, -0.8 * h, h)           # smaller than the spot: some hits fall outside
    return sc, src, res, win, bmo.spot_stats(res, sc["spot"], bins=(48, 64), window=win)


@pytest.mark.gpu
@pytest.mark.parametrize("W", [2, 3, 8])
def test_c2_aligned_slices_equal_one_trace(bmo, c2_whole, W):
    from bmo_b200 import parallel as par
    sc, src, _, win, whole = c2_whole
    assert whole["hits"] > 0.9 * len(src) and whole["outside"] > 0
    parts = [_trace(bmo, sc["system"], src.shard(*par.spot_shard_slice(len(src), r, W))) for r in range(W)]
    _same_stats(bmo.spot_stats(parts, sc["spot"], bins=(48, 64), window=win), whole)


@pytest.mark.gpu
def test_c2_unaligned_random_cuts_equal_one_trace(bmo, c2_whole):
    sc, src, _, win, whole = c2_whole
    rng = np.random.default_rng(11)
    edges = [0] + sorted(rng.choice(np.arange(1, len(src)), 5, replace=False).tolist()) + [len(src)]
    parts = [_trace(bmo, sc["system"], src.shard(a, b - a)) for a, b in zip(edges[:-1], edges[1:])]
    _same_stats(bmo.spot_stats(parts, sc["spot"], bins=(48, 64), window=win), whole)
    # one result in a list is bmo_spot_stats
    _same_stats(bmo.spot_stats([c2_whole[2]], sc["spot"], bins=(48, 64), window=win), whole)


# ---- 3. against numpy ----------------------------------------------------------------------------------------------------
def _det(res, obj):
    return next(i for i, o in enumerate(res.dsys.flat.objects) if o is obj)


@pytest.mark.gpu
def test_splitter_system_traced_as_two_bundles_against_numpy(bmo):
    system, sds = splitter_scene(bmo)
    src = bmo.PointSource((0.0, 0.0, 0.0), (0.0, 1.0, 0.0), 0.05, LAM, num_rings=12, num_rays=1 << 13, b1=(1.0, 0.0, 0.0), on_device=True)
    parts = [_trace(bmo, system, src.shard(0, 3001)), _trace(bmo, system, src.shard(3001, len(src) - 3001))]
    assert all(p.n_beams > p.n_roots for p in parts)
    spots = [p.spots() for p in parts]
    obj = np.concatenate([s[0] for s in spots])
    xz = np.concatenate([s[1] for s in spots])
    win = (-5e-3, 4e-3, -3e-3, 6e-3)
    seen = 0
    for sd in sds:
        ref = np_stats(obj, xz, _det(parts[0], sd), win, 16, 12)
        _check_stats(bmo.spot_stats(parts, sd, bins=(16, 12), window=win), ref)
        seen += ref["hits"]
    assert seen == int((obj >= 0).sum()) and seen > 0


@pytest.mark.gpu
def test_ray_result_mixed_with_beamlet_result_against_numpy(bmo):
    from tests import scenes
    sc = scenes.doublet_spot(bmo)
    rays = _trace(bmo, sc["system"], _disc(bmo, 4096))
    pos, _ = scenes.fibonacci_disc(1024, diameter=15e-3)
    bb = bmo.BeamletBundle.from_params(pos, (0.0, 1.0, 0.0), LAM, w0=0.2e-3)
    beamlets = bmo.solve_system_(sc["system"], bb, retrace=False, collect_spots=False)
    assert rays.R == 1 and beamlets.R == 3
    win = (-1e-3, 1e-3, -1e-3, 1e-3)
    for order in ([rays, beamlets], [beamlets, rays, beamlets]):
        spots = [r.spots() for r in order]
        ref = np_stats(np.concatenate([s[0] for s in spots]), np.concatenate([s[1] for s in spots]), _det(rays, sc["spot"]), win, 50, 40)
        assert ref["hits"] > 4096
        _check_stats(bmo.spot_stats(order, sc["spot"], bins=(50, 40), window=win), ref)


# ---- 4. refusals -----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_refused_arguments_leave_the_context_usable(bmo, c2_whole):
    from bmo_b200 import _lib as L
    lib = L.lib()
    sc, src, res, win, whole = c2_whole
    system, _ = splitter_scene(bmo)
    split = _trace(bmo, system, src.shard(0, 4096))
    info = L.bmo_spot_info()
    det = _det(res, sc["spot"])
    two = (C.c_void_p * 2)(res.h, res.h)
    assert lib.bmo_spot_stats_results(0, two, det, None, 0, 0, C.byref(info), None, 0) == -1
    assert lib.bmo_spot_stats_results(2, None, det, None, 0, 0, C.byref(info), None, 0) == -1
    assert lib.bmo_spot_stats_results(2, (C.c_void_p * 2)(res.h, None), det, None, 0, 0, C.byref(info), None, 0) == -1
    assert lib.bmo_spot_stats_results(2, two, 0, None, 0, 0, C.byref(info), None, 0) == -1           # the doublet
    # object 3 is a Spotdetector of the splitter system, not of C2 (two objects)
    mixed = (C.c_void_p * 2)(split.h, res.h)
    assert lib.bmo_spot_stats_results(2, mixed, 3, None, 0, 0, C.byref(info), None, 0) == -1
    assert lib.bmo_spot_stats_results(1, mixed, 3, None, 0, 0, C.byref(info), None, 0) == 0
    assert lib.bmo_spot_stats_results(2, two, det, L.ptr(np.array([1e-3, -1e-3, 0.0, 1e-3])), 4, 4, C.byref(info),
                                      L.ptr(np.zeros(16, np.int64)), 0) == -1
    assert lib.bmo_spot_stats_results(2, two, det, None, 4, 4, C.byref(info), L.ptr(np.zeros(16, np.int64)), 0) == -1
    ctx, h = L.context(0), C.c_void_p()
    n = src.desc.n_rays
    for first, count in [(-1, 10), (0, 0), (5, -1), (n - 9, 10), (n, 1), (1, (1 << 63) - 1), (0, n + 1)]:
        assert lib.bmo_source_create_slice(ctx, C.byref(src.desc), first, count, C.byref(h)) == -1, (first, count)
    with pytest.raises(ValueError):
        src.shard(n - 9, 10)
    # the context still traces and reduces
    _same_stats(bmo.spot_stats([_trace(bmo, sc["system"], src.shard(0, n))], sc["spot"], bins=(48, 64), window=win), whole)


# ---- 5. one rank -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_one_rank_communicator_equals_spot_stats(bmo, c2_whole):
    import torch  # noqa: F401  (libnccl.so.2 comes with torch)
    from bmo_b200 import _lib as L
    from bmo_b200 import parallel as par
    sc, src, res, win, whole = c2_whole
    comm = par.FieldComm(0, 1, par.FieldComm.unique_id(), 0)
    try:
        det = _det(res, sc["spot"])
        _same_stats(comm.spot_stats(res, det, 48, 64, win), whole)
        plain = bmo.spot_stats(res, sc["spot"])
        _same_stats(comm.spot_stats(res, det), plain)
        _same_stats(par.solve_spot_sharded(sc["system"], src, sc["spot"], bins=(48, 64), window=win, comm=comm), whole)
        # a rank without rays: the statistics of no entries
        empty = comm.spot_stats(None, det, 4, 4, win)
        assert empty["hits"] == 0 and empty["outside"] == 0 and not empty["counts"].any() and math.isnan(empty["rms"])
        with pytest.raises(L.BmoError, match="libbmo error -1"):
            comm.spot_stats(res, 0, 0, 0, None)
        with pytest.raises(L.BmoError, match="libbmo error -1"):
            comm.spot_stats(res, det, 4, 4, None)
        # device histogram
        import torch
        counts = torch.zeros((64, 48), dtype=torch.int64, device="cuda:0")
        torch.cuda.synchronize()
        info = L.bmo_spot_info()
        L.check(L.lib().bmo_spot_stats_sharded(comm.h, res.h, det, L.ptr(np.array(win)), 48, 64, C.byref(info),
                                               C.c_void_p(counts.data_ptr()), L.INPUT_DEVICE))
        assert np.array_equal(counts.cpu().numpy(), whole["counts"]) and info.hits == whole["hits"]
    finally:
        comm.free()


# ---- 6. several GPUs ---------------------------------------------------------------------------------------------------------
N_RAYS = 1 << 20
WIN_FRAC = (-0.5, 0.35, -0.4, 0.5)      # window in units of the spot's max_r: smaller than the spot


def _rank_main(rank, world_size, uid, tmp, mode):
    sys.path.insert(0, ROOT)
    import torch
    torch.cuda.set_device(rank)
    import __graft_entry__ as ge
    m = ge.load_package()
    from bmo_b200 import _lib as L
    from bmo_b200 import parallel as par
    from tests import scenes
    comm = par.FieldComm(rank, world_size, uid, device=rank)
    sc = scenes.doublet_spot(m)
    src = _disc(m, N_RAYS)
    win = tuple(f * float(np.load(os.path.join(tmp, "scale.npy"))) for f in WIN_FRAC)
    out = {}
    if mode:
        first, count = par.spot_shard_slice(N_RAYS, rank, world_size)
        if mode == "unaligned" and rank == 0:
            count -= 1                  # rank 0 ends one ray short of its block boundary
        nx, nz = (16, 64) if mode == "shape" and rank == world_size - 1 else (64, 16)   # the last rank's histogram is transposed
        res = m.solve_system_(sc["system"], src.shard(first, count), retrace=False, keep_segments=False, collect_spots=False)
        t0 = time.perf_counter()
        try:
            comm.spot_stats(res, 1, nx, nz, win)
            out["rc"] = 0
        except L.BmoError as e:
            out["rc"], out["msg"] = int(str(e).split()[2].rstrip(":")), str(e)
        out["seconds"] = time.perf_counter() - t0
    else:
        st = par.solve_spot_sharded(sc["system"], src, sc["spot"], bins=(48, 64), window=win, comm=comm)
        out = {k: np.asarray(v) for k, v in st.items()}
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
def test_ranks_equal_one_gpu_trace(bmo, c2_whole, tmp_path):
    import torch  # noqa: F401
    if _gpus() < 2:
        pytest.skip(f"needs >= 2 GPUs, this box has {_gpus()}")
    sc, src, res, _, _ = c2_whole
    scale = bmo.spot_stats(res, sc["spot"])["max_r"]
    np.save(tmp_path / "scale.npy", scale)
    win = tuple(f * scale for f in WIN_FRAC)
    whole = bmo.spot_stats(res, sc["spot"], bins=(48, 64), window=win)
    assert len(src) == N_RAYS and whole["outside"] > 0
    for w in sorted({2, min(4, _gpus())}):
        for got in _spawn(w, tmp_path, None):
            _same_stats({k: got[k] for k in FIELDS}, whole)


@pytest.mark.gpu
@pytest.mark.parametrize("mode, words", [("unaligned", "spot_shard_slice"), ("shape", "histogram shape")])
def test_disagreeing_rank_refuses_on_every_rank(bmo, c2_whole, tmp_path, mode, words):
    """One rank with an unaligned shard, or with another histogram shape than the others: every rank returns BMO_EINVAL
    promptly and the processes exit cleanly."""
    import torch  # noqa: F401
    if _gpus() < 2:
        pytest.skip(f"needs >= 2 GPUs, this box has {_gpus()}")
    np.save(tmp_path / "scale.npy", 1e-3)
    w = min(4, _gpus())
    outs = _spawn(w, tmp_path, mode, timeout=240)
    for o in outs:
        assert o["rc"] == -1, o
        assert o["seconds"] < 30, o
        assert words in o["msg"], o
