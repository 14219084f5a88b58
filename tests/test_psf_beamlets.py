"""PSFDetector records of GaussianBeamlet solves (reference: Gaussian.jl:124-135 and PSFDetector.jl:77-89).

A beamlet that ends on a PSFDetector goes through the generic triple interact3d: the detector's interact3d(::Beam, ::Ray) runs
for the chief, the waist and the divergence beam in that order, and each call pushes one record (hit, dir, optical_path_length
of its own Beam, |dir . normal|, 2 pi / lambda).  A beamsplitter links only the chief beams of its children to the parent
(Gaussian.jl:107-111), so the chief's OPL runs through every ancestor and the waist's and divergence's count their own rays.

CPU: the oracle's restatement of that definition.  GPU: bmo_psf_collect of beamlet results through the C ABI against the oracle
(records 1e-9 relative, maps 1e-8 relative L2), a splitter cavity deeper than 64 generations, torn and clipped beamlets,
accumulation with ray solves, retrace, the sharded map, and a Photodetector in the same system."""
import math
import os
import sys
import time

import numpy as np
import pytest

from tests import scenes
from tests.scenes import INCH
from tests.test_psf import D_BEAM, LAM, _airy, _OF

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REC_TOL = 1e-9      # hit records, relative
FIELD_TOL = 1e-8    # intensity maps and detector fields, relative L2
W0 = 0.2e-3


def _rel_l2(a, b):
    return float(np.linalg.norm((a - b).ravel()) / np.linalg.norm(b.ravel()))


def _same(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and a.tobytes() == b.tobytes()


def _last_hit(r):
    return r["pos"][-1] + r["t"][-1] * r["dir"][-1]


def _own_opl(r):
    """optical_path_length of a beam without a parent: its rays' t * n in order, up to the first ray without a hit."""
    s = 0.0
    for t, n in zip(r["t"], r["n"]):
        if not np.isfinite(t):
            break
        s += t * n
    return s


# ---- CPU: the definition, in the oracle ----------------------------------------------------------------------------------
def test_oracle_beamlet_pushes_chief_waist_divergence(orc):
    sc = _airy(_OF())
    g = orc.gaussian_beamlet([1e-3, -10e-3, 2e-3], [0.0, 1.0, 0.0], LAM, w0=W0, support=(1.0, 0.0, 0.0))
    orc.solve_system_(sc["system"], g)
    data = sc["psf"].psf_data()
    assert data.shape == (3, 9)
    (b,) = orc.gauss_export(sc["system"], g)
    for k, name in enumerate(("chief", "waist", "div")):
        r = b[name]
        assert np.array_equal(data[k, 0:3], _last_hit(r)), name
        assert np.array_equal(data[k, 3:6], r["dir"][-1]), name
        assert data[k, 6] == _own_opl(r), name
        assert data[k, 7] == abs(float(np.dot(r["dir"][-1], r["nrm"][-1]))), name
        assert data[k, 8] == 2 * math.pi / LAM
    assert not np.array_equal(data[1, 0:3], data[0, 0:3]) and not np.array_equal(data[2, 3:6], data[0, 3:6])


def test_oracle_beamlet_opl_behind_a_splitter(orc):
    """The child's chief record carries the stem's OPL, its waist and divergence records only their own path."""
    F = _OF()
    bs = F.ThinBeamsplitter(INCH, reflectance=0.5)
    bs.zrotate3d_(math.radians(45))
    psfd = F.PSFDetector(10e-3); psfd.translate3d_([0.0, 0.1, 0.0])
    sys_ = F.System([bs, psfd])
    g = orc.gaussian_beamlet([0.0, -0.1, 0.0], [0.0, 1.0, 0.0], LAM, w0=1e-3, support=(1.0, 0.0, 0.0))
    orc.solve_system_(sys_, g)
    data = psfd.psf_data()
    assert data.shape == (3, 9)
    tree = orc.gauss_export(sys_, g)
    root = tree[0]
    child = next(b for b in tree if b["parent"] == 0 and len(b["chief"]["t"]) and np.isfinite(b["chief"]["t"][-1]))
    assert abs(data[0, 6] - 0.2) < 1e-12                                           # stem 0.1 + child 0.1
    assert data[0, 6] == _own_opl(root["chief"]) + _own_opl(child["chief"])
    for k, name in ((1, "waist"), (2, "div")):
        assert data[k, 6] == _own_opl(child[name]), name
        assert abs(data[k, 6] - 0.1) < 2e-3, name                                  # no stem: ~0.1, not ~0.2
        assert np.array_equal(data[k, 0:3], _last_hit(child[name]))


# ---- GPU helpers ---------------------------------------------------------------------------------------------------------
def _lattice(n_side, diameter=D_BEAM, y0=-10e-3):
    """n_side^2 beamlet positions on a square lattice, clipped to a disc of `diameter`."""
    u = (np.arange(n_side) + 0.5) / n_side * diameter - diameter / 2
    x, z = np.meshgrid(u, u, indexing="ij")
    keep = x ** 2 + z ** 2 <= (diameter / 2) ** 2
    pos = np.zeros((int(keep.sum()), 3))
    pos[:, 0], pos[:, 1], pos[:, 2] = x[keep], y0, z[keep]
    return pos


def _oracle_beamlets(orc, osys, pos, d, w0=W0):
    """The oracle solving the beamlets one after another (its PSFDetector pushes in that order)."""
    g = np.zeros((len(pos), 14))
    g[:, 0:3] = pos; g[:, 3:6] = d; g[:, 6] = LAM; g[:, 7] = w0; g[:, 8] = 1.0; g[:, 9] = 1e-3; g[:, 10] = 0.0; g[:, 11] = 1.0
    orc.bulk_trace_beamlets(osys, g, r_max=100, nthreads=1)


def _bundle(bmo, pos, d=(0.0, 1.0, 0.0), w0=W0):
    return bmo.BeamletBundle.from_params(pos, d, LAM, w0=w0, support=(1.0, 0.0, 0.0))


def _check_records(got, ref):
    assert got.shape == ref.shape, (got.shape, ref.shape)
    scale = max(1.0, np.abs(ref[:, 0:3]).max())
    assert np.abs(got[:, 0:6] - ref[:, 0:6]).max() <= REC_TOL * scale
    assert np.abs(got[:, 6] - ref[:, 6]).max() <= REC_TOL * np.abs(ref[:, 6]).max()      # optical path length
    assert np.abs(got[:, 7] - ref[:, 7]).max() <= REC_TOL
    assert np.array_equal(got[:, 8], ref[:, 8])


def _sorted(rec):
    """Records ordered by hit x, then z, then OPL (rounded to 1e-9), for sets whose push order differs."""
    return rec[np.lexsort(np.round(rec[:, [6, 2, 0]], 9).T)]


# ---- 1. the Airy scene ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_gpu_beamlet_lattice_records_and_maps(bmo, orc):
    sc, osc = _airy(scenes._ProductFactory(bmo)), _airy(_OF())
    pos = _lattice(38)
    assert len(pos) >= 1024
    res = bmo.solve_system_(sc["system"], _bundle(bmo, pos))
    _oracle_beamlets(orc, osc["system"], pos, (0.0, 1.0, 0.0))
    got, ref = sc["psf"].data, osc["psf"].psf_data()
    absorbed = int((res.beams()["status"] == 2).sum())
    assert absorbed == len(pos) and got.shape[0] == 3 * absorbed
    _check_records(got, ref)                                       # row by row: beamlet order, then chief, waist, divergence
    n = 96
    for center in ("centroid", "bbox"):
        a, b = np.array(sc["psf"].calc_local_lims(3.0, center)), osc["psf"].psf_lims(3.0, center)
        assert np.abs(a - b).max() <= 1e-12 * np.abs(b).max() + 1e-15
        x, z, I = sc["psf"].intensity(n=n, crop_factor=3, center=center)
        xo, zo, Io = osc["psf"].psf_intensity(n=n, crop_factor=3, center=center)
        assert np.abs(x - xo).max() <= 1e-15 and np.abs(z - zo).max() <= 1e-15
        assert _rel_l2(I, Io) <= FIELD_TOL, center
    kw = dict(n=64, x_min=-4e-4, x_max=5e-4, z_min=-3e-4, z_max=4e-4, x0_shift=2e-6, z0_shift=-1e-6)
    x, z, I = sc["psf"].intensity(**kw)
    xo, zo, Io = osc["psf"].psf_intensity(**kw)
    assert np.abs(x - xo).max() <= 1e-15 and Io.max() > 0
    assert _rel_l2(I, Io) <= FIELD_TOL


@pytest.mark.gpu
def test_gpu_single_gaussian_beamlet(bmo, orc):
    sc, osc = _airy(scenes._ProductFactory(bmo)), _airy(_OF())
    p = [1e-3, -10e-3, 2e-3]
    bmo.solve_system_(sc["system"], bmo.GaussianBeamlet(p, [0.0, 1.0, 0.0], LAM, W0, support=(1.0, 0.0, 0.0)))
    orc.solve_system_(osc["system"], orc.gaussian_beamlet(p, [0.0, 1.0, 0.0], LAM, w0=W0, support=(1.0, 0.0, 0.0)))
    got, ref = sc["psf"].data, osc["psf"].psf_data()
    assert got.shape == (3, 9)
    _check_records(got, ref)


# ---- 2. beamsplitter, mirror and lens ------------------------------------------------------------------------------------
def _splitter(F):
    bs = F.ThinBeamsplitter(INCH, reflectance=0.5); bs.zrotate3d_(math.radians(45))
    m = F.SquarePlanoMirror2D(INCH); m.zrotate3d_(math.radians(90)); m.translate3d_([-0.05, 0.0, 0.0])
    lens = F.SphericalLens(0.1, math.inf, 2e-3, INCH, 1.5); lens.translate3d_([0.0, 0.03, 0.0])
    psfd = F.PSFDetector(10e-3); psfd.translate3d_([0.0, 0.2, 0.0])
    return dict(system=F.System([bs, m, lens, psfd]), psf=psfd)


def _splitter_beamlets(n=64):
    rng = np.random.default_rng(3)
    pos = np.zeros((n, 3)); pos[:, 0] = rng.uniform(-2e-3, 2e-3, n); pos[:, 2] = rng.uniform(-2e-3, 2e-3, n); pos[:, 1] = -0.1
    return pos


@pytest.mark.gpu
def test_gpu_beamlets_through_beamsplitter_children(bmo, orc):
    sc, osc = _splitter(scenes._ProductFactory(bmo)), _splitter(_OF())
    pos = _splitter_beamlets()
    bmo.solve_system_(sc["system"], _bundle(bmo, pos))
    _oracle_beamlets(orc, osc["system"], pos, (0.0, 1.0, 0.0))
    got, ref = sc["psf"].data, osc["psf"].psf_data()
    assert got.shape == ref.shape and got.shape[0] >= 3 * len(pos)
    assert ref[0::3, 6].min() > 0.25 and ref[1::3, 6].max() < 0.25     # chief OPL with the stem, waist / divergence without
    _check_records(_sorted(got), _sorted(ref))     # push order differs (waves vs the beam tree): sets keyed by hit point
    x, z, I = sc["psf"].intensity(n=48, crop_factor=2)
    xo, zo, Io = osc["psf"].psf_intensity(n=48, crop_factor=2)
    assert _rel_l2(I, Io) <= FIELD_TOL


# ---- 3. a splitter cavity deeper than 64 generations ---------------------------------------------------------------------
CAVITY_GAP, CAVITY_TAN = 2e-3, 0.08


def _cavity(F):
    """Two parallel thin beamsplitters 2 mm apart; a tilted beamlet walks 0.16 mm along x per round trip, and a child escapes
    through the upper splitter towards the detector on every one, until the beamlet walks off the splitters' edge."""
    b1 = F.ThinBeamsplitter(INCH, reflectance=0.5)
    b2 = F.ThinBeamsplitter(INCH, reflectance=0.5); b2.translate3d_([0.0, CAVITY_GAP, 0.0])
    psfd = F.PSFDetector(60e-3); psfd.translate3d_([0.0, CAVITY_GAP + 0.02, 0.0])
    return dict(system=F.System([b1, b2, psfd]), psf=psfd)


@pytest.mark.gpu
def test_gpu_chief_opl_through_a_deep_cavity(bmo, orc):
    sc, osc = _cavity(scenes._ProductFactory(bmo)), _cavity(_OF())
    pos = np.array([[-11.5e-3, -10e-3, z] for z in (-2e-3, 0.0, 3e-3)])
    d = np.array([CAVITY_TAN, 1.0, 0.0]) / math.hypot(CAVITY_TAN, 1.0)
    res = bmo.solve_system_(sc["system"], _bundle(bmo, pos, d, w0=0.3e-3))
    _oracle_beamlets(orc, osc["system"], pos, d, w0=0.3e-3)
    got, ref = sc["psf"].data, osc["psf"].psf_data()
    # generation of every beamlet that reached the detector
    b = res.beams()
    depth = np.zeros(res.n_beams, np.int64)
    for i in range(res.n_roots, res.n_beams):
        depth[i] = depth[b["parent"][i]] + 1
    seg = res.segments()
    on = [i for i in range(res.n_beams) if b["status"][i] == 2 and b["nseg"][i] > 0
          and seg["obj"][(b["first"][i] + b["nseg"][i] - 1) * 3] == 2]
    assert len(on) * 3 == got.shape[0]
    assert depth[on].max() > 64 and (depth[on] > 64).sum() >= 10, depth[on].max()
    _check_records(_sorted(got), _sorted(ref))
    assert got[0::3, 6].max() > 64 * CAVITY_GAP       # chief OPL through more than 64 passes of the cavity


# ---- 4. torn and clipped beamlets ----------------------------------------------------------------------------------------
def _edge(F, behind):
    psfd = F.PSFDetector(10e-3); psfd.translate3d_([0.0, 0.1, 0.0])
    objs = [psfd]
    back = None
    if behind:      # a second detector behind the edge: the waist ray hits another shape than the chief (torn)
        back = F.PSFDetector(40e-3); back.translate3d_([0.0, 0.12, 0.0])
        objs.append(back)
    return dict(system=F.System(objs), psf=psfd, back=back)


@pytest.mark.gpu
@pytest.mark.parametrize("behind", [False, True])
def test_gpu_beamlet_across_the_detector_edge(bmo, orc, behind):
    w0 = 1e-3
    pos = np.array([[0.0, 0.0, 1e-3], [5e-3 - w0 / 2, 0.0, 0.0]])     # one inside, one with its waist ray past the edge x = 5 mm
    sc, osc = _edge(scenes._ProductFactory(bmo), behind), _edge(_OF(), behind)
    res = bmo.solve_system_(sc["system"], _bundle(bmo, pos, w0=w0))
    _oracle_beamlets(orc, osc["system"], pos, (0.0, 1.0, 0.0), w0=w0)
    st = res.beams()["status"]
    assert st[0] == 2 and st[1] == (6 if behind else 5)               # BMO_ST_TORN / BMO_ST_CLIPPED
    got, ref = sc["psf"].data, osc["psf"].psf_data()
    assert ref.shape[0] == 3 and got.shape[0] == 3
    _check_records(got, ref)
    if behind:
        assert len(sc["back"]) == osc["back"].psf_data().shape[0] == 0


# ---- 5. accumulation with ray solves -------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_gpu_ray_then_beamlet_solves_accumulate(bmo):
    rays_pos, rays_d = scenes.fibonacci_disc(500, diameter=D_BEAM, y0=-10e-3)
    blt = _lattice(16)
    both, only_r, only_b = (_airy(scenes._ProductFactory(bmo)) for _ in range(3))
    bmo.solve_system_(both["system"], bmo.RayBundle(rays_pos, rays_d, LAM))
    bmo.solve_system_(both["system"], _bundle(bmo, blt))
    bmo.solve_system_(only_r["system"], bmo.RayBundle(rays_pos, rays_d, LAM))
    bmo.solve_system_(only_b["system"], _bundle(bmo, blt))
    assert len(only_b["psf"]) == 3 * len(blt)
    assert _same(both["psf"].data, np.concatenate([only_r["psf"].data, only_b["psf"].data]))
    both["psf"].empty_()
    assert len(both["psf"]) == 0
    bmo.solve_system_(both["system"], _bundle(bmo, blt))
    assert _same(both["psf"].data, only_b["psf"].data)


# ---- 6. retrace ----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_gpu_retraced_beamlets_match_a_fresh_oracle_solve(bmo, orc, monkeypatch):
    from bmo_b200 import solver
    sc, osc = _airy(scenes._ProductFactory(bmo)), _airy(_OF())
    pos = _lattice(12)
    bundle = _bundle(bmo, pos)
    bmo.solve_system_(sc["system"], bundle)
    before = sc["psf"].data
    sc["psf"].empty_()
    move = [0.3e-3, 0.2e-3, -0.2e-3]
    sc["lens"].translate3d_(move)
    osc["lens"].translate3d_(move)
    calls, orig = [], solver.retrace
    monkeypatch.setattr(solver, "retrace", lambda *a, **k: calls.append(1) or orig(*a, **k))
    bmo.solve_system_(sc["system"], bundle, retrace=True)
    assert calls, "the second solve did not retrace the stored solution"
    _oracle_beamlets(orc, osc["system"], pos, (0.0, 1.0, 0.0))
    got, ref = sc["psf"].data, osc["psf"].psf_data()
    assert got.shape == before.shape and not np.array_equal(got, before)
    _check_records(got, ref)


# ---- 7. the sharded map --------------------------------------------------------------------------------------------------
def _one_rank(bmo):
    import torch  # noqa: F401  (libnccl.so.2 comes with torch)
    from bmo_b200 import parallel as par
    return par.FieldComm(0, 1, par.FieldComm.unique_id(), 0)


MAP_KW = dict(n=64, crop_factor=3.0, center="bbox")


@pytest.mark.gpu
def test_one_rank_solve_psf_sharded_beamlet_bundle(bmo):
    from bmo_b200 import parallel as par
    pos = _lattice(24)
    ref_sc, sc = _airy(scenes._ProductFactory(bmo)), _airy(scenes._ProductFactory(bmo))
    bmo.solve_system_(ref_sc["system"], _bundle(bmo, pos), retrace=False)
    ref = ref_sc["psf"].intensity(**MAP_KW)
    comm = _one_rank(bmo)
    try:
        got = par.solve_psf_sharded(sc["system"], _bundle(bmo, pos), sc["psf"], comm=comm, **MAP_KW)
    finally:
        comm.free()
    assert len(sc["psf"]) == 3 * len(pos)
    for a, b in zip(got, ref):
        assert _same(a, b)


def _rank_main(rank, world_size, uid, tmp):
    sys.path.insert(0, ROOT)
    import torch
    torch.cuda.set_device(rank)
    import __graft_entry__ as ge
    m = ge.load_package()
    from bmo_b200 import parallel as par
    comm = par.FieldComm(rank, world_size, uid, device=rank)
    sc = _airy(scenes._ProductFactory(m))
    xs, zs, I = par.solve_psf_sharded(sc["system"], _bundle(m, _lattice(24)), sc["psf"], comm=comm, **MAP_KW)
    comm.free()
    np.save(os.path.join(tmp, f"rank{rank}.npy"), dict(xs=xs, zs=zs, I=I), allow_pickle=True)


def _gpus():
    import torch
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


@pytest.mark.gpu
def test_ranks_beamlet_bundle_equal_one_gpu_map(bmo, tmp_path):
    if _gpus() < 2:
        pytest.skip(f"needs >= 2 GPUs, this box has {_gpus()}")
    import torch.multiprocessing as mp
    from bmo_b200 import parallel as par
    sc = _airy(scenes._ProductFactory(bmo))
    bmo.solve_system_(sc["system"], _bundle(bmo, _lattice(24)), retrace=False)
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


# ---- 8. a Photodetector next to the PSFDetector --------------------------------------------------------------------------
def _pd_and_psf(F):
    """A splitter sends each beamlet's transmitted child to a PSFDetector and its reflected child to a Photodetector."""
    bs = F.ThinBeamsplitter(INCH, reflectance=0.5); bs.zrotate3d_(math.radians(45))
    psfd = F.PSFDetector(10e-3); psfd.translate3d_([0.0, 0.1, 0.0])
    pd = F.Photodetector(8e-3, 64); pd.zrotate3d_(math.radians(90)); pd.translate3d_([0.1, 0.0, 0.0])
    return dict(system=F.System([bs, psfd, pd]), psf=psfd, pd=pd)


@pytest.mark.gpu
def test_gpu_collecting_leaves_the_photodetector_field_alone(bmo, monkeypatch):
    from bmo_b200 import solver
    pos = _splitter_beamlets(32) * 0.5
    a = _pd_and_psf(scenes._ProductFactory(bmo))
    bmo.solve_system_(a["system"], _bundle(bmo, pos))
    assert len(a["psf"]) == 3 * len(pos)
    assert np.abs(a["pd"].field).max() > 0
    b = _pd_and_psf(scenes._ProductFactory(bmo))
    monkeypatch.setattr(solver, "_collect_psfs", lambda dsys, res: None)
    bmo.solve_system_(b["system"], _bundle(bmo, pos))
    assert len(b["psf"]) == 0
    assert _same(a["pd"].field, b["pd"].field)
