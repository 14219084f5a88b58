"""Photodetector fields (K4) and PSFDetector maps (K6) pixel by pixel against the extended-precision reference tests/xref.py.

Every pixel is held to the bound of xref's error model (what binary64 can give that pixel), not to one relative L2 number of the
whole map: a wrong dim pixel, a wrong partial tile or a wrong regime (waist plane, far field, beam tails, long paths, pixels on
an earlier chief segment) fails here even where the bright pixels dominate the L2 norm.

CPU: xref against mpmath at 40 digits, xref against closed-form Gaussian-beam optics, and the double oracle inside every bound
with a margin of at least 4 (the rehearsal of the error model).  GPU: both K4 kernels (pd_field_fast and the reference-order
pd_field) and K6 per pixel, and the PSF records of a ray tree deeper than 64 splitter generations."""
import math

import numpy as np
import pytest

from tests import scenes, scenes2 as s2, xref
from tests.test_psf import LAM, _airy, _disc, _OF
from tests.test_psf_beamlets import CAVITY_TAN, _cavity, _lattice, _sorted

LD_TOL = 64 * float(np.finfo(np.longdouble).eps)
MARGIN = 4.0            # the oracle's worst error / bound must stay below 1 / MARGIN
W0 = 50e-6
ZR = math.pi * W0 ** 2 / LAM
Z0 = 1e4 * ZR + 0.1     # distance from the beamlet's start to its waist: planes at -1e4 z_R still lie ahead of the start
OFFSETS = [0.0, 1e-6, -1e-6, 1e-2, -1e-2, 1.0, -1.0, 1e2, -1e2, 1e4, -1e4]


def _ratio(err, bound, what):
    r, k = xref.worst_ratio(err, bound)
    print(f"xref {what}: worst error / bound {r:.3g}")
    return r, k


# ---- scenes: one free-space beamlet through its waist, and a detector behind a fold mirror ---------------------------------
def _waist(F, off, n=33, half=3.0, lam=LAM, w0=W0, z0=Z0, dist=None):
    """A Photodetector `off` Rayleigh lengths behind the waist of a beamlet that starts at the origin along +y; the window spans
    +-half beam radii.  `dist` places the detector at an absolute distance instead."""
    zr = math.pi * w0 ** 2 / lam
    y = z0 + off * zr if dist is None else dist
    w = w0 * math.sqrt(1 + ((y - z0) / zr) ** 2)
    pd = F.Photodetector(2 * half * w, n)
    pd.translate3d_([0.0, y, 0.0])
    return dict(system=F.System([pd]), pd=pd, w=w, half=half * w, lam=lam, w0=w0, z0=z0)


FOLD_BEAM = dict(pos=(0.0, -0.05, 0.0), dir=(0.0, 1.0, 0.0), lam=1e-6, w0=2e-3)


def _fold(F, n):
    """test_gpu_configs.test_pd_tilted_detector_behind_fold_mirror: a detector tilted by 35 degrees 4 mm behind a fold mirror,
    so that part of its pixels project onto the chief segment in front of the mirror."""
    m = F.SquarePlanoMirror2D(2 * s2.INCH)
    m.zrotate3d_(np.radians(45))
    pd = F.Photodetector(30e-3, n)
    pd.zrotate3d_(float(np.radians(-90) + np.radians(35)))     # the mirror folds +y into +x
    pd.translate3d_([4e-3, 0.0, 0.0])
    return dict(system=F.System([m, pd]), pd=pd)


def _fold_positions(k, seed=7):
    rng = np.random.default_rng(seed)
    pos = np.zeros((k, 3)); pos[:, 1] = FOLD_BEAM["pos"][1]
    pos[:, 0] = rng.uniform(-1.5e-3, -0.1e-3, k)
    pos[:, 2] = rng.uniform(-1.5e-3, 1.5e-3, k)
    return pos


# ---- CPU: the reference itself --------------------------------------------------------------------------------------------
def _oracle_waist(orc, off, **kw):
    sc = _waist(scenes._OracleFactory(), off, **kw)
    g = orc.gaussian_beamlet([0.0, 0.0, 0.0], [0.0, 1.0, 0.0], sc["lam"], w0=sc["w0"], z0=sc["z0"], support=(1.0, 0.0, 0.0))
    orc.solve_system_(sc["system"], g)
    return sc, xref.beamlets_from_oracle(orc.gauss_export(sc["system"], g), 0)


def _oracle_pd(orc, sc, bl, n):
    pos, dirm = sc["pd"].pose()
    p1, (ii, jj) = xref.pd_pixels(pos, dirm, -sc["half"], sc["half"], n)
    return sc["pd"].pd_field(n)[ii, jj], xref.pd_field(bl, p1), p1


def test_xref_matches_mpmath(orc):
    """xref's longdouble restatement against the same code at 40 digits, on seeded pixel-term pairs at the waist plane, next to
    it, in the far field and in the beam tails (K4), and on PSF records of the Airy scene (K6).  Longdouble forms a phase of
    k z ~ 1e9 rad to ~1e-10 rad, so each pixel is held to the tighter of 1/64 of the bound B it sets and 64 longdouble
    roundings of its largest phase: 64 eps_ld (Phi + 1) S."""
    rng = np.random.default_rng(11)
    for off in (0.0, 1e-6, -1.0, 1e4, -1e4):
        sc, bl = _oracle_waist(orc, off, n=17, half=30.0 if off == -1.0 else 3.0)
        pos, dirm = sc["pd"].pose()
        ij = rng.integers(0, 17, (2, 40))
        p1, _ = xref.pd_pixels(pos, dirm, -sc["half"], sc["half"], 17, (ij[0], ij[1]))
        a, b = xref.pd_field(bl, p1), xref.pd_field(bl, p1, xref.MP)
        d = np.abs(xref._f(a["re"] - b["re"].astype(np.longdouble)) + 1j * xref._f(a["im"] - b["im"].astype(np.longdouble)))
        assert (d <= np.minimum(a["B"] / 64, LD_TOL * (a["PHI"] + 1) * a["S"])).all(), off
    F = _OF()
    sc = _airy(F)
    pos, d = _disc(200)
    for p in pos:
        orc.solve_system_(sc["system"], orc.beam(p, [0.0, 1.0, 0.0], LAM))
    rec = sc["psf"].psf_data()
    xs, zs, _ = sc["psf"].psf_intensity(n=9, crop_factor=3, center="bbox")
    ppos, pdir = sc["psf"].pose()
    p, _ = xref.psf_pixels(ppos, pdir, xs, zs, (np.arange(9), (np.arange(9) * 5) % 9))
    a, b = xref.psf_field(rec, p), xref.psf_field(rec, p, xref.MP)
    dd = np.abs(xref._f(a["re"] - b["re"].astype(np.longdouble)) + 1j * xref._f(a["im"] - b["im"].astype(np.longdouble)))
    assert (dd <= np.minimum(a["B"] / 64, LD_TOL * (a["PHI"] + 1) * a["S"])).all()


def test_xref_closed_form_gaussian_beam(orc):
    """On the chief ray of a free-space beamlet xref's w, R and Gouy phase are those of a Gaussian beam of waist w0 and Rayleigh
    length z_R' = w0 / tan(lambda / (pi w0)) (the divergence ray's slope, Gaussian.jl:215-256): w = w0 sqrt(1 + (z/z_R')^2),
    R = z / (z^2 + z_R'^2), psi = -atan(z / z_R')."""
    zr = W0 / math.tan(LAM / (math.pi * W0))
    for off in OFFSETS:
        sc, bl = _oracle_waist(orc, off)
        pos, dirm = sc["pd"].pose()
        p1, _ = xref.pd_pixels(pos, dirm, -sc["half"], sc["half"], 33, (np.array([16]), np.array([16])))
        t = xref.pd_terms(bl[0], p1)
        z = float(pos[1]) - Z0
        assert abs(t["w"][0] - W0 * math.sqrt(1 + (z / zr) ** 2)) <= 1e-12 * t["w"][0], off
        tol_z = 4 * math.ulp(Z0)          # the waist sits where binary64 inputs put it: z0 and the divergence ray's start
        assert abs(t["R"][0] - z / (z * z + zr * zr)) <= 1e-9 * abs(z / (z * z + zr * zr)) + tol_z / zr ** 2, off
        assert abs(t["psi"][0] + math.atan(z / zr)) <= 1e-9, off


def test_oracle_within_bound_waist_tails_long_paths(orc):
    """The rehearsal of K4's error model: the double oracle meets every per-pixel bound with a margin of at least 4 at planes
    {0, +-1e-6, +-1e-2, +-1, +-1e2, +-1e4} z_R from the waist, in tails where r^2/w^2 passes 708, and along paths with k z from
    1e6 to 1.6e9 rad."""
    cases = [dict(off=o) for o in OFFSETS] + [dict(off=1.0, half=40.0, n=65)]
    cases += [dict(off=0.0, lam=lam, w0=2e-3, z0=0.0, dist=dist) for lam in (400e-9, 1.6e-6) for dist in (0.25, 100.0)]
    worst = 0.0
    for c in cases:
        off = c.pop("off")
        n = c.get("n", 33)
        sc, bl = _oracle_waist(orc, off, **c)
        ref, X, _ = _oracle_pd(orc, sc, bl, n)
        r, k = xref.worst_ratio(np.abs(ref - X["A"]), X["B"])
        assert r <= 1 / MARGIN, (off, c, r, k)
        worst = max(worst, r)
        if c.get("half") == 40.0:
            assert (np.abs(X["A"]) < 1e-300).any() and (np.abs(ref) == 0).any()    # exp(-r^2/w^2) below binary64's range
    print(f"oracle K4 worst error / bound {worst:.3g}")


def test_oracle_within_bound_fold_mirror(orc):
    """Same for the tilted detector behind a fold mirror, where xref finds pixels on the earlier chief segment."""
    n = 33
    sc = _fold(scenes._OracleFactory(), n)
    bl = []
    for p in _fold_positions(5):
        g = orc.gaussian_beamlet(list(p), FOLD_BEAM["dir"], FOLD_BEAM["lam"], w0=FOLD_BEAM["w0"], support=(1.0, 0.0, 0.0))
        orc.solve_system_(sc["system"], g)
        bl += xref.beamlets_from_oracle(orc.gauss_export(sc["system"], g), 1)
    pos, dirm = sc["pd"].pose()
    p1, (ii, jj) = xref.pd_pixels(pos, dirm, -15e-3, 15e-3, n)
    X = xref.pd_field(bl, p1)
    assert len(bl) == 5 and X["earlier"].any() and not X["earlier"].all()
    r, _ = xref.worst_ratio(np.abs(sc["pd"].pd_field(n)[ii, jj] - X["A"]), X["B"])
    assert r <= 1 / MARGIN, r


def test_oracle_within_bound_dense_expander(orc):
    """Same for the 4096 overlapping beamlets through the expander of test_gpu_pd_dense_overlap, on pixels out to the far tails
    (|A| ~ 5e-268 at pixel (119, 120)), where a height's error along the chief dominates the bound."""
    n = 128
    sc = s2.expander_oracle(n)
    lat = s2.beamlet_lattice(64)
    bl = []
    for p in lat["pos"]:
        g = orc.gaussian_beamlet(p, lat["dir"], lat["lam"], lat["w0"], M2=lat["M2"], P0=lat["P0"], support=lat["support"])
        orc.solve_system_(sc["system"], g)
        bl += xref.beamlets_from_oracle(orc.gauss_export(sc["system"], g), 2)
    assert len(bl) == len(lat["pos"])
    rng = np.random.default_rng(5)
    ii = np.concatenate([rng.integers(0, n, 12), [0, n - 1, 119]])
    jj = np.concatenate([rng.integers(0, n, 12), [n - 1, 0, 120]])
    pos, dirm = sc["pd"].pose()
    p1, _ = xref.pd_pixels(pos, dirm, -20e-3, 20e-3, n, (ii, jj))
    X = xref.pd_field(bl, p1)
    assert np.abs(X["A"]).min() < 1e-260
    r, _ = xref.worst_ratio(np.abs(sc["pd"].pd_field(n)[ii, jj] - X["A"]), X["B"])
    assert r <= 1 / MARGIN, r


def _airy_moved(F, offset):
    sc = _airy(F)
    g = F.ObjectGroup([sc["lens"], sc["psf"]])
    g.translate3d_([offset, 0.0, 0.0])
    sc["system"] = F.System([g])
    return sc


@pytest.mark.parametrize("offset", [0.0, 1.0, 10.0])
def test_oracle_within_bound_psf(orc, offset):
    """K6's error model rehearsed on the Airy scene moved 0, 1 and 10 m from the world origin, bbox window and an explicit
    window with shifts."""
    sc = _airy_moved(_OF(), offset)
    pos, d = _disc(400)
    for p in pos + np.array([offset, 0.0, 0.0]):
        orc.solve_system_(sc["system"], orc.beam(p, [0.0, 1.0, 0.0], LAM))
    rec = sc["psf"].psf_data()
    ppos, pdir = sc["psf"].pose()
    for n, kw in ((64, dict(crop_factor=5, center="bbox")),
                  (33, dict(x_min=-2e-5, x_max=3e-5, z_min=-1e-5, z_max=1e-5, x0_shift=2e-6, z0_shift=-1e-6))):
        xs, zs, I = sc["psf"].psf_intensity(n=n, **kw)
        p, (ii, jj) = xref.psf_pixels(ppos, pdir, xs, zs)
        X = xref.psf_field(rec, p)
        r, _ = xref.worst_ratio(np.abs(I[ii, jj] - X["I"]), xref.intensity_bound(X["A"], X["B"]))
        assert r <= 1 / MARGIN, (n, r)


# ---- GPU: K4 --------------------------------------------------------------------------------------------------------------
def _pd_gpu(bmo, sc, bundle, ref_order):
    dsys = bmo.upload_system(sc["system"], [float(bundle.lam[0])])
    res = bmo.trace_beamlets(dsys, bundle.rays, np.zeros(len(bundle.rays), np.int32), bundle.w0, bundle.E0)
    res.lams = [float(bundle.lam[0])]
    idx = dsys.flat.object_index(sc["pd"])
    n = sc["pd"].n
    field = np.zeros((n, n), np.complex128, order="F")
    bmo.pd_accumulate(dsys, res, idx, field, reference_order=ref_order)
    return res, idx, field


def _check_pd(bmo, sc, bundle, ref_order, what, ij=None):
    res, idx, field = _pd_gpu(bmo, sc, bundle, ref_order)
    pd = sc["pd"]
    bl = xref.beamlets_from_result(res, idx)
    assert len(bl) == len(bundle.rays), (len(bl), len(bundle.rays))
    p1, (ii, jj) = xref.pd_pixels(pd.position(), pd.orientation(), pd.lo, pd.hi, pd.n, ij)
    X = xref.pd_field(bl, p1)
    kern = "pd_field" if ref_order else "pd_field_fast"
    r, k = _ratio(np.abs(field[ii, jj] - X["A"]), X["B"], f"{kern} {what}")
    assert r <= 1.0, (what, kern, r, int(ii[k]), int(jj[k]), complex(field[ii[k], jj[k]]), complex(X["A"][k]), X["B"][k])
    return X


def _waist_bundle(bmo, sc):
    return bmo.BeamletBundle.from_params(np.zeros((1, 3)), (0.0, 1.0, 0.0), sc["lam"], sc["w0"], z0=sc["z0"], support=(1.0, 0.0, 0.0))


@pytest.mark.gpu
@pytest.mark.parametrize("ref_order", [False, True])
@pytest.mark.parametrize("off", OFFSETS)
def test_gpu_pd_through_the_waist(bmo, off, ref_order):
    sc = _waist(scenes._ProductFactory(bmo), off)
    _check_pd(bmo, sc, _waist_bundle(bmo, sc), ref_order, f"waist {off:g} z_R")


@pytest.mark.gpu
@pytest.mark.parametrize("ref_order", [False, True])
def test_gpu_pd_tails_and_long_paths(bmo, ref_order):
    sc = _waist(scenes._ProductFactory(bmo), 1.0, n=65, half=40.0)
    X = _check_pd(bmo, sc, _waist_bundle(bmo, sc), ref_order, "tails r^2/w^2 > 708")
    assert (np.abs(X["A"]) < 1e-300).any()
    for lam in (400e-9, 1.6e-6):
        for dist in (0.25, 100.0):
            sc = _waist(scenes._ProductFactory(bmo), 0.0, lam=lam, w0=2e-3, z0=0.0, dist=dist)
            _check_pd(bmo, sc, _waist_bundle(bmo, sc), ref_order, f"lambda {lam:g} at {dist:g} m")


def _fold_bundle(bmo, k):
    return bmo.BeamletBundle.from_params(_fold_positions(k), FOLD_BEAM["dir"], FOLD_BEAM["lam"], FOLD_BEAM["w0"], support=(1.0, 0.0, 0.0))


@pytest.mark.gpu
@pytest.mark.parametrize("ref_order", [False, True])
@pytest.mark.parametrize("k", [47, 48, 49, 97])
def test_gpu_pd_fold_mirror_deferred_pairs(bmo, k, ref_order):
    """Beamlet counts either side of PDF_BATCH = 48: the fast kernel defers the pairs on an earlier segment per batch."""
    sc = _fold(scenes._ProductFactory(bmo), 33)
    X = _check_pd(bmo, sc, _fold_bundle(bmo, k), ref_order, f"fold mirror, {k} beamlets")
    assert X["earlier"].any() and not X["earlier"].all()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 31, 33, 257])
def test_gpu_pd_map_sizes(bmo, n):
    """Partial 32 x 8 tiles and the n = 1 LinRange; n = 257 is checked on its last tile row and column plus a sample."""
    sc = _fold(scenes._ProductFactory(bmo), n)
    for ref_order in (False, True):
        _check_pd(bmo, sc, _fold_bundle(bmo, 49), ref_order, f"n = {n}", xref.edge_sample(n))


@pytest.mark.gpu
def test_gpu_pd_dense_overlap(bmo):
    """4096 overlapping beamlets through the expander (accumulation error), on a seeded sample of pixels."""
    n = 128
    sc = s2.expander(bmo, n)
    lat = s2.beamlet_lattice(64)
    bundle = bmo.BeamletBundle.from_params(lat["pos"], lat["dir"], lat["lam"], lat["w0"], M2=lat["M2"], P0=lat["P0"], support=lat["support"])
    rng = np.random.default_rng(5)
    ij = (rng.integers(0, n, 96), rng.integers(0, n, 96))
    _check_pd(bmo, sc, bundle, False, "4096 beamlets", ij)


@pytest.mark.gpu
@pytest.mark.parametrize("ref_order", [False, True])
def test_gpu_pd_pose_sweep(bmo, ref_order):
    """bmo_pd_accumulate_poses: the detector moves along the folded beam from pose to pose, and the poses hold 47, 97 and 49
    beamlets, so every pose's record range starts off a multiple of PDF_BATCH = 48."""
    from bmo_b200 import _lib as L, sweep, solver
    import ctypes as C
    counts = [47, 97, 49]
    P, n = len(counts), 33
    sc = _fold(scenes._ProductFactory(bmo), n)
    base = np.array(sc["pd"].position(), dtype=np.float64)

    def apply_pose(p):
        sc["pd"].translate_to3d_([float(x) for x in base + np.array([1e-3 * p, 0.0, 0.0])])
    f0, (prims, verts, bounds, det_pos, det_dir) = sweep.flatten_poses(sc["system"], [FOLD_BEAM["lam"]], P, apply_pose)
    dsys = solver.DeviceSystem(f0, 0)
    L.check(L.lib().bmo_system_set_poses(dsys.h, P, L.ptr(prims), L.ptr(verts), L.ptr(bounds), L.ptr(det_pos), L.ptr(det_dir)))
    bundles = [_fold_bundle(bmo, k) for k in counts]
    rays = np.ascontiguousarray(np.concatenate([b.rays.reshape(-1, 18) for b in bundles]))
    w0 = np.ascontiguousarray(np.concatenate([b.w0 for b in bundles]))
    E0 = np.concatenate([b.E0 for b in bundles])
    e = np.ascontiguousarray(np.stack([E0.real, E0.imag], axis=-1))
    pose_id = np.ascontiguousarray(np.repeat(np.arange(P, dtype=np.int32), counts))
    lam_ids = np.zeros(len(rays), np.int32)
    h = C.c_void_p()
    L.check(L.lib().bmo_trace_beamlets(dsys.h, rays.shape[0], L.ptr(rays), L.ptr(lam_ids), L.ptr(w0), L.ptr(e), L.ptr(pose_id), 100, 0,
                                       C.byref(h)))
    res = solver.TraceResult(dsys, h)
    res.lams = [FOLD_BEAM["lam"]]
    assert res.n_beams == res.n_roots == len(rays)
    idx = f0.object_index(sc["pd"])
    fields = np.zeros((P, n * n * 2))
    L.check(L.lib().bmo_pd_accumulate_poses(dsys.h, res.h, idx, P, L.ptr(fields), L.PD_REFERENCE_ORDER if ref_order else 0))
    kern = "pd_field" if ref_order else "pd_field_fast"
    for p in range(P):
        field = (fields[p, 0::2] + 1j * fields[p, 1::2]).reshape(n, n, order="F")
        bl = xref.beamlets_from_result(res, idx, keep=pose_id == p)
        assert len(bl) == counts[p]
        det = sweep.get_pose_tables(dsys, p)[3][idx]
        p1, (ii, jj) = xref.pd_pixels(det[0:3], det[3:12].reshape(3, 3), sc["pd"].lo, sc["pd"].hi, n)
        X = xref.pd_field(bl, p1)
        assert X["earlier"].any()
        r, k = _ratio(np.abs(field[ii, jj] - X["A"]), X["B"], f"{kern} pose {p} of a sweep, {counts[p]} beamlets")
        assert r <= 1.0, (p, kern, r, int(ii[k]), int(jj[k]))


# ---- GPU: K6 --------------------------------------------------------------------------------------------------------------
def _check_psf(psf, rec, xs, zs, I, what, ij=None):
    p, (ii, jj) = xref.psf_pixels(psf.position(), psf.orientation(), xs, zs, ij)
    X = xref.psf_field(rec, p)
    r, k = _ratio(np.abs(I[ii, jj] - X["I"]), xref.intensity_bound(X["A"], X["B"]), f"psf_intensity {what}")
    assert r <= 1.0, (what, r, int(ii[k]), int(jj[k]), float(I[ii[k], jj[k]]), float(X["I"][k]))
    return r


def _airy_gpu(bmo, offset=0.0, n_rays=1000):
    sc = _airy_moved(scenes._ProductFactory(bmo), offset)
    pos, d = _disc(n_rays)
    bmo.solve_system_(sc["system"], bmo.RayBundle(pos + np.array([offset, 0.0, 0.0]), d, LAM))
    return sc


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 33, 160, 257])
def test_gpu_psf_airy_per_pixel(bmo, n):
    sc = _airy_gpu(bmo)
    psf = sc["psf"]
    rec = psf.data
    ij = xref.edge_sample(n)
    for center in ("centroid", "bbox"):
        xs, zs, I = psf.intensity(n=n, crop_factor=5, center=center)
        _check_psf(psf, rec, xs, zs, I, f"n = {n} {center}", ij)
    kw = dict(x_min=-2e-5, x_max=3e-5, z_min=-1e-5, z_max=1e-5, x0_shift=2e-6, z0_shift=-1e-6)
    xs, zs, I = psf.intensity(n=n, **kw)
    _check_psf(psf, rec, xs, zs, I, f"n = {n} window + shifts", ij)


@pytest.mark.gpu
def test_gpu_psf_column_bands(bmo):
    """bmo_psf_intensity_cols on bands whose j0 / j1 are not multiples of the 8-row tile."""
    import ctypes as C
    from bmo_b200 import _lib as L, solver
    sc = _airy_gpu(bmo)
    psf, n = sc["psf"], 160
    dsys, oi = solver._psf_dsys(psf)
    lims = solver.psf_window(solver.psf_lims(psf, 5.0, "bbox"))
    xs, zs = solver.psf_axes(n, lims)
    rec = psf.data
    for j0, j1 in ((0, 13), (13, 101), (101, 160), (77, 78)):
        out = np.zeros((n, j1 - j0), order="F")
        L.check(L.lib().bmo_psf_intensity_cols(dsys.h, C.c_void_p(psf._psf), oi, 0, n, L.ptr(lims), 0.0, 0.0, j0, j1, L.ptr(out), 0))
        I = np.zeros((n, n)); I[:, j0:j1] = out
        jj, ii = np.meshgrid(np.arange(j0, j1), np.arange(n))
        _check_psf(psf, rec, xs, zs, I, f"columns [{j0}, {j1})", (ii.ravel(), jj.ravel()))


@pytest.mark.gpu
@pytest.mark.parametrize("offset", [0.0, 1.0, 10.0])
def test_gpu_psf_far_from_the_origin(bmo, offset):
    """K6 folds k (opl - hit . dir) into one constant, so its phase rounding grows with |hit|; the bound's Phi carries k |hit|."""
    sc = _airy_gpu(bmo, offset)
    xs, zs, I = sc["psf"].intensity(n=64, crop_factor=5, center="bbox")
    _check_psf(sc["psf"], sc["psf"].data, xs, zs, I, f"scene moved {offset:g} m")


@pytest.mark.gpu
def test_gpu_psf_beamlet_records(bmo):
    sc = _airy(scenes._ProductFactory(bmo))
    bmo.solve_system_(sc["system"], bmo.BeamletBundle.from_params(_lattice(12), (0.0, 1.0, 0.0), LAM, w0=0.2e-3, support=(1.0, 0.0, 0.0)))
    rec = sc["psf"].data
    assert rec.shape[0] == 3 * len(_lattice(12))
    xs, zs, I = sc["psf"].intensity(n=64, crop_factor=3, center="centroid")
    _check_psf(sc["psf"], rec, xs, zs, I, "beamlet records")


# ---- GPU: ray PSF records deeper than 64 splitter generations -------------------------------------------------------------
@pytest.mark.gpu
def test_gpu_ray_opl_through_a_deep_cavity(bmo, orc):
    """The cavity of test_psf_beamlets traced with plain rays: their PSF records take optical_path_length(beam) through every
    ancestor (Beam.jl:137-149), more than 64 generations of them."""
    sc, osc = _cavity(scenes._ProductFactory(bmo)), _cavity(_OF())
    pos = np.array([[-11.5e-3, -10e-3, z] for z in (-2e-3, 0.0, 3e-3)])
    d = np.array([CAVITY_TAN, 1.0, 0.0]) / math.hypot(CAVITY_TAN, 1.0)
    res = bmo.solve_system_(sc["system"], bmo.RayBundle(pos, d, LAM))
    for p in pos:
        orc.solve_system_(osc["system"], orc.beam(p, d, LAM))
    got, ref = sc["psf"].data, osc["psf"].psf_data()
    b, seg = res.beams(), res.segments()
    depth = np.zeros(res.n_beams, np.int64)
    for i in range(res.n_roots, res.n_beams):
        depth[i] = depth[b["parent"][i]] + 1
    on = [i for i in range(res.n_beams) if b["status"][i] == 2 and b["nseg"][i] > 0 and seg["obj"][b["first"][i] + b["nseg"][i] - 1] == 2]
    assert len(on) == got.shape[0] == ref.shape[0]
    assert depth[on].max() > 64 and (depth[on] > 64).sum() >= 10, depth[on].max()
    got, ref = _sorted(got), _sorted(ref)
    assert np.abs(got[:, 6] - ref[:, 6]).max() <= 1e-12 * np.abs(ref[:, 6]).max()          # optical path length
    assert np.abs(got[:, 0:6] - ref[:, 0:6]).max() <= 1e-9 * max(1.0, np.abs(ref[:, 0:3]).max())
    assert np.abs(got[:, 7] - ref[:, 7]).max() <= 1e-12
    assert np.array_equal(got[:, 8], ref[:, 8])
    assert got[:, 6].max() > 64 * 2e-3
    xs, zs, I = sc["psf"].intensity(n=48, crop_factor=2)
    _check_psf(sc["psf"], sc["psf"].data, xs, zs, I, "ray cavity")
