"""TEST INFRASTRUCTURE ONLY -- extended-precision reference of the two detector kernels, with a per-pixel error model.

K4 (Photodetector field, bmo_detector.cu) and K6 (PSFDetector intensity, bmo_psf.cu) are restated here in numpy `longdouble`
(x86-64: 64-bit significand, eps = 1.08e-19) on the same binary64 inputs the kernels read -- the segment table of the traced
beamlets, the 9-column PSF records, the detector pose -- so that a comparison isolates the kernels' arithmetic from the tracer:

  K4  I(i, j) -> sum_b electric_field(gauss_b, r, z) sqrt(proj_b)  with the pixel grid of Photodetector.jl:78-103 (LinRange
      lerpi, transposed orientation), point_on_beam with its earlier-segment loop (Beam.jl:177-205), gauss_parameters
      (Gaussian.jl:298-353: line_plane_distance3d, angle3d, the NaN guards and the R < 0 flip) and electric_field with ref_phi
      (Gaussian.jl:381-392, OpticUtils.jl:87-89).  tan(pi/2 - acos(c)) is taken as c / sqrt(1 - c^2) and E0 (w0_b / w0) w0 / w
      as E0 w0_b / w: identical values, without the cancellations the literal forms would cost in extended precision.
  K6  I[i, j] = | sum_h proj_h cis(k_h (opl_h + (p_ij - hit_h) . dir_h)) |^2   (PSFDetector.jl:190-237).

Every function is written against a backend (LD: numpy longdouble arrays, MP: numpy object arrays of mpmath numbers), so the
same code evaluated at 40 digits validates the longdouble restatement (tests/test_detector_xref.py).

Error model.  Besides the value A of a pixel, `pd_field` / `psf_field` return
  S  = sum_h |term_h|                      (magnitudes of the complex terms)
  B  = a bound on |A_binary64 - A|         (what a binary64 implementation of the operation can be held to)
with
  B = sum_h |term_h| beta_h + C_N n_terms EPS S + U
  beta_h = C_PHI EPS Phi_h + C_G G_h + C_A (EPS + DELTA) D_h
where EPS = 2^-53 and DELTA = 1e-13 (K4's one-Newton-step rcp13 / rsqrt13, bmo_detector.cu; 0 for K6):
  Phi_h  largest phase magnitude binary64 must form: K4 k (|l0| + |l1| + |temp| + |p0| + |p1|) + |ref_phi| + k r^2 |R| / 2
         + |psi|; K6 k (|opl| + |hit| + |p|) -- K6 folds k (opl - hit . dir) into one constant (bmo_psf.cu), so its rounding
         grows with |hit| where the reference's k (opl + (p - hit) . dir) does not.
  G_h    (K4) phase and amplitude error carried by the Gaussian parameters: the ray heights y = ray_pos + il ray_dir - point
         are differences of world coordinates (absolute error EPS (|ray_pos| + |il| + |point|)), the slopes m come from a dot
         product of near-orthogonal unit vectors (absolute error EPS (1 + m^2)^(3/2)), and a height's error along the chief
         turns the angle between height and ray (error (ey / y) (1 + m^2)^(3/2) in m, so ey (1 + m^2)^(3/2) in y m: the
         dominant term at the waist plane and in the far tails); propagated to w, R and psi:
         amplitude (1 + 2 r^2 / w^2) dw / w, curvature phase k r^2 / 2 dR, Gouy phase d(sin psi) / cos psi.
  D_h    (K4) relative-error amplification of the reciprocal / square roots: 1 + 2 r^2 / w^2 + k r^2 |R| + 1 / cos psi.
  U      underflow: exp(-r^2/w^2) is flushed to 0 below -708 (binary64 has nothing there but subnormals):
         sum_h |E0_h w0_h / w_h sqrt(proj_h)| exp(-708).
The constants were fixed once from the double oracle (test_oracle_within_bound): each is about four times the largest ratio
the oracle reached for its term, so the oracle meets the whole bound with a margin of at least 4.
  C_PHI = 8   phase: about six roundings form it (the l1 dot product, z = l0 + l1, k z, + psi + curvature + ref_phi); the
              oracle reached 1.6 EPS Phi (a far-tail pixel of the fold-mirror scene, where the phase term is all of the bound)
  C_G   = 4   Gaussian parameters: two roundings per height / slope, propagated once (the oracle reached 0.1 of the bound at a
              far-tail pixel of 256 overlapping beamlets through the expander, where this term is all of it)
  C_A   = 8   reciprocal / square root approximations: up to four of them enter one factor (rw twice, id / iw, spsi)
  C_N   = 2   the n-term complex sum and the final |A|^2
Intensities: |dI| <= 2 |A| B + B^2.
"""
import math

import numpy as np

EPS = 2.0 ** -53
DELTA = 1e-13
C_PHI, C_G, C_A, C_N = 8.0, 4.0, 8.0, 2.0
EXP_FLOOR = math.exp(-708.0)
TWO_PI_F64 = 6.283185307179586      # Float64(2pi): the reference's k = 2pi / lambda and ref_phi use this binary64 constant


# ---- backends -----------------------------------------------------------------------------------------------------------
class LD:
    """numpy longdouble."""
    @staticmethod
    def arr(x): return np.asarray(x, dtype=np.float64).astype(np.longdouble)
    sqrt, exp, cos, sin, arctan2, isnan = np.sqrt, np.exp, np.cos, np.sin, np.arctan2, np.isnan
    HALF_PI = np.longdouble("1.570796326794896619231321691639751442")


class MP:
    """numpy object arrays of mpmath mpf (40 digits by default)."""
    import mpmath as _mp
    _mp.mp.dps = 40
    @staticmethod
    def arr(x):
        a = np.asarray(x, dtype=np.float64)
        return np.vectorize(lambda v: MP._mp.mpf(float(v)), otypes=[object])(a) if a.ndim else MP._mp.mpf(float(a))
    sqrt = staticmethod(np.vectorize(lambda v: MP._mp.sqrt(v) if v >= 0 else MP._mp.nan, otypes=[object]))
    exp = staticmethod(np.vectorize(lambda v: MP._mp.exp(v), otypes=[object]))
    cos = staticmethod(np.vectorize(lambda v: MP._mp.cos(v), otypes=[object]))
    sin = staticmethod(np.vectorize(lambda v: MP._mp.sin(v), otypes=[object]))
    arctan2 = staticmethod(np.vectorize(lambda y, x: MP._mp.atan2(y, x), otypes=[object]))
    isnan = staticmethod(np.vectorize(lambda v: bool(MP._mp.isnan(v)), otypes=[bool]))
    HALF_PI = _mp.pi / 2


def _dot(a, b):
    return a[..., 0] * b[..., 0] + a[..., 1] * b[..., 1] + a[..., 2] * b[..., 2]


def _f(x):
    return np.asarray(x, dtype=np.float64) if not isinstance(x, np.ndarray) or x.dtype != object else x.astype(np.float64)


def lin(n, lo, hi):
    """LinRange(lo, hi, n) in binary64 (Base.lerpi), as the kernels and the reference index it."""
    t = np.arange(n) / (n - 1) if n > 1 else np.zeros(1)
    return (1 - t) * lo + t * hi


# ---- K4: Photodetector ----------------------------------------------------------------------------------------------------
def beamlets_from_result(res, pd_index, keep=None):
    """Beamlets of a device result (TraceResult of a beamlet trace) that ended on object `pd_index`, as pd_field input; `keep`
    (bool per beam) selects some of them, e.g. the beams of one pose of a sweep."""
    b, seg = res.beams(), res.segments()
    lam = np.asarray(res.lams, dtype=np.float64)[b["lam_id"]]
    tree = []
    for i in range(res.n_beams):
        f, n = int(b["first"][i]), int(b["nseg"][i])
        rows = (f + np.arange(n))[:, None] * 3 + np.arange(3)[None, :]
        tree.append(dict(parent=int(b["parent"][i]), lam=float(lam[i]), w0=float(b["w0"][i]), E0=complex(b["E0"][i]),
                         pos=seg["pos"][rows], dir=seg["dir"][rows], n=seg["n"][rows[:, 0]], t=seg["t"][rows[:, 0]],
                         nrm=seg["nrm"][rows[:, 0]], obj=seg["obj"][rows], ok=b["status"][i] == 2 and (keep is None or keep[i])))
    return _leaves(tree, pd_index)


def beamlets_from_oracle(tree_export, pd_index):
    """Same from orc.gauss_export(system, g) (BFS list of dicts with chief / waist / div ray records)."""
    tree = []
    for g in tree_export:
        c, w, d = g["chief"], g["waist"], g["div"]
        n = len(c["t"])
        tree.append(dict(parent=g["parent"], lam=g["lam"], w0=g["w0"], E0=complex(g["E0"]),
                         pos=np.stack([c["pos"], w["pos"][:n], d["pos"][:n]], axis=1),
                         dir=np.stack([c["dir"], w["dir"][:n], d["dir"][:n]], axis=1), n=c["n"], t=c["t"], nrm=c["nrm"],
                         obj=np.stack([c["obj"], w["obj"][:n], d["obj"][:n]], axis=1), ok=True))
    return _leaves(tree, pd_index)


def _leaves(tree, pd_index):
    """The rays (t, n) of every beam's ancestors, root first, up to each one's first ray without a hit (their length and OPL
    enter length(gauss) and optical_path_length(gauss), Beam.jl:125-149), and the beams whose three last rays ended on the
    detector."""
    for g in tree:
        own = []
        for t, nn in zip(g["t"], g["n"]):
            if not np.isfinite(t):
                break
            own.append((t, nn))
        p = g["parent"]
        g["anc"] = tree[p]["anc"] + tree[p]["own"] if p >= 0 else []
        g["own"] = own
    return [g for g in tree if g["ok"] and len(g["t"]) and np.isfinite(g["t"][-1]) and (g["obj"][-1] == pd_index).all()]


def pd_pixels(pos, dirm, lo, hi, n, ij=None):
    """World coordinates of pixels (i, j) (binary64, the reference's arithmetic): p1 = dir' (x, 0, y) + pos."""
    x = lin(n, lo, hi)
    if ij is None:
        jj, ii = np.meshgrid(np.arange(n), np.arange(n))
        ii, jj = ii.ravel(order="F"), jj.ravel(order="F")
    else:
        ii, jj = ij
    dirm = np.asarray(dirm, dtype=np.float64)
    return (dirm[0][None, :] * x[ii][:, None] + dirm[2][None, :] * x[jj][:, None]) + np.asarray(pos)[None, :], (ii, jj)


def pd_terms(g, p1, M=LD):
    """Every term electric_field(gauss, r, z) sqrt(proj) of one beamlet at pixels p1 (m, 3) -> dict(re, im, mag = |term|, beta,
    floor, idx = chief segment of point_on_beam, w, R, psi, z)."""
    ns = len(g["t"])
    P = M.arr(g["pos"]); Dd = M.arr(g["dir"]); T = M.arr(g["t"]); N = M.arr(g["n"])
    lam = M.arr(g["lam"]); k = M.arr(TWO_PI_F64) / lam
    anc = np.array(g["anc"], dtype=np.float64).reshape(-1, 2)
    at, an = M.arr(anc[:, 0]), M.arr(anc[:, 1])
    plen, popl = M.arr(0.0) + sum(at), M.arr(0.0) + sum(at * an)
    L = plen + sum(T[s] for s in range(ns))                         # length(gauss)
    OPL = popl + sum(T[s] * N[s] for s in range(ns))                # optical_path_length(gauss)
    l0 = L - T[ns - 1]
    ref_phi = (OPL - L) / lam * M.arr(TWO_PI_F64)
    p0, d0 = P[ns - 1, 0], Dd[ns - 1, 0]
    q = M.arr(p1)
    l1 = _dot(q - p0, d0[None, :])
    v = q - (p0[None, :] + l1[:, None] * d0[None, :])
    r2 = _dot(v, v)
    z = l0 + l1
    # point_on_beam (Beam.jl:177-205): first earlier segment with z < temp, else the last one
    temps = [plen]
    for s in range(ns - 1):
        temps.append(temps[-1] + T[s])
    idx = np.full(len(l1), ns - 1)
    for s in range(ns - 2, -1, -1):
        idx = np.where(z < temps[s + 1], s, idx)
    start = np.array([temps[s] for s in idx], dtype=object if M is MP else np.longdouble)
    point = P[idx, 0] + (z - start)[:, None] * Dd[idx, 0]
    cd = Dd[idx, 0]
    ys, ms, mag = [], [], []
    for ray in (2, 1):                                               # divergence, then waist (Gaussian.jl:310-325)
        rp, rd = P[idx, ray], Dd[idx, ray]
        il = _dot(point - rp, cd) / _dot(cd, rd)                     # line_plane_distance3d
        y0 = rp + il[:, None] * rd - point
        y = M.sqrt(_dot(y0, y0))
        c = _dot(y0, rd) / (y * M.sqrt(_dot(rd, rd)))                # cos angle3d(y0 / y, ray dir)
        c = np.where(c > 1, 1, np.where(c < -1, -1, c))
        m = c / M.sqrt(1 - c * c)                                    # tan(pi/2 - acos(c))
        ys.append(y); ms.append(m)
        mag.append(np.abs(_f(rp)).sum(axis=1) + np.abs(_f(il)) + np.abs(_f(point)).sum(axis=1))
    (yd, yw), (md, mw) = ys, ms
    E = yd * md + yw * mw
    F2 = md * md + mw * mw
    w2 = yd * yd + yw * yw
    R = E / w2
    Rz = E * E / (w2 * F2)
    with np.errstate(divide="ignore", invalid="ignore"):
        psi = -M.arctan2(np.ones_like(Rz), M.sqrt(1 / Rz - 1))
    R = np.where(M.isnan(R), 0, R)
    psi = np.where(M.isnan(psi), 0, psi)
    psi = np.where(R < 0, -psi, psi)
    w = M.sqrt(w2)
    C = M.arr(g["E0"].real), M.arr(g["E0"].imag)
    nrm, dl = M.arr(g["nrm"][ns - 1]), d0
    sq = M.sqrt(abs(_dot(dl, nrm)))
    amp = M.arr(g["w0"]) * sq / w * M.exp(-r2 / w2)
    ph = k * z + psi + k * r2 * R / 2 + ref_phi
    cs, sn = M.cos(ph), M.sin(ph)
    re = (C[0] * cs - C[1] * sn) * amp
    im = (C[0] * sn + C[1] * cs) * amp
    # ---- error model (binary64 magnitudes) ----
    f = _f
    kf, r2f, Rf, wf, psif = float(k), f(r2), f(R), f(w), f(psi)
    ydf, ywf, mdf, mwf = f(yd), f(yw), f(md), f(mw)
    Ff = np.sqrt(mdf ** 2 + mwf ** 2)
    cpsi = np.maximum(np.abs(np.cos(psif)), 1e-300)
    phi = (kf * (abs(float(l0)) + np.abs(f(l1)) + float(max(abs(float(t)) for t in temps)) + np.abs(_f(g["pos"][ns - 1, 0])).sum()
                 + np.abs(_f(p1)).sum(axis=1)) + abs(float(ref_phi)) + kf * r2f * np.abs(Rf) / 2 + np.abs(psif))
    ey = EPS * np.maximum(mag[0], mag[1]) + EPS * wf                 # absolute error of the ray heights
    # A height's error along the chief changes cos(angle3d) by ey / y, and m = c / sqrt(1 - c^2) by (ey / y) (1 + m^2)^(3/2):
    # the product y m, which E sums, carries ey (1 + m^2)^(3/2) whatever the height.  F is formed from the same slopes, and its
    # error cannot move sin psi by more than sin psi itself.
    gd, gw = (1 + mdf ** 2) ** 1.5, (1 + mwf ** 2) ** 1.5
    emd = (EPS + ey / np.maximum(ydf, 1e-300)) * gd
    emw = (EPS + ey / np.maximum(ywf, 1e-300)) * gw
    eE = ey * (np.abs(mdf) + np.abs(mwf)) + (EPS * ydf + ey) * gd + (EPS * ywf + ey) * gw + EPS * (np.abs(ydf * mdf) + np.abs(ywf * mwf))
    eF = (np.abs(mdf) * emd + np.abs(mwf) * emw) / np.maximum(Ff, 1e-300)
    spsi = np.abs(np.sin(psif))
    dpsi = (eE / (wf * Ff) + spsi * ey / wf + spsi * np.minimum(eF / np.maximum(Ff, 1e-300), 1.0)) / cpsi
    G = (1 + 2 * r2f / wf ** 2) * ey / wf + kf * r2f / 2 * (eE / wf ** 2 + 2 * np.abs(Rf) * ey / wf) + dpsi
    D = 1 + 2 * r2f / wf ** 2 + kf * r2f * np.abs(Rf) + 1 / cpsi
    beta = C_PHI * EPS * phi + C_G * G + C_A * (EPS + DELTA) * D
    floor = abs(g["E0"]) * g["w0"] * float(np.sqrt(abs(np.dot(g["dir"][ns - 1, 0], g["nrm"][ns - 1])))) / wf * EXP_FLOOR
    return dict(re=re, im=im, mag=np.hypot(f(re), f(im)), beta=beta, floor=floor, idx=idx, w=wf, R=Rf, psi=psif, z=f(z), phi=phi)


def pd_field(beamlets, p1, M=LD):
    """Field of the beamlets at pixels p1 (m, 3): dict(re, im (backend sums), A (complex128 of them), S, B, PHI (largest phase
    of any term), n_terms, earlier: pixels at which some beamlet's z falls on an earlier chief segment)."""
    m = len(p1)
    re = np.zeros(m, dtype=np.longdouble if M is LD else object); im = np.zeros_like(re)
    S = np.zeros(m); B = np.zeros(m); U = np.zeros(m); PHI = np.zeros(m); earlier = np.zeros(m, bool)
    for g in beamlets:
        t = pd_terms(g, p1, M)
        re = re + t["re"]; im = im + t["im"]
        S += t["mag"]; B += t["mag"] * t["beta"]; U += t["floor"]; PHI = np.maximum(PHI, t["phi"])
        earlier |= t["idx"] < len(g["t"]) - 1
    n = len(beamlets)
    B = B + C_N * max(n, 1) * EPS * S + U
    return dict(re=re, im=im, A=_f(re) + 1j * _f(im) if M is LD else None, S=S, B=B, PHI=PHI, n_terms=n, earlier=earlier)


# ---- K6: PSFDetector ------------------------------------------------------------------------------------------------------
def psf_pixels(pos, dirm, xs, zs, ij=None):
    """p = origin + x e1 + z e2 (PSFDetector.jl:226; e1, e2 = orientation columns 1 and 3) in binary64."""
    n = len(xs)
    if ij is None:
        jj, ii = np.meshgrid(np.arange(len(zs)), np.arange(n))
        ii, jj = ii.ravel(order="F"), jj.ravel(order="F")
    else:
        ii, jj = ij
    dirm = np.asarray(dirm, dtype=np.float64)
    return (np.asarray(pos)[None, :] + xs[ii][:, None] * dirm[:, 0][None, :]) + zs[jj][:, None] * dirm[:, 2][None, :], (ii, jj)


def psf_field(rec, p, M=LD, chunk=2048):
    """Amplitude sum_h proj_h cis(k_h (opl_h + (p - hit_h) . dir_h)) at pixels p (m, 3) -> dict(A, I, S, B, n_terms)."""
    rec = np.asarray(rec, dtype=np.float64)
    hit, d, opl, proj, k = M.arr(rec[:, 0:3]), M.arr(rec[:, 3:6]), M.arr(rec[:, 6]), M.arr(rec[:, 7]), M.arr(rec[:, 8])
    m, nh = len(p), len(rec)
    out_re, out_im = [], []
    for a in range(0, m, chunk):
        q = M.arr(p[a:a + chunk])
        l = _dot(q[:, None, :] - hit[None, :, :], d[None, :, :])
        ph = k[None, :] * (opl[None, :] + l)
        out_re.append((proj[None, :] * M.cos(ph)).sum(axis=1)); out_im.append((proj[None, :] * M.sin(ph)).sum(axis=1))
    re, im = np.concatenate(out_re), np.concatenate(out_im)
    S = np.full(m, float(np.abs(rec[:, 7]).sum()))
    phi = rec[:, 8][None, :] * (np.abs(rec[:, 6])[None, :] + np.abs(rec[:, 0:3]).sum(axis=1)[None, :]
                                + np.abs(p).sum(axis=1)[:, None])
    B = (np.abs(rec[:, 7])[None, :] * C_PHI * EPS * phi).sum(axis=1) + C_N * max(nh, 1) * EPS * S
    A = _f(re) + 1j * _f(im) if M is LD else None
    out = dict(re=re, im=im, A=A, S=S, B=B, PHI=phi.max(axis=1), n_terms=nh)
    if M is LD:
        out["I"] = _f(re * re + im * im)
    return out


def intensity_bound(A, B):
    """|I - |A|^2| <= 2 |A| B + B^2 for |A_binary64 - A| <= B."""
    return 2 * np.abs(A) * B + B * B


def worst_ratio(err, bound):
    """Largest err / bound and the index where it occurs."""
    r = np.asarray(err) / np.asarray(bound)
    k = int(np.argmax(r))
    return float(r[k]), k


def edge_sample(n, seed=0, extra=512, tile=(32, 8)):
    """(i, j) pixel indices of an n x n map: every pixel for n <= 128, otherwise the last partial tile row and column (tiles of
    32 x 8 pixels) plus `extra` seeded pixels."""
    if n <= 128:
        jj, ii = np.meshgrid(np.arange(n), np.arange(n))
        return ii.ravel(order="F"), jj.ravel(order="F")
    ri = np.arange((n - 1) // tile[0] * tile[0], n)
    rj = np.arange((n - 1) // tile[1] * tile[1], n)
    a = [(i, j) for i in ri for j in range(n)] + [(i, j) for j in rj for i in range(n)]
    rng = np.random.default_rng(seed)
    a += list(zip(rng.integers(0, n, extra), rng.integers(0, n, extra)))
    a = np.unique(np.array(a), axis=0)
    return a[:, 0], a[:, 1]
