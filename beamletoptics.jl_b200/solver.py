"""`solve_system!` on the GPU (reference: src/System.jl:444-475).

`solve_system_(system, beam)` flattens the system at call time (poses are static during a trace,
docs/src/basics/elements.md), uploads the tables, runs the wavefront tracer of libbmo.so and puts
the results where the reference puts them: `Beam.rays` / `.children`, `Spotdetector.data`,
`Photodetector.field`.  With `retrace=True` (the reference's default) a beam that already holds a
solution is re-validated against the previously hit objects first (retrace_system!,
System.jl:188-428 -> bmo_retrace); a fresh beam is traced non-sequentially.
"""
import ctypes as C
import weakref

import numpy as np

from . import _lib as L
from . import beams as bm
from . import components as co
from .flatten import FlatSystem


class DeviceSystem:
    """Uploaded copy of a flattened System (bmo_sys)."""

    def __init__(self, flat, device=0):
        self.flat = flat
        self.device = device
        self.ctx = L.context(device)
        h = C.c_void_p()
        L.check(L.lib().bmo_system_upload(self.ctx, C.byref(flat.tables), C.byref(h)))
        self.h = h
        self.n_poses = 1
        self._results = weakref.WeakSet()    # results traced through this system

    def free(self):
        """Results are released first: whatever order the garbage collector finalises a reference cycle
        in, a bmo_result never outlives the bmo_sys it was traced through."""
        for r in list(self._results):
            r.free()
        if self.h:
            L.lib().bmo_system_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class TraceResult:
    """Device-resident result of one trace (bmo_result) with lazy host views."""

    def __init__(self, dsys, handle):
        self.dsys, self.h = dsys, handle
        info = L.bmo_result_info()
        L.check(L.lib().bmo_result_get_info(handle, C.byref(info)))
        self.n_roots, self.n_beams, self._n_segments = info.n_roots, info.n_beams, info.n_segments
        self.interactions, self.R, self.polarized, self.waves = info.interactions, info.rays_per_beam, bool(info.polarized), info.waves
        self._beams = self._segs = self._spots = None
        dsys._results.add(self)
        self.keep = self.R == 3      # segment table kept (set by the trace wrappers; beamlet traces always keep it)

    @property
    def n_segments(self):
        if self._n_segments < 0:     # spot-only trace: the segment count is computed on demand
            self.beams()
            info = L.bmo_result_info()
            L.check(L.lib().bmo_result_get_info(self.h, C.byref(info)))
            self._n_segments = info.n_segments
        return self._n_segments

    def free(self):
        if self.h:
            L.lib().bmo_result_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

    def beams(self):
        if self._beams is None:
            nb = self.n_beams
            d = dict(parent=np.zeros(nb, np.int32), slot=np.zeros(nb, np.int32), nseg=np.zeros(nb, np.int32),
                     status=np.zeros(nb, np.int32), first=np.zeros(nb, np.int64), lam_id=np.zeros(nb, np.int32))
            w0 = E0 = None
            if self.R == 3:
                w0, E0 = np.zeros(nb), np.zeros(2 * nb)
            L.check(L.lib().bmo_result_beams(self.h, L.ptr(d["parent"]), L.ptr(d["slot"]), L.ptr(d["nseg"]), L.ptr(d["status"]),
                                            L.ptr(d["first"]), L.ptr(w0), L.ptr(E0), L.ptr(d["lam_id"])))
            if self.R == 3:
                d["w0"], d["E0"] = w0, E0[0::2] + 1j * E0[1::2]
            d["e0_warn"] = (d["status"] >> 8) & 1      # E0 orthogonality check (atol 1e-14) failed along the beam
            d["status"] = d["status"] & 0xff
            self._beams = d
        return self._beams

    def segments(self):
        """Beam-major segment table: arrays of `n_segments * R` rows (Gaussian: chief, waist, div interleaved)."""
        if self._segs is None:
            rows = self.n_segments * self.R
            d = dict(pos=np.zeros((rows, 3)), dir=np.zeros((rows, 3)), n=np.zeros(rows), t=np.zeros(rows), nrm=np.zeros((rows, 3)),
                     obj=np.zeros(rows, np.int32), part=np.zeros(rows, np.int32))
            E0 = np.zeros((rows, 6)) if self.polarized else None
            L.check(L.lib().bmo_result_segments(self.h, L.ptr(d["pos"]), L.ptr(d["dir"]), L.ptr(d["n"]), L.ptr(d["t"]), L.ptr(d["nrm"]),
                                               L.ptr(d["obj"]), L.ptr(d["part"]), L.ptr(E0)))
            if self.polarized:
                d["E0"] = E0[:, 0::2] + 1j * E0[:, 1::2]
            self._segs = d
        return self._segs

    def spots(self):
        if self._spots is None:
            n = self.n_beams * self.R
            obj, xz = np.zeros(n, np.int32), np.zeros((n, 2))
            L.check(L.lib().bmo_result_spots(self.h, L.ptr(obj), L.ptr(xz)))
            self._spots = (obj, xz)
        return self._spots

    def bfs_order(self):
        """Beam ids in the reference's processing order: root by root, FIFO over each beam tree
        (System.jl:444-461 = level order, children as [transmitted, reflected])."""
        b = self.beams()
        parent, slot = b["parent"], b["slot"]
        nb = self.n_beams
        if nb == self.n_roots:
            return np.arange(nb)
        root = np.arange(nb)
        depth = np.zeros(nb, np.int64)
        code = np.zeros(nb, np.int64)      # path of 0/1 choices, MSB first
        for i in range(self.n_roots, nb):   # children always have larger ids than their parent
            p = parent[i]
            root[i], depth[i], code[i] = root[p], depth[p] + 1, code[p] * 2 + slot[i]
        return np.lexsort((code, depth, root))


def _lambda_ids(lams):
    uniq, inv = np.unique(np.asarray(lams, dtype=np.float64), return_inverse=True)
    return [float(x) for x in uniq], np.ascontiguousarray(inv.astype(np.int32))


def upload_system(system, lambdas, device=0, norm_zero_rule=1):
    return DeviceSystem(FlatSystem(system, lambdas, norm_zero_rule), device)


def _tables_key(flat, device):
    """Everything bmo_system_upload reads, as bytes: two flattenings with the same key are the same device system."""
    t = flat.tables
    parts = [bytes(memoryview(flat._prims)) if flat.n_prims else b"", bytes(memoryview(flat._parts)), bytes(memoryview(flat._objs)),
             bytes(memoryview(flat._meshes)) if flat.n_meshes else b"", flat._verts.tobytes(), flat._faces.tobytes(), flat._lams.tobytes(),
             flat._ntab.tobytes(), flat._jones.tobytes(), flat._ext.tobytes() if t.n_ext else b"",
             np.array([t.n_system, float(t.norm_zero_rule), float(device)]).tobytes()]
    import hashlib
    h = hashlib.blake2b(digest_size=16)
    for b in parts:
        h.update(len(b).to_bytes(8, "little")); h.update(b)
    return h.digest()


def cached_system(system, lambdas, device=0, norm_zero_rule=1):
    """upload_system with a one-entry cache on the System: poses are static during a trace and usually between the solves
    of a loop as well (the reference keeps its objects; a Michelson scan moves one mirror per step), so the flattened tables
    are hashed and the uploaded copy -- BVH included -- is reused while they do not change.  Moving an object changes the
    key and triggers a fresh upload."""
    flat = FlatSystem(system, lambdas, norm_zero_rule)
    key = _tables_key(flat, device)
    hit = getattr(system, "_device", None)
    if hit is not None and hit[0] == key and hit[1].h:
        dsys = hit[1]
        # the host objects the ids map back to are those of this flattening (same objects unless the list was rebuilt)
        dsys.flat.objects, dsys.flat.part_owner = flat.objects, flat.part_owner
        if dsys.n_poses != 1:     # a sweep left stacked pose tables behind: restore the uploaded ones
            L.check(L.lib().bmo_system_set_poses(dsys.h, 1, None, None, None, None, None))
            dsys.n_poses = 1
        return dsys
    dsys = DeviceSystem(flat, device)
    try:
        system._device = (key, dsys)
    except AttributeError:
        pass
    return dsys


def trace_rays(dsys, pos, dir, lam_id, E0=None, pose_id=None, r_max=100, keep_segments=True, device_inputs=False, uniform_dir=False):
    """Thin wrapper of bmo_trace_rays.  With device_inputs=True pos/dir/lam_id/E0/pose_id are integer
    device pointers (e.g. torch tensors' data_ptr()) and `n` must be given as pos=(ptr, n); uniform_dir=True then
    says that `dir` points at one direction for every ray (BMO_UNIFORM_DIR)."""
    flags = L.KEEP_SEGMENTS if keep_segments else 0
    h = C.c_void_p()
    if device_inputs:
        (ppos, n) = pos
        flags |= L.INPUT_DEVICE | (L.UNIFORM_DIR if uniform_dir else 0)
        L.check(L.lib().bmo_trace_rays(dsys.h, n, L.ptr(ppos), L.ptr(dir), L.ptr(lam_id), L.ptr(E0), L.ptr(pose_id), r_max, flags, C.byref(h)))
    else:
        pos = np.ascontiguousarray(pos, dtype=np.float64)
        dir = np.ascontiguousarray(dir, dtype=np.float64)
        if dir.ndim == 1:
            flags |= L.UNIFORM_DIR
        lam_id = None if lam_id is None else np.ascontiguousarray(lam_id, dtype=np.int32)
        e = None
        if E0 is not None:
            ec = np.ascontiguousarray(E0, dtype=np.complex128)
            e = np.ascontiguousarray(np.stack([ec.real, ec.imag], axis=-1).reshape(pos.shape[0], 6))
        pid = None if pose_id is None else np.ascontiguousarray(pose_id, dtype=np.int32)
        L.check(L.lib().bmo_trace_rays(dsys.h, pos.shape[0], L.ptr(pos), L.ptr(dir), L.ptr(lam_id), L.ptr(e), L.ptr(pid), r_max, flags, C.byref(h)))
    res = TraceResult(dsys, h)
    res.keep = bool(keep_segments)
    return res


def trace_rays_spots(dsys, pos, dir, lam_id, E0=None, pose_id=None, r_max=100, want_objects=True):
    """bmo_trace_rays_spots: trace a bundle through a splitter-free system and return the Spotdetector
    hits (det_object (n,), xz (n, 2)) and the TraceResult -- host copies pipelined with the waves.
    `dir` of shape (3,) is one direction for the whole bundle (BMO_UNIFORM_DIR), `lam_id=None` means lambdas[0] for
    every ray; with want_objects=False only xz comes back (NaN where no Spotdetector was reached)."""
    pos = np.ascontiguousarray(pos, dtype=np.float64)
    dir = np.ascontiguousarray(dir, dtype=np.float64)
    flags = L.UNIFORM_DIR if dir.ndim == 1 else 0
    lam_id = None if lam_id is None else np.ascontiguousarray(lam_id, dtype=np.int32)
    n = pos.shape[0]
    e = None
    if E0 is not None:
        ec = np.ascontiguousarray(E0, dtype=np.complex128)
        e = np.ascontiguousarray(np.stack([ec.real, ec.imag], axis=-1).reshape(n, 6))
    pid = None if pose_id is None else np.ascontiguousarray(pose_id, dtype=np.int32)
    obj, xz = (np.zeros(n, np.int32) if want_objects else None), np.zeros((n, 2))
    h = C.c_void_p()
    L.check(L.lib().bmo_trace_rays_spots(dsys.h, n, L.ptr(pos), L.ptr(dir), L.ptr(lam_id), L.ptr(e), L.ptr(pid), r_max, flags,
                                         L.ptr(obj), L.ptr(xz), C.byref(h)))
    return obj, xz, TraceResult(dsys, h)


def trace_beamlets(dsys, rays, lam_id, w0, E0, pose_id=None, r_max=100, device_inputs=False):
    """Thin wrapper of bmo_trace_beamlets.  With device_inputs=True rays/lam_id/w0/E0/pose_id are integer device pointers
    (lam_id and pose_id may be None) and `n` must be given as rays=(ptr, n), as in trace_rays."""
    h = C.c_void_p()
    if device_inputs:
        (prays, n) = rays
        L.check(L.lib().bmo_trace_beamlets(dsys.h, n, L.ptr(prays), L.ptr(lam_id), L.ptr(w0), L.ptr(E0), L.ptr(pose_id), r_max, L.INPUT_DEVICE,
                                           C.byref(h)))
        return TraceResult(dsys, h)
    rays = np.ascontiguousarray(rays, dtype=np.float64).reshape(-1, 18)
    lam_id = np.ascontiguousarray(lam_id, dtype=np.int32)
    w0 = np.ascontiguousarray(w0, dtype=np.float64)
    ec = np.ascontiguousarray(E0, dtype=np.complex128)
    e = np.ascontiguousarray(np.stack([ec.real, ec.imag], axis=-1))
    pid = None if pose_id is None else np.ascontiguousarray(pose_id, dtype=np.int32)
    L.check(L.lib().bmo_trace_beamlets(dsys.h, rays.shape[0], L.ptr(rays), L.ptr(lam_id), L.ptr(w0), L.ptr(e), L.ptr(pid), r_max, 0, C.byref(h)))
    return TraceResult(dsys, h)


def retrace(dsys, prev, r_max=100, keep_segments=True):
    """bmo_retrace: solve_system!(system, beam; retrace=true) for beams that already hold the solution
    `prev` (a TraceResult with its segment table); `dsys` is the system after the kinematic changes."""
    flags = L.KEEP_SEGMENTS if keep_segments else 0
    h = C.c_void_p()
    L.check(L.lib().bmo_retrace(dsys.h, prev.h, int(r_max), flags, C.byref(h)))
    res = TraceResult(dsys, h)
    res.keep = bool(keep_segments) or res.R == 3
    return res


def _root_signature(beam):
    """What a retrace starts from: the state of the first ray(s) of the beam as the host holds it now.  retrace_system!
    re-validates the stored path starting at `first(rays(beam))` (System.jl:188-199) and a Gaussian beamlet's E0 / w0 are read
    from the (mutable) beamlet, so a host that has changed them (`polarization!`, `electric_field!`, test/runtests.jl:2405,
    2846-2849) expects the new values to travel down the tree."""
    if isinstance(beam, bm.GaussianBeamlet):
        return (tuple(np.asarray(beam.rays18(), dtype=np.float64).ravel().tolist()), float(beam.w0), complex(beam.E0), float(beam.lam))
    if isinstance(beam, bm.Beam):
        r = beam.rays[0]
        return (tuple(r.pos), tuple(r.dir), float(r.lam), tuple(complex(x) for x in r.E0) if r.polarized else None)
    if isinstance(beam, bm.BeamletBundle):
        return (hash(np.ascontiguousarray(beam.rays).tobytes()), hash(np.ascontiguousarray(beam.w0).tobytes()), hash(np.ascontiguousarray(beam.E0).tobytes()))
    if isinstance(beam, bm.DeviceSource):
        return (beam.signature(),)
    if isinstance(beam, bm.RayBundle):
        e = None if beam.E0 is None else hash(np.ascontiguousarray(beam.E0).tobytes())
        return (hash(np.ascontiguousarray(beam.pos).tobytes()), hash(np.ascontiguousarray(beam.dir).tobytes()), e)
    return None


def _previous_solution(beam, dsys, lams):
    """The stored solution of `beam` if it can be retraced through `dsys` (same object / part structure and
    wavelength table, root rays as they were when it was stored), else None: the device keeps the roots of the stored
    solution, so a beam whose first ray / E0 / w0 was changed on the host is traced afresh (same result: the reference's
    retrace re-interacts every stored ray with the new values)."""
    prev = getattr(beam, "_solution", None)
    if prev is None or prev.h is None or not prev.keep:
        return None
    if getattr(prev, "_root_sig", None) != _root_signature(beam):
        return None
    pf, nf = prev.dsys.flat, dsys.flat
    if prev.dsys.device != dsys.device or len(pf.objects) != len(nf.objects) or pf.tables.n_parts != nf.tables.n_parts:
        return None
    if list(getattr(prev, "lams", [])) != list(lams):
        return None
    return prev


def pd_accumulate(dsys, result, pd_index, field, pose=0, reference_order=False):
    """field: (n, n) complex128 Fortran-ordered host array; the beamlet fields are ADDED to it.
    reference_order=True evaluates every pixel-beamlet pair in the reference's operation order
    (BMO_PD_REFERENCE_ORDER) instead of the strength-reduced default kernel."""
    assert field.flags["F_CONTIGUOUS"] and field.dtype == np.complex128
    flags = L.PD_REFERENCE_ORDER if reference_order else 0
    L.check(L.lib().bmo_pd_accumulate(dsys.h, result.h, int(pd_index), int(pose), L.ptr(field), flags))


# ---- rebuilding the reference's host objects from the segment table --------------------------------
def _mk_ray(seg, row, flat, polarized, lam):
    if polarized:
        r = bm.PolarizedRay.__new__(bm.PolarizedRay)
        r.E0 = tuple(complex(x) for x in seg["E0"][row])
    else:
        r = bm.Ray.__new__(bm.Ray)
    r.pos, r.dir = tuple(seg["pos"][row]), tuple(seg["dir"][row])
    r.lam, r.n = lam, float(seg["n"][row])
    t = float(seg["t"][row])
    if np.isfinite(t):
        part = int(seg["part"][row])
        r.intersection = bm.Intersection(t, tuple(seg["nrm"][row]), flat.objects[int(seg["obj"][row])], flat.part_owner[part].shape)
    else:
        r.intersection = None
    return r


def _rebuild_beam(beam, res, flat, root=0):
    b, seg = res.beams(), res.segments()
    lam = beam.rays[0].lam
    pol = res.polarized
    objs = {root: beam}
    beam.children = []
    ids = [root] + [i for i in range(res.n_roots, res.n_beams)]
    # roots of other rays are not part of this tree
    owner = {root: True}
    for i in ids:
        if i != root:
            if not owner.get(int(b["parent"][i]), False):
                continue
            owner[i] = True
            nb = bm.Beam.__new__(bm.Beam)
            nb.parent, nb.children = objs[int(b["parent"][i])], []
            objs[i] = nb
        tgt = objs[i]
        f, n = int(b["first"][i]), int(b["nseg"][i])
        tgt.rays = [_mk_ray(seg, f + k, flat, pol, lam) for k in range(n)]
    for i in sorted(objs):
        if i != root:
            objs[int(b["parent"][i])].children.append(objs[i])   # slot 0 (transmitted) is numbered before slot 1
    return objs


def _rebuild_gauss(g, res, flat, root=0):
    b, seg = res.beams(), res.segments()
    objs = {root: g}
    g.children = []
    for i in [root] + list(range(res.n_roots, res.n_beams)):
        if i != root:
            p = int(b["parent"][i])
            if p not in objs:
                continue
            ng = bm.GaussianBeamlet._raw(bm.Beam.__new__(bm.Beam), bm.Beam.__new__(bm.Beam), bm.Beam.__new__(bm.Beam),
                                         g.lam, float(b["w0"][i]), complex(b["E0"][i]))
            ng.parent = objs[p]
            for bb in (ng.chief, ng.waist, ng.divergence):
                bb.parent, bb.children = None, []
            ng.chief.parent = objs[p].chief          # Gaussian.jl:107-111
            objs[p].children.append(ng)
            objs[i] = ng
        tgt = objs[i]
        f, n = int(b["first"][i]), int(b["nseg"][i])
        for r, bb in enumerate((tgt.chief, tgt.waist, tgt.divergence)):
            bb.rays = [_mk_ray(seg, (f + k) * 3 + r, flat, False, g.lam) for k in range(n)]
    return objs


def _collect_spots(system_flat, res):
    """Append Spotdetector hits in the reference's push! order."""
    obj, xz = res.spots()
    if not (obj >= 0).any():
        return
    order = res.bfs_order()
    R = res.R
    idx = (order[:, None] * R + np.arange(R)[None, :]).ravel()
    for oi, o in enumerate(system_flat.objects):
        if isinstance(o, co.Spotdetector):
            sel = idx[obj[idx] == oi]
            if sel.size:
                o.data = np.concatenate([o.data, xz[sel]])


def solve_system_(system, beam, r_max=100, retrace=True, device=0, norm_zero_rule=1, keep_segments=True, collect_spots=True):
    """solve_system!(system, beam; r_max, retrace) for a Beam, GaussianBeamlet, RayBundle, DeviceSource, BeamletBundle or
    DeviceBeamletSource (System.jl:444-468).  Returns the TraceResult (the reference returns nothing).
    collect_spots=False leaves Spotdetector.data alone: the hits stay on the device for spot_stats / TraceResult.spots."""
    if isinstance(beam, (list, tuple)):
        return [solve_system_(system, b, r_max, retrace, device, norm_zero_rule, keep_segments, collect_spots) for b in beam]
    if isinstance(beam, bm.Beam):
        r0 = beam.rays[0]
        lams, lam_id = _lambda_ids([r0.lam])
        dsys = cached_system(system, lams, device, norm_zero_rule)
        prev = _previous_solution(beam, dsys, lams) if retrace else None
        if prev is not None:
            res = globals()["retrace"](dsys, prev, r_max)
        else:
            E0 = np.array([r0.E0]) if r0.polarized else None
            res = trace_rays(dsys, np.array([r0.pos]), np.array([r0.dir]), lam_id, E0, None, r_max, True)
        res.lams = lams
        beam._solution = res
        res._root_sig = _root_signature(beam)
        _rebuild_beam(beam, res, dsys.flat)
        if collect_spots:
            _collect_spots(dsys.flat, res)
        _collect_psfs(dsys, res)
        return res
    if isinstance(beam, bm.GaussianBeamlet):
        lams, lam_id = _lambda_ids([beam.lam])
        dsys = cached_system(system, lams, device, norm_zero_rule)
        prev = _previous_solution(beam, dsys, lams) if retrace else None
        if prev is not None:
            res = globals()["retrace"](dsys, prev, r_max)
        else:
            res = trace_beamlets(dsys, np.array([beam.rays18()]), lam_id, np.array([beam.w0]), np.array([beam.E0]), None, r_max)
        res.lams = lams
        beam._solution = res
        res._root_sig = _root_signature(beam)
        _rebuild_gauss(beam, res, dsys.flat)
        if collect_spots:
            _collect_spots(dsys.flat, res)
        _collect_psfs(dsys, res)
        _accumulate_pds(dsys, res)
        return res
    if isinstance(beam, bm.RayBundle):
        lams, lam_id = _lambda_ids(beam.lam)
        dsys = cached_system(system, lams, device, norm_zero_rule)
        splitters = any(o.kind in ("thin_bs", "plate_bs", "cube_bs") for o in dsys.flat.objects)
        has_psf = any(isinstance(o, co.PSFDetector) for o in dsys.flat.objects)
        keep_segments = keep_segments or has_psf       # the PSF records are rebuilt from the segment table
        # collimated single-wavelength bundles ship one direction and no wavelength ids (24 B per ray instead of 52)
        bdir = beam.dir[0] if getattr(beam, "uniform_dir", False) and len(beam) else beam.dir
        blam = None if len(lams) == 1 else lam_id
        prev = _previous_solution(beam, dsys, lams) if retrace else None
        if prev is not None:
            res = globals()["retrace"](dsys, prev, r_max, keep_segments)
        elif not keep_segments and not splitters and collect_spots:   # one beam per ray: fused trace + Spotdetector read-back (pipelined copies)
            obj, xz, res = trace_rays_spots(dsys, beam.pos, bdir, blam, beam.E0, None, r_max)
            res._spots = (obj, xz)
        else:
            res = trace_rays(dsys, beam.pos, bdir, blam, beam.E0, None, r_max, keep_segments)
        res.lams = lams
        beam.result = beam._solution = res
        res._root_sig = _root_signature(beam)
        if collect_spots:
            _collect_spots(dsys.flat, res)
        if has_psf:
            _collect_psfs(dsys, res)
        return res
    if isinstance(beam, bm.DeviceBeamletSource):
        lams, _ = _lambda_ids([beam.lam])
        dsys = cached_system(system, lams, device, norm_zero_rule)
        prev = _previous_solution(beam, dsys, lams) if retrace else None
        if prev is not None:
            res = globals()["retrace"](dsys, prev, r_max)
        else:      # the beamlets never leave the device: bmo_source -> bmo_trace_beamlets(BMO_INPUT_DEVICE)
            n, rays, w0, E0 = beam.device_beamlets(device)
            res = trace_beamlets(dsys, (rays, n), None, w0, E0, None, r_max, device_inputs=True)
        res.lams = lams
        beam.result = beam._solution = res
        res._root_sig = _root_signature(beam)
        if collect_spots:
            _collect_spots(dsys.flat, res)
        _collect_psfs(dsys, res)
        _accumulate_pds(dsys, res)
        return res
    if isinstance(beam, bm.DeviceSource):
        lams, _ = _lambda_ids([beam.lam])
        dsys = cached_system(system, lams, device, norm_zero_rule)
        has_psf = any(isinstance(o, co.PSFDetector) for o in dsys.flat.objects)
        keep_segments = keep_segments or has_psf       # the PSF records are rebuilt from the segment table
        prev = _previous_solution(beam, dsys, lams) if retrace else None
        if prev is not None:
            res = globals()["retrace"](dsys, prev, r_max, keep_segments)
        else:      # the rays never leave the device: bmo_source -> bmo_trace_rays(BMO_INPUT_DEVICE)
            n, ppos, pdir, uniform = beam.device_arrays(device)
            res = trace_rays(dsys, (ppos, n), pdir, None, None, None, r_max, keep_segments, device_inputs=True, uniform_dir=uniform)
        res.lams = lams
        beam.result = beam._solution = res
        res._root_sig = _root_signature(beam)
        if collect_spots:
            _collect_spots(dsys.flat, res)
        if has_psf:
            _collect_psfs(dsys, res)
        return res
    if isinstance(beam, bm.BeamletBundle):
        lams, lam_id = _lambda_ids(beam.lam)
        dsys = cached_system(system, lams, device, norm_zero_rule)
        prev = _previous_solution(beam, dsys, lams) if retrace else None
        if prev is not None:
            res = globals()["retrace"](dsys, prev, r_max)
        else:
            res = trace_beamlets(dsys, beam.rays, lam_id, beam.w0, beam.E0, None, r_max)
        res.lams = lams
        beam.result = beam._solution = res
        res._root_sig = _root_signature(beam)
        if collect_spots:
            _collect_spots(dsys.flat, res)
        _collect_psfs(dsys, res)
        _accumulate_pds(dsys, res)
        return res
    raise TypeError(f"cannot trace {type(beam).__name__}")


def _spot_args(objs, detector, bins, window, what):
    """(object index, nx, nz, window array) of a spot_stats call on a system with objects `objs`; the window defaults to the
    detector's face."""
    if isinstance(detector, (int, np.integer)):
        oi = int(detector)
    else:
        oi = next((i for i, o in enumerate(objs) if o is detector), -1)
        if oi < 0:
            raise L.BmoError(f"{what}: the detector is not part of the traced system")
    nx = nz = 0
    if bins is not None:
        nx, nz = (int(bins), int(bins)) if np.ndim(bins) == 0 else (int(bins[0]), int(bins[1]))
        if window is None and 0 <= oi < len(objs) and hasattr(objs[oi], "hw"):
            hw = objs[oi].hw
            window = (-hw, hw, -hw, hw)
    win = None if window is None else np.ascontiguousarray(window, dtype=np.float64)
    return oi, nx, nz, win


def _spot_dict(info, counts):
    out = dict(hits=int(info.hits), centroid=(info.centroid[0], info.centroid[1]), rms=info.rms, max_r=info.max_r,
               lo=(info.lo[0], info.lo[1]), hi=(info.hi[0], info.hi[1]), outside=int(info.outside))
    if counts is not None:
        out["counts"] = counts
    return out


def spot_stats(result, detector, bins=None, window=None):
    """Spot diagram of `detector` (a Spotdetector of the traced system, or its object index) reduced on the device
    (bmo_spot_stats): dict of hits, centroid (x, z), rms, max_r (largest distance from the detector origin), lo / hi
    (x, z) and outside (hits outside `window`).  With `bins` (n or (nx, nz)) also "counts", an (nz, nx) int64 histogram
    over `window` = (x_lo, x_hi, z_lo, z_hi), by default the detector's face.  The statistics cover every spot entry of the
    result on that detector (chief, waist and divergence rays of a beamlet result), whether or not they were collected.
    `result` may be a list of results traced on one device (bmo_spot_stats_results): the spot diagram of all their entries,
    in list order, as the reference's Spotdetector accumulates over several solve_system! calls until empty!; a bundle
    traced in splitter-free pieces gives the bits of tracing it once."""
    results = list(result) if isinstance(result, (list, tuple)) else [result]
    if not results:
        raise L.BmoError("spot_stats: no result")
    oi, nx, nz, win = _spot_args(results[0].dsys.flat.objects, detector, bins, window, "spot_stats")
    for r in results[1:]:
        if _spot_args(r.dsys.flat.objects, detector, None, None, "spot_stats")[0] != oi:
            raise L.BmoError("spot_stats: the detector has another object index in another result's system")
    counts = None if bins is None else np.zeros((max(nz, 0), max(nx, 0)), np.int64)
    info = L.bmo_spot_info()
    if isinstance(result, (list, tuple)):
        hs = (C.c_void_p * len(results))(*[r.h for r in results])
        L.check(L.lib().bmo_spot_stats_results(len(results), hs, oi, L.ptr(win), nx, nz, C.byref(info), L.ptr(counts), 0))
    else:
        L.check(L.lib().bmo_spot_stats(result.h, oi, L.ptr(win), nx, nz, C.byref(info), L.ptr(counts), 0))
    return _spot_dict(info, counts)


def spot_stats_poses(result, detector, n_poses, bins=None, window=None):
    """spot_stats for every pose of a pose sweep (bmo_spot_stats_poses): pose p covers the beams traced with pose id p
    (children inherit their root's pose).  Returns a dict of arrays: hits (P,), outside (P,), centroid (P, 2), rms (P,),
    max_r (P,), lo / hi (P, 2) and, with `bins`, counts (P, nz, nx) over `window` (by default the detector's face).  Pose p
    has the bits spot_stats gives for a one-pose solve that lists the pose's hits in the same order, which a system
    without beamsplitters always does."""
    oi, nx, nz, win = _spot_args(result.dsys.flat.objects, detector, bins, window, "spot_stats_poses")
    P = int(n_poses)
    counts = None if bins is None else np.zeros((max(P, 0), max(nz, 0), max(nx, 0)), np.int64)
    info = (L.bmo_spot_info * max(P, 1))()
    L.check(L.lib().bmo_spot_stats_poses(result.h, oi, P, L.ptr(win), nx, nz, info, L.ptr(counts), 0))
    return _spot_pose_dict(info, P, counts)


def _spot_pose_dict(info, P, counts):
    """spot_stats_poses's dict of the first P entries of a bmo_spot_info array (and the (P, nz, nx) counts or None)."""
    a = np.frombuffer(info, dtype=np.dtype([("hits", np.int64), ("outside", np.int64), ("centroid", np.float64, 2), ("rms", np.float64),
                                            ("max_r", np.float64), ("lo", np.float64, 2), ("hi", np.float64, 2)]))[:P]
    out = {k: np.array(a[k]) for k in ("hits", "outside", "centroid", "rms", "max_r", "lo", "hi")}
    if counts is not None:
        out["counts"] = counts
    return out


# ---- PSFDetector (PSFDetector.jl) -----------------------------------------------------------------------
def _collect_psfs(dsys, res):
    """interact3d(::PSFDetector, ::Beam, ::Ray) of every beam that ended on a PSF detector (push! order is
    irrelevant for the sums that use the data); a GaussianBeamlet pushes three records: chief, waist, divergence."""
    for oi, o in enumerate(dsys.flat.objects):
        if isinstance(o, co.PSFDetector):
            h = C.c_void_p(o._psf) if o._psf else C.c_void_p()
            n = C.c_int64(0)
            L.check(L.lib().bmo_psf_collect(dsys.h, res.h, oi, C.byref(h), C.byref(n)))
            o._psf, o._dsys, o._index = h.value, dsys, oi


def psf_count(psf):
    if not psf._psf:
        return 0
    n = C.c_int64(0)
    L.check(L.lib().bmo_psf_count(C.c_void_p(psf._psf), C.byref(n)))
    return int(n.value)


def psf_data(psf):
    n = psf_count(psf)
    out = np.zeros((n, 9))
    if n:
        L.check(L.lib().bmo_psf_data(C.c_void_p(psf._psf), L.ptr(out)))
    return out


def psf_free(psf):
    if psf._psf:
        L.lib().bmo_psf_free(C.c_void_p(psf._psf))
    psf._psf = None


def _psf_dsys(psf):
    """(system, object index) of the solve that filled the detector: lims / intensity use the detector's
    pose at that solve."""
    if not psf._psf:
        raise L.BmoError("the PSFDetector holds no data (solve_system_ first)")
    return psf._dsys, psf._index


def psf_lims(psf, crop_factor=1.0, center="centroid"):
    dsys, oi = _psf_dsys(psf)
    lims = np.zeros(4)
    L.check(L.lib().bmo_psf_lims(dsys.h, C.c_void_p(psf._psf), oi, 0, float(crop_factor), 0 if center == "centroid" else 1, L.ptr(lims)))
    return tuple(float(x) for x in lims)


def psf_intensity(psf, n=100, crop_factor=1.0, center="centroid", x_min=np.inf, x_max=np.inf, z_min=np.inf, z_max=np.inf,
                  x0_shift=0.0, z0_shift=0.0):
    dsys, oi = _psf_dsys(psf)
    lims = psf_window(psf_lims(psf, crop_factor, center), x_min, x_max, z_min, z_max)
    I = np.zeros((n, n), order="F")
    L.check(L.lib().bmo_psf_intensity(dsys.h, C.c_void_p(psf._psf), oi, 0, int(n), L.ptr(lims), float(x0_shift), float(z0_shift), L.ptr(I), 0))
    return psf_axes(n, lims, x0_shift, z0_shift) + (I,)


def psf_window(lims, x_min=np.inf, x_max=np.inf, z_min=np.inf, z_max=np.inf):
    """The (x_min, x_max, z_min, z_max) float64 array intensity(psf; ...) sums over: calc_local_lims's `lims`, with each axis
    replaced where both of its bounds are given (PSFDetector.jl:202-205)."""
    lims = [float(v) for v in lims]
    if x_min != np.inf and x_max != np.inf:
        lims[0], lims[1] = float(x_min), float(x_max)
    if z_min != np.inf and z_max != np.inf:
        lims[2], lims[3] = float(z_min), float(z_max)
    return np.array(lims, dtype=np.float64)


def psf_axes(n, lims, x0_shift=0.0, z0_shift=0.0):
    """(xs, zs) of an n x n intensity map over the window `lims`: LinRange(lo, hi, n) .+ shift (PSFDetector.jl:202-211)."""
    t = np.arange(n) / (n - 1) if n > 1 else np.zeros(1)
    xs = ((1 - t) * lims[0] + t * lims[1]) + x0_shift
    zs = ((1 - t) * lims[2] + t * lims[3]) + z0_shift
    return xs, zs


def _accumulate_pds(dsys, res):
    for oi, o in enumerate(dsys.flat.objects):
        if isinstance(o, co.Photodetector):
            if not o.field.flags["F_CONTIGUOUS"]:
                o.field = np.asfortranarray(o.field)
            pd_accumulate(dsys, res, oi, o.field)
