"""Batched kinematic pose sweeps (BASELINE config 5): many `translate3d!/rotate3d!` poses of one
system traced in a single launch, one Photodetector interferogram or one spot diagram per pose.

The reference solves one pose at a time (move -> empty!(pd) -> solve_system! -> optical_power(pd),
test/runtests.jl:2092-2120; likewise empty!(sd) -> solve_system! -> sd.data for a Spotdetector).  Here
every pose is flattened on the host with the unchanged kinematic API (or computed on the device from a
KinProgram), the tables are stacked and uploaded once (bmo_system_set_poses), every beamlet or ray is
replicated per pose with a pose id, and the detector kernel writes fields[pose] / the spot reduction
writes the statistics of each pose.
"""
import ctypes as C

import numpy as np

from . import _lib as L
from . import beams as bm
from .flatten import FlatSystem
from .solver import DeviceSystem, _lambda_ids, spot_stats_poses, trace_beamlets, trace_rays


def flatten_poses(system, lambdas, n_poses, apply_pose, norm_zero_rule=1):
    """apply_pose(p) moves the host objects into pose p.  Returns (flat of pose 0, stacked tables)."""
    flats = []
    for p in range(n_poses):
        apply_pose(p)
        flats.append(FlatSystem(system, lambdas, norm_zero_rule))
    f0 = flats[0]
    for f in flats[1:]:
        if (f.n_prims, f.n_parts, f.n_objects, f._verts.shape) != (f0.n_prims, f0.n_parts, f0.n_objects, f0._verts.shape):
            raise ValueError("poses must not change the topology of the system")
    arrs = [f.pose_arrays() for f in flats]
    prims = np.concatenate([a[0] for a in arrs]) if f0.n_prims else np.zeros(8, dtype=np.uint8)
    verts = np.concatenate([a[1] for a in arrs]) if f0._verts.size else np.zeros((1, 3))
    bounds = np.concatenate([a[2] for a in arrs])
    det_pos = np.concatenate([a[3] for a in arrs])
    det_dir = np.concatenate([a[4] for a in arrs])
    return f0, tuple(np.ascontiguousarray(x) for x in (prims, verts, bounds, det_pos, det_dir))


def solve_pose_sweep(system, beam, n_poses, apply_pose, pd, r_max=100, device=0, want_fields=True):
    """Trace `beam` (GaussianBeamlet, BeamletBundle or DeviceBeamletSource) through `n_poses` poses of `system`.
    Returns dict(fields=(n_poses, n, n) complex, power=(n_poses,), result=TraceResult)."""
    lams, lam_id, beam = _beamlet_lambdas(beam)
    f0, (prims, verts, bounds, det_pos, det_dir) = flatten_poses(system, lams, n_poses, apply_pose)
    dsys = DeviceSystem(f0, device)
    L.check(L.lib().bmo_system_set_poses(dsys.h, n_poses, L.ptr(prims), L.ptr(verts), L.ptr(bounds), L.ptr(det_pos), L.ptr(det_dir)))
    res = _trace_beamlet_sweep(dsys, beam, lam_id, n_poses, r_max)
    pd_index = f0.object_index(pd)
    n = pd.n
    # one call: per-pose fields accumulated and integrated on the device; the fields only come back when asked for
    fields = np.zeros((n_poses, n * n * 2)) if want_fields else None
    power = np.zeros(n_poses)
    L.check(L.lib().bmo_pd_sweep(dsys.h, res.h, pd_index, n_poses, L.ptr(fields), L.ptr(power), 0))
    out = dict(power=power, result=res, dsys=dsys)
    if want_fields:
        z = fields[:, 0::2] + 1j * fields[:, 1::2]
        out["fields"] = z.reshape(n_poses, n, n).transpose(0, 2, 1)   # stored column-major [i + n*j] -> [pose, i, j]
    return out


# ---- K5: the same sweep with the poses computed on the device --------------------------------------------
class KinProgram:
    """A kinematic program for `bmo_system_apply_poses`: the calls `translate3d_(obj, offsets[p])`,
    `translate_to3d_(obj, targets[p])`, `rotate3d_(obj, axis, thetas[p])` recorded once for all poses p.
    Each call is expanded into micro-ops on the kinematic tree exactly as the host classes recurse
    (components.MultiShapeObject, shapes.UnionSDF, shapes.Mesh); the per-pose operands (offset vectors,
    Rodrigues matrices from `linalg.rotate3d`, i.e. the host's cos / sin) go into the parameter table."""

    TRANSLATE, TRANSLATE_TO, ROT_FRAME, ROT_LEAF, PIVOT = range(5)

    def __init__(self, flat, n_poses):
        self.flat, self.n_poses = flat, int(n_poses)
        self.nodes, self.prim_bounds, self.node_of = flat.kinematics()
        self.ops, self.params = [], []

    def _node(self, obj):
        try:
            return self.node_of[id(obj)]
        except KeyError:
            raise KeyError(f"{type(obj).__name__} is not part of the flattened system") from None

    def _param(self, rows):
        rows = np.asarray(rows, dtype=np.float64).reshape(self.n_poses, -1)
        p = np.zeros((self.n_poses, 9))
        p[:, :rows.shape[1]] = rows
        self.params.append(p)
        return len(self.params) - 1

    def translate3d_(self, obj, offsets):
        self.ops.append((self.TRANSLATE, self._node(obj), 0, self._param(offsets)))

    def translate_to3d_(self, obj, targets):
        self.ops.append((self.TRANSLATE_TO, self._node(obj), 0, self._param(targets)))

    def rotate3d_(self, obj, axis, thetas):
        from . import linalg as la
        thetas = np.broadcast_to(np.asarray(thetas, dtype=np.float64), (self.n_poses,))
        R = [[x for row in la.rotate3d(axis, float(t)) for x in row] for t in thetas]
        self._rotate(self._node(obj), self._param(R))

    def _rotate(self, a, k):
        nd = self.nodes[a]
        if nd.kind in (0, 2):        # ObjectGroup / UnionSDF: own frame first, then every child rotates and moves about the pivot
            self.ops.append((self.ROT_FRAME, a, 0, k))
        if nd.kind in (0, 1, 2):
            c = a + 1
            while c < a + nd.size:
                self._rotate(c, k)
                self.ops.append((self.PIVOT, c, a, k))
                c += self.nodes[c].size
        else:
            self.ops.append((self.ROT_LEAF, a, 0, k))

    def param_table(self, first=0, count=None):
        """Rows [first, first + count) of the parameter table ([pose][param][9]; count=None: to the last pose)."""
        first = int(first)
        count = self.n_poses - first if count is None else int(count)
        if first < 0 or count < 1 or first + count > self.n_poses:
            raise ValueError(f"KinProgram: poses [{first}, {first + count}) outside [0, {self.n_poses})")
        if not self.params:
            return np.zeros((count, 0, 9))
        return np.ascontiguousarray(np.stack([p[first:first + count] for p in self.params], axis=1))

    def apply(self, dsys, first=0, count=None):
        """Install the kinematic tree (once per DeviceSystem) and run the program for poses [first, first + count) (count=None:
        to the last pose): dsys then holds them as its poses 0 .. count - 1, each with the bits of the same pose of the whole
        program (the device computes every pose from its own row of the parameter table)."""
        params = self.param_table(first, count)
        lib = L.lib()
        if getattr(dsys, "_kin_installed", None) is not self.flat:
            L.check(lib.bmo_system_set_kinematics(dsys.h, len(self.nodes), C.byref(self.nodes), L.ptr(self.prim_bounds)))
            dsys._kin_installed = self.flat
        ops = (L.bmo_kin_op * max(len(self.ops), 1))(*[L.bmo_kin_op(*o) for o in self.ops])
        L.check(lib.bmo_system_apply_poses(dsys.h, params.shape[0], len(self.ops), C.byref(ops), len(self.params), L.ptr(params)))


def get_pose_tables(dsys, pose):
    """Tables of one pose as the device holds them (bmo_system_get_pose): prims (ctypes array), vertices, bounds, det_pose."""
    f = dsys.flat
    prims = (L.bmo_prim * max(f.n_prims, 1))()
    verts = np.zeros((max(f._verts.shape[0], 1), 3))
    bounds = np.zeros((f.n_parts, 10))
    det = np.zeros((f.n_objects, 12))
    L.check(L.lib().bmo_system_get_pose(dsys.h, int(pose), C.byref(prims), L.ptr(verts), L.ptr(bounds), L.ptr(det)))
    return prims, verts[:f._verts.shape[0]], bounds, det


def solve_pose_sweep_device(system, beam, n_poses, program, pd, r_max=100, device=0, want_fields=True):
    """solve_pose_sweep with the poses produced on the device: `program(prog)` records the kinematic calls of the
    sweep on a KinProgram (e.g. `prog.translate3d_(mirror, offsets)`); the host objects are not moved."""
    lams, lam_id, beam = _beamlet_lambdas(beam)
    f0 = FlatSystem(system, lams)
    dsys = DeviceSystem(f0, device)
    prog = KinProgram(f0, n_poses)
    program(prog)
    prog.apply(dsys)
    res = _trace_beamlet_sweep(dsys, beam, lam_id, n_poses, r_max)
    pd_index = f0.object_index(pd)
    n = pd.n
    fields = np.zeros((n_poses, n * n * 2)) if want_fields else None
    power = np.zeros(n_poses)
    L.check(L.lib().bmo_pd_sweep(dsys.h, res.h, pd_index, n_poses, L.ptr(fields), L.ptr(power), 0))
    out = dict(power=power, result=res, dsys=dsys)
    if want_fields:
        z = fields[:, 0::2] + 1j * fields[:, 1::2]
        out["fields"] = z.reshape(n_poses, n, n).transpose(0, 2, 1)
    return out


# ---- spot diagrams over poses ------------------------------------------------------------------------------
def tile_ray_bundle(beam, n_poses):
    """A RayBundle tiled pose-major for a sweep: (pos (n P, 3), dir ((3,) uniform or (n P, 3)), lam (n P,), pose_id (n P,)),
    ray i is ray i mod n and pose_id[i] = i // n -- the layout bmo_source_create_poses gives a DeviceSource."""
    n = len(beam)
    pos = np.ascontiguousarray(np.tile(beam.pos, (n_poses, 1)))
    if getattr(beam, "uniform_dir", False) and n:
        dir = np.ascontiguousarray(beam.dir[0])
    else:
        dir = np.ascontiguousarray(np.tile(beam.dir, (n_poses, 1)))
    lam = np.ascontiguousarray(np.tile(np.broadcast_to(np.asarray(beam.lam, dtype=np.float64), (n,)), n_poses))
    pose_id = np.ascontiguousarray(np.repeat(np.arange(n_poses, dtype=np.int32), n))
    return pos, dir, lam, pose_id


def _trace_spot_sweep(dsys, beam, lam_id, n_poses, r_max):
    """Trace `beam` once per pose of `dsys` (segments not kept): a DeviceSource is tiled on the device, a RayBundle on
    the host."""
    if isinstance(beam, bm.DeviceSource):
        n, ppos, pdir, uniform, pid = beam.device_arrays(dsys.device, n_poses)
        return trace_rays(dsys, (ppos, n), pdir, None, None, pid, r_max, False, device_inputs=True, uniform_dir=uniform)
    pos, dir, _, pose_id = tile_ray_bundle(beam, n_poses)
    lam = None if len(dsys.flat.lambdas) == 1 else np.tile(lam_id, n_poses)
    E0 = None if beam.E0 is None else np.tile(beam.E0, (n_poses, 1))
    return trace_rays(dsys, pos, dir, lam, E0, pose_id, r_max, False)


def _beamlet_lambdas(beam):
    """(lambdas, lambda ids, beam) of a pose sweep's beamlets; a GaussianBeamlet becomes a one-beamlet BeamletBundle."""
    if isinstance(beam, bm.DeviceBeamletSource):
        return _lambda_ids([beam.lam]) + (beam,)
    if isinstance(beam, bm.GaussianBeamlet):
        beam = bm.BeamletBundle(np.array([beam.rays18()]), [beam.lam], [beam.w0], [beam.E0])
    return _lambda_ids(beam.lam) + (beam,)


def _trace_beamlet_sweep(dsys, beam, lam_id, n_poses, r_max):
    """Trace the beamlets of `beam` once per pose of `dsys`: a DeviceBeamletSource is tiled on the device, a BeamletBundle on
    the host, both pose-major with pose_id[i] = i // len(beam)."""
    if isinstance(beam, bm.DeviceBeamletSource):
        n, rays, w0, E0, pid = beam.device_beamlets(dsys.device, n_poses)
        return trace_beamlets(dsys, (rays, n), None, w0, E0, pid, r_max, device_inputs=True)
    nb = len(beam)
    rays = np.tile(beam.rays.reshape(nb, 18), (n_poses, 1))
    pose_id = np.repeat(np.arange(n_poses, dtype=np.int32), nb)
    return trace_beamlets(dsys, rays, np.tile(lam_id, n_poses), np.tile(beam.w0, n_poses), np.tile(beam.E0, n_poses), pose_id, r_max)


def _beam_lambdas(beam):
    if isinstance(beam, bm.DeviceSource):
        return _lambda_ids([beam.lam])
    if not isinstance(beam, bm.RayBundle):
        raise TypeError(f"a spot sweep traces a RayBundle or a DeviceSource, not {type(beam).__name__}")
    return _lambda_ids(beam.lam)


def solve_spot_sweep(system, beam, n_poses, apply_pose, detector, bins=None, window=None, r_max=100, device=0):
    """Spot diagrams of `detector` (a Spotdetector) over `n_poses` poses of `system`: apply_pose(p) moves the host objects
    into pose p (flatten_poses), the rays of `beam` (RayBundle or DeviceSource) are traced once per pose in one call and
    reduced per pose on the device (spot_stats_poses).  Replaces the loop move -> empty!(sd) -> solve_system! -> sd.data.
    Returns dict(stats=spot_stats_poses(...), result=TraceResult, dsys=DeviceSystem); the host objects are left in the
    last pose."""
    lams, lam_id = _beam_lambdas(beam)
    f0, (prims, verts, bounds, det_pos, det_dir) = flatten_poses(system, lams, n_poses, apply_pose)
    dsys = DeviceSystem(f0, device)
    L.check(L.lib().bmo_system_set_poses(dsys.h, n_poses, L.ptr(prims), L.ptr(verts), L.ptr(bounds), L.ptr(det_pos), L.ptr(det_dir)))
    dsys.n_poses = n_poses
    res = _trace_spot_sweep(dsys, beam, lam_id, n_poses, r_max)
    return dict(stats=spot_stats_poses(res, detector, n_poses, bins, window), result=res, dsys=dsys)


def solve_spot_sweep_device(system, beam, n_poses, program, detector, bins=None, window=None, r_max=100, device=0):
    """solve_spot_sweep with the poses produced on the device: `program(prog)` records the kinematic calls of the sweep on
    a KinProgram (e.g. `prog.translate3d_(detector, offsets)`); the host objects are not moved.  A DeviceSource is tiled
    on the device (bmo_source_create_poses), so no per-ray data crosses the bus."""
    lams, lam_id = _beam_lambdas(beam)
    f0 = FlatSystem(system, lams)
    dsys = DeviceSystem(f0, device)
    prog = KinProgram(f0, n_poses)
    program(prog)
    prog.apply(dsys)
    dsys.n_poses = n_poses
    res = _trace_spot_sweep(dsys, beam, lam_id, n_poses, r_max)
    return dict(stats=spot_stats_poses(res, detector, n_poses, bins, window), result=res, dsys=dsys)
