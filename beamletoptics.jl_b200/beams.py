"""Ray / beam data model of the reference (layer L2) on the host.

Single beams mirror the reference's objects (`Ray`, `Beam`, `GaussianBeamlet`); bundles
(`RayBundle`, `BeamletBundle`) are the structure-of-arrays form the GPU path consumes -- a
`CollimatedSource` of a million rays is one bundle, not a million Python objects.
Citations: /root/reference/src.
"""
import copy
import ctypes as C
import math

import numpy as np

from . import linalg as la

Z_VACUUM = 376.730313668   # Constants.jl:6


class Intersection:
    """AbstractTypes/AbstractRay.jl:13-18"""
    __slots__ = ("object", "shape", "t", "n")

    def __init__(self, t, n, obj=None, shape=None):
        self.t, self.n, self.object, self.shape = t, n, obj, shape


class Ray:
    """Rays.jl:14-42 (dir is normalised, n = 1)."""
    polarized = False

    def __init__(self, pos, dir, lam=1000e-9, n=1.0, normalize=True):
        self.pos = la.v3(pos)
        self.dir = la.normalize(la.v3(dir)) if normalize else la.v3(dir)
        self.intersection = None
        self.lam = float(lam)
        self.n = float(n)

    def length(self): return math.inf if self.intersection is None else self.intersection.t
    def optical_path_length(self): return math.inf if self.intersection is None else self.intersection.t * self.n


class PolarizedRay(Ray):
    """PolarizedRays.jl:37-95: E0 must be orthogonal to dir (atol 1e-14)."""
    polarized = True

    def __init__(self, pos, dir, lam=1000e-9, E0=None, n=1.0, normalize=True):
        super().__init__(pos, dir, lam, n, normalize)
        if E0 is None:
            E0 = (math.sqrt(2 * 1 * Z_VACUUM), 0.0, 0.0)   # [electric_field(1), 0, 0]
        self.E0 = tuple(complex(x) for x in E0)
        d = sum(self.dir[k] * self.E0[k] for k in range(3))
        if abs(d) > 1e-14:
            raise ValueError("Ray dir. and E0 must be orthogonal.")


class Beam:
    """Beam.jl:13-17"""

    def __init__(self, ray_or_pos, dir=None, lam=None, E0=None):
        if isinstance(ray_or_pos, Ray):
            ray = ray_or_pos
        elif E0 is not None:
            ray = PolarizedRay(ray_or_pos, dir, 1000e-9 if lam is None else lam, E0)
        else:
            ray = Ray(ray_or_pos, dir, 1000e-9 if lam is None else lam)
        self.rays = [ray]
        self.parent = None
        self.children = []

    def length(self):   # Beam.jl:125-169
        l = 0.0
        for r in self.rays:
            if r.intersection is None:
                break
            l += r.length()
        return l + (self.parent.length() if self.parent is not None else 0.0)

    def optical_path_length(self):   # :137-149
        l0 = self.parent.optical_path_length() if self.parent is not None else 0.0
        for r in self.rays:
            if r.intersection is None:
                break
            l0 += r.optical_path_length()
        return l0

    def leaves(self):
        out, q = [], [self]
        while q:
            b = q.pop(0)
            if not b.children:
                out.append(b)
            q.extend(b.children)
        return out


class GaussianBeamlet:
    """Gaussian.jl:33-42 / 215-256.  `support` must be given for reproducible results (the
    reference draws a random orthogonal vector when it is omitted)."""

    def __init__(self, position, direction, lam=1e-6, w0=1e-3, M2=1.0, P0=1e-3, z0=0.0, support=None):
        d = la.normalize(la.v3(direction))
        if support is None:
            rng = np.random.default_rng()
            nw = tuple(rng.random(3))
            nn = la.norm(d)
            nw = la.sub(nw, la.scale(1.0 / (nn * nn), la.scale(la.dot(nw, d), d)))
            support = nw
        s1 = la.normalize(la.v3(support))
        tant = math.tan(M2 * lam / (math.pi * w0))
        pos = la.v3(position)
        self.chief = Beam(Ray(pos, d, lam))
        self.waist = Beam(Ray(la.add(pos, la.scale(w0, s1)), d, lam))
        dz = -z0 * tant
        self.divergence = Beam(Ray(la.add(pos, la.scale(dz, s1)), la.normalize(la.add(d, la.scale(tant, s1))), lam))  # normalised twice, like the reference
        self.lam = float(lam)
        self.w0 = float(w0)
        I0 = 2 * P0 / (math.pi * (w0 * w0))
        self.E0 = complex(math.sqrt(2 * I0 * Z_VACUUM), 0.0)
        self.parent = None
        self.children = []

    @classmethod
    def _raw(cls, chief, waist, div, lam, w0, E0):
        g = cls.__new__(cls)
        g.chief, g.waist, g.divergence, g.lam, g.w0, g.E0 = chief, waist, div, lam, w0, E0
        g.parent, g.children = None, []
        return g

    def length(self): return self.chief.length()
    def optical_path_length(self): return self.chief.optical_path_length()

    def rays18(self):
        out = []
        for b in (self.chief, self.waist, self.divergence):
            r = b.rays[0]
            out.extend(r.pos + r.dir)
        return out

    def leaves(self):
        out, q = [], [self]
        while q:
            b = q.pop(0)
            if not b.children:
                out.append(b)
            q.extend(b.children)
        return out


# ---- bundles (SoA) -----------------------------------------------------------------------------
class RayBundle:
    """N independent root rays: pos/dir (N,3), lam (N,), optional E0 (N,3) complex -> PolarizedRays."""

    def __init__(self, pos, dir, lam=1000e-9, E0=None, normalize=True):
        self.pos = np.ascontiguousarray(pos, dtype=np.float64).reshape(-1, 3)
        d = np.ascontiguousarray(dir, dtype=np.float64)
        self.uniform_dir = d.ndim == 1      # one direction for the whole bundle (collimated sources): shipped once (BMO_UNIFORM_DIR)
        if d.ndim == 1:
            d = np.broadcast_to(d, self.pos.shape)
        d = np.array(d, dtype=np.float64)
        if normalize:   # inv(norm) * d like Ray(pos, dir, lam)
            inv = 1.0 / np.sqrt(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1] + d[:, 2] * d[:, 2])
            d = d * inv[:, None]
        self.dir = np.ascontiguousarray(d)
        self.uniform_lam = np.ndim(lam) == 0
        self.lam = np.ascontiguousarray(np.broadcast_to(np.asarray(lam, dtype=np.float64), (self.pos.shape[0],)))
        self.E0 = None
        if E0 is not None:
            e = np.asarray(E0, dtype=np.complex128)
            if e.ndim == 1:
                e = np.broadcast_to(e, self.pos.shape)
            self.E0 = np.ascontiguousarray(e)
        self.result = None

    def __len__(self): return self.pos.shape[0]


class BeamletBundle:
    """N root Gaussian beamlets in SoA form: rays (N,3,6) = chief/waist/divergence pos+dir."""

    def __init__(self, rays, lam, w0, E0):
        self.rays = np.ascontiguousarray(rays, dtype=np.float64).reshape(-1, 3, 6)
        n = self.rays.shape[0]
        self.lam = np.ascontiguousarray(np.broadcast_to(np.asarray(lam, dtype=np.float64), (n,)))
        self.w0 = np.ascontiguousarray(np.broadcast_to(np.asarray(w0, dtype=np.float64), (n,)))
        self.E0 = np.ascontiguousarray(np.broadcast_to(np.asarray(E0, dtype=np.complex128), (n,)))
        self.result = None

    def __len__(self): return self.rays.shape[0]

    @classmethod
    def from_params(cls, position, direction, lam=1e-6, w0=1e-3, M2=1.0, P0=1e-3, z0=0.0, support=(1.0, 0.0, 0.0)):
        """Vectorised GaussianBeamlet constructor (Gaussian.jl:215-256) for (N,3) positions."""
        pos = np.ascontiguousarray(position, dtype=np.float64).reshape(-1, 3)
        n = pos.shape[0]
        out = np.zeros((n, 3, 6))
        w0a = np.broadcast_to(np.asarray(w0, dtype=np.float64), (n,))
        lama = np.broadcast_to(np.asarray(lam, dtype=np.float64), (n,))
        P0a = np.broadcast_to(np.asarray(P0, dtype=np.float64), (n,))
        d = la.normalize(la.v3(direction))
        s1 = la.normalize(la.v3(support))
        dv, sv = np.array(la.normalize(d)), np.array(s1)   # Ray(pos, dir, lam) normalises `dir` a second time
        for i in range(n):
            tant = math.tan(M2 * lama[i] / (math.pi * w0a[i]))
            out[i, 0, :3] = pos[i]; out[i, 0, 3:] = dv
            out[i, 1, :3] = pos[i] + sv * w0a[i]; out[i, 1, 3:] = dv
            dd = la.normalize(la.normalize(la.add(d, la.scale(tant, s1))))
            out[i, 2, :3] = pos[i] + sv * (-z0 * tant); out[i, 2, 3:] = dd
        I0 = 2 * P0a / (math.pi * (w0a * w0a))
        E0 = np.sqrt(2 * I0 * Z_VACUUM).astype(np.complex128)
        return cls(out, lama, w0a, E0)


# ---- sources (BeamGroups.jl) -------------------------------------------------------------------
def _basis(dir, b1):
    d = la.normalize(la.v3(dir))
    if b1 is None:   # the reference's normal3d(dir): random Gram-Schmidt
        rng = np.random.default_rng()
        nw = tuple(rng.random(3))
        nn = la.norm(d)
        b1 = la.normalize(la.sub(nw, la.scale(1.0 / (nn * nn), la.scale(la.dot(nw, d), d))))
    return d, la.v3(b1)


def _bundle_dir(d):
    """The direction RayBundle stores for the unit vector `d` (it normalises once more)."""
    return tuple(float(x) for x in RayBundle(np.zeros(3), np.array(d)).dir[0])


def source_rings(kind, d, b1, size, num_rings, num_rays):
    """Ring layout of CollimatedSource (kind "collimated", size = diameter) and PointSource ("point", size = theta):
    [(first, count, start, rot)] for rings 1 .. num_rings - 1.  Ray 0 is the centre / axis; ring rays
    [first, first + count) are start, rot * start, rot * (rot * start), ... with rot = rotate3d(d, 2 pi / count); start is
    the ring's first offset r * b1 (collimated) or first direction (point).  A ring of count 0 is skipped (rot = identity).
    The host constructors expand this table and the device descriptor (DeviceSource) carries it, so both use one layout."""
    m = num_rays - 1
    if kind == "collimated":
        radii = [(size / 2) * i / (num_rings - 1) for i in range(1, num_rings)]
        starts = [la.scale(r, b1) for r in radii]
        circm = [r * 2 * math.pi for r in radii]
    else:
        b2 = la.normalize(la.cross(d, b1))
        step = size / (num_rings - 1)
        starts = [la.matvec(la.rotate3d(b2, step * i), d) for i in range(1, num_rings)]
        circm = [la.norm(la.sub(nd, la.scale(la.dot(nd, d), d))) * 2 * math.pi for nd in starts]
    ds = sum(circm) / m
    counts = [int(round(c / ds)) for c in circm]
    counts[-1] += m - sum(counts)
    rings, first = [], 1
    for start, count in zip(starts, counts):
        rings.append((first, count, start, la.rotate3d(d, 2 * math.pi / count) if count else la.IDENTITY))
        first += count
    return rings


def _expand_rings(rings, emit):
    """Host expansion of a ring table: emit(v) for every ring ray in ray order (serial recurrence v <- rot v)."""
    for _, count, v, rot in rings:
        for _ in range(count):
            emit(v)
            v = la.matvec(rot, v)


class DeviceSource:
    """A source whose rays are generated on the GPU (bmo_source_create) from a descriptor: the basis, the ring table and
    every transcendental are computed here by the code that builds the host bundles.  One bmo_source is created per
    (device, n_poses, first, count) on first use -- n_poses > 1 tiles the rays pose-major for a pose sweep
    (bmo_source_create_poses), a shard (`shard(first, count)`) holds the rays [first, first + count) of the source
    (bmo_source_create_slice); `pos` / `dir` download the untiled rays for inspection.  solve_system_ traces it from the
    device pointers, so no per-ray data crosses the bus.  The handles belong to the per-process contexts of _lib.context,
    which live until the process ends, so freeing them from __del__ never outlives the context."""

    def __init__(self, kind, n, pos, dir, lam, rings=(), e1=(0.0, 0.0, 0.0), e2=(0.0, 0.0, 0.0), radius=0.0, phi0=0.0, direction=None):
        from . import _lib as L
        self.kind, self.n, self.lam = kind, int(n), float(lam)
        self.direction = la.v3(dir if direction is None else direction)   # as the constructor was given it (beamlets' from_params)
        self.uniform_dir = kind != L.SRC_POINT
        self.E0 = None
        self._rings = (L.bmo_source_ring * max(1, len(rings)))()
        for i, (first, count, start, rot) in enumerate(rings):
            self._rings[i].first, self._rings[i].count = int(first), int(count)
            self._rings[i].start[:] = [float(x) for x in start]
            self._rings[i].rot[:] = [float(rot[r][c]) for r in range(3) for c in range(3)]
        desc = L.bmo_source_desc()
        desc.kind, desc.n_rays, desc.n_rings = kind, self.n, len(rings)
        desc.pos[:], desc.dir[:], desc.e1[:], desc.e2[:] = la.v3(pos), la.v3(dir), la.v3(e1), la.v3(e2)
        desc.radius, desc.phi0 = float(radius), float(phi0)
        # what the rays depend on, without the pointer: the root signature of a retrace
        self._sig = bytes(desc) + bytes(memoryview(self._rings))[:len(rings) * C.sizeof(L.bmo_source_ring)] + np.float64(self.lam).tobytes()
        desc.rings = self._rings
        self.desc = desc
        self.first = 0               # this source holds the rays [first, first + n) of the descriptor's desc.n_rays
        self._handles = {}
        self._host = None
        self.result = None

    def __len__(self): return self.n

    def signature(self): return self._sig

    def shard(self, first, count):
        """The rays [first, first + count) of this source as a DeviceSource of their own (bmo_source_create_slice): bit for
        bit the same rays as those of the whole source, so that tracing the shards of a splitter-free system gives the
        whole source's hits.  Offsets are relative to this source."""
        first, count = int(first), int(count)
        if first < 0 or count < 1 or first + count > self.n:
            raise ValueError(f"shard [{first}, {first + count}) is not a non-empty part of the {self.n} rays")
        s = copy.copy(self)
        s.first, s.n = self.first + first, count
        s._sig = self._sig + np.array([s.first, s.n], np.int64).tobytes()
        s._handles, s._host, s.result = {}, None, None
        s.__dict__.pop("_solution", None)
        return s

    def handle(self, device=0, n_poses=1):
        """The bmo_source of this descriptor on `device`, tiled `n_poses` times (created on first use)."""
        from . import _lib as L
        key = (int(device), int(n_poses), self.first, self.n)
        if key not in self._handles:
            whole = (self.first, self.n) == (0, self.desc.n_rays)
            if not whole and key[1] != 1:
                raise ValueError("a shard of a source is traced with one pose")
            h = C.c_void_p()
            L.check(self._create(L.context(device), key[1], whole, h))
            self._handles[key] = h
        return self._handles[key]

    def _create(self, ctx, n_poses, whole, h):
        from . import _lib as L
        if whole:
            return L.lib().bmo_source_create_poses(ctx, C.byref(self.desc), n_poses, C.byref(h))
        return L.lib().bmo_source_create_slice(ctx, C.byref(self.desc), self.first, self.n, C.byref(h))

    def beamlets(self, w0, M2=1.0, P0=1e-3, z0=0.0, support=(1.0, 0.0, 0.0)):
        """GaussianBeamlets on the rays of this source, generated on the GPU (bmo_source_create_beamlets): beamlet i has the
        bits of BeamletBundle.from_params(P, self.direction, self.lam, w0, M2, P0, z0, support) at the position P of ray i as
        `rays()` gives it.  A point source is refused (its rays have no common direction)."""
        from . import _lib as L
        if self.kind == L.SRC_POINT:
            raise ValueError("a point source has no beamlet source: its rays differ in direction")
        return DeviceBeamletSource(self, beamlet_desc(self.direction, self.lam, w0, M2, P0, z0, support))

    def device_arrays(self, device=0, n_poses=None):
        """(n, pos, dir, uniform_dir): device pointers for bmo_trace_rays with BMO_INPUT_DEVICE.  With `n_poses` the rays
        are tiled pose-major and the tuple ends with the pose-id pointer, (n * n_poses, pos, dir, uniform_dir, pose_id);
        pose_id is None for one pose."""
        from . import _lib as L
        h = self.handle(device, 1 if n_poses is None else n_poses)
        n, p, d, u = C.c_int64(), C.c_void_p(), C.c_void_p(), C.c_int32()
        L.check(L.lib().bmo_source_device(h, C.byref(n), C.byref(p), C.byref(d), C.byref(u)))
        if n_poses is None:
            return int(n.value), p.value, d.value, bool(u.value)
        npo, pid = C.c_int32(), C.c_void_p()
        L.check(L.lib().bmo_source_pose_ids(h, C.byref(npo), C.byref(pid)))
        return int(n.value), p.value, d.value, bool(u.value), pid.value

    def rays(self, device=0, n_poses=1):
        """Host copies (pos (n * n_poses, 3), dir (n * n_poses, 3)) of the rays generated on `device` (bmo_source_rays)."""
        from . import _lib as L
        m = self.n * int(n_poses)
        pos, dir = np.zeros((m, 3)), np.zeros((m, 3))
        L.check(L.lib().bmo_source_rays(self.handle(device, n_poses), L.ptr(pos), L.ptr(dir)))
        return pos, dir

    def _download(self):
        if self._host is None:
            self._host = self.rays(next(iter(self._handles), (0,))[0])
        return self._host

    @property
    def pos(self): return self._download()[0]

    @property
    def dir(self): return self._download()[1]

    def free(self):
        from . import _lib as L
        for h in self._handles.values():
            L.lib().bmo_source_free(h)
        self._handles = {}

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def beamlet_desc(direction, lam, w0, M2=1.0, P0=1e-3, z0=0.0, support=(1.0, 0.0, 0.0)):
    """The bmo_beamlet_desc of GaussianBeamlets with these parameters: the constants BeamletBundle.from_params forms, by its
    code.  ValueError for w0 <= 0 and for non-finite input or constants."""
    from . import _lib as L
    vals = [lam, w0, M2, P0, z0] + list(la.v3(direction)) + list(la.v3(support))
    if not all(math.isfinite(float(v)) for v in vals):
        raise ValueError("beamlet parameters must be finite")
    if not float(w0) > 0:
        raise ValueError(f"w0 must be > 0, not {w0}")
    if la.norm(la.v3(direction)) == 0 or la.norm(la.v3(support)) == 0:
        raise ValueError("direction and support must not be zero vectors")
    w0a, lama, P0a = np.float64(w0), np.float64(lam), np.float64(P0)
    d = la.normalize(la.v3(direction))
    s1 = la.normalize(la.v3(support))
    tant = math.tan(M2 * lama / (math.pi * w0a))
    I0 = 2 * P0a / (math.pi * (w0a * w0a))
    b = L.bmo_beamlet_desc()
    b.dv[:] = [float(x) for x in la.normalize(d)]
    b.dd[:] = [float(x) for x in la.normalize(la.normalize(la.add(d, la.scale(tant, s1))))]
    b.s[:] = [float(x) for x in s1]
    b.w0, b.div_offset = float(w0a), float(-z0 * tant)
    b.E0[:] = [float(np.sqrt(2 * I0 * Z_VACUUM)), 0.0]
    if not all(math.isfinite(x) for x in list(b.dv) + list(b.dd) + list(b.s) + [b.div_offset, b.E0[0]]):
        raise ValueError("beamlet constants are not finite")
    return b


class DeviceBeamletSource(DeviceSource):
    """GaussianBeamlets generated on the GPU on the rays of a DeviceSource (DeviceSource.beamlets): the source's descriptor
    plus one bmo_beamlet_desc, expanded by bmo_source_create_beamlets per (device, n_poses, first, count) like the ray source's
    handles.  `shard(first, count)` gives the beamlets [first, first + count); solve_system_, the pose sweeps and the sharded
    solves trace it from the device pointers, so no per-beamlet data crosses the bus."""

    def __init__(self, source, bdesc):
        self.__dict__.update(source.__dict__)
        self.bdesc = bdesc
        self.w0, self.E0 = float(bdesc.w0), complex(bdesc.E0[0], bdesc.E0[1])
        self._sig = source._sig + bytes(bdesc)
        self._handles, self._host, self.result = {}, None, None
        self.__dict__.pop("_solution", None)

    def _create(self, ctx, n_poses, whole, h):
        from . import _lib as L
        return L.lib().bmo_source_create_beamlets(ctx, C.byref(self.desc), C.byref(self.bdesc), n_poses, self.first, self.n, C.byref(h))

    def device_beamlets(self, device=0, n_poses=None):
        """(n, rays, w0, E0): device pointers for bmo_trace_beamlets with BMO_INPUT_DEVICE.  With `n_poses` the beamlets are
        tiled pose-major and the tuple ends with the pose-id pointer (None for one pose)."""
        from . import _lib as L
        h = self.handle(device, 1 if n_poses is None else n_poses)
        n, r, w, e = C.c_int64(), C.c_void_p(), C.c_void_p(), C.c_void_p()
        L.check(L.lib().bmo_source_beamlets_device(h, C.byref(n), C.byref(r), C.byref(w), C.byref(e)))
        if n_poses is None:
            return int(n.value), r.value, w.value, e.value
        npo, pid = C.c_int32(), C.c_void_p()
        L.check(L.lib().bmo_source_pose_ids(h, C.byref(npo), C.byref(pid)))
        return int(n.value), r.value, w.value, e.value, pid.value

    def beamlets(self, device=0, n_poses=1):
        """Host copies (rays (n * n_poses, 3, 6), w0 (n * n_poses,), E0 (n * n_poses,) complex) of the beamlets generated on
        `device` (bmo_source_beamlets)."""
        from . import _lib as L
        m = self.n * int(n_poses)
        rays, w0, e = np.zeros((m, 3, 6)), np.zeros(m), np.zeros((m, 2))
        L.check(L.lib().bmo_source_beamlets(self.handle(device, n_poses), L.ptr(rays), L.ptr(w0), L.ptr(e)))
        return rays, w0, e.view(np.complex128).reshape(m)


def UniformDiscSource(pos, dir, diameter, lam=1e-6, num_rays=1000, e1=None, on_device=False):
    """BeamGroups.jl:222-245 (Fibonacci disc); `e1` fixes the reference's random in-plane basis.  on_device=True returns a
    DeviceSource whose positions are computed on the GPU (within a few ulp of these: CUDA's sin / cos)."""
    d, e1 = _basis(dir, e1)
    e2 = la.normalize(la.cross(d, e1))
    R = diameter / 2
    phi0 = 2 * math.pi / (1 + math.sqrt(5))
    if on_device:
        from . import _lib as L
        b = DeviceSource(L.SRC_DISC, num_rays, pos, _bundle_dir(d), lam, e1=e1, e2=e2, radius=R, phi0=phi0, direction=dir)
        b.diameter = float(diameter)
        return b
    k = np.arange(num_rays, dtype=np.float64)
    rho = np.sqrt((k + 0.5) / num_rays)
    phi = k * phi0
    r = R * rho
    x = (r * np.cos(phi))[:, None] * np.array(e1) + (r * np.sin(phi))[:, None] * np.array(e2)
    p = np.array(la.v3(pos)) + x
    b = RayBundle(p, np.array(d), lam)
    b.diameter = float(diameter)
    return b


def CollimatedSource(pos, dir, diameter, lam=1e-6, num_rings=10, num_rays=None, b1=None, on_device=False):
    """BeamGroups.jl:152-195 (concentric rings).  on_device=True returns a DeviceSource with bit-identical rays."""
    if num_rays is None:
        num_rays = 100 * num_rings
    if num_rays < num_rings * 20:
        raise ValueError("No. of rays should be atleast 20x no. of rings")
    d, b1 = _basis(dir, b1)
    p0 = la.v3(pos)
    rings = source_rings("collimated", d, b1, diameter, num_rings, num_rays)
    if on_device:
        from . import _lib as L
        b = DeviceSource(L.SRC_COLLIMATED, num_rays, p0, _bundle_dir(d), lam, rings=rings, direction=dir)
    else:
        pts = [p0]
        _expand_rings(rings, lambda v: pts.append(la.add(p0, v)))
        b = RayBundle(np.array(pts), np.array(d), lam)
    b.diameter = float(diameter)
    return b


def PointSource(pos, dir, theta, lam=1e-6, num_rings=10, num_rays=None, b1=None, on_device=False):
    """BeamGroups.jl:51-100 (cone of concentric fans).  on_device=True returns a DeviceSource with bit-identical rays."""
    if num_rays is None:
        num_rays = 100 * num_rings
    if num_rays < num_rings * 20:
        raise ValueError("No. of rays should be atleast 20x no. of rings")
    if theta >= math.pi:
        raise ValueError("Point source opening half-angle must be <= pi")
    d, b1 = _basis(dir, b1)
    rings = source_rings("point", d, b1, theta, num_rings, num_rays)
    if on_device:
        from . import _lib as L
        b = DeviceSource(L.SRC_POINT, num_rays, pos, _bundle_dir(d), lam, rings=rings)
    else:
        dirs = [d]
        _expand_rings(rings, dirs.append)
        n = len(dirs)
        b = RayBundle(np.tile(np.array(la.v3(pos)), (n, 1)), np.array(dirs), lam)
    b.NA = math.sin(theta)
    return b
