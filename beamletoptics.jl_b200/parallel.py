"""Multi-GPU layer of the trace path (SURVEY 8(e)): one process per GPU, `torch.distributed` for the
plumbing (NCCL over NVLink on the GPU box, gloo in the CPU tests).

Rays, beamlets and poses are independent, the system tables are small and replicated, so the path
shards without a data-path collective: every rank traces its slice of the bundle on its own GPU and
owns the corresponding slice of the outputs.  The exchange steps are the Photodetector and the spot
diagram.  Each rank accumulates *its* beamlets onto a full n x n complex128 partial field and the partial
fields are summed with one all-reduce of 2 n^2 doubles (the reference adds the beamlet fields serially into
`pd.field`, Photodetector.jl:103; addition order across ranks changes the sum at the 1e-16 level).  A spot
diagram of a DeviceSource sharded with spot_shard_slice is reduced where the hits are (solve_spot_sharded:
bmo_spot_stats_sharded all-gathers per-block partials, not hits) and has the bits of the unsharded solve.  A PSFDetector map
is sharded by pixel columns (solve_psf_sharded): the ranks all-gather their hit records in rank order, each sums all records
into its band of columns, and the bands are all-gathered; for a splitter-free system the map has the bits of one solve.  A
Photodetector pose sweep is sharded by pose range (solve_pose_sweep_sharded): each rank traces its poses into fields of its own,
which never leave it, and only the powers are all-gathered; every pose has the bits of the one-GPU sweep.  A spot-diagram pose
sweep is sharded the same way (solve_spot_sweep_sharded): each rank reduces its own poses, whose hits never leave it, and the
per-pose statistics and histograms are all-gathered; every pose has the bits of the one-GPU sweep.
"""
import ctypes as C
import math
import os

import numpy as np

from . import _lib as L
from . import beams as bm


class FieldComm:
    """bmo_comm (include/bmo.h): the NCCL communicator behind the C ABI, one per process and GPU.  The 128-byte id
    made by rank 0 (`FieldComm.unique_id()`) has to reach every rank by some host transport; `from_torch` uses the
    process group torchrun set up, a Julia host would use Distributed / MPI / a file."""

    def __init__(self, rank, world_size, id_bytes, device=0):
        self.rank, self.world_size, self.device = int(rank), int(world_size), int(device)
        buf = (C.c_uint8 * L.COMM_ID_BYTES).from_buffer_copy(bytes(id_bytes))
        h = C.c_void_p()
        L.check(L.lib().bmo_comm_init(L.context(device), self.world_size, self.rank, buf, C.byref(h)))
        self.h = h

    @staticmethod
    def unique_id():
        buf = (C.c_uint8 * L.COMM_ID_BYTES)()
        L.check(L.lib().bmo_comm_unique_id(buf))
        return bytes(buf)

    @classmethod
    def from_torch(cls, device=None, group=None):
        import torch.distributed as dist
        rank, ws = dist.get_rank(group), dist.get_world_size(group)
        box = [cls.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0, group=group)
        return cls(rank, ws, box[0], world()[2] if device is None else device)

    def nccl_version(self):
        v = C.c_int32(0)
        L.check(L.lib().bmo_comm_info(self.h, None, None, C.byref(v)))
        return int(v.value)

    def allreduce(self, field, n_complex=None, sync=True):
        """Sum `field` over all ranks in place (bmo_pd_allreduce).  field: complex128 / float64 numpy array (host, staged
        through the GPU by the library), or an integer device pointer together with n_complex."""
        if isinstance(field, int):
            L.check(L.lib().bmo_pd_allreduce(self.h, C.c_void_p(field), int(n_complex), L.INPUT_DEVICE | (L.COMM_SYNC if sync else 0)))
            return field
        assert field.dtype in (np.complex128, np.float64) and (field.flags["C_CONTIGUOUS"] or field.flags["F_CONTIGUOUS"])
        n = field.size if field.dtype == np.complex128 else field.size // 2
        L.check(L.lib().bmo_pd_allreduce(self.h, L.ptr(field), int(n), 0))
        return field

    def spot_stats(self, result, det_object, nx=0, nz=0, window=None):
        """bmo_spot_stats_sharded, collective: every rank passes the TraceResult of its shard (None for a rank without rays)
        and receives the spot statistics of all ranks' entries in rank order, as solver.spot_stats's dict ("counts": an
        (nz, nx) int64 histogram over `window` when nx > 0).  BmoError on every rank if any rank's arguments are refused."""
        from .solver import _spot_dict
        counts = np.zeros((nz, nx), np.int64) if nx else None
        win = None if window is None else np.ascontiguousarray(window, dtype=np.float64)
        info = L.bmo_spot_info()
        L.check(L.lib().bmo_spot_stats_sharded(self.h, None if result is None else result.h, int(det_object), L.ptr(win), int(nx), int(nz),
                                               C.byref(info), L.ptr(counts), 0))
        return _spot_dict(info, counts)

    def psf_intensity(self, detector, n=100, crop_factor=1.0, center="centroid", x_min=math.inf, x_max=math.inf, z_min=math.inf,
                      z_max=math.inf, x0_shift=0.0, z0_shift=0.0):
        """PSFDetector.intensity over all ranks, collective: every rank passes its detector (after a solve, with or without hits
        of its own) and receives (xs, zs, I) of the records of all ranks in rank order.  The records are all-gathered
        (bmo_psf_allgather), the window is calc_local_lims of the gathered records with the x_min / z_min overrides of
        PSFDetector.intensity, and bmo_psf_intensity_sharded computes this rank's band of pixel columns and all-gathers the
        bands.  BmoError on every rank if any rank's arguments are refused."""
        from .solver import psf_axes, psf_window
        if detector._dsys is None:
            raise L.BmoError("FieldComm.psf_intensity: the PSFDetector was not solved on this rank")
        dsys, oi = detector._dsys, detector._index
        lib = L.lib()
        all_ = C.c_void_p()
        L.check(lib.bmo_psf_allgather(self.h, C.c_void_p(detector._psf) if detector._psf else None, C.byref(all_)))
        try:
            lims = np.zeros(4)
            L.check(lib.bmo_psf_lims(dsys.h, all_, oi, 0, float(crop_factor), 0 if center == "centroid" else 1, L.ptr(lims)))
            lims = psf_window(lims, x_min, x_max, z_min, z_max)
            I = np.zeros((n, n), order="F")
            L.check(lib.bmo_psf_intensity_sharded(self.h, dsys.h, all_, oi, 0, int(n), L.ptr(lims), float(x0_shift), float(z0_shift),
                                                  L.ptr(I), 0))
        finally:
            lib.bmo_psf_free(all_)
        return psf_axes(n, lims, x0_shift, z0_shift) + (I,)

    def pd_sweep(self, dsys, result, pd_index, n_poses, first, count, want_fields=True):
        """bmo_pd_sweep_sharded, collective: this rank's `dsys` holds poses [first, first + count) of an n_poses-pose sweep as its
        poses 0 .. count - 1 and `result` is their trace (None on a rank without poses).  Returns (power (n_poses,) of every
        rank's poses in pose order, this rank's fields (count, n, n) complex or None).  BmoError on every rank if any rank's
        arguments are refused."""
        from . import components as co
        objs = dsys.flat.objects
        n = objs[pd_index].n if 0 <= pd_index < len(objs) and isinstance(objs[pd_index], co.Photodetector) else 0   # else refused
        fields = np.zeros((count, n * n * 2)) if want_fields and count > 0 and n > 0 else None
        power = np.zeros(max(int(n_poses), 0))
        L.check(L.lib().bmo_pd_sweep_sharded(self.h, dsys.h, None if result is None else result.h, int(pd_index), int(n_poses), int(first),
                                             int(count), L.ptr(fields), L.ptr(power), 0))
        if not want_fields:
            return power, None
        if fields is None:
            return power, np.zeros((0, n, n), np.complex128)
        z = fields[:, 0::2] + 1j * fields[:, 1::2]
        return power, z.reshape(count, n, n).transpose(0, 2, 1)   # stored column-major [i + n*j] -> [pose, i, j]

    def spot_sweep(self, result, det_object, n_poses, first, count, nx=0, nz=0, window=None):
        """bmo_spot_stats_poses_sharded, collective: `result` is this rank's trace of poses [first, first + count) of an n_poses-pose
        sweep, traced as its poses 0 .. count - 1 (None on a rank without poses).  Returns, on every rank, solver.spot_stats_poses's
        dict of all n_poses poses in pose order ("counts": (n_poses, nz, nx) int64 histograms over `window` when nx > 0).  BmoError
        on every rank if any rank's arguments are refused."""
        from .solver import _spot_pose_dict
        P = int(n_poses)
        counts = np.zeros((max(P, 0), max(int(nz), 0), max(int(nx), 0)), np.int64) if nx else None
        win = None if window is None else np.ascontiguousarray(window, dtype=np.float64)
        info = (L.bmo_spot_info * max(P, 1))()
        L.check(L.lib().bmo_spot_stats_poses_sharded(self.h, None if result is None else result.h, int(det_object), P, int(first), int(count),
                                                     L.ptr(win), int(nx), int(nz), info, L.ptr(counts), 0))
        return _spot_pose_dict(info, P, counts)

    def free(self):
        if self.h:
            L.lib().bmo_comm_free(self.h)
            self.h = None


_default_comm = None


def default_comm(group=None):
    """The process-wide FieldComm: created on first use from the torch.distributed group (NCCL backends only), or a
    one-rank communicator on GPU LOCAL_RANK when this process is not part of a process group of several ranks."""
    global _default_comm
    if _default_comm is None:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
            _default_comm = FieldComm.from_torch(group=group)
        else:
            _default_comm = FieldComm(0, 1, FieldComm.unique_id(), world()[2])
    return _default_comm


def world():
    """(rank, world_size, local_rank) of this process; (0, 1, 0) outside torchrun."""
    return int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))


def shard_slice(n, rank, world_size):
    """Contiguous slice [start, stop) of rank `rank`: sizes differ by at most one, order preserved
    (sequential lens stacks: equal count = equal work)."""
    base, rem = divmod(n, world_size)
    start = rank * base + min(rank, rem)
    return start, start + base + (1 if rank < rem else 0)


def spot_shard_slice(n_rays, rank, world_size, R=1):
    """(first, count): the contiguous rays of rank `rank` for bmo_spot_stats_sharded.  Every slice but the last holds a
    multiple of BMO_SPOT_PER(n_rays * R) entries (R per ray), so no block of the spot reduction crosses a rank boundary, and
    the slices are as even as that allows: they are cut in units of the fewest rays that fill whole blocks (per / gcd(per,
    R) rays, at most `per`), the extra units go to the last ranks, and sizes differ by at most one unit.  A rank may get no
    rays when there are fewer units than ranks."""
    n_rays, rank, world_size = int(n_rays), int(rank), int(world_size)
    if not (0 <= rank < world_size) or n_rays < 0:
        raise ValueError(f"spot_shard_slice: rank {rank} of {world_size}, {n_rays} rays")
    per = L.spot_per(n_rays * R)
    unit = per // math.gcd(per, R)
    base, rem = divmod(-(-n_rays // unit), world_size)

    def start(k):   # first unit of rank k: ranks world_size - rem ... world_size - 1 take base + 1 units
        return k * base + max(0, k - (world_size - rem))
    first = min(n_rays, start(rank) * unit)
    stop = n_rays if rank == world_size - 1 else min(n_rays, start(rank + 1) * unit)
    return first, stop - first


def shard_interleaved(n, rank, world_size):
    """Round-robin indices rank, rank + W, ... for branching workloads (C4): the branch depth varies
    with the ray position, so interleaving equalises the work where contiguous blocks would not."""
    return np.arange(rank, n, world_size)


def shard_bundle(bundle, rank, world_size, interleaved=False):
    """This rank's part of a RayBundle / BeamletBundle (+ the global indices it holds)."""
    n = len(bundle)
    idx = shard_interleaved(n, rank, world_size) if interleaved else np.arange(*shard_slice(n, rank, world_size))
    if isinstance(bundle, bm.RayBundle):
        part = bm.RayBundle(bundle.pos[idx], bundle.dir[idx], bundle.lam[idx], None if bundle.E0 is None else bundle.E0[idx], normalize=False)
    elif isinstance(bundle, bm.BeamletBundle):
        part = bm.BeamletBundle(bundle.rays[idx], bundle.lam[idx], bundle.w0[idx], bundle.E0[idx])
    else:
        raise TypeError(f"cannot shard {type(bundle).__name__}")
    return part, idx


def allreduce_field(field, group=None, comm=None):
    """Sum the ranks' partial Photodetector fields in place.  With a FieldComm (or an NCCL process group, for which the
    process-wide FieldComm is used) the sum runs through the C ABI (bmo_pd_allreduce: NCCL inside libbmo.so); the
    torch.distributed path remains for gloo (CPU tests).  `field`: complex128 numpy array or a torch tensor (float64 view
    of re/im pairs, or complex128) that lives where the backend wants it."""
    import torch
    import torch.distributed as dist
    if comm is None and dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1 and dist.get_backend(group) == "nccl":
        comm = default_comm(group)
    if comm is not None:
        if isinstance(field, np.ndarray):
            return comm.allreduce(field)
        t = torch.view_as_real(field) if field.is_complex() else field
        assert t.is_cuda and t.is_contiguous() and t.dtype == torch.float64
        torch.cuda.current_stream(t.device).synchronize()      # the library reduces on its own stream
        comm.allreduce(int(t.data_ptr()), t.numel() // 2, sync=True)
        return field
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return field
    if isinstance(field, np.ndarray):
        assert field.dtype == np.complex128
        flat = np.ascontiguousarray(field.T if field.flags["F_CONTIGUOUS"] and field.ndim == 2 else field)
        t = torch.from_numpy(flat.view(np.float64).reshape(-1))
        if dist.get_backend(group) == "nccl":
            g = t.cuda()
            dist.all_reduce(g, op=dist.ReduceOp.SUM, group=group)
            t.copy_(g.cpu())
        else:
            dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
        out = flat.T if flat is not field and field.ndim == 2 and field.flags["F_CONTIGUOUS"] else flat
        if out is not field:
            field[...] = out
        return field
    t = torch.view_as_real(field) if field.is_complex() else field
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return field


def gather_rows(local, idx, n_total, group=None):
    """Assemble per-ray outputs (e.g. Spotdetector hits) of all ranks in global ray order on every rank."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return local
    parts = [None] * dist.get_world_size(group)
    dist.all_gather_object(parts, (np.asarray(idx), np.asarray(local)), group=group)
    out = np.full((n_total,) + np.asarray(local).shape[1:], np.nan, dtype=np.asarray(local).dtype)
    for i, v in parts:
        out[i] = v
    return out


def solve_spot_sharded(system, source, detector, bins=None, window=None, comm=None, r_max=100):
    """The spot diagram of a DeviceSource traced across all ranks: this rank traces source.shard(*spot_shard_slice(...)) on
    its GPU (the hits stay there) and bmo_spot_stats_sharded reduces every rank's hits.  Returns, on every rank, the dict
    spot_stats gives for one unsharded solve of the whole source on one GPU -- bit for bit when the system has no
    beamsplitters.  `comm`: a FieldComm (default: default_comm(), a one-rank communicator outside torchrun); the rank
    traces on the communicator's GPU.  `bins` / `window` as in spot_stats."""
    from .solver import _lambda_ids, _spot_args, cached_system, solve_system_
    comm = default_comm() if comm is None else comm
    first, count = spot_shard_slice(len(source), comm.rank, comm.world_size)
    res = None
    if count:
        res = solve_system_(system, source.shard(first, count), r_max=r_max, retrace=False, device=comm.device, keep_segments=False,
                            collect_spots=False)
    dsys = res.dsys if res is not None else cached_system(system, _lambda_ids([source.lam])[0], comm.device)
    oi, nx, nz, win = _spot_args(dsys.flat.objects, detector, bins, window, "solve_spot_sharded")
    return comm.spot_stats(res, oi, nx, nz, win)


def psf_shard_band(n, rank, world_size):
    """Pixel columns [j0, j1) of rank `rank` in bmo_psf_intensity_sharded: bands of B = ceil(n / world_size) columns in rank
    order, the last one cut at n; ranks past the last column get an empty band."""
    B = -(-int(n) // int(world_size))
    return min(n, rank * B), min(n, (rank + 1) * B)


def solve_psf_sharded(system, source, detector, n=100, crop_factor=1.0, center="centroid", x_min=math.inf, x_max=math.inf,
                      z_min=math.inf, z_max=math.inf, x0_shift=0.0, z0_shift=0.0, comm=None, r_max=100):
    """The intensity map of `detector` (a PSFDetector of `system`) for a DeviceSource, DeviceBeamletSource, RayBundle or BeamletBundle
    traced across all ranks: this rank traces its shard_slice of the source (DeviceSource.shard, which builds only those rays or
    beamlets on the device / shard_bundle) on the communicator's GPU, its records are
    appended to the detector as by solve_system_, and FieldComm.psf_intensity makes the map of all ranks' records.  Returns
    (xs, zs, I) on every rank: for a system without beamsplitters the bits of solve_system_ of the whole source followed by
    detector.intensity(...) on one GPU.  `comm`: a FieldComm (default: default_comm(), a one-rank communicator outside
    torchrun).  A rank with an empty slice traces nothing and contributes no records."""
    from .solver import _lambda_ids, cached_system, solve_system_
    comm = default_comm() if comm is None else comm
    first, stop = shard_slice(len(source), comm.rank, comm.world_size)
    if isinstance(source, bm.DeviceSource):
        part = source.shard(first, stop - first) if stop > first else None
        lams = [source.lam]
    else:
        part = shard_bundle(source, comm.rank, comm.world_size)[0] if stop > first else None
        lams = source.lam
    if part is not None:
        solve_system_(system, part, r_max=r_max, retrace=False, device=comm.device)
    elif detector._dsys is None:          # no rays here: the detector's system and index for the collective
        dsys = cached_system(system, _lambda_ids(lams)[0], comm.device)
        detector._dsys, detector._index = dsys, next(i for i, o in enumerate(dsys.flat.objects) if o is detector)
    return comm.psf_intensity(detector, n, crop_factor, center, x_min, x_max, z_min, z_max, x0_shift, z0_shift)


def solve_pose_sweep_sharded(system, beam, n_poses, pd, program=None, apply_pose=None, comm=None, want_fields=True, r_max=100):
    """A Photodetector pose sweep (solve_pose_sweep_device / solve_pose_sweep) across all ranks: this rank sweeps its shard_slice
    [first, first + count) of the n_poses poses on the communicator's GPU and bmo_pd_sweep_sharded gathers the powers.  Exactly one
    of `program` (records the kinematic calls of the whole sweep on a KinProgram; the rank applies its rows) and `apply_pose`
    (apply_pose(p) moves the host objects into pose p; called for the rank's p only) is given.  `beam`: GaussianBeamlet,
    BeamletBundle or DeviceBeamletSource, tiled `count` times.  Returns, on every rank, dict(power=(n_poses,), fields=(count, n, n)
    complex of this rank's poses or None, first=first, result=TraceResult or None, dsys=DeviceSystem): pose p's power and field
    have the bits of the one-GPU sweep (DESIGN §14).  `comm`: a FieldComm (default: default_comm())."""
    from . import sweep as sw
    n_poses = _check_sweep_args("solve_pose_sweep_sharded", n_poses, program, apply_pose)
    comm = default_comm() if comm is None else comm
    first, stop = shard_slice(n_poses, comm.rank, comm.world_size)
    count = stop - first
    lams, lam_id, beam = sw._beamlet_lambdas(beam)
    f0, dsys = _pose_range_system(system, lams, n_poses, first, count, program, apply_pose, comm.device)
    res = sw._trace_beamlet_sweep(dsys, beam, lam_id, count, r_max) if count else None
    power, fields = comm.pd_sweep(dsys, res, f0.object_index(pd), n_poses, first, count, want_fields)
    return dict(power=power, fields=fields, first=first, result=res, dsys=dsys)


def solve_spot_sweep_sharded(system, beam, n_poses, detector, program=None, apply_pose=None, bins=None, window=None, comm=None, r_max=100):
    """A spot-diagram pose sweep (solve_spot_sweep_device / solve_spot_sweep) across all ranks: this rank sweeps its shard_slice
    [first, first + count) of the n_poses poses on the communicator's GPU and bmo_spot_stats_poses_sharded gathers the statistics.
    Exactly one of `program` (records the kinematic calls of the whole sweep on a KinProgram; the rank applies its rows) and
    `apply_pose` (apply_pose(p) moves the host objects into pose p; called for the rank's p only) is given.  `beam`: RayBundle or
    DeviceSource, traced once per local pose.  `bins` / `window` as in spot_stats_poses.  Returns, on every rank,
    dict(stats=spot_stats_poses's dict of all n_poses poses, first=first, result=TraceResult or None, dsys=DeviceSystem): pose p has
    the bits of the one-GPU sweep (DESIGN §15).  `comm`: a FieldComm (default: default_comm())."""
    from . import sweep as sw
    from .solver import _spot_args
    n_poses = _check_sweep_args("solve_spot_sweep_sharded", n_poses, program, apply_pose)
    comm = default_comm() if comm is None else comm
    first, stop = shard_slice(n_poses, comm.rank, comm.world_size)
    count = stop - first
    lams, lam_id = sw._beam_lambdas(beam)
    f0, dsys = _pose_range_system(system, lams, n_poses, first, count, program, apply_pose, comm.device)
    oi, nx, nz, win = _spot_args(f0.objects, detector, bins, window, "solve_spot_sweep_sharded")
    res = sw._trace_spot_sweep(dsys, beam, lam_id, count, r_max) if count else None
    stats = comm.spot_sweep(res, oi, n_poses, first, count, nx, nz, win)
    return dict(stats=stats, first=first, result=res, dsys=dsys)


def _check_sweep_args(what, n_poses, program, apply_pose):
    """n_poses as an int, once exactly one of program and apply_pose is given and there is at least one pose."""
    if (program is None) == (apply_pose is None):
        raise ValueError(f"{what}: give exactly one of program and apply_pose")
    n_poses = int(n_poses)
    if n_poses < 1:
        raise ValueError(f"{what}: n_poses = {n_poses}, at least one pose is needed")
    return n_poses


def _pose_range_system(system, lams, n_poses, first, count, program, apply_pose, device):
    """(FlatSystem, DeviceSystem on `device`) of a sweep's poses [first, first + count), held as the system's poses 0 .. count - 1,
    each with the bits of the same pose of the whole sweep: `program` records the kinematic calls of all n_poses poses on a
    KinProgram and its rows [first, first + count) are applied on the device, or apply_pose(p) moves the host objects into pose p
    for those p only.  With count == 0 the system is uploaded as it is."""
    from . import sweep as sw
    from .flatten import FlatSystem
    from .solver import DeviceSystem
    if apply_pose is not None and count:
        f0, (prims, verts, bounds, det_pos, det_dir) = sw.flatten_poses(system, lams, count, lambda k: apply_pose(first + k))
        dsys = DeviceSystem(f0, device)
        L.check(L.lib().bmo_system_set_poses(dsys.h, count, L.ptr(prims), L.ptr(verts), L.ptr(bounds), L.ptr(det_pos), L.ptr(det_dir)))
    else:
        f0 = FlatSystem(system, lams)
        dsys = DeviceSystem(f0, device)
        if count:
            prog = sw.KinProgram(f0, n_poses)
            program(prog)
            prog.apply(dsys, first, count)
    return f0, dsys


def solve_system_sharded(system, bundle, r_max=100, interleaved=False, keep_segments=False, group=None, comm=None):
    """solve_system! of a bundle across all ranks: this rank traces its shard on GPU LOCAL_RANK; every
    Photodetector of `system` ends up with the field of the *whole* bundle on every rank (all-reduce);
    Spotdetector data stay rank-local (disjoint slices).  A DeviceSource or DeviceBeamletSource is cut into contiguous
    shard_slice parts, each rank building only its own on the device (interleaved=True is refused: a device shard is
    contiguous).  Returns (TraceResult of the shard, indices)."""
    from . import components as co
    from .solver import solve_system_
    rank, ws, local = world()
    if isinstance(bundle, bm.DeviceSource):
        if interleaved:
            raise ValueError("a device source is sharded in contiguous slices, not interleaved")
        start, stop = shard_slice(len(bundle), rank, ws)
        part, idx = (bundle.shard(start, stop - start) if stop > start else None), np.arange(start, stop)
    else:
        part, idx = shard_bundle(bundle, rank, ws, interleaved)
    pds = [o for o in system.leaves() if isinstance(o, co.Photodetector)]
    before = [pd.field.copy() for pd in pds]
    for pd in pds:                       # accumulate this rank's beamlets onto a zeroed partial field
        pd.field[...] = 0
    res = solve_system_(system, part, r_max=r_max, device=local, keep_segments=keep_segments) if part is not None and len(part) else None
    for pd, old in zip(pds, before):
        allreduce_field(pd.field, group, comm)
        pd.field += old                  # the reference's `+=` onto whatever the detector already held
    return res, idx
