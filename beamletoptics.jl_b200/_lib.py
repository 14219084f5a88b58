"""ctypes binding of libbmo.so (the C ABI declared in include/bmo.h).

There is no CPU fallback: if the shared library is missing, or no sm_100 GPU is present when a
trace is requested, the call raises.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BMO_LIB") or os.path.join(_HERE, "libbmo.so")   # BMO_LIB: another build of the same library (A/B timing)

KEEP_SEGMENTS = 1
INPUT_DEVICE = 2
PD_REFERENCE_ORDER = 4
UNIFORM_DIR = 8
COMM_SYNC = 16
COMM_ID_BYTES = 128
SRC_DISC, SRC_COLLIMATED, SRC_POINT = 0, 1, 2     # bmo_source_kind
SPOT_SLICE, SPOT_MAX_BLOCKS = 4096, 1024          # BMO_SPOT_PER


def spot_per(m):
    """BMO_SPOT_PER(m): entries per block of the spot reduction over m entries, 4096 * max(1, ceil(m / (4096 * 1024)))."""
    return SPOT_SLICE * max(1, -(-int(m) // (SPOT_SLICE * SPOT_MAX_BLOCKS)))

STATUS_NAMES = ["ACTIVE", "MISS", "ABSORBED", "RMAX", "SPLIT", "CLIPPED", "TORN", "ERROR"]


class BmoError(RuntimeError):
    pass


class bmo_prim(C.Structure):
    _fields_ = [("type", C.c_int32), ("reserved", C.c_int32), ("pos", C.c_double * 3), ("tdir", C.c_double * 9), ("par", C.c_double * 4),
                ("ext_first", C.c_int32), ("ext_count", C.c_int32)]


class bmo_part(C.Structure):
    _fields_ = [("object", C.c_int32), ("role", C.c_int32), ("shape_kind", C.c_int32), ("first", C.c_int32), ("count", C.c_int32),
                ("n_row", C.c_int32), ("reflectance", C.c_double), ("transmittance", C.c_double), ("bound", C.c_double * 10)]


class bmo_object(C.Structure):
    _fields_ = [("kind", C.c_int32), ("first_part", C.c_int32), ("n_parts", C.c_int32), ("pd_n", C.c_int32),
                ("pos", C.c_double * 3), ("dir", C.c_double * 9), ("pd_lo", C.c_double), ("pd_hi", C.c_double)]


class bmo_mesh(C.Structure):
    _fields_ = [("first_vertex", C.c_int64), ("n_vertices", C.c_int64), ("first_face", C.c_int64), ("n_faces", C.c_int64),
                ("f32", C.c_int32), ("reserved", C.c_int32)]


class bmo_tables(C.Structure):
    _fields_ = [("n_prims", C.c_int32), ("prims", C.POINTER(bmo_prim)),
                ("n_parts", C.c_int32), ("parts", C.POINTER(bmo_part)),
                ("n_objects", C.c_int32), ("objects", C.POINTER(bmo_object)),
                ("n_meshes", C.c_int32), ("meshes", C.POINTER(bmo_mesh)),
                ("n_vertices", C.c_int64), ("vertices", C.POINTER(C.c_double)),
                ("n_faces", C.c_int64), ("faces", C.POINTER(C.c_int32)),
                ("n_lambda", C.c_int32), ("lambdas", C.POINTER(C.c_double)),
                ("n_rows", C.c_int32), ("n_table", C.POINTER(C.c_double)),
                ("n_system", C.c_double),
                ("n_ext", C.c_int64), ("ext", C.POINTER(C.c_double)),
                ("n_jones", C.c_int32), ("jones", C.POINTER(C.c_double)),
                ("norm_zero_rule", C.c_int32), ("reserved", C.c_int32)]


class bmo_kin_node(C.Structure):
    _fields_ = [("kind", C.c_int32), ("size", C.c_int32), ("pos_ref", C.c_int32), ("index", C.c_int32), ("flags", C.c_int32),
                ("object", C.c_int32), ("pos", C.c_double * 3), ("dir", C.c_double * 9)]


class bmo_kin_op(C.Structure):
    _fields_ = [("kind", C.c_int32), ("node", C.c_int32), ("pivot", C.c_int32), ("param", C.c_int32)]


class bmo_counters(C.Structure):
    _fields_ = [("interactions", C.c_int64), ("sdf_evals", C.c_int64), ("tri_tests", C.c_int64), ("waves", C.c_int64),
                ("kernel_launches", C.c_int64), ("px_beamlets", C.c_int64), ("trace_ms", C.c_double), ("pd_ms", C.c_double),
                ("trace_step_ms", C.c_double), ("trace_step_launches", C.c_int64), ("scatter_ms", C.c_double),
                ("scatter_bytes", C.c_double), ("pd_field_ms", C.c_double),
                ("psf_pairs", C.c_int64), ("psf_ms", C.c_double)]


class bmo_result_info(C.Structure):
    _fields_ = [("n_roots", C.c_int64), ("n_beams", C.c_int64), ("n_segments", C.c_int64), ("interactions", C.c_int64),
                ("rays_per_beam", C.c_int32), ("polarized", C.c_int32), ("waves", C.c_int32), ("reserved", C.c_int32)]


class bmo_source_ring(C.Structure):
    _fields_ = [("first", C.c_int64), ("count", C.c_int64), ("start", C.c_double * 3), ("rot", C.c_double * 9)]


class bmo_source_desc(C.Structure):
    _fields_ = [("kind", C.c_int32), ("reserved", C.c_int32), ("n_rays", C.c_int64), ("n_rings", C.c_int64),
                ("rings", C.POINTER(bmo_source_ring)), ("pos", C.c_double * 3), ("dir", C.c_double * 3), ("e1", C.c_double * 3),
                ("e2", C.c_double * 3), ("radius", C.c_double), ("phi0", C.c_double)]


class bmo_beamlet_desc(C.Structure):
    _fields_ = [("dv", C.c_double * 3), ("dd", C.c_double * 3), ("s", C.c_double * 3), ("w0", C.c_double), ("div_offset", C.c_double),
                ("E0", C.c_double * 2)]


class bmo_spot_info(C.Structure):
    _fields_ = [("hits", C.c_int64), ("outside", C.c_int64), ("centroid", C.c_double * 2), ("rms", C.c_double), ("max_r", C.c_double),
                ("lo", C.c_double * 2), ("hi", C.c_double * 2)]


# every symbol include/bmo.h declares (checked by tests/test_abi.py)
EXPORTS = [
    "bmo_init", "bmo_shutdown", "bmo_last_error", "bmo_set_stream", "bmo_counters_get", "bmo_counters_reset",
    "bmo_system_upload", "bmo_system_free", "bmo_system_set_poses", "bmo_trace_rays", "bmo_trace_rays_spots", "bmo_trace_beamlets",
    "bmo_retrace", "bmo_psf_collect", "bmo_psf_count", "bmo_psf_data", "bmo_psf_lims", "bmo_psf_intensity", "bmo_psf_free",
    "bmo_result_get_info", "bmo_result_beams", "bmo_result_segments", "bmo_result_spots", "bmo_result_spots_device",
    "bmo_result_free", "bmo_pd_accumulate", "bmo_pd_accumulate_poses", "bmo_pd_power", "bmo_pd_sweep", "bmo_measure_fp64_peak",
    "bmo_system_set_kinematics", "bmo_system_apply_poses", "bmo_system_get_pose",
    "bmo_debug_normals", "bmo_trim",
    "bmo_source_create", "bmo_source_device", "bmo_source_rays", "bmo_source_free", "bmo_spot_stats",
    "bmo_source_create_poses", "bmo_source_pose_ids", "bmo_spot_stats_poses",
    "bmo_source_create_slice", "bmo_spot_stats_results", "bmo_spot_stats_sharded",
    "bmo_psf_intensity_cols", "bmo_psf_allgather", "bmo_psf_intensity_sharded", "bmo_pd_sweep_sharded",
    "bmo_spot_stats_poses_sharded",
    "bmo_source_create_beamlets", "bmo_source_beamlets_device", "bmo_source_beamlets",
    "bmo_comm_unique_id", "bmo_comm_init", "bmo_comm_init_local", "bmo_comm_info", "bmo_pd_allreduce", "bmo_pd_allreduce_local", "bmo_comm_free",
]

_lib = None
_vp, _dp, _ip = C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int32)


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise BmoError(f"{LIB_PATH} not found: build it with __graft_entry__.build() (there is no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        L.bmo_last_error.restype = C.c_char_p
        L.bmo_init.argtypes = [C.c_int32, C.POINTER(_vp)]
        L.bmo_shutdown.argtypes = [_vp]
        L.bmo_set_stream.argtypes = [_vp, _vp]
        L.bmo_counters_get.argtypes = [_vp, C.POINTER(bmo_counters)]
        L.bmo_counters_reset.argtypes = [_vp]
        L.bmo_system_upload.argtypes = [_vp, C.POINTER(bmo_tables), C.POINTER(_vp)]
        L.bmo_system_free.argtypes = [_vp]
        L.bmo_system_set_poses.argtypes = [_vp, C.c_int32, _vp, _vp, _vp, _vp, _vp]
        L.bmo_trace_rays.argtypes = [_vp, C.c_int64, _vp, _vp, _vp, _vp, _vp, C.c_int32, C.c_uint32, C.POINTER(_vp)]
        L.bmo_trace_rays_spots.argtypes = [_vp, C.c_int64, _vp, _vp, _vp, _vp, _vp, C.c_int32, C.c_uint32, _vp, _vp, C.POINTER(_vp)]
        L.bmo_trace_beamlets.argtypes = [_vp, C.c_int64, _vp, _vp, _vp, _vp, _vp, C.c_int32, C.c_uint32, C.POINTER(_vp)]
        L.bmo_retrace.argtypes = [_vp, _vp, C.c_int32, C.c_uint32, C.POINTER(_vp)]
        L.bmo_result_get_info.argtypes = [_vp, C.POINTER(bmo_result_info)]
        L.bmo_result_beams.argtypes = [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]
        L.bmo_result_segments.argtypes = [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]
        L.bmo_result_spots.argtypes = [_vp, _vp, _vp]
        L.bmo_result_spots_device.argtypes = [_vp, C.POINTER(_vp), C.POINTER(_vp)]
        L.bmo_result_free.argtypes = [_vp]
        L.bmo_pd_accumulate.argtypes = [_vp, _vp, C.c_int32, C.c_int32, _vp, C.c_uint32]
        L.bmo_pd_accumulate_poses.argtypes = [_vp, _vp, C.c_int32, C.c_int32, _vp, C.c_uint32]
        L.bmo_pd_power.argtypes = [_vp, C.c_int32, C.c_int32, _vp, _vp, C.c_uint32]
        L.bmo_pd_sweep.argtypes = [_vp, _vp, C.c_int32, C.c_int32, _vp, _vp, C.c_uint32]
        L.bmo_psf_collect.argtypes = [_vp, _vp, C.c_int32, C.POINTER(_vp), C.POINTER(C.c_int64)]
        L.bmo_psf_count.argtypes = [_vp, C.POINTER(C.c_int64)]
        L.bmo_psf_data.argtypes = [_vp, _vp]
        L.bmo_psf_lims.argtypes = [_vp, _vp, C.c_int32, C.c_int32, C.c_double, C.c_int32, _vp]
        L.bmo_psf_intensity.argtypes = [_vp, _vp, C.c_int32, C.c_int32, C.c_int32, _vp, C.c_double, C.c_double, _vp, C.c_uint32]
        L.bmo_psf_free.argtypes = [_vp]
        L.bmo_measure_fp64_peak.argtypes = [_vp, _dp]
        L.bmo_trim.argtypes = [_vp, C.POINTER(C.c_int64)]
        L.bmo_debug_normals.argtypes = [_vp, C.c_int64, _vp, _vp, _vp, _vp]
        L.bmo_system_set_kinematics.argtypes = [_vp, C.c_int32, _vp, _vp]
        L.bmo_system_apply_poses.argtypes = [_vp, C.c_int32, C.c_int32, _vp, C.c_int32, _vp]
        L.bmo_system_get_pose.argtypes = [_vp, C.c_int32, _vp, _vp, _vp, _vp]
        L.bmo_source_create.argtypes = [_vp, C.POINTER(bmo_source_desc), C.POINTER(_vp)]
        L.bmo_source_device.argtypes = [_vp, C.POINTER(C.c_int64), C.POINTER(_vp), C.POINTER(_vp), _ip]
        L.bmo_source_rays.argtypes = [_vp, _vp, _vp]
        L.bmo_source_free.argtypes = [_vp]
        L.bmo_spot_stats.argtypes = [_vp, C.c_int32, _vp, C.c_int32, C.c_int32, C.POINTER(bmo_spot_info), _vp, C.c_uint32]
        L.bmo_source_create_poses.argtypes = [_vp, C.POINTER(bmo_source_desc), C.c_int32, C.POINTER(_vp)]
        L.bmo_source_pose_ids.argtypes = [_vp, _ip, C.POINTER(_vp)]
        L.bmo_spot_stats_poses.argtypes = [_vp, C.c_int32, C.c_int32, _vp, C.c_int32, C.c_int32, C.POINTER(bmo_spot_info), _vp, C.c_uint32]
        L.bmo_comm_unique_id.argtypes = [_vp]
        L.bmo_comm_init.argtypes = [_vp, C.c_int32, C.c_int32, _vp, C.POINTER(_vp)]
        L.bmo_comm_init_local.argtypes = [C.c_int32, C.POINTER(_vp), C.POINTER(_vp)]
        L.bmo_comm_info.argtypes = [_vp, _ip, _ip, _ip]
        L.bmo_pd_allreduce.argtypes = [_vp, _vp, C.c_int64, C.c_uint32]
        L.bmo_pd_allreduce_local.argtypes = [C.c_int32, C.POINTER(_vp), C.POINTER(_vp), C.c_int64, C.c_uint32]
        L.bmo_comm_free.argtypes = [_vp]
        L.bmo_source_create_slice.argtypes = [_vp, C.POINTER(bmo_source_desc), C.c_int64, C.c_int64, C.POINTER(_vp)]
        L.bmo_spot_stats_results.argtypes = [C.c_int32, C.POINTER(_vp), C.c_int32, _vp, C.c_int32, C.c_int32, C.POINTER(bmo_spot_info), _vp, C.c_uint32]
        L.bmo_spot_stats_sharded.argtypes = [_vp, _vp, C.c_int32, _vp, C.c_int32, C.c_int32, C.POINTER(bmo_spot_info), _vp, C.c_uint32]
        L.bmo_psf_intensity_cols.argtypes = [_vp, _vp, C.c_int32, C.c_int32, C.c_int32, _vp, C.c_double, C.c_double, C.c_int32, C.c_int32, _vp,
                                             C.c_uint32]
        L.bmo_psf_allgather.argtypes = [_vp, _vp, C.POINTER(_vp)]
        L.bmo_psf_intensity_sharded.argtypes = [_vp, _vp, _vp, C.c_int32, C.c_int32, C.c_int32, _vp, C.c_double, C.c_double, _vp, C.c_uint32]
        L.bmo_pd_sweep_sharded.argtypes = [_vp, _vp, _vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _vp, _vp, C.c_uint32]
        L.bmo_spot_stats_poses_sharded.argtypes = [_vp, _vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _vp, C.c_int32, C.c_int32,
                                                   C.POINTER(bmo_spot_info), _vp, C.c_uint32]
        L.bmo_source_create_beamlets.argtypes = [_vp, C.POINTER(bmo_source_desc), C.POINTER(bmo_beamlet_desc), C.c_int32, C.c_int64, C.c_int64,
                                                 C.POINTER(_vp)]
        L.bmo_source_beamlets_device.argtypes = [_vp, C.POINTER(C.c_int64), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp)]
        L.bmo_source_beamlets.argtypes = [_vp, _vp, _vp, _vp]
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise BmoError(f"libbmo error {rc}: {lib().bmo_last_error().decode()}")


def ptr(a):
    """void* of a numpy array (None -> NULL) or pass an int device pointer through."""
    if a is None:
        return None
    if isinstance(a, int):
        return C.c_void_p(a)
    return a.ctypes.data_as(C.c_void_p)


_ctx = {}


def context(device=0):
    """One bmo_ctx per (process, device)."""
    if device not in _ctx:
        h = _vp()
        check(lib().bmo_init(int(device), C.byref(h)))
        _ctx[device] = h
    return _ctx[device]


def counters(device=0):
    c = bmo_counters()
    check(lib().bmo_counters_get(context(device), C.byref(c)))
    return {k: getattr(c, k) for k, _ in bmo_counters._fields_}


def counters_reset(device=0):
    check(lib().bmo_counters_reset(context(device)))


def trim(device=0):
    """bmo_trim: hand parked / pooled device memory back to the driver; returns the bytes released from the free list."""
    n = C.c_int64(0)
    check(lib().bmo_trim(context(device), C.byref(n)))
    return int(n.value)


def set_stream(stream_ptr, device=0):
    check(lib().bmo_set_stream(context(device), C.c_void_p(stream_ptr)))


def measure_fp64_peak(device=0):
    v = C.c_double(0)
    check(lib().bmo_measure_fp64_peak(context(device), C.byref(v)))
    return v.value
