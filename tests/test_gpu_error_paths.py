"""Error paths of the C ABI on the GPU: a refused or failed call leaves its objects as they were and frees what it
allocated.

(a) bmo_system_apply_poses refuses a kinematic tree whose per-node frames do not fit one block's shared memory before it
    touches the system: the pose tables and the traces through them stay what they were.
(b) Argument refusals that come after device work (bad lambda ids seen by the trace kernels, the kinematic refusal) leave
    the stream-ordered pool's used bytes where they were.  The pool is read through the driver API; torch's caching
    allocator does not use the device's default pool, and every buffer here stays below the 64 MiB from which libbmo
    bypasses the pool.
(c) Contexts are created, used by a pipelined trace (auxiliary streams) and shut down over and over."""
import ctypes as C

import numpy as np
import pytest

from tests import scenes

LAM = 707e-9


@pytest.fixture(scope="module")
def pool_used():
    """Bytes of device 0's default memory pool in use, after a device synchronise."""
    import torch
    cu = C.CDLL("libcuda.so.1")
    assert cu.cuInit(0) == 0
    dev, pool = C.c_int(), C.c_void_p()
    assert cu.cuDeviceGet(C.byref(dev), 0) == 0
    assert cu.cuDeviceGetDefaultMemPool(C.byref(pool), dev) == 0
    CU_MEMPOOL_ATTR_USED_MEM_CURRENT = 7

    def used():
        torch.cuda.synchronize()
        v = C.c_uint64()
        assert cu.cuMemPoolGetAttribute(pool, CU_MEMPOOL_ATTR_USED_MEM_CURRENT, C.byref(v)) == 0
        return v.value
    return used


def _bundle(n):
    pos, d = scenes.fibonacci_disc(n)
    return np.ascontiguousarray(pos), np.ascontiguousarray(d)


def _spots(L, dsys, pos, d, pose_ids):
    """Spotdetector hits of one host-input trace (segments not kept)."""
    h = C.c_void_p()
    L.check(L.lib().bmo_trace_rays(dsys.h, len(pos), L.ptr(pos), L.ptr(d), None, None, L.ptr(pose_ids), 100, 0, C.byref(h)))
    obj, xz = np.zeros(len(pos), np.int32), np.zeros((len(pos), 2))
    L.check(L.lib().bmo_result_spots(h, L.ptr(obj), L.ptr(xz)))
    L.lib().bmo_result_free(h)
    return obj, xz


@pytest.mark.gpu
def test_refused_kinematic_program_leaves_the_system_intact(bmo, pool_used):
    from bmo_b200 import _lib as L
    from bmo_b200 import sweep
    P = 3
    sc = scenes.doublet_spot(bmo)
    dsys = bmo.upload_system(sc["system"], [LAM])
    prog = sweep.KinProgram(dsys.flat, P)
    prog.translate3d_(sc["spot"], np.array([[0.0, 0.0, 0.0], [1e-4, 0.0, 0.0], [0.0, 0.0, 2e-4]]))
    prog.apply(dsys)
    pos, d = _bundle(4096)
    pose_ids = np.repeat(np.arange(P, dtype=np.int32), -(-len(pos) // P))[:len(pos)]
    before = [sweep.get_pose_tables(dsys, p) for p in range(P)]
    spots = _spots(L, dsys, pos, d, pose_ids)

    # childless groups after the tree: accepted by bmo_system_set_kinematics, but 2134 nodes * 96 B > the 200 KB the kernel may use
    nodes = list(prog.nodes)
    for i in range(len(nodes), 2134):
        nodes.append(L.bmo_kin_node(kind=0, size=1, pos_ref=i, index=-1, flags=0, object=-1))
    tab = (L.bmo_kin_node * len(nodes))(*nodes)
    lib = L.lib()
    L.check(lib.bmo_system_set_kinematics(dsys.h, len(nodes), C.byref(tab), L.ptr(prog.prim_bounds)))
    ops = (L.bmo_kin_op * len(prog.ops))(*[L.bmo_kin_op(*o) for o in prog.ops])
    params = np.ascontiguousarray(np.stack(prog.params, axis=1))
    used = pool_used()
    assert lib.bmo_system_apply_poses(dsys.h, P, len(prog.ops), C.byref(ops), len(prog.params), L.ptr(params)) == -1   # BMO_EINVAL
    assert b"too large for one block's shared memory" in lib.bmo_last_error()
    assert pool_used() == used

    for p in range(P):
        after = sweep.get_pose_tables(dsys, p)
        assert bytes(after[0]) == bytes(before[p][0])
        for a, b in zip(after[1:], before[p][1:]):
            assert a.tobytes() == b.tobytes()
    again = _spots(L, dsys, pos, d, pose_ids)
    assert np.array_equal(again[0], spots[0]) and again[1].tobytes() == spots[1].tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("scene", ["lean", "splitter"])
def test_refused_trace_frees_what_it_allocated(bmo, pool_used, scene):
    """A lambda id outside the system's table is seen by the trace kernels, so the call is refused after all its device work:
    through the whole-solve kernel (lean doublet) and through the wave loop (Michelson with its cube beamsplitter)."""
    from bmo_b200 import _lib as L
    system = scenes.doublet_spot(bmo)["system"] if scene == "lean" else scenes.michelson(bmo, pd_n=16)["system"]
    dsys = bmo.upload_system(system, [LAM])
    n = 4096
    pos, d = _bundle(n)
    if scene == "splitter":
        pos[:, 1] = 0.0
        pos *= 1e-2
        d[:] = (0.0, 1.0, 0.0)
    lam = np.zeros(n, np.int32)
    lam[n // 2] = 1
    lib = L.lib()
    for _ in range(2):      # the second call runs with the sizes the first one recorded (bmo_sys::hints)
        used = pool_used()
        L.counters_reset(0)
        h = C.c_void_p()
        assert lib.bmo_trace_rays(dsys.h, n, L.ptr(pos), L.ptr(d), L.ptr(lam), None, None, 100, 0, C.byref(h)) == -1
        assert b"lambda_id outside" in lib.bmo_last_error()
        launches = L.counters(0)["kernel_launches"]
        assert (launches == 1) if scene == "lean" else (launches > 2)     # solve_rays_persistent alone / the wave loop
        assert pool_used() == used


@pytest.mark.gpu
def test_contexts_come_and_go(bmo):
    from bmo_b200 import _lib as L
    lib = L.lib()
    flat = bmo.upload_system(scenes.doublet_spot(bmo)["system"], [LAM]).flat
    n = 512 * 1024          # host inputs of a splitter-free system: 4 sub-batches, 3 of them on auxiliary streams
    pos, d = _bundle(n)
    for _ in range(20):
        ctx, sys_, res = C.c_void_p(), C.c_void_p(), C.c_void_p()
        L.check(lib.bmo_init(0, C.byref(ctx)))
        L.check(lib.bmo_system_upload(ctx, C.byref(flat.tables), C.byref(sys_)))
        L.check(lib.bmo_trace_rays(sys_, n, L.ptr(pos), L.ptr(d), None, None, None, 100, 0, C.byref(res)))
        info = L.bmo_result_info()
        L.check(lib.bmo_result_get_info(res, C.byref(info)))
        assert info.interactions > 0
        assert lib.bmo_result_free(res) == 0
        assert lib.bmo_system_free(sys_) == 0
        assert lib.bmo_shutdown(ctx) == 0
    res = bmo.trace_rays(bmo.upload_system(scenes.doublet_spot(bmo)["system"], [LAM]), pos[:1024], d[:1024], None, keep_segments=False)
    assert res.interactions > 0     # the process's own context still traces
