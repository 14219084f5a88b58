"""The whole-solve kernel (solve_rays_persistent) against the wavefront path it replaces for plain rays through splitter-free
lens systems whose segments are not kept.  The two paths are selected per process (BMO_PERSIST is read once), so each side
runs the same cases in a subprocess of its own and the outputs are compared bit for bit: per-ray spots, detector ids, segment
counts and status words, the result info (interactions, waves) and the device counters (SDF evaluations, triangle tests,
interactions).  Calls outside the kernel's scope -- a system with a beamsplitter, a call that keeps its segment table, a
Gaussian beamlet bundle -- must launch exactly what they launched before.

Run directly (python tests/test_gpu_persistent.py OUT.npz) it is the worker: it traces every case and writes OUT.npz."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if __name__ == "__main__":
    sys.path.insert(0, ROOT)     # the worker imports this repository's tests package, not another one on the path
LAMS = [707e-9, 587.6e-9, 486.1e-9]


def lens_stack(m, k=37):
    """k biconvex lenses on the y axis, a flat two-triangle mirror mesh at 45 degrees behind them, a Spotdetector in the folded
    beam.  With k = 37 the staged tables (144 B per primitive, 208 B per part with its bounds and part word) come to 24096 B:
    just under the 24 KB the lean kernels allow, and more than a block could add to 25 KB of static scratch within 48 KB."""
    import math
    objs, y = [], 0.0
    for _ in range(k):
        lens = m.SphericalLens(0.2, -0.2, 4e-3, 25.4e-3, 1.5)
        lens.translate3d_((0.0, y, 0.0))
        objs.append(lens)
        y += 12e-3
    mirror = m.Mirror(m.QuadraticFlatMesh(40e-3))
    mirror.zrotate3d_(math.radians(45))
    mirror.translate3d_((0.0, y + 0.03, 0.0))
    sd = m.Spotdetector(50e-3)
    sd.zrotate3d_(math.radians(90))
    sd.translate3d_((0.05, y + 0.03, 0.0))
    return m.System(objs + [mirror, sd])


def _cases():
    """(name, system, kwargs) of every device-input trace; kwargs: pos, dir, lam, pose (host arrays or None), uniform, r_max."""
    from tests import scenes
    out = []
    c2_pos, c2_dir = scenes.fibonacci_disc(1 << 20)
    out.append(("c2", "doublet", dict(pos=c2_pos, dir=c2_dir, lam=np.zeros(1 << 20, np.int32))))
    pos, d = scenes.fibonacci_disc(1 << 16)
    out.append(("c2_uniform_dir", "doublet", dict(pos=pos, dir=d[0], lam=None, uniform=True)))
    rng = np.random.default_rng(3)
    dj = d + rng.normal(scale=2e-3, size=d.shape)
    dj /= np.linalg.norm(dj, axis=1, keepdims=True)
    lam = rng.integers(0, len(LAMS), size=len(pos)).astype(np.int32)
    out.append(("per_ray_dir_lambdas", "doublet", dict(pos=pos, dir=dj, lam=lam)))
    out.append(("device_pose_ids", "doublet", dict(pos=pos, dir=dj, lam=lam, pose=np.zeros(len(pos), np.int32))))
    out.append(("rotated_doublet", "doublet_rot", dict(pos=pos, dir=d, lam=None)))
    big, bd = scenes.fibonacci_disc(1 << 17, diameter=40e-3)     # overfilled pupil: most rays miss everything
    for r_max in (1, 2, 3, 100):
        out.append((f"overfilled_rmax{r_max}", "doublet", dict(pos=big, dir=bd, lam=None, r_max=r_max)))
    sp, sdir = scenes.fibonacci_disc(1 << 14)
    out.append(("lens_stack_mirror", "stack", dict(pos=sp, dir=sdir, lam=None)))
    for n in (1, 127, 129):
        out.append((f"n{n}", "doublet", dict(pos=pos[:n], dir=dj[:n], lam=lam[:n])))
    return out


def _worker(path):
    import ctypes as C
    import torch
    import __graft_entry__ as ge
    ge.build_libbmo()
    m = ge.load_package()
    from bmo_b200 import _lib as L
    from tests import scenes
    from tests import scenes2 as s2
    dev = 0
    systems = {"doublet": m.upload_system(scenes.doublet_spot(m)["system"], LAMS, device=dev),
               "doublet_rot": m.upload_system(scenes.doublet_spot(m, rotate=True)["system"], LAMS, device=dev),
               "stack": m.upload_system(lens_stack(m), LAMS, device=dev)}
    out = {}

    def run(name, dsys, pos, dir, lam=None, pose=None, uniform=False, r_max=100, keep=False):
        t = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda()
        pd, dd, ld, qd = t(pos), t(dir), t(lam), t(pose)
        p = lambda x: None if x is None else C.c_void_p(x.data_ptr())
        flags = L.INPUT_DEVICE | (L.UNIFORM_DIR if uniform else 0) | (L.KEEP_SEGMENTS if keep else 0)
        L.counters_reset(dev)
        h = C.c_void_p()
        L.check(L.lib().bmo_trace_rays(dsys.h, len(pos), p(pd), p(dd), p(ld), None, p(qd), r_max, flags, C.byref(h)))
        res = m.solver.TraceResult(dsys, h)
        c = L.counters(dev)
        obj, xz = res.spots()
        b = res.beams()
        out.update({f"{name}/spot_object": obj, f"{name}/spot_xz": xz, f"{name}/nseg": b["nseg"], f"{name}/status": b["status"],
                    f"{name}/parent": b["parent"], f"{name}/lam": b["lam_id"],
                    f"{name}/info": np.array([res.n_roots, res.n_beams, res.interactions, res.waves], np.int64),
                    f"{name}/counters": np.array([c["interactions"], c["sdf_evals"], c["tri_tests"], c["waves"]], np.int64),
                    f"{name}/launches": np.array([c["kernel_launches"]], np.int64)})
        res.free()

    for name, sysname, kw in _cases():
        run(name, systems[sysname], **kw)
    # calls the kernel does not take: their launches must not change
    pos, d = scenes.fibonacci_disc(4096)
    run("kept_segments", systems["doublet"], pos, d, keep=True)
    mi = scenes.michelson(m)
    msys = m.upload_system(mi["system"], [scenes.MICHELSON_BEAM["lam"]], device=dev)
    mpos = np.zeros((512, 3)); mpos[:, 0] = np.linspace(-1e-3, 1e-3, 512)
    mdir = np.zeros((512, 3)); mdir[:, 1] = 1.0
    L.counters_reset(dev)
    mres = m.trace_rays(msys, mpos, mdir, np.zeros(512, np.int32), keep_segments=False)
    out["splitter/launches"] = np.array([L.counters(dev)["kernel_launches"]], np.int64)
    out["splitter/info"] = np.array([mres.n_beams, mres.interactions, mres.waves], np.int64)
    out["splitter/nseg"] = mres.beams()["nseg"]
    mres.free()
    sc = s2.expander(m, 16)
    lat = s2.beamlet_lattice(8)
    bundle = m.BeamletBundle.from_params(lat["pos"], lat["dir"], lat["lam"], lat["w0"], M2=lat["M2"], P0=lat["P0"], support=lat["support"])
    L.counters_reset(dev)
    m.solve_system_(sc["system"], bundle)
    out["beamlets/launches"] = np.array([L.counters(dev)["kernel_launches"]], np.int64)
    out["beamlets/field"] = sc["pd"].field
    # n = 0 and ids outside the tables are refused, and the context stays usable
    errs = []
    for kw in (dict(n=0), dict(lam=7), dict(pose=3)):
        n = kw.get("n", 256)
        pos, d = scenes.fibonacci_disc(max(n, 1))
        lam = np.zeros(max(n, 1), np.int32); lam[n // 2] = kw.get("lam", 0)
        pose = np.zeros(max(n, 1), np.int32); pose[n // 3] = kw.get("pose", 0)
        pd, dd, ld, qd = (torch.from_numpy(a).cuda() for a in (pos, d, lam, pose))
        h = C.c_void_p()
        errs.append(L.lib().bmo_trace_rays(systems["doublet"].h, n, C.c_void_p(pd.data_ptr()), C.c_void_p(dd.data_ptr()),
                                           C.c_void_p(ld.data_ptr()), None, C.c_void_p(qd.data_ptr()), 100, L.INPUT_DEVICE, C.byref(h)))
    out["invalid/rc"] = np.array(errs, np.int64)
    pos, d = scenes.fibonacci_disc(1000)
    run("after_invalid", systems["doublet"], pos, d, lam=np.zeros(1000, np.int32))
    # host inputs small enough for one sub-batch take the kernel too (spots copied back by the same call)
    obj, xz, res = m.solver.trace_rays_spots(systems["doublet"], pos, d[0], None)
    out.update({"host_spots/obj": obj, "host_spots/xz": xz, "host_spots/info": np.array([res.interactions, res.waves], np.int64)})
    res.free()
    np.savez(path, **out)


def _run_side(tmp_path, persist):
    path = str(tmp_path / f"persist{persist}.npz")
    env = dict(os.environ, BMO_PERSIST=str(persist))
    r = subprocess.run([sys.executable, os.path.abspath(__file__), path], env=env, cwd=ROOT, capture_output=True, text=True, timeout=1800)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
    return dict(np.load(path))


@pytest.fixture(scope="module")
def sides(tmp_path_factory):
    tmp = tmp_path_factory.mktemp("persistent")
    return _run_side(tmp, 0), _run_side(tmp, 1)


@pytest.mark.gpu
def test_same_keys(sides):
    old, new = sides
    assert sorted(old) == sorted(new)


@pytest.mark.gpu
@pytest.mark.parametrize("name", [c[0] for c in _cases()] + ["after_invalid", "host_spots"])
def test_persistent_bitwise(sides, name):
    old, new = sides
    keys = [k for k in old if k.startswith(name + "/") and k != name + "/launches"]
    assert keys
    for k in keys:
        a, b = old[k], new[k]
        assert a.dtype == b.dtype and a.shape == b.shape, k
        assert np.array_equal(np.ascontiguousarray(a).view(np.uint8), np.ascontiguousarray(b).view(np.uint8)), k   # bit for bit, NaN included
    if name + "/launches" in new:
        assert int(new[name + "/launches"][0]) == 1                         # the whole solve in one launch
        assert int(old[name + "/launches"][0]) > 1


@pytest.mark.gpu
def test_c2_outputs_are_physical(sides):
    _, new = sides
    info = new["c2/info"]
    assert info[2] == 4 * (1 << 20) and info[3] == 4                        # 4 interactions per ray, 4 waves
    assert (new["c2/spot_object"] >= 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["kept_segments", "splitter", "beamlets"])
def test_other_calls_keep_their_launches(sides, name):
    old, new = sides
    for k in old:
        if k.startswith(name + "/"):
            assert np.array_equal(np.ascontiguousarray(old[k]).view(np.uint8), np.ascontiguousarray(new[k]).view(np.uint8)), k


def test_lens_stack_tables_fill_the_lean_limit():
    """The stack's tables need more dynamic shared memory than 48 KB minus 25 KB of static scratch leaves, and no more than the
    lean gate allows: a persistent kernel with that much scratch could not launch for it."""
    sys.path.insert(0, ROOT)
    import __graft_entry__ as ge
    m = ge.load_package()
    from bmo_b200 import flatten
    t = flatten.FlatSystem(lens_stack(m), LAMS).tables
    smem = t.n_prims * 144 + t.n_parts * (120 + 10 * 8 + 8)
    assert 48 * 1024 - 25088 < smem <= 24 * 1024


@pytest.mark.gpu
def test_lens_stack_runs_both_branches(sides):
    _, new = sides
    assert new["lens_stack_mirror/counters"][2] > 0                           # triangle tests of the mirror mesh
    assert new["lens_stack_mirror/info"][2] > 37 * (1 << 14)                  # most rays cross the stack: refractive interactions


@pytest.mark.gpu
def test_invalid_ids_are_refused(sides):
    old, new = sides
    assert np.array_equal(old["invalid/rc"], new["invalid/rc"])
    assert (new["invalid/rc"] != 0).all()


if __name__ == "__main__":
    _worker(sys.argv[1])
