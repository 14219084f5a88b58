"""Sources generated on the device (bmo_source_*) and the spot-diagram reduction (bmo_spot_stats).

CPU: the ring table of CollimatedSource / PointSource, expanded by a restatement of the device recurrence (one lane per
ring, serial in the ray index), gives the host constructors' rays bit for bit, and the new C structs have the header's
layout.  GPU: ring sources equal the host constructors bit for bit, discs agree to a few ulp, tracing a device source gives
exactly what tracing the host copy of its rays gives, and bmo_spot_stats agrees with numpy on bmo_result_spots."""
import ctypes as C
import math
import os
import shutil
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LAM = 707e-9


# ---- CPU: one ring layout for host and device ------------------------------------------------------------------------
def restate_rings(desc, n):
    """The device's source_rings in numpy: every ring is a lane; ray j of a ring is start, then v <- rot v with
    ((a0 v0 + a1 v1) + a2 v2), no contraction.  Point directions get RayBundle's renormalisation."""
    from bmo_b200 import _lib as L
    p, d = np.array(desc.pos[:]), np.array(desc.dir[:])
    pos, dirs = np.empty((n, 3)), np.empty((n, 3))
    pos[0], dirs[:] = p, d
    rings = [desc.rings[i] for i in range(desc.n_rings) if desc.rings[i].count > 0]
    first = np.array([g.first for g in rings], np.int64)
    count = np.array([g.count for g in rings], np.int64)
    V = np.array([g.start[:] for g in rings]).reshape(-1, 3)
    A = np.array([g.rot[:] for g in rings]).reshape(-1, 3, 3)
    for j in range(int(count.max()) if len(rings) else 0):
        live = count > j
        idx, v = first[live] + j, V[live]
        if desc.kind == L.SRC_POINT:
            inv = 1.0 / np.sqrt(v[:, 0] * v[:, 0] + v[:, 1] * v[:, 1] + v[:, 2] * v[:, 2])
            pos[idx], dirs[idx] = p, v * inv[:, None]
        else:
            pos[idx] = p + v
        V = (A[:, :, 0] * V[:, 0:1] + A[:, :, 1] * V[:, 1:2]) + A[:, :, 2] * V[:, 2:3]
    return pos, dirs


def _same(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and np.array_equal(a.view(np.int64), b.view(np.int64))


RING_CASES = [
    ("collimated", dict(pos=(0.0, -0.05, 0.0), dir=(0.0, 1.0, 0.0), diameter=20e-3, num_rings=10, num_rays=None, b1=(1.0, 0.0, 0.0))),
    ("collimated", dict(pos=(0.01, 0.02, -0.03), dir=(0.3, 0.5, -0.2), diameter=5e-3, num_rings=7, num_rays=3001, b1=(1.0, 0.0, 0.0))),
    ("collimated", dict(pos=(0.0, 0.0, 0.0), dir=(0.0, 0.0, 1.0), diameter=1e-3, num_rings=40, num_rays=20000, b1=(0.0, 1.0, 0.0))),
    ("collimated", dict(pos=(1.0, 2.0, 3.0), dir=(-1.0, 1.0, 1.0), diameter=25.4e-3, num_rings=2, num_rays=40, b1=(1.0, 1.0, 0.0))),
    ("point", dict(pos=(0.0, 0.0, 0.0), dir=(0.0, 1.0, 0.0), theta=0.3, num_rings=10, num_rays=None, b1=(1.0, 0.0, 0.0))),
    ("point", dict(pos=(0.1, -0.2, 0.3), dir=(0.3, 0.5, -0.2), theta=1.0, num_rings=13, num_rays=5000, b1=(1.0, 0.0, 0.0))),
    ("point", dict(pos=(0.0, 0.0, 0.0), dir=(0.0, 0.0, 1.0), theta=math.pi - 1e-3, num_rings=30, num_rays=20000, b1=(0.0, 1.0, 0.0))),
    ("point", dict(pos=(0.0, 0.0, 0.0), dir=(1.0, 0.0, 0.0), theta=math.pi - 1e-12, num_rings=5, num_rays=500, b1=(0.0, 0.0, 1.0))),
]


def _make(m, kind, kw, on_device):
    kw = dict(kw)
    if kind == "collimated":
        return m.CollimatedSource(kw.pop("pos"), kw.pop("dir"), kw.pop("diameter"), LAM, on_device=on_device, **kw)
    return m.PointSource(kw.pop("pos"), kw.pop("dir"), kw.pop("theta"), LAM, on_device=on_device, **kw)


@pytest.mark.parametrize("case", range(len(RING_CASES)))
def test_ring_table_restated_equals_host_constructor(bmo, case):
    kind, kw = RING_CASES[case]
    host = _make(bmo, kind, kw, False)
    src = _make(bmo, kind, kw, True)          # descriptor only: nothing is created on a device until it is traced
    assert isinstance(src, bmo.DeviceSource) and len(src) == len(host)
    assert sum(src.desc.rings[i].count for i in range(src.desc.n_rings)) == len(host) - 1
    pos, dirs = restate_rings(src.desc, len(src))
    assert _same(pos, host.pos)
    assert _same(dirs, host.dir)
    assert src.uniform_dir == host.uniform_dir


def test_ring_layout_is_contiguous_and_skips_empty_rings(bmo):
    from bmo_b200 import beams
    rings = beams.source_rings("point", (0.0, 0.0, 1.0), (1.0, 0.0, 0.0), math.pi - 1e-3, 30, 20000)
    nxt = 1
    for first, count, _, _ in rings:
        assert first == nxt and count >= 0
        nxt += count
    assert nxt == 20000


def test_disc_descriptor_matches_host_basis(bmo):
    host = bmo.UniformDiscSource((0.0, -0.05, 0.0), (0.0, 2.0, 0.0), 20e-3, LAM, num_rays=1000, e1=(1.0, 0.0, 0.0))
    src = bmo.UniformDiscSource((0.0, -0.05, 0.0), (0.0, 2.0, 0.0), 20e-3, LAM, num_rays=1000, e1=(1.0, 0.0, 0.0), on_device=True)
    assert tuple(src.desc.dir) == tuple(host.dir[0]) and src.desc.n_rings == 0
    assert src.desc.radius == 10e-3 and src.desc.phi0 == 2 * math.pi / (1 + math.sqrt(5))


def test_new_struct_layouts_match_header(bmo):
    from bmo_b200 import _lib as L
    sizes = {"bmo_source_ring": C.sizeof(L.bmo_source_ring), "bmo_source_desc": C.sizeof(L.bmo_source_desc),
             "bmo_spot_info": C.sizeof(L.bmo_spot_info)}
    assert sizes == {"bmo_source_ring": 2 * 8 + 12 * 8, "bmo_source_desc": 4 + 4 + 8 + 8 + 8 + 12 * 8 + 2 * 8,
                     "bmo_spot_info": 2 * 8 + 8 * 8}
    cc = shutil.which("cc") or shutil.which("gcc")
    if cc is None:
        return
    src = ('#include <stdio.h>\n#include <stddef.h>\n#include "bmo.h"\nint main(void) { printf("%zu %zu %zu %zu %zu\\n", '
           'sizeof(bmo_source_ring), sizeof(bmo_source_desc), sizeof(bmo_spot_info), offsetof(bmo_source_desc, pos), '
           'offsetof(bmo_spot_info, rms)); return 0; }\n')
    import tempfile
    with tempfile.TemporaryDirectory() as td:
        with open(os.path.join(td, "s.c"), "w") as f:
            f.write(src)
        subprocess.run([cc, "-I", os.path.join(ROOT, "include"), "-o", os.path.join(td, "s"), os.path.join(td, "s.c")], check=True)
        got = [int(x) for x in subprocess.run([os.path.join(td, "s")], check=True, capture_output=True, text=True).stdout.split()]
    assert got == [sizes["bmo_source_ring"], sizes["bmo_source_desc"], sizes["bmo_spot_info"],
                   L.bmo_source_desc.pos.offset, L.bmo_spot_info.rms.offset]


# ---- GPU ---------------------------------------------------------------------------------------------------------------
def _rays_equal_host(m, host, src):
    pos, dirs = src.rays()
    return _same(pos, host.pos) and _same(dirs, host.dir)


@pytest.mark.gpu
@pytest.mark.parametrize("case", range(len(RING_CASES)))
def test_ring_sources_on_device_bit_identical(bmo, case):
    kind, kw = RING_CASES[case]
    assert _rays_equal_host(bmo, _make(bmo, kind, kw, False), _make(bmo, kind, kw, True))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["collimated", "point"])
def test_ring_sources_on_device_bit_identical_2p20(bmo, kind):
    kw = (dict(pos=(0.0, -0.05, 0.0), dir=(0.1, 1.0, 0.0), diameter=20e-3, num_rings=10, num_rays=1 << 20, b1=(1.0, 0.0, 0.0))
          if kind == "collimated" else
          dict(pos=(0.0, 0.0, 0.0), dir=(0.0, 1.0, 0.1), theta=3.0, num_rings=64, num_rays=1 << 20, b1=(1.0, 0.0, 0.0)))
    assert _rays_equal_host(bmo, _make(bmo, kind, kw, False), _make(bmo, kind, kw, True))


@pytest.mark.gpu
def test_disc_on_device_within_ulp_bound(bmo):
    args = ((0.01, -0.05, 0.02), (0.2, 1.0, -0.1), 20e-3, LAM)
    kw = dict(num_rays=1 << 20, e1=(1.0, 0.0, 0.0))
    host = bmo.UniformDiscSource(*args, **kw)
    src = bmo.UniformDiscSource(*args, on_device=True, **kw)
    pos, dirs = src.rays()
    assert _same(dirs, host.dir)
    R = 10e-3
    bound = 4 * 2.0 ** -52 * (np.abs(host.pos) + R)
    err = np.abs(pos - host.pos)
    assert (err <= bound).all(), f"worst {float((err / bound).max()):.3f} of the bound"
    same = int(np.all(pos.view(np.int64) == host.pos.view(np.int64), axis=1).sum())
    print(f"disc 2^20: {same} of {len(pos)} rays bit-identical to the host constructor, worst error {float((err / bound).max()):.3f} of the bound")


def _outputs(res):
    obj, xz = res.spots()
    b = res.beams()
    out = dict(obj=obj, xz=xz, nseg=b["nseg"], status=b["status"], parent=b["parent"], slot=b["slot"],
               info=np.array([res.n_roots, res.n_beams, res.n_segments, res.interactions, res.R, res.waves]))
    if res.keep:
        for k, v in res.segments().items():
            out["seg_" + k] = v
    return out


def _assert_same_outputs(a, b):
    assert a.keys() == b.keys()
    for k in a:
        assert _same(a[k], b[k]), k


def _host_copy(m, src):
    pos, dirs = src.rays()
    return m.RayBundle(pos, dirs[0].copy() if src.uniform_dir else dirs, src.lam, normalize=False)


@pytest.mark.gpu
@pytest.mark.parametrize("collect", [True, False])
def test_trace_device_source_c2_matches_host_copy(bmo, collect):
    from tests import scenes
    sc = scenes.doublet_spot(bmo)
    src = bmo.UniformDiscSource((0.0, -0.05, 0.0), (0.0, 1.0, 0.0), 20e-3, LAM, num_rays=1 << 20, e1=(1.0, 0.0, 0.0), on_device=True)
    host = _host_copy(bmo, src)
    rh = bmo.solve_system_(sc["system"], host, keep_segments=False, collect_spots=collect)
    data_h = sc["spot"].data.copy()
    sc["spot"].empty_()
    rd = bmo.solve_system_(sc["system"], src, keep_segments=False, collect_spots=collect)
    assert not rd.keep
    _assert_same_outputs(_outputs(rh), _outputs(rd))
    if collect:
        assert len(data_h) > 0 and _same(sc["spot"].data, data_h)
    else:
        assert len(data_h) == 0 and len(sc["spot"].data) == 0
    # the same rays through the low-level wrapper, host inputs against the source's device pointers
    n, p, d, u = src.device_arrays()
    dsys = rd.dsys
    a = bmo.trace_rays(dsys, host.pos, host.dir[0], None, keep_segments=False)
    b = bmo.trace_rays(dsys, (p, n), d, None, keep_segments=False, device_inputs=True, uniform_dir=u)
    _assert_same_outputs(_outputs(a), _outputs(b))


def splitter_scene(m):
    """A 45-degree thin beamsplitter with a Spotdetector in the transmitted beam and one on either side of it."""
    bs = m.ThinBeamsplitter(30e-3)
    bs.zrotate3d_(math.radians(45))
    bs.translate3d_((0.0, 0.05, 0.0))
    sds = [m.Spotdetector(20e-3) for _ in range(3)]
    sds[0].translate3d_((0.0, 0.1, 0.0))
    for sd, x in zip(sds[1:], (0.05, -0.05)):
        sd.zrotate3d_(math.radians(90))
        sd.translate3d_((x, 0.05, 0.0))
    return m.System([bs] + sds), sds


@pytest.mark.gpu
@pytest.mark.parametrize("collect", [True, False])
def test_trace_device_source_splitter_keep_segments_matches_host_copy(bmo, collect):
    system, sds = splitter_scene(bmo)
    src = bmo.PointSource((0.0, 0.0, 0.0), (0.0, 1.0, 0.0), 0.05, LAM, num_rings=12, num_rays=1 << 16, b1=(1.0, 0.0, 0.0), on_device=True)
    host = _host_copy(bmo, src)
    rh = bmo.solve_system_(system, host, keep_segments=True, collect_spots=collect)
    data_h = [sd.data.copy() for sd in sds]
    for sd in sds:
        sd.empty_()
    rd = bmo.solve_system_(system, src, keep_segments=True, collect_spots=collect)
    assert rd.keep and rd.n_beams > rd.n_roots        # the splitter made children
    _assert_same_outputs(_outputs(rh), _outputs(rd))
    for sd, dh in zip(sds, data_h):
        assert _same(sd.data, dh)
        assert collect or len(dh) == 0
    if collect:
        assert sum(len(dh) > 0 for dh in data_h) >= 2


@pytest.mark.gpu
def test_trace_device_source_michelson_keep_segments(bmo):
    from tests import scenes
    sc = scenes.michelson(bmo)
    src = bmo.CollimatedSource((0.0, 0.0, 0.0), (0.0, 1.0, 0.0), 2e-3, 632.8e-9, num_rings=5, num_rays=4096, b1=(1.0, 0.0, 0.0), on_device=True)
    host = _host_copy(bmo, src)
    rh = bmo.solve_system_(sc["system"], host, keep_segments=True)
    rd = bmo.solve_system_(sc["system"], src, keep_segments=True)
    assert rd.n_beams > rd.n_roots
    _assert_same_outputs(_outputs(rh), _outputs(rd))
    # a second solve retraces the stored solution (same descriptor = same roots)
    rr = bmo.solve_system_(sc["system"], src, keep_segments=True)
    a, b = _outputs(rd), _outputs(rr)
    for k in ("obj", "xz", "nseg", "status"):
        assert _same(a[k], b[k]), k
    assert all(_same(a[k], b[k]) for k in a if k.startswith("seg_"))


# ---- spot statistics -------------------------------------------------------------------------------------------------
def np_stats(obj, xz, det, window=None, nx=0, nz=0):
    sel = obj == det
    x, z = xz[sel, 0], xz[sel, 1]
    out = dict(hits=int(sel.sum()))
    if out["hits"]:
        cx, cz = x.mean(), z.mean()
        out.update(centroid=(cx, cz), rms=math.sqrt(((x - cx) ** 2 + (z - cz) ** 2).sum() / len(x)),
                   max_r=np.sqrt(x * x + z * z).max(), lo=(x.min(), z.min()), hi=(x.max(), z.max()))
    out["outside"] = 0
    if window is not None:
        xl, xh, zl, zh = window
        inside = (x >= xl) & (x <= xh) & (z >= zl) & (z <= zh)
        out["outside"] = int((~inside).sum())
        if nx:
            i = np.minimum(np.floor((x[inside] - xl) / (xh - xl) * nx), nx - 1).astype(np.int64)
            j = np.minimum(np.floor((z[inside] - zl) / (zh - zl) * nz), nz - 1).astype(np.int64)
            c = np.zeros((nz, nx), np.int64)
            np.add.at(c, (j, i), 1)
            out["counts"] = c
    return out


def _check_stats(got, ref):
    assert got["hits"] == ref["hits"] and got["outside"] == ref["outside"]
    if ref["hits"] == 0:
        for k in ("rms", "max_r"):
            assert math.isnan(got[k])
        assert all(math.isnan(v) for v in got["centroid"] + got["lo"] + got["hi"])
    else:
        assert got["max_r"] == ref["max_r"] and got["lo"] == ref["lo"] and got["hi"] == ref["hi"]
        # relative to the spot's size: a centroid near the origin is a cancelling sum
        for g, r in zip(got["centroid"], ref["centroid"]):
            assert abs(g - r) <= 1e-12 * max(abs(r), ref["max_r"]), (g, r)
        assert abs(got["rms"] - ref["rms"]) <= 1e-12 * ref["rms"], (got["rms"], ref["rms"])
    if "counts" in ref:
        assert np.array_equal(got["counts"], ref["counts"])


def _same_stats(a, b):
    ka = sorted(a)
    return ka == sorted(b) and all(_same(np.asarray(a[k], dtype=np.float64), np.asarray(b[k], dtype=np.float64)) for k in ka)


@pytest.fixture(scope="module")
def c2_result(bmo):
    from tests import scenes
    sc = scenes.doublet_spot(bmo)
    src = bmo.UniformDiscSource((0.0, -0.05, 0.0), (0.0, 1.0, 0.0), 20e-3, LAM, num_rays=1 << 20, e1=(1.0, 0.0, 0.0), on_device=True)
    res = bmo.solve_system_(sc["system"], src, keep_segments=False, collect_spots=False)
    return sc, res


@pytest.mark.gpu
def test_spot_stats_c2_against_numpy(bmo, c2_result):
    sc, res = c2_result
    obj, xz = res.spots()
    det = next(i for i, o in enumerate(res.dsys.flat.objects) if o is sc["spot"])
    ref = np_stats(obj, xz, det)
    assert ref["hits"] > 0.9 * len(obj)
    got = bmo.spot_stats(res, sc["spot"])
    _check_stats(got, ref)
    a = 0.5 * ref["max_r"]
    win = (-a, 0.7 * a, -0.8 * a, a)      # smaller than the spot: some hits fall outside
    ref = np_stats(obj, xz, det, win, 256, 200)
    g1 = bmo.spot_stats(res, sc["spot"], bins=(256, 200), window=win)
    assert ref["outside"] > 0
    _check_stats(g1, ref)
    g2 = bmo.spot_stats(res, det, bins=(256, 200), window=win)
    assert _same_stats(g1, g2)                     # two calls: the same bits
    # the same histogram into a device buffer
    import torch
    from bmo_b200 import _lib as L
    cd = torch.full((200, 256), 7, dtype=torch.int64, device="cuda")
    info = L.bmo_spot_info()
    w = np.array(win)
    L.check(L.lib().bmo_spot_stats(res.h, det, L.ptr(w), 256, 200, C.byref(info), L.ptr(cd.data_ptr()), L.INPUT_DEVICE))
    torch.cuda.synchronize()
    assert np.array_equal(cd.cpu().numpy(), ref["counts"])
    assert info.hits == g1["hits"] and info.rms == g1["rms"] and info.outside == g1["outside"]
    # default window: the detector's face
    hw = sc["spot"].hw
    _check_stats(bmo.spot_stats(res, sc["spot"], bins=64), np_stats(obj, xz, det, (-hw, hw, -hw, hw), 64, 64))


@pytest.mark.gpu
def test_spot_stats_two_detectors_and_empty(bmo):
    system, sds = splitter_scene(bmo)
    src = bmo.PointSource((0.0, 0.0, 0.0), (0.0, 1.0, 0.0), 0.05, LAM, num_rings=12, num_rays=1 << 16, b1=(1.0, 0.0, 0.0), on_device=True)
    res = bmo.solve_system_(system, src, keep_segments=False, collect_spots=False)
    obj, xz = res.spots()
    objs = res.dsys.flat.objects
    hits = []
    for sd in sds:
        det = next(i for i, o in enumerate(objs) if o is sd)
        ref = np_stats(obj, xz, det, (-5e-3, 4e-3, -3e-3, 6e-3), 32, 48)
        got = bmo.spot_stats(res, sd, bins=(32, 48), window=(-5e-3, 4e-3, -3e-3, 6e-3))
        _check_stats(got, ref)
        hits.append(got["hits"])
    assert sum(h > 0 for h in hits) >= 2 and 0 in hits    # transmitted + reflected, and the detector on the wrong side is empty
    assert sum(hits) == int((obj >= 0).sum())


@pytest.mark.gpu
def test_spot_stats_beamlet_result(bmo):
    from tests import scenes
    sc = scenes.doublet_spot(bmo)
    pos, _ = scenes.fibonacci_disc(4096, diameter=15e-3)
    bb = bmo.BeamletBundle.from_params(pos, (0.0, 1.0, 0.0), LAM, w0=0.2e-3)
    res = bmo.solve_system_(sc["system"], bb, collect_spots=False)
    assert res.R == 3
    obj, xz = res.spots()
    assert len(obj) == 3 * res.n_beams
    det = next(i for i, o in enumerate(res.dsys.flat.objects) if o is sc["spot"])
    ref = np_stats(obj, xz, det, (-1e-3, 1e-3, -1e-3, 1e-3), 50, 50)
    assert ref["hits"] > 4096          # waist and divergence rays count too
    _check_stats(bmo.spot_stats(res, sc["spot"], bins=50, window=(-1e-3, 1e-3, -1e-3, 1e-3)), ref)


@pytest.mark.gpu
def test_malformed_descriptors_and_stats_arguments_are_refused(bmo, c2_result):
    from bmo_b200 import _lib as L
    lib = L.lib()
    ctx = L.context(0)

    def create(src, mutate):
        d = L.bmo_source_desc.from_buffer_copy(src.desc)
        d.rings = src.desc.rings
        rings = (L.bmo_source_ring * max(1, d.n_rings)).from_buffer_copy(src._rings)
        if d.n_rings:
            d.rings = C.cast(rings, C.POINTER(L.bmo_source_ring))
        mutate(d, rings)
        h = C.c_void_p()
        rc = lib.bmo_source_create(ctx, C.byref(d), C.byref(h))
        if rc == 0:
            lib.bmo_source_free(h)
        return rc

    col = bmo.CollimatedSource((0.0, -0.05, 0.0), (0.0, 1.0, 0.0), 20e-3, LAM, num_rings=5, num_rays=1000, b1=(1.0, 0.0, 0.0), on_device=True)
    disc = bmo.UniformDiscSource((0.0, -0.05, 0.0), (0.0, 1.0, 0.0), 20e-3, LAM, num_rays=1000, e1=(1.0, 0.0, 0.0), on_device=True)
    assert create(col, lambda d, r: None) == 0 and create(disc, lambda d, r: None) == 0
    bad = [
        (col, lambda d, r: setattr(d, "kind", 7)),
        (col, lambda d, r: setattr(d, "n_rays", 0)),
        (disc, lambda d, r: setattr(d, "n_rays", -5)),
        (col, lambda d, r: d.pos.__setitem__(0, math.nan)),
        (disc, lambda d, r: setattr(d, "radius", math.inf)),
        (col, lambda d, r: r[0].rot.__setitem__(4, math.nan)),
        (col, lambda d, r: setattr(r[1], "first", r[1].first + 1)),
        (col, lambda d, r: setattr(d, "n_rays", d.n_rays + 1)),
        (col, lambda d, r: setattr(r[0], "count", -1)),
    ]
    for src, mutate in bad:
        assert create(src, mutate) == -1
    sc, res = c2_result
    det = next(i for i, o in enumerate(res.dsys.flat.objects) if o is sc["spot"])
    info = L.bmo_spot_info()
    counts = np.zeros(16, np.int64)
    good = np.array([-1e-3, 1e-3, -1e-3, 1e-3])
    for d_obj, win, nx, nz, cnt in [
        (0, None, 0, 0, None),                                   # the doublet is not a Spotdetector
        (99, None, 0, 0, None),
        (-1, None, 0, 0, None),
        (det, np.array([-1e-3, math.nan, -1e-3, 1e-3]), 4, 4, counts),
        (det, np.array([1e-3, -1e-3, -1e-3, 1e-3]), 4, 4, counts),
        (det, None, 4, 4, counts),                                # a histogram needs a window
        (det, good, 0, 4, counts),
        (det, good, 4, -1, counts),
    ]:
        assert lib.bmo_spot_stats(res.h, d_obj, L.ptr(win), nx, nz, C.byref(info), L.ptr(cnt), 0) == -1
    # the context still traces and reduces
    r2 = bmo.solve_system_(sc["system"], col, keep_segments=False, collect_spots=False)
    assert r2.n_beams == 1000 and bmo.spot_stats(r2, sc["spot"])["hits"] > 0
    assert bmo.spot_stats(res, sc["spot"])["hits"] > 0
