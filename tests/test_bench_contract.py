"""bench.py prints exactly one JSON line on stdout with the keys the driver reads.  The reference arm runs on the CPU
(oracle port on the host cores, bounded sample); our arm needs the GPU."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
             "data", "config", "e2e"}


def _run(*args):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines            # one JSON line, nothing else on stdout
    return json.loads(lines[0])


def test_reference_arm_line():
    d = _run("--impl", "reference", "--steps", "1", "--warmup", "0")
    assert BASE_KEYS <= set(d) and d["impl"] == "reference"
    assert d["metric"] == "ray-surface interactions/s" and d["unit"] == "interactions/s" and d["higher_is_better"] is True
    assert d["config"]["workload"].startswith("C2") and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["value"] > 0


@pytest.mark.gpu
def test_our_arm_line():
    d = _run("--steps", "3", "--warmup", "3", "--no-detector", "--no-extras", "--no-cpu-baseline", "--rays", str(1 << 18))
    assert BASE_KEYS <= set(d) and "impl" not in d
    assert d["dtype"] == "f64" and d["scaling"] == "weak" and d["vs_baseline"] is None and d["n_gpus"] == 1
    assert d["gpu_launches"] > 0
    r = d["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(r) and 0 < r["frac"] < 1
    e = d["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and e["value"] < d["value"]
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])


def test_dump_sample_is_fixed_and_bounded(tmp_path):
    import bench
    assert np.array_equal(bench.sample_index(10, 16, seed=1), np.arange(10))
    a, b = bench.sample_index(1 << 22, 1 << 12, seed=2), bench.sample_index(1 << 22, 1 << 12, seed=2)
    assert np.array_equal(a, b) and len(np.unique(a)) == 1 << 12 and np.all(np.diff(a) > 0) and a[-1] < 1 << 22
    with pytest.raises(SystemExit):
        bench.dump_outputs(str(tmp_path / "big"), {"x": np.zeros(bench.DUMP_BYTES // 8 + 1)})
    assert not (tmp_path / "big").exists()


@pytest.mark.gpu
def test_dump_outputs(tmp_path, orc):
    """--dump-outputs with more rays than the per-ray cap: a fixed sample of the last step's outputs, both trace legs agreeing
    with each other and, on a few rays, with the CPU oracle bit for bit."""
    n = (1 << 20) + 4096
    out = tmp_path / "out"
    _run("--steps", "2", "--warmup", "3", "--no-extras", "--no-cpu-baseline", "--rays", str(n), "--c3-side", "16", "--c3-pixels", "256",
         "--dump-outputs", str(out))
    g = {f.stem: np.load(f) for f in out.glob("*.npy")}
    assert set(g) == {"spot_xz", "spot_object", "nseg", "interactions", "ray_index", "e2e_spot_xz", "e2e_interactions",
                      "detector_field", "detector_pixel_index"}
    assert all(a.dtype in (np.float32, np.float64) for a in g.values()) and sum(a.nbytes for a in g.values()) <= 64 << 20
    idx = g["ray_index"].astype(np.int64)
    assert len(idx) == 1 << 20 and np.all(np.diff(idx) > 0) and idx[-1] < n
    assert np.array_equal(g["spot_xz"], g["e2e_spot_xz"], equal_nan=True) and g["interactions"][0] == g["e2e_interactions"][0] > 0
    assert g["detector_field"].shape == (256 * 256, 2) and np.array_equal(g["detector_pixel_index"], np.arange(256 * 256))
    assert np.abs(g["detector_field"]).max() > 0
    import bench
    from tests import scenes
    pos, d = bench.rays_for_rank(0, n)
    k = idx[::16384]
    osc = scenes.doublet_spot_oracle()
    ref = orc.bulk_trace_rays(osc["system"], np.ascontiguousarray(pos[k]), np.ascontiguousarray(d[k]), bench.LAMBDA, want_segments=False, spot=osc["spot"])
    assert np.array_equal(ref["spot"], g["spot_xz"][::16384], equal_nan=True)
