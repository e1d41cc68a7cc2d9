"""bench.py's contract: the reference arm (`--impl reference`) runs the compiled reference (the oracle port where the
reference sources are absent) on the host cores and prints ONE JSON line with the keys a reader of the line expects;
without a CUDA device the product arm refuses to run instead of falling back to a CPU path; on the GPU,
`--dump-outputs` writes the accumulators of the timed steps."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

import oracle_lib

ROOT = Path(__file__).resolve().parent.parent


def test_reference_arm_prints_the_contract_line():
    kind = "reference" if oracle_lib.load_ref() is not None else "port"
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "path-tracing throughput" and d["unit"] == "Mpaths/s"
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 1 and d["higher_is_better"] is True
    assert d["vs_baseline"] is None and d["dtype"] == "f32" and d["data"] == "synthetic" and d["scaling"] == "weak"
    assert "configs[1]" in d["config"]["workload"] and d["value"] > 0 and d["ms_per_step"] > 0
    # the line says itself that the CPU leg renders a sample frame, not the 1024x1024 job
    assert d["config"]["same_config"] is False and d["config"]["sample_width"] == 128 and d["config"]["job_width"] == 1024
    assert "128x128 sample frame" in d["config"]["workload"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == kind and cb["cores"] >= 1 and cb["value"] == d["value"] and "128x128" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "Mpaths/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0 and 100 < d["rays_per_path"] < 130   # the reference traces zero-weight children too


def test_product_arm_fails_loudly_without_a_gpu(lib, has_gpu):
    if has_gpu:
        pytest.skip("a GPU is present")
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", "1", "--warmup", "1", "--no-cpu-baseline"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode != 0
    assert not [l for l in r.stdout.splitlines() if l.startswith("{") and '"value"' in l]


@pytest.mark.gpu
def test_dump_outputs_writes_the_accumulators_of_the_timed_steps(tmp_path):
    """`--steps K` timed steps: the dumped count holds exactly the camera paths of the K steps (per pixel it follows
    GridRenderPlane's row mapping, so it is not uniform), and the dumped sums give the image mean the line reports."""
    steps = 2
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", str(steps), "--warmup", "3", "--e2e-steps", "1",
                        "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert d["steps"] == steps
    files = sorted(p.name for p in tmp_path.iterdir())
    assert files == ["count.npy", "sum.npy", "sumsq.npy"]
    assert sum(p.stat().st_size for p in tmp_path.iterdir()) <= 64 << 20
    s, q, c = (np.load(tmp_path / f) for f in ("sum.npy", "sumsq.npy", "count.npy"))
    assert s.dtype == q.dtype == c.dtype == np.float32 and s.shape == q.shape == c.shape == (1024, 1024)
    assert c.sum(dtype=np.float64) == steps * d["config"]["paths_per_step_per_gpu"]
    assert np.isfinite(s).all() and (q >= 0).all() and s.sum() > 0
    assert abs(s.sum(dtype=np.float64) / c.sum(dtype=np.float64) - d["image_mean"]) <= 1e-6 * d["image_mean"]


def test_dump_outputs_samples_frames_above_the_limit(tmp_path, monkeypatch):
    """Frames larger than the limit (the c4 workload's 3840x2160, for one) are written as a seeded pixel sample with its
    flat indices, the same sample on every run, within the limit."""
    import bench

    h, w = 60, 80
    acc = {"sum": np.arange(h * w, dtype=np.float32).reshape(h, w), "sumsq": np.ones((h, w), np.float32),
           "count": np.full((h, w), 3, np.uint32)}
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 4096 + 20 * 1000)
    for d in (tmp_path / "a", tmp_path / "b"):
        bench.dump_outputs(d, acc)
        assert sum(p.stat().st_size for p in d.iterdir()) <= bench.DUMP_LIMIT_BYTES
    a = {n: np.load(tmp_path / "a" / f"{n}.npy") for n in ("sum", "sumsq", "count", "pixel_index")}
    assert a["pixel_index"].dtype == np.float64 and a["sum"].dtype == a["count"].dtype == np.float32
    idx = a["pixel_index"].astype(np.int64)
    assert len(idx) == 1000 and (np.diff(idx) > 0).all() and idx[-1] < h * w
    assert np.array_equal(a["sum"], acc["sum"].reshape(-1)[idx]) and (a["count"] == 3).all()
    assert np.array_equal(a["pixel_index"], np.load(tmp_path / "b" / "pixel_index.npy"))
