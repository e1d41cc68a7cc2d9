"""The reference-facing C++ host classes (ipt_b200/host/device_plugins.hpp): build check on CPU, behaviour on the GPU."""
import json
import shutil
import subprocess
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
HOST = ROOT / "ipt_b200" / "host"


@pytest.fixture(scope="module")
def host_demo(lib):
    subprocess.run(["make", "-C", str(HOST), "check"], check=True, capture_output=True)
    return HOST / "host_demo"


def test_host_classes_build_and_refuse_to_run_without_a_device(host_demo, has_gpu):
    if has_gpu:
        pytest.skip("a GPU is present")
    r = subprocess.run([str(host_demo)], capture_output=True, text=True)
    out = json.loads(r.stdout)
    assert r.returncode == 3 and "no CPU fallback" in out["error"]


def test_host_classes_compile_against_the_reference_headers():
    import oracle_lib

    if oracle_lib.REF_SRC is None or not (oracle_lib.REF_SRC / "src" / "tracer_interfaces.h").exists():
        pytest.skip("no reference sources here (IPT_REFERENCE)")
    r = subprocess.run(["make", "-C", str(HOST), "check-reference", f"REF={oracle_lib.REF_SRC}"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert "compile against the reference's own tracer_interfaces.h" in r.stdout


@pytest.mark.gpu
@pytest.mark.parametrize("scene", ["box", "cornell"])
def test_render_sample_through_the_cpp_interfaces(scene, host_demo, oracle, tmp_path):
    import oracle_lib
    from ipt_b200 import capi

    png = tmp_path / "result.png"
    r = subprocess.run([str(host_demo), scene, "4", str(png)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    multi, session, first, last = r.stdout.strip().splitlines()
    multi = json.loads(multi)   # ipt_b200::render_sample(scene, plane, params, devices): same passes on two device slots
    session = json.loads(session)  # ipt_b200::ProgressiveSession: the interactive loop headless, checkpoint / resume in C++
    assert session["session_spp"] == [8, 8, 2] and session["session_counters_equal"] == 64 * 64 and session["session_max_rel"] < 2e-5
    assert session["session_refused"] == 1 and abs(session["session_cutoff"] - 1.01 * 2.0) < 1e-5   # wheel: sqrt(2)^2
    stage = json.loads(first)
    assert stage["display_max"] == 1.0 and stage["orbit_round_trip_error"] < 1e-5   # DevicePlane::display, DeviceCamera::orbit
    from test_output_host import decode_png_gray8
    img = decode_png_gray8(png.read_bytes())                                         # DevicePlane::save == Gui::save
    assert img.shape == (96, 96) and img.max() == 255 and len(np.unique(img)) > 30
    out = json.loads(last)
    assert out["paths"] == 96 * 96 * 4 and out["rays"] > out["paths"]
    assert multi["multi_paths"] == out["paths"] and multi["multi_rays"] == out["rays"]
    assert multi["multi_counters_equal"] == 96 * 96 and multi["multi_max_rel"] < 2e-5     # float atomics order only
    sd = capi.SceneDescription(scene)
    p = capi.default_params(width=96, height=96, pass_count=4)
    o = oracle.render(sd.ptr, p, oracle_lib.RNG_PHILOX, 0)
    mean = o["sum"].sum() / o["counters"].sum()
    assert out["count_device_plane"] == 96 * 96 * 4
    assert abs(out["mean_device_plane"] - mean) < 0.02 * mean          # same Philox stream; ulp-level flips only
    assert abs(out["mean_foreign_plane"] * out["cells_foreign_plane"] / (96 * 96) - mean) < 0.05 * mean
    # single-ray virtuals against the oracle
    co, cd = oracle.camera_rays(sd.ptr, np.array([[0.5, 0.3]], np.float32))
    t = oracle.trace_batch(sd.ptr, co, cd)
    assert out["hit"] == 1
    assert np.allclose(out["hit_pos"], t["pos"][0], atol=0) and np.allclose(out["hit_normal"], t["normal"][0], atol=0)
    assert abs(out["sdf_value_at_normal"] - 1 / np.pi) < 1e-6 or scene == "cornell"
    assert out["sdf_sample_dot_normal"] >= 0
    assert out["light_hit"] in (0, 1)
    lv = oracle.light_ddf_value(sd.ptr, [0.2, -0.8, -1.0], [[0, 0, 1]])[0]
    assert abs(out["light_ddf_value"] - lv) <= 1e-4 * max(lv, 1e-6)


def test_dropin_binary_builds_against_reference_headers(lib):
    import oracle_lib

    if oracle_lib.REF_SRC is None or not oracle_lib.REF_SRC.exists():
        pytest.skip("no reference sources here (IPT_REFERENCE)")
    exe = oracle_lib.build_dropin()
    assert exe is not None and exe.exists()


@pytest.mark.gpu
def test_reference_estimator_runs_on_ipt_b200_objects(lib):
    """oracle/ab_dropin.cpp: the reference's compiled ray_power_recursive calls Geometry::traceRay /
    Lighting::traceRayToLight / distributionInPoint / Ddf::sample / Ddf::value on ipt_b200's host objects (every call
    evaluated on the GPU): single-ray results equal the reference's own objects to the bit, the estimate agrees
    statistically."""
    import oracle_lib

    exe = oracle_lib.build_dropin()
    if exe is None:
        pytest.skip("oracle/_ref/ab_dropin not available (built where IPT_REFERENCE names the reference sources)")
    r = subprocess.run([str(exe), "box", "1500"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    out = json.loads(r.stdout.strip().splitlines()[-1])
    assert out["geometry_equal"] == out["rays"] and out["geometry_hits"] > 0.5 * out["rays"]
    assert out["light_equal"] == out["rays"] and out["light_hits"] > 50
    assert abs(out["mean_reference_objects"] - out["mean_ipt_b200_objects"]) < 4 * out["standard_error"] + 1e-4
    assert out["mean_reference_objects"] > 0
    # the reference's GeometrySphereInBox + SimpleCamera + GridRenderPlane through ipt_b200::render_sample == DevicePlane
    assert out["grid_cells"] > 0.9 * 80 * 80 and out["grid_counters_equal"] == 80 * 80
    assert out["grid_cells_equal"] == out["grid_cells"] and out["grid_max_rel"] <= 1e-5
    assert out["grid_max_rel_two_devices"] < 2e-5
    assert abs(out["grid_max_value"] - out["device_max_value"]) <= 1e-5 * out["device_max_value"]
