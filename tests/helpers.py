"""Shared input generators for the parity tests."""
from __future__ import annotations

from pathlib import Path

import numpy as np

SCENES_REFERENCE = ["box", "fractal", "smallpt", "square", "corner", "openspheres"]
SCENES_ANALYTIC = SCENES_REFERENCE + ["cornell", "mixedlights"]

# (box centre, half extent) of the region secondary rays start from, per scene
REGION = {
    "box": ((0, 0, 0), 1.0), "mixedlights": ((0, 0, 0), 1.0), "cornell": ((0, 0, 0), 1.0), "corner": ((0, 0, 0), 1.0), "square": ((0, 0, -0.5), 1.0),
    "openspheres": ((0, 0, -0.6), 0.6), "fractal": ((0, 0, 0), 2.5), "smallpt": ((50, 40, 80), 45.0),
}


def unit_dirs(rng, n):
    v = rng.normal(size=(n, 3)).astype(np.float32)
    v /= np.linalg.norm(v, axis=1, keepdims=True).astype(np.float32)
    return v.astype(np.float32)


def ray_batch(scene_name, camera_rays_fn, n_cam_side=96, n_random=20000, seed=7):
    """A fixed ray batch: jittered camera rays over the whole frame + random rays inside the scene volume +
    rays starting ON surfaces-ish (points on the unit box walls) to exercise the epsilon branches."""
    rng = np.random.default_rng(seed)
    ix, iy = np.meshgrid(np.arange(n_cam_side), np.arange(n_cam_side))
    xy = np.stack([(ix.ravel() + rng.random(ix.size)) / n_cam_side, (iy.ravel() + rng.random(iy.size)) / n_cam_side], 1).astype(np.float32)
    xy = np.minimum(xy, np.float32(0.99999994))
    co, cd = camera_rays_fn(xy)
    c, h = REGION.get(scene_name.split(":")[0], ((0, 0, 0), 1.0))
    o = (np.asarray(c, np.float32) + (rng.random((n_random, 3)).astype(np.float32) * 2 - 1) * np.float32(h)).astype(np.float32)
    d = unit_dirs(rng, n_random)
    # axis-aligned and wall-grazing cases
    o2 = o[:2000].copy()
    o2[:, 2] = np.float32(-1.0)
    d2 = unit_dirs(rng, len(o2))
    d3 = np.zeros((600, 3), np.float32)
    for a in range(3):
        d3[a * 200:(a + 1) * 200, a] = np.where(rng.random(200) < 0.5, -1, 1)
    o3 = o[:600]
    d3 = d3[: len(o3)]
    return np.concatenate([co, o, o2, o3]), np.concatenate([cd, d, d2, d3]), xy


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def oracle_render_parallel(scene, passes, seed, use_bvh=0, workers=None, timeout=900, **kw):
    """The oracle's Philox-mode render (test infrastructure: the CPU checker) of `passes` passes, split into contiguous pass
    ranges over single-threaded worker PROCESSES started from scratch (tests/oracle_worker.py; a fork of a process that has
    initialised CUDA is not safe). Philox counters are keyed by (pixel, pass, node), so the ranges are disjoint streams and
    the merged accumulators equal a single render. Returns dict(sum, sumsq, count, rays)."""
    import json
    import os
    import subprocess
    import sys
    import tempfile
    from pathlib import Path

    workers = max(1, min(workers or (os.cpu_count() or 1), passes))
    base, extra = divmod(passes, workers)
    worker = str(Path(__file__).resolve().parent / "oracle_worker.py")
    with tempfile.TemporaryDirectory() as tmp:
        procs, begin = [], 0
        for r in range(workers):
            n = base + (1 if r < extra else 0)
            out = os.path.join(tmp, f"part{r}.npz")
            procs.append((subprocess.Popen([sys.executable, worker, scene, json.dumps(kw), str(seed), str(begin), str(n), str(use_bvh), out],
                                           stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True), out))
            begin += n
        parts = []
        try:
            for pr, out in procs:
                log, _ = pr.communicate(timeout=timeout)
                assert pr.returncode == 0, log[-2000:]
                parts.append(dict(np.load(out)))
        finally:
            for pr, _ in procs:
                if pr.poll() is None:
                    pr.kill()
    return dict(sum=sum(p["sum"] for p in parts), sumsq=sum(p["sumsq"] for p in parts), count=sum(p["count"] for p in parts),
                rays=int(sum(int(p["rays"]) for p in parts)))


def block_sums(a, block):
    """Sums of block x block cells (frames whose sides are multiples of `block`)."""
    H, W = a.shape
    return a.reshape(H // block, block, W // block, block).sum((1, 3))


# ---------------------------------------------------------------------------------------------------------------------
# stored copies of the compiled reference's outputs (tests/golden/pin_live.npz, made by make_golden.py `pins`)
# ---------------------------------------------------------------------------------------------------------------------
PINS = Path(__file__).resolve().parent / "golden" / "pin_live.npz"


def digest(a):
    """sha256 of an array's bytes: bit-exact equality of frames too large to store."""
    import hashlib

    return np.array(hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest())


def assert_same_record(got: dict, want: dict, what=""):
    """Bit-exact equality of two records (same keys, dtypes, shapes and bytes)."""
    assert sorted(got) == sorted(want), (what, sorted(got), sorted(want))
    for k in want:
        a, b = np.asarray(got[k]), np.asarray(want[k])
        assert a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes(), (what, k)


def reference_record(pins, ref, key: str, from_ref):
    """What the compiled reference gives for `key`. Where the reference is built (`ref` not None) it is run live and the
    stored copy must equal it; elsewhere the stored copy stands in for it."""
    stored = {k[len(key) + 2:]: pins[k] for k in pins.files if k.startswith(key + "__")}
    assert stored, f"{key} missing from {PINS.name}: rerun `python tests/golden/make_golden.py pins`"
    if ref is None:
        return stored
    live = {k: np.asarray(v) for k, v in from_ref(ref).items()}
    assert_same_record(stored, live, f"stored {key} vs the live reference")
    return live


# ---------------------------------------------------------------------------------------------------------------------
# scenes built in Python on top of a sample scene
# ---------------------------------------------------------------------------------------------------------------------
def custom_scene(base="box", prims=None, lights=None, materials=None, triangles=None, triangle_material=None):
    """A library-owned description of `base` with some of its arrays replaced by Python-built ones (kept alive by the
    description)."""
    from ipt_b200 import capi

    sd = capi.SceneDescription(base)
    keep = []
    if prims is not None:
        arr = (capi.Prim * len(prims))(*prims)
        sd.desc.prims, sd.desc.n_prims = arr, len(prims)
        keep.append(arr)
    if lights is not None:
        arr = (capi.Light * len(lights))(*lights)
        sd.desc.lights, sd.desc.n_lights = arr, len(lights)
        keep.append(arr)
    if materials is not None:
        arr = (capi.Material * len(materials))(*materials)
        sd.desc.materials, sd.desc.n_materials = arr, len(materials)
        keep.append(arr)
    if triangles is not None:
        tris = np.ascontiguousarray(triangles, np.float32).reshape(-1, 9)
        sd.desc.triangles, sd.desc.n_triangles = tris.ctypes.data_as(capi.f32p), tris.shape[0]
        keep.append(tris)
    if triangle_material is not None:
        sd.desc.triangle_material = triangle_material
    sd._keep = keep
    return sd


def make_light(kind, position, x_axis=(0, 0, 0), y_axis=(0, 0, 0), radius=0.0, power=1.0):
    from ipt_b200 import capi

    l = capi.Light()
    l.kind = kind
    l.position[:] = [float(v) for v in position]; l.x_axis[:] = [float(v) for v in x_axis]; l.y_axis[:] = [float(v) for v in y_axis]
    l.radius = radius; l.power = power
    return l
