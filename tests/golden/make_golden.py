"""Generates the golden fixtures under tests/golden/ from the UNMODIFIED reference (oracle/_ref/libipt_ref.so,
compiled from /root/reference by `make -C oracle ref`). Run here, where /root/reference exists; the fixtures travel to
the GPU box, the reference sources do not.

    python tests/golden/make_golden.py

Fixtures:
  kat_<scene>.npz    bit-exact known answers of the reference's own functions on a fixed ray batch:
                     Camera::sampleRay, Geometry::traceRay (hit, position, normal, curvature),
                     Lighting::traceRayToLight (hit, position, power), ray_power_preview, camera fields, light fields.
  ddf_kat.npz        Ddf::value known answers (src/libddf/test_ddf.cpp:181-223 and a direction sweep),
                     AreaLight KAT (src/lighting/test_lighting.cpp:130-144), GridRenderPlane::addRay KAT.
  output_kat.npz     the output stage (src/gui.cpp): normalize(), glare(), the pixel bytes of Gui::save and the arrow-key
                     camera orbit on two input images (`python tests/golden/make_golden.py output`).
  image_<scene>.npz  sum / sumsq / count of the reference estimator (ray_power_recursive, n_rays=16, depth_max=4)
                     over P passes at WxH with libc drand48, merged over forked workers seeded 1000+rank.
  pin_live.npz       what the bit-exact pins of tests/test_oracle_pin_live.py and tests/test_output_host.py compare the
                     oracle with (`python tests/golden/make_golden.py pins`): whole drand48 passes (sha256 of pixels and
                     counters, ray count, 4096 sampled pixels), mixture / DDF / light-DDF sample sequences, and the
                     output stage on random ragged images. Recorded from the compiled reference. Where its sources are
                     not at hand, `pins --from-oracle` records the oracle instead, which those pins held bit-identical
                     to the reference; the file says which in `source`, and wherever the reference is built the tests
                     check every stored array against it live.
"""
from __future__ import annotations

import multiprocessing as mp
import sys
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE.parent))
sys.path.insert(0, str(HERE.parent.parent))

IMAGE_JOBS = {  # scene: (W, H, passes). 2048 passes: SURVEY 8d's tolerances (99.7 % within 3 sigma, |mean z| < 0.1, block relRMSE
    # < 1 %) need a golden whose own noise is well below them; the sizes keep each job to a few minutes on 8 cores.
    "box": (96, 96, 2048),
    "cornell": (96, 96, 2048),
    "corner": (96, 96, 2048),
    "openspheres": (96, 96, 2048),
    # cheap scenes with rare bright paths: many more passes, so that the golden's own per-pixel variance estimates are sound
    "fractal": (96, 96, 65536),
    "square": (96, 96, 32768),
    "smallpt": (64, 64, 2048),
    "mixedlights": (64, 64, 2048),
    # many lights: CollectionLighting::distributionInPoint is O(L^2) per hit in the reference (SURVEY S11), 29 paths/s per
    # core at L = 1024 -> a coarse frame of the whole view
    "lightgrid:32x32": (20, 20, 768),
}
WORKERS = 8


def _image_worker(args):
    scene, W, H, passes, rank = args
    import oracle_lib

    ref = oracle_lib.load_ref()
    h = ref.scene(scene)
    ref.set_tree(16, 4)
    ref.seed(1000 + rank)
    r = ref.render(h, passes, W, H, verbatim=False)
    return r["sum"], r["sumsq"], r["counters"], r["rays"]


def make_images():
    only = sys.argv[2:] if len(sys.argv) > 2 else None
    for key, (W, H, passes) in IMAGE_JOBS.items():
        if only and key not in only:
            continue
        scene = key.split("@")[0]
        per = passes // WORKERS
        with mp.get_context("fork").Pool(WORKERS) as pool:
            parts = pool.map(_image_worker, [(scene, W, H, per, k) for k in range(WORKERS)])
        s = sum(p[0] for p in parts)
        q = sum(p[1] for p in parts)
        c = sum(p[2] for p in parts)
        rays = sum(p[3] for p in parts)
        np.savez_compressed(HERE / f"image_{key.replace('@', '_').replace(':', '_')}.npz", sum=s.astype(np.float32), sumsq=q.astype(np.float32), count=c.astype(np.uint32),
                            passes=per * WORKERS, rays=rays, n_rays=16, depth_max=4)
        print(scene, "mean", s.sum() / c.sum(), "rays/path", rays / (W * H * per * WORKERS))


def make_kats():
    import oracle_lib
    from helpers import SCENES_ANALYTIC, ray_batch

    ref = oracle_lib.load_ref()
    for scene in SCENES_ANALYTIC + ["lightgrid:4x5"]:
        h = ref.scene(scene)
        o, d, xy = ray_batch(scene, lambda xy: ref.camera_rays(h, xy), n_cam_side=24, n_random=1500)
        co, cd = ref.camera_rays(h, xy)
        g = ref.trace_geometry(h, o, d)
        l = ref.trace_light(h, o, d)
        lights = np.stack([ref.light_fields(h, i) for i in range(ref.light_count(h))])
        preview = ref.preview_batch(h, o, d)
        np.savez_compressed(HERE / f"kat_{scene.replace(':', '_')}.npz", xy=xy, cam_o=co, cam_d=cd, o=o, d=d, hit=g["hit"], pos=g["pos"],
                            normal=g["normal"], curvature=g["curvature"], lhit=l["hit"], lpos=l["pos"], lpower=l["power"],
                            camera=ref.camera_fields(h), lights=lights, preview=preview)
        print(scene, "rays", len(o), "hits", int(g["hit"].sum()), "light hits", int(l["hit"].sum()))


def make_ddf_kat():
    import oracle_lib

    ref = oracle_lib.load_ref()
    rng = np.random.default_rng(3)
    v = rng.normal(size=(512, 3)).astype(np.float32)
    v /= np.linalg.norm(v, axis=1, keepdims=True).astype(np.float32)
    fixed = np.array([[0, 0, 1], [1, 0, 0], [0, 0, -1], [0, 1, 0], [-1, 0, 0]], np.float32)  # test_ddf.cpp:185-215 directions
    dirs = np.concatenate([fixed, v]).astype(np.float32)
    out = {"dirs": dirs}
    for kind, nm in [(0, "spherical"), (1, "upperhalf"), (2, "cosine"), (40, "power40")]:
        out[nm] = ref.ddf_value(kind, dirs)
    tos = np.array([[0, 0, 1], [0, 0, -1], [1, 0, 0], [0, -1, 0], [0.6, 0.0, 0.8], [-0.48, 0.6, -0.64]], np.float32)
    out["tos"] = tos
    out["cosine_rotated"] = np.stack([ref.ddf_value(2, dirs, to=t) for t in tos])
    out["power40_rotated"] = np.stack([ref.ddf_value(40, dirs, to=t) for t in tos])
    # AreaLight KAT (src/lighting/test_lighting.cpp:130-144)
    area, hit, sp = ref.arealight([1, 1, 1], [-1, -1, -1], [0, -1, 0], 4.0, False, [0, 0, 0.1], [1.1, 0, 0])
    out["arealight"] = np.array([area, float(hit), sp], np.float32)
    area, hit, sp = ref.arealight([0, 0, 1], [1, 0, 0], [0, 1, 0], 2.0, True, [0.2, 0.2, 0], [0, 0, 1])  # back face: miss
    out["arealight_tri_back"] = np.array([area, float(hit), sp], np.float32)
    area, hit, sp = ref.arealight([0, 0, 1], [0, 1, 0], [1, 0, 0], 2.0, True, [0.2, 0.2, 0], [0, 0, 1])
    out["arealight_tri_front"] = np.array([area, float(hit), sp], np.float32)
    # GridRenderPlane::addRay KAT incl. the row mapping quirk (SURVEY S5)
    x = rng.random(4000).astype(np.float32); y = rng.random(4000).astype(np.float32); val = rng.random(4000).astype(np.float32)
    pix, cnt, mx = ref.plane_addray(16, 12, x, y, val)
    out.update(plane_x=x, plane_y=y, plane_v=val, plane_pixels=pix, plane_counters=cnt, plane_max=np.float32(mx))
    np.savez_compressed(HERE / "ddf_kat.npz", **out)
    print("ddf kat", {k: np.asarray(vv).shape for k, vv in out.items()})


def output_inputs():
    """Input images of the output-stage KAT (also used by the GPU tests): a synthetic HDR-like image with ragged size and the
    committed reference render of the box scene (light visible -> real glare sources)."""
    rng = np.random.default_rng(5)
    a = (rng.random((48, 70)).astype(np.float32) ** 6 * np.float32(4.0)).astype(np.float32)
    a[rng.random(a.shape) < 0.25] = 0
    g = np.load(HERE / "image_box.npz")
    b = (g["sum"] / np.maximum(g["count"], 1)).astype(np.float32)
    b = np.ascontiguousarray(b[::2, 1::2][:61])  # 61x64 subsample keeps the bright light pixels
    return {"synthetic": a, "box": b}


def make_output_kat():
    """Output stage (src/gui.cpp): normalize(), glare(), Gui::save bytes and the arrow-key camera orbit, from the compiled reference."""
    import oracle_lib

    ref = oracle_lib.load_ref()
    out = {}
    for name, img in output_inputs().items():
        out[f"{name}_image"] = img
        out[f"{name}_normalize"] = ref.image_normalize(img)
        out[f"{name}_bytes"] = ref.image_save_bytes(img)
        cut = [1.01, 0.25] if name == "synthetic" else [1.01, float(np.float32(img.max()) * np.float32(0.5))]
        out[f"{name}_cutoffs"] = np.array(cut, np.float32)
        out[f"{name}_glare"] = np.stack([ref.image_glare(img, c) for c in np.array(cut, np.float32)])
        print(name, img.shape, "bright", [(img > c).sum() for c in cut])
    keys = np.array([0, 0, 2, 1, 3, 3, 1, 1, 2, 0], np.int32)
    cam = np.zeros((len(keys) + 1, 4, 3), np.float32)
    pos, d = np.array([0.0, -3.0, 0.1], np.float32), np.array([0.0, 0.8111071, -0.5848977], np.float32)
    cam[0, 0], cam[0, 1] = pos, d
    for i, k in enumerate(keys):
        cam[i + 1] = ref.camera_orbit(cam[i, 0], cam[i, 1], int(k))
    out["orbit_keys"], out["orbit_cameras"] = keys, cam
    np.savez_compressed(HERE / "output_kat.npz", **out)


def make_pins():
    import oracle_lib
    import test_oracle_pin_live as P
    import test_output_host as O

    ref = oracle_lib.load_ref()
    if ref is None and "--from-oracle" not in sys.argv:
        raise SystemExit("the compiled reference (oracle/_ref/libipt_ref.so) is not built; `pins --from-oracle` records the oracle")
    side, chk = ("ref", ref) if ref is not None else ("oracle", oracle_lib.load_oracle())
    records = {P.pass_key(*c): P.pass_record(side, chk, *c) for c in P.PASS_CASES}
    records.update({f"mix_{s}": P.mix_record(side, chk, s) for s in P.MIX_SCENES})
    records.update({f"ddf_{k}": P.ddf_record(side, chk, k) for k in P.DDF_KINDS})
    records.update({f"light_{s}": P.light_record(side, chk, s) for s in P.LIGHT_SCENES})
    records["output"] = O.output_record(chk)
    out = {f"{key}__{k}": v for key, rec in records.items() for k, v in rec.items()}
    out["source"] = np.array("reference" if ref is not None else "oracle")
    np.savez_compressed(HERE / "pin_live.npz", **out)
    print("pin_live.npz:", len(out), "arrays from the", out["source"])


if __name__ == "__main__":
    what = sys.argv[1] if len(sys.argv) > 1 else "all"
    if what in ("all", "kats"):
        make_kats()
        make_ddf_kat()
    if what in ("all", "images"):
        make_images()
    if what in ("all", "kats", "output"):
        make_output_kat()
    if what in ("all", "pins"):
        make_pins()
