"""GPU parity tests proper: the CUDA path, called through the C ABI, against the CPU oracle on the same inputs.

Bar (BASELINE.json north_star): hit primitive IDs bit-exact, hit distances within 1e-5 relative (we require
bit-exact), per-pixel radiance within float tolerance when both sides draw the same Philox numbers.
"""
import numpy as np
import pytest

import oracle_lib
from helpers import SCENES_ANALYTIC, bits, custom_scene, ray_batch
from ipt_b200 import capi

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def scenes(lib):
    cache = {}

    def get(name):
        if name not in cache:
            sd = capi.SceneDescription(name)
            cache[name] = (sd, capi.Scene(sd))
        return cache[name]

    yield get
    for sd, sc in cache.values():
        sc.close()


@pytest.mark.parametrize("name", SCENES_ANALYTIC)
def test_camera_rays_bit_exact(name, scenes, oracle):
    sd, sc = scenes(name)
    rng = np.random.default_rng(1)
    xy = rng.random((50000, 2)).astype(np.float32)
    o_g, d_g = sc.camera_rays(xy)
    o_c, d_c = oracle.camera_rays(sd.ptr, xy)
    assert np.array_equal(bits(o_g), bits(o_c))
    assert np.array_equal(bits(d_g), bits(d_c))


@pytest.mark.parametrize("name", SCENES_ANALYTIC + ["lightgrid:4x5"])
def test_trace_batch_bit_exact(name, scenes, oracle):
    """Primary + secondary ray batch: primitive id, t, nearest light, light hit position and the
    light-vs-surface decision of main.cpp:111-128 are all bit-identical to the oracle."""
    sd, sc = scenes(name)
    o, d, _ = ray_batch(name, lambda xy: oracle.camera_rays(sd.ptr, xy))
    g = sc.trace_batch(o, d)
    c = oracle.trace_batch(sd.ptr, o, d)
    assert (c["prim"] != capi.IPT_NO_HIT).sum() > 1000, "degenerate batch"
    assert np.array_equal(g["prim"], c["prim"])
    assert np.array_equal(bits(g["t"]), bits(c["t"]))
    assert np.array_equal(g["light"], c["light"])
    assert np.array_equal(bits(g["light_pos"]), bits(c["light_pos"]))
    assert np.array_equal(g["outcome"], c["outcome"])


@pytest.mark.parametrize("name", ["smallpt", "box", "cornell", "fractal", "openspheres"])
def test_rays_starting_on_surfaces_bit_exact(name, scenes, oracle):
    """Three generations of rays that START on a surface (the hit point of the previous generation, random directions in
    the hemisphere of its normal): the regime every secondary ray of a render lives in. GeometrySmallPt's radius-1000
    spheres with eps = 1e-4 (GeometrySmallPt.cpp:17-22) make 11 % of such rays hit the very wall they start on, decided by
    the float rounding of the start point; the device agrees with the oracle bit for bit there too."""
    sd, sc = scenes(name)
    rng = np.random.default_rng(3)
    o, d = oracle.camera_rays(sd.ptr, rng.random((20000, 2)).astype(np.float32))
    first = oracle.trace_batch(sd.ptr, o, d)
    hit = first["outcome"] == 1
    pos, nrm = first["pos"][hit], first["normal"][hit]
    assert len(pos) > 1000
    self_hits = 0
    for generation in range(3):
        v = rng.normal(size=pos.shape).astype(np.float32)
        v /= np.linalg.norm(v, axis=1, keepdims=True).astype(np.float32)
        flip = (v * nrm).sum(1) < 0
        v[flip] = -v[flip]
        v = np.ascontiguousarray(v, np.float32)
        g = sc.trace_batch(pos, v)
        c = oracle.trace_batch(sd.ptr, pos, v)
        assert np.array_equal(g["prim"], c["prim"]) and np.array_equal(bits(g["t"]), bits(c["t"]))
        assert np.array_equal(g["outcome"], c["outcome"]) and np.array_equal(g["light"], c["light"])
        self_hits += int(((c["t"] < 1e-2) & (c["outcome"] == 1)).sum())
        ok = c["outcome"] == 1
        pos, nrm = c["pos"][ok], c["normal"][ok]
    if name == "smallpt":
        assert self_hits > 1000  # the self-intersection regime is really exercised


def _render_pair(sd, sc, oracle, **kw):
    p = capi.default_params(**kw)
    s, q, cnt, st = sc.render_host(p)
    o = oracle.render(sd.ptr, p, oracle_lib.RNG_PHILOX, 0)
    return p, s, q, cnt, st, o


@pytest.mark.parametrize("name,res", [("box", 96), ("cornell", 96), ("corner", 64), ("square", 64), ("smallpt", 64),
                                       ("fractal", 64), ("openspheres", 64), ("lightgrid:3x3", 48)])
def test_two_level_render_matches_oracle_per_pixel(name, res, scenes, oracle):
    """depth_max=2, schedule 16/8: camera ray, first hit, 16 mixture samples, their trace and emission. Both sides draw
    the same Philox numbers, every intersection input up to the first hit is bit-identical, so pixels agree to float
    rounding. (Deeper levels start from directions that differ in the last ulp -- CUDA vs glibc sin/cos -- and the
    reference's box-plane test `abs(point.x) > 1.0f` on the plane's own axis (geometric_utils.cpp:18) flips on such
    differences, so deeper trees are compared statistically below.)"""
    sd, sc = scenes(name)
    p, s, q, cnt, st, o = _render_pair(sd, sc, oracle, width=res, height=res, pass_count=2, depth_max=2, schedule=[16, 8],
                                       flags=capi.FLAG_KEEP_ZERO_WEIGHT)
    assert np.array_equal(cnt.astype(np.uint64), o["counters"])
    assert st.paths == res * res * 2
    # sum and sumsq (what checkpoints and bench.py --dump-outputs carry) against the oracle's double accumulators; a square
    # doubles relative differences, hence twice the bound on the sumsq total
    for got, ref, total in ((s, o["sum"], 1e-4), (q, o["sumsq"], 2e-4)):
        scale = max(ref.max(), 1e-12)
        err = np.abs(got - ref) / scale
        assert (err > 1e-5).mean() < 4e-3, f"{(err > 1e-5).sum()} pixels differ"
        assert abs(got.sum() - ref.sum()) <= total * max(ref.sum(), 1e-9)
    assert abs(int(st.rays) - int(o["rays"])) <= 2e-4 * o["rays"] + 2
    assert st.rays_at_depth[0] == o["rays_at_depth"][0] == res * res * 2


def test_gui_plane_two_level_render_matches_oracle_per_pixel(scenes, oracle):
    """IPT_PLANE_GUI (Gui::addRay's cell mapping, gui.cpp:168-172) through the whole render: counters, sum and sumsq per
    cell against the oracle, which maps its samples the same way."""
    sd, sc = scenes("cornell")
    p, s, q, cnt, st, o = _render_pair(sd, sc, oracle, width=64, height=48, pass_count=2, depth_max=2, schedule=[16, 8],
                                       plane_mode=capi.PLANE_GUI, flags=capi.FLAG_KEEP_ZERO_WEIGHT)
    assert np.array_equal(cnt.astype(np.uint64), o["counters"])
    for got, ref, total in ((s, o["sum"], 1e-4), (q, o["sumsq"], 2e-4)):
        scale = max(ref.max(), 1e-12)
        err = np.abs(got - ref) / scale
        assert (err > 1e-5).mean() < 4e-3, f"{(err > 1e-5).sum()} pixels differ"
        assert abs(got.sum() - ref.sum()) <= total * max(ref.sum(), 1e-9)


@pytest.mark.parametrize("name,res", [("box", 96), ("cornell", 96), ("corner", 64), ("smallpt", 48), ("lightgrid:3x3", 48)])
def test_full_tree_render_matches_oracle_with_common_random_numbers(name, res, scenes, oracle):
    """Reference schedule 16/8/4/2, depth 4, same Philox numbers: the large majority of pixels is identical to float
    rounding; the rest (ulp-level branch flips, see above) must be unbiased."""
    sd, sc = scenes(name)
    p, s, q, cnt, st, o = _render_pair(sd, sc, oracle, width=res, height=res, pass_count=2, flags=capi.FLAG_KEEP_ZERO_WEIGHT)
    ref = o["sum"]
    scale = max(ref.max(), 1e-12)
    diff = s - ref
    same = np.abs(diff) / scale <= 1e-5
    print(f"CRN_FULL_TREE {name} identical={same.mean():.4f}")
    # smallpt is sampled in the reference's operation order (ipt_shading.cuh: make_basis_exact), the others with contracted
    # arithmetic after the first random number
    assert same.mean() > (0.85 if name == "smallpt" else 0.5)
    # flips are rare events on both sides with the same distribution: the mean difference is noise around 0
    d = diff[~same]
    if d.size > 20:
        assert abs(d.mean()) < 5 * d.std() / np.sqrt(d.size)
    assert abs(s.sum() - ref.sum()) < 0.01 * ref.sum()
    assert abs(int(st.rays) - int(o["rays"])) < 1e-2 * o["rays"]
    for k in range(4):
        assert abs(int(st.rays_at_depth[k]) - int(o["rays_at_depth"][k])) <= 1e-2 * o["rays_at_depth"][k] + 4


def test_zero_weight_pruning_preserves_the_image(scenes):
    sd, sc = scenes("box")
    a = sc.render_host(capi.default_params(width=64, height=64, pass_count=2))
    b = sc.render_host(capi.default_params(width=64, height=64, pass_count=2, flags=capi.FLAG_KEEP_ZERO_WEIGHT))
    assert np.allclose(a[0], b[0], rtol=1e-5, atol=1e-7)
    assert a[3].rays <= b[3].rays and a[3].zero_weight_pruned > 0


@pytest.mark.parametrize("name,kw", [("box", {}), ("cornell", {}), ("smallpt", {}), ("mixedlights", {}), ("lightgrid:3x3", {}),
                                     ("lightgrid:5x6", {}),  # > 8 lights: light LBVH, last-level rays regrouped before the walk
                                     ("box", dict(depth_max=2, schedule=[5, 3])), ("box", dict(depth_max=1)),
                                     ("cornell", dict(depth_max=3, schedule=[4, 0, 2]))])
def test_fused_last_level_equals_queued_last_level(name, kw, scenes):
    """The shade kernels that trace their own children (default on analytic scenes: every depth, shadow rays at the last)
    against the queue + k_extend path, for the last level only (IPT_FLAG_NO_FUSED_TRACE) and for all levels
    (IPT_FLAG_NO_FUSED_LAST_LEVEL): same rays, same hits; sums equal up to the order of the float atomics."""
    sd, sc = scenes(name)
    base = dict(width=64, height=64, pass_count=3, plane_mode=capi.PLANE_LINEAR)
    base.update(kw)
    a = sc.render_host(capi.default_params(**base))
    m = sc.render_host(capi.default_params(flags=capi.FLAG_NO_FUSED_TRACE, **base))
    b = sc.render_host(capi.default_params(flags=capi.FLAG_NO_FUSED_LAST_LEVEL, **base))
    for x in (m, b):
        assert np.allclose(a[0], x[0], rtol=2e-5, atol=1e-7) and np.allclose(a[1], x[1], rtol=5e-5, atol=1e-7)
        assert np.array_equal(a[2], x[2])
        for f in ("rays", "light_hits", "surface_hits", "misses", "failed_samples", "zero_weight_pruned", "nonfinite_dropped"):
            assert getattr(a[3], f) == getattr(x[3], f), f
        assert list(a[3].rays_at_depth) == list(x[3].rays_at_depth)
    assert b[3].rays_resolved_in_shade == 0
    if base.get("depth_max", 4) >= 2 and base.get("schedule", [1])[-1] != 0:
        assert a[3].kernel_launches <= m[3].kernel_launches < b[3].kernel_launches
        assert a[3].rays_resolved_in_shade == a[3].rays - a[3].paths      # everything but the camera rays
        assert m[3].rays_resolved_in_shade <= a[3].rays_resolved_in_shade


def test_batching_and_tiles_are_invisible(scenes):
    """Philox counters are keyed by (pixel, pass, node): batch size, tiles and pass ranges must not change the result."""
    sd, sc = scenes("box")
    full = sc.render_host(capi.default_params(width=64, height=48, pass_count=4, plane_mode=capi.PLANE_LINEAR))
    small = sc.render_host(capi.default_params(width=64, height=48, pass_count=4, plane_mode=capi.PLANE_LINEAR, batch_paths=1000))
    assert np.allclose(full[0], small[0], rtol=1e-5, atol=1e-7)
    assert np.array_equal(full[2], small[2])
    plane = capi.Plane(sc, 64, 48)
    for (x0, y0, w, h) in [(0, 0, 32, 48), (32, 0, 32, 20), (32, 20, 32, 28)]:
        for (pb, pc) in [(0, 3), (3, 1)]:
            plane.render(capi.default_params(width=64, height=48, pass_begin=pb, pass_count=pc, plane_mode=capi.PLANE_LINEAR,
                                             tile_x0=x0, tile_y0=y0, tile_w=w, tile_h=h))
    s, q, c = plane.download()
    assert np.allclose(full[0], s, rtol=1e-5, atol=1e-7)
    assert np.array_equal(full[2], c)
    plane.close()


def test_grid_plane_mapping_matches_addray(scenes, oracle):
    """GridRenderPlane::addRay maps loop rows H-2 and H-1 both to image row 0 and never writes row H-1 (SURVEY S5)."""
    sd, sc = scenes("box")
    p = capi.default_params(width=40, height=40, pass_count=3)
    s, q, cnt, st = sc.render_host(p)
    assert (cnt[0] == 6).all() and (cnt[39] == 0).all() and (cnt[1:39] == 3).all()
    pl = capi.Plane(sc, 40, 40)
    pl.render(p)
    pix, counters, mx = pl.resolve()
    assert np.allclose(pix, np.where(cnt > 0, s / np.maximum(cnt, 1), 0), rtol=1e-6)
    assert mx == pytest.approx(pix.max())
    pl.close()


def test_depth_and_schedule_variants(scenes, oracle):
    sd, sc = scenes("box")
    for depth_max, schedule in [(1, [16]), (2, [4, 2]), (3, [3, 3, 3]), (8, [1] * 8), (5, [2, 2, 0, 2, 2])]:
        p = capi.default_params(width=48, height=48, pass_count=2, depth_max=depth_max, schedule=schedule, flags=capi.FLAG_KEEP_ZERO_WEIGHT)
        s, q, cnt, st = sc.render_host(p)
        o = oracle.render(sd.ptr, p, oracle_lib.RNG_PHILOX, 0)
        scale = max(o["sum"].max(), 1e-12)
        assert (np.abs(s - o["sum"]) / scale > 1e-4).mean() < (1e-3 if depth_max <= 2 else 0.05), (depth_max, schedule)
        assert abs(s.sum() - o["sum"].sum()) <= 0.02 * max(o["sum"].sum(), 1e-9), (depth_max, schedule)
        assert abs(int(st.rays) - int(o["rays"])) <= 3e-3 * o["rays"] + 4


def test_no_lights_scene(lib, oracle):
    """unite() degenerates to the sdf alone when there are no lights (ddf.cpp:209-210): everything is black, rays still counted."""
    sd = capi.SceneDescription("box")
    sd.desc.n_lights = 0
    sc = capi.Scene(sd)
    p = capi.default_params(width=32, height=32, pass_count=1, schedule=[4, 2, 1, 1])
    s, q, cnt, st = sc.render_host(p)
    o = oracle.render(sd.ptr, p, oracle_lib.RNG_PHILOX, 0)
    assert s.max() == 0.0 and o["sum"].max() == 0.0
    assert abs(int(st.rays) - int(o["rays"])) <= 1e-2 * o["rays"] + 4
    sd.desc.n_lights = 1
    sc.close()


def test_checkpoint_resume_equals_uninterrupted_render(scenes, tmp_path):
    """Accumulators saved after 3 passes and restored into a fresh plane, then 5 more passes == 8 passes at once."""
    from ipt_b200 import checkpoint

    sd, sc = scenes("cornell")
    kw = dict(width=80, height=60, seed=11)
    a = capi.Plane(sc, 80, 60)
    a.render(capi.default_params(pass_begin=0, pass_count=3, **kw))
    checkpoint.save(tmp_path / "ck.npz", a, next_pass=3, seed=11)
    a.close()
    b = capi.Plane(sc, 80, 60)
    meta = checkpoint.load(tmp_path / "ck.npz", b)
    assert int(meta["next_pass"]) == 3 and int(meta["seed"]) == 11
    b.render(capi.default_params(pass_begin=3, pass_count=5, **kw))
    s1, q1, c1 = b.download()
    b.close()
    s2, q2, c2, _ = sc.render_host(capi.default_params(pass_begin=0, pass_count=8, **kw))
    assert np.array_equal(c1, c2)
    assert np.allclose(s1, s2, rtol=1e-5, atol=1e-6) and np.allclose(q1, q2, rtol=1e-5, atol=1e-6)


def test_plane_add_rays_matches_gridrenderplane(scenes):
    """RenderPlane::addRay itself on the device, against the reference's GridRenderPlane (golden) incl. its row mapping."""
    from pathlib import Path

    g = np.load(Path(__file__).resolve().parent / "golden" / "ddf_kat.npz")
    sd, sc = scenes("box")
    pl = capi.Plane(sc, 16, 12)
    pl.add_rays(g["plane_x"], g["plane_y"], g["plane_v"])
    pix, cnt, mx = pl.resolve()
    assert np.array_equal(cnt, g["plane_counters"])
    assert np.allclose(pix, g["plane_pixels"], rtol=2e-6)  # sum/count vs the reference's float running mean
    assert mx == pytest.approx(float(g["plane_max"]), rel=1e-3) or mx <= float(g["plane_max"])  # running max >= final max
    pl.close()


def test_many_lights_through_the_light_lbvh(lib, oracle):
    """CollectionLighting with many emitters (BASELINE configs[4]): light sets > 8 go through an LBVH on the device;
    the reference scans linearly. Nearest light id / position must stay bit-exact, the mixture density equal."""
    name = "lightgrid:12x12"
    sd = capi.SceneDescription(name)
    sc = capi.Scene(sd)
    rng = np.random.default_rng(4)
    # rays from the floor / sphere region up towards the ceiling grid, plus generic rays
    n = 30000
    o = np.stack([rng.uniform(-0.95, 0.95, n), rng.uniform(-0.95, 0.95, n), rng.uniform(-0.99, 0.5, n)], 1).astype(np.float32)
    tgt = np.stack([rng.uniform(-1, 1, n), rng.uniform(-1, 1, n), np.full(n, 0.99)], 1).astype(np.float32)
    # a third of the rays aims inside an emitter (they are 0.01 wide), some through two of them in a row
    lights = np.array([list(sd.desc.lights[i].position) for i in range(sd.desc.n_lights)], np.float32)
    pick = rng.integers(0, len(lights), n // 3)
    tgt[: n // 3] = lights[pick] + np.stack([rng.uniform(0, 0.01, n // 3), rng.uniform(0, 0.01, n // 3), np.zeros(n // 3)], 1).astype(np.float32)
    d = tgt - o
    d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
    g = sc.trace_batch(o, d)
    c = oracle.trace_batch(sd.ptr, o, d)
    assert (c["light"] != capi.IPT_NO_HIT).sum() > 2000
    assert np.array_equal(g["light"], c["light"]) and np.array_equal(bits(g["light_pos"]), bits(c["light_pos"]))
    assert np.array_equal(g["outcome"], c["outcome"]) and np.array_equal(g["prim"], c["prim"])
    pos = np.array([0.1, -0.3, -1.0], np.float32)
    w = d[:4000]
    assert np.allclose(sc.light_ddf_value(pos, w), oracle.light_ddf_value(sd.ptr, pos, w), rtol=2e-4, atol=1e-6)
    p = capi.default_params(width=48, height=48, pass_count=2, depth_max=2, schedule=[16, 8], flags=capi.FLAG_KEEP_ZERO_WEIGHT)
    s, q, cnt, st = sc.render_host(p)
    ref = oracle.render(sd.ptr, p, oracle_lib.RNG_PHILOX, 0)
    scale = max(ref["sum"].max(), 1e-12)
    assert (np.abs(s - ref["sum"]) / scale > 1e-5).mean() < 4e-3
    assert abs(s.sum() - ref["sum"].sum()) <= 1e-4 * ref["sum"].sum()
    sc.close()


def test_edge_cases_and_argument_validation(scenes, oracle):
    """Empty and ragged inputs, extreme parameters, and the error codes of the C ABI."""
    sd, sc = scenes("box")
    # empty batches
    assert sc.trace_batch(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.float32))["prim"].shape == (0,)
    assert sc.preview_batch(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.float32)).shape == (0,)
    # zero passes: nothing accumulated, no error
    s, q, c, st = sc.render_host(capi.default_params(width=16, height=16, pass_count=0))
    assert st.paths == 0 and c.sum() == 0
    # ragged frame, 1x1 tile in the last row/column, batch of one path
    p = capi.default_params(width=37, height=23, pass_count=3, plane_mode=capi.PLANE_LINEAR, tile_x0=36, tile_y0=22, tile_w=1, tile_h=1, batch_paths=1)
    s, q, c, st = sc.render_host(p)
    assert st.paths == 3 and c[22, 36] == 3 and c.sum() == 3
    o = oracle.render(sd.ptr, p, oracle_lib.RNG_PHILOX, 0)
    assert np.array_equal(c.astype(np.uint64), o["counters"])
    # the deepest tree the ABI allows, one child per hit
    p = capi.default_params(width=24, height=24, pass_count=2, depth_max=16, schedule=[1] * 16)
    s, q, c, st = sc.render_host(p)
    assert st.rays_at_depth[15] <= st.rays_at_depth[1] and np.isfinite(s).all()
    # GUI plane mapping (Gui::addRay, gui.cpp:168-172): yi = H - y*H, clamped: unlike GridRenderPlane every row is hit once per pass
    s, q, c, st = sc.render_host(capi.default_params(width=20, height=20, pass_count=2, plane_mode=capi.PLANE_GUI))
    assert c.sum() == 800 and (c == 2).all()
    # errors: every one is reported through the status code + ipt_last_error, nothing falls back
    for bad in [dict(depth_max=0), dict(depth_max=17), dict(width=16, height=16, tile_x0=10, tile_w=10, tile_h=4), dict(plane_mode=7),
                dict(depth_max=4, schedule=[60000, 60000, 60000, 2])]:
        with pytest.raises(capi.IptError) as e:
            sc.render_host(capi.default_params(**{**dict(width=16, height=16), **bad}))
        assert e.value.code in (1, 4), bad
    pl = capi.Plane(sc, 8, 8)
    with pytest.raises(capi.IptError):
        pl.render(capi.default_params(width=16, height=16))  # plane / frame size mismatch
    pl.close()
    # scene descriptions are validated: a box plane must be an axis-aligned unit vector
    sd2 = capi.SceneDescription("box")
    sd2.desc.prims[0].p[1] = 0.5
    with pytest.raises(capi.IptError):
        capi.Scene(sd2)
    sd2.desc.prims[0].p[1] = 0.0
    sd2.desc.prims[5].material = 9
    with pytest.raises(capi.IptError):
        capi.Scene(sd2)


def test_every_light_kind_in_one_collection(lib, oracle):
    """CollectionLighting with all five Light classes at once (lighting.h:16-73, CollectionLighting.cpp:36-55): square,
    triangle, sphere, inverted sphere ("outer light") and point light. Mixed kinds take the linear multi-light path."""
    sd = capi.SceneDescription("mixedlights")
    sc = capi.Scene(sd)
    o, d, _ = ray_batch("box", lambda xy: oracle.camera_rays(sd.ptr, xy), n_cam_side=64, n_random=20000)
    g = sc.trace_batch(o, d); c = oracle.trace_batch(sd.ptr, o, d)
    for k in range(4):
        assert (c["light"] == k).sum() > 10, f"light {k} never hit"
    assert (c["light"] == 4).sum() == 0  # a point light is never hit (lighting.h:41-43)
    assert np.array_equal(g["light"], c["light"]) and np.array_equal(bits(g["light_pos"]), bits(c["light_pos"]))
    assert np.array_equal(g["outcome"], c["outcome"]) and np.array_equal(g["prim"], c["prim"]) and np.array_equal(bits(g["t"]), bits(c["t"]))
    pos = np.array([0.1, -0.3, -1.0], np.float32)
    w = d[:5000]
    assert np.allclose(sc.light_ddf_value(pos, w), oracle.light_ddf_value(sd.ptr, pos, w), rtol=3e-4, atol=1e-6)
    p = capi.default_params(width=64, height=64, pass_count=2, depth_max=2, schedule=[16, 8], flags=capi.FLAG_KEEP_ZERO_WEIGHT)
    s, q, cnt, st = sc.render_host(p)
    ref = oracle.render(sd.ptr, p, oracle_lib.RNG_PHILOX, 0)
    scale = max(ref["sum"].max(), 1e-12)
    # the dome lies behind every wall, so here an ulp-level hit/miss flip of the reference's plane test
    # (geometric_utils.cpp:18) changes a pixel even at the last level: most pixels identical, the rest unbiased
    assert (np.abs(s - ref["sum"]) / scale > 1e-5).mean() < 0.25
    assert abs(s.sum() - ref["sum"].sum()) <= 5e-3 * ref["sum"].sum()
    # full tree: statistical agreement
    p4 = capi.default_params(width=48, height=48, pass_count=8)
    s4, _, _, _ = sc.render_host(p4)
    r4 = oracle.render(sd.ptr, p4, oracle_lib.RNG_PHILOX, 0)
    assert abs(s4.sum() - r4["sum"].sum()) < 0.03 * r4["sum"].sum()
    sc.close()


@pytest.mark.parametrize("name", ["lightgrid:2x2", "lightgrid:2x4"])
def test_few_lights_take_the_linear_path(name, lib, oracle):
    """2..8 lights: scanned linearly on the device (no light LBVH), like CollectionLighting.cpp:23-34."""
    sd = capi.SceneDescription(name)
    sc = capi.Scene(sd)
    p = capi.default_params(width=48, height=48, pass_count=2, depth_max=2, schedule=[16, 8], flags=capi.FLAG_KEEP_ZERO_WEIGHT)
    s, q, cnt, st = sc.render_host(p)
    ref = oracle.render(sd.ptr, p, oracle_lib.RNG_PHILOX, 0)
    scale = max(ref["sum"].max(), 1e-12)
    assert (np.abs(s - ref["sum"]) / scale > 1e-5).mean() < 4e-3
    assert abs(int(st.rays) - int(ref["rays"])) <= 2e-4 * ref["rays"] + 2
    sc.close()


def test_many_spheres_take_the_generic_primitive_scan(lib, oracle):
    """More primitives than fit the kernel-parameter tables (24 inline / 8 unrolled spheres): the ordered scan over the
    global primitive array must give the same bits, including ties resolved towards the lower index."""
    rng = np.random.default_rng(9)
    prims = []
    for k in range(5):
        pr = capi.Prim(); pr.kind = 0; pr.material = 0
        pr.p[:] = [(1, 0, 0), (0, 1, 0), (0, 0, 1), (-1, 0, 0), (0, 0, -1)][k]
        prims.append(pr)
    for k in range(40):
        pr = capi.Prim(); pr.kind = 1; pr.material = 0
        pr.p[:] = [float(v) for v in rng.uniform(-0.8, 0.8, 3)]
        pr.radius = float(rng.uniform(0.05, 0.2)); pr.curvature = 1.0 / pr.radius
        prims.append(pr)
    prims.append(prims[7])  # an exact duplicate: the first one must keep winning
    sd = custom_scene(prims=prims)
    sc = capi.Scene(sd)
    o, d, _ = ray_batch("box", lambda xy: oracle.camera_rays(sd.ptr, xy), n_cam_side=64, n_random=20000)
    g = sc.trace_batch(o, d); c = oracle.trace_batch(sd.ptr, o, d)
    assert np.array_equal(g["prim"], c["prim"]) and np.array_equal(bits(g["t"]), bits(c["t"])) and np.array_equal(g["outcome"], c["outcome"])
    assert (c["prim"] == 45).sum() == 0 and (c["prim"] >= 5).sum() > 1000
    p = capi.default_params(width=48, height=48, pass_count=2, depth_max=2, schedule=[16, 8], flags=capi.FLAG_KEEP_ZERO_WEIGHT)
    s, q, cnt, st = sc.render_host(p)
    ref = oracle.render(sd.ptr, p, oracle_lib.RNG_PHILOX, 0)
    scale = max(ref["sum"].max(), 1e-12)
    assert (np.abs(s - ref["sum"]) / scale > 1e-5).mean() < 6e-3
    sc.close()


def test_four_threads_on_one_scene_like_main_cpp(scenes):
    """main.cpp:258-277 calls render_sample from four threads on one Scene. Concurrent callers of one ipt_scene are
    serialised by the library; every thread must get exactly the result of a sequential call."""
    import threading

    sd, sc = scenes("cornell")
    jobs = [capi.default_params(width=64, height=64, pass_begin=8 * k, pass_count=8, seed=3) for k in range(4)]
    expect = [sc.render_host(p) for p in jobs]
    got = [None] * 4

    def work(k):
        for _ in range(3):
            got[k] = sc.render_host(jobs[k])

    threads = [threading.Thread(target=work, args=(k,)) for k in range(4)]
    [t.start() for t in threads]
    [t.join() for t in threads]
    for k in range(4):
        assert np.array_equal(got[k][2], expect[k][2])
        assert np.allclose(got[k][0], expect[k][0], rtol=1e-5, atol=1e-6)
