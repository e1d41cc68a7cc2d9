"""GPU checks of ipt_scene_update_lights (Scene.update_lights): the light tables, the light LBVH and lights_inside_box
derived on the device equal what ipt_scene_create derives on the host. Updating a scene with its own lights changes
nothing; after moving and re-powering the lights, a rebuilt scene equals a fresh scene of the new lights bit for bit, and a
refitted one equals it except for the light tree's traversal counters and the summation order of the all-hits density. The light
sets and rays are those of test_gpu_dispatch_matrix.py; every case runs for host and device input and for refit and
rebuild."""
import ctypes as C

import numpy as np
import pytest

from helpers import bits, custom_scene, ray_batch
from ipt_b200 import capi
from test_gpu_dispatch_matrix import (BOX_ORIGINS, LIGHT_POINTS, ROWS, TRIANGLE, aimed_rays, box_light_moved, copy_light, diamonds,
                                      light_arrays, scene_lights)

pytestmark = pytest.mark.gpu

UPDATE_ROWS = ["L1-diamonds", "L2-triangles", "L2-mixed", "L3-duplicates", "L4-skewed", "L5-eight", "L5-nine", "L6-sphere",
               "S1-dome", "S1-point", "B1-near-wall", "M1-lbvh", "M1-mixedlights"]
LIGHTSET_ROWS = [k for k in UPDATE_ROWS if ROWS[k].lightset]
FORMS = [pytest.param(False, id="refit"), pytest.param(True, id="rebuild")]
INPUTS = ["host", "device"]
# not compared: timings, and the mesh traversal counters, which the persistent k_extend_mesh kernel makes vary from run to
# run (as in test_gpu_mesh_update.py)
TIMINGS = {"ms_total", "ms_generate", "ms_extend", "ms_shade", "ms_accumulate", "bvh_nodes_visited", "triangles_tested"}
# the light tree's traversal counters: leaf records tested and nodes visited depend on its topology, which a refit keeps
REFIT_FREE = {"light_bvh_nodes_visited", "lights_tested"}
MIX_RAY = (np.array([0.05, -0.1, 0.2], np.float32), np.array([0.3, 0.2, -1.0], np.float32))  # hits the box's back wall


def light_records(lights):
    """The lights as an (n, 12) array of ipt_light records (column 0: the kind's bit pattern)."""
    arr = (capi.Light * len(lights))(*lights)
    return np.frombuffer(arr, np.int32).reshape(len(lights), 12).copy()


def as_input(lights, src, dtype="float32"):
    if src == "host":
        return list(lights)
    import torch

    rec = light_records(lights)
    return torch.from_numpy(rec.view(np.float32) if dtype == "float32" else rec).to("cuda:0")


def copies(lights):
    return [copy_light(l) for l in lights]


def move_lights(lights, seed, amp=0.05):
    """Every light moved, rotated about its centre and rescaled (area lights), moved and rescaled (spheres) or moved
    (points), with new powers: about a tenth of them 0 (never light 0, whose zero power would make every weight NaN) and
    one 10^4 times brighter. A light that would leave the margin of test_light_sets_stay_inside_the_box keeps its place."""
    rng = np.random.default_rng(seed)
    n = len(lights)
    out = copies(lights)
    hot = int(rng.integers(0, n))
    for i, l in enumerate(out):
        p, xa, ya = (np.array(v, np.float64) for v in (l.position, l.x_axis, l.y_axis))
        if l.kind <= TRIANGLE:
            ax = rng.normal(size=3); ax /= np.linalg.norm(ax)
            th = rng.uniform(-0.4, 0.4)
            K = np.array([[0, -ax[2], ax[1]], [ax[2], 0, -ax[0]], [-ax[1], ax[0], 0]])
            R = np.eye(3) + np.sin(th) * K + (1 - np.cos(th)) * K @ K
            s = rng.uniform(0.8, 1.2)
            c = p + 0.5 * (xa + ya) + rng.uniform(-amp, amp, 3)
            xa2, ya2 = s * (R @ xa), s * (R @ ya)
            p2 = c - 0.5 * (xa2 + ya2)
            corners = np.stack([p2, p2 + xa2, p2 + ya2, p2 + xa2 + ya2])
            if np.abs(corners).max() < 0.98:
                l.position[:], l.x_axis[:], l.y_axis[:] = p2.tolist(), xa2.tolist(), ya2.tolist()
        else:
            if np.abs(p).max() + l.radius < 0.9:
                l.position[:] = (p + rng.uniform(-amp, amp, 3)).tolist()
            l.radius = float(l.radius * rng.uniform(0.9, 1.1))
        l.power = float(rng.uniform(0.2, 3.0))
        if i > 0 and n > 2 and rng.random() < 0.1:
            l.power = 0.0
    out[hot].power = float(max(out[hot].power, 0.5) * 1e4)
    return out


def rays_for(sd, oracle, lights, origins, region="box"):
    o1, d1, _ = ray_batch(region, lambda xy: oracle.camera_rays(sd.ptr, xy), n_cam_side=32, n_random=6000)
    o2, d2 = aimed_rays(lights, origins, max_lights=150)
    return np.concatenate([o1, o2]), np.concatenate([d1, d2])


def outputs(sc, o, d, lights, render=True):
    """Everything compared: traces, the light mixture's value and samples, the mixture at a surface hit, dispatch, and
    a two-level render with a fixed seed."""
    out = dict(trace=sc.trace_batch(o, d), dispatch=sc.dispatch())
    rng = np.random.default_rng(5)
    vals = []
    for pt in LIGHT_POINTS:
        p = np.array(pt, np.float32)
        _, w = aimed_rays(lights, p[None], max_lights=100)
        v = rng.normal(size=(1000, 3))
        w = np.concatenate([w[::3], v / np.linalg.norm(v, axis=1, keepdims=True)]).astype(np.float32)
        vals.append(sc.light_ddf_value(p, w))
    out["ddf_value"] = np.concatenate(vals)
    out["ddf_sample"] = sc.light_ddf_sample(np.array(LIGHT_POINTS[0], np.float32), 20000, seed=99)
    out["mix"] = sc.mix_sample(*MIX_RAY, 20000, seed=7)
    if render:
        p = capi.default_params(width=32, height=32, pass_count=2, depth_max=2, schedule=[16, 8], seed=11, flags=capi.FLAG_KEEP_ZERO_WEIGHT)
        out["render"] = sc.render_host(p)
    return out


def assert_outputs_equal(a, b, refit=False):
    """Bit for bit; after a refit the all-hits density (ddf value, mixture value, render sums) to its last bits, and the
    light tree's traversal counters are free."""
    for k in ("prim", "light", "outcome"):
        assert np.array_equal(a["trace"][k], b["trace"][k]), k
    for k in ("t", "light_pos"):
        assert np.array_equal(bits(a["trace"][k]), bits(b["trace"][k])), k
    assert a["dispatch"] == b["dispatch"]
    assert np.array_equal(bits(a["ddf_sample"]), bits(b["ddf_sample"]))
    (wa, ma, sa), (wb, mb, sb) = a["mix"], b["mix"]
    assert np.array_equal(bits(wa), bits(wb)) and np.array_equal(bits(sa), bits(sb))
    if refit:
        assert np.allclose(a["ddf_value"], b["ddf_value"], rtol=4e-6, atol=0, equal_nan=True)
        assert np.allclose(ma, mb, rtol=4e-6, atol=0, equal_nan=True)
    else:
        assert np.array_equal(bits(a["ddf_value"]), bits(b["ddf_value"]))
        assert np.array_equal(bits(ma), bits(mb))
    if "render" in a and "render" in b:
        (s1, q1, c1, st1), (s2, q2, c2, st2) = a["render"], b["render"]
        assert np.array_equal(c1, c2)
        x, y = st1.as_dict(), st2.as_dict()
        for name in x:
            if name not in TIMINGS and not (refit and name in REFIT_FREE):
                assert x[name] == y[name], name
        # the fused-vs-queued tolerance of test_path_variants_agree: the float atomics add in another order
        assert np.allclose(s1, s2, rtol=2e-5, atol=1e-7) and np.allclose(q1, q2, rtol=5e-5, atol=1e-7)


def row_scene(name):
    sd = ROWS[name].build()
    return sd, copies(scene_lights(sd)), capi.Scene(sd)


@pytest.mark.parametrize("rebuild", FORMS)
@pytest.mark.parametrize("src", INPUTS)
@pytest.mark.parametrize("name", UPDATE_ROWS)
def test_identity(name, src, rebuild, lib, oracle):
    """Updating a scene with its own lights changes no output, including the light tree's node visits."""
    r = ROWS[name]
    sd, lights, sc = row_scene(name)
    o, d = rays_for(sd, oracle, lights, r.origins, r.region)
    before = outputs(sc, o, d, lights)
    sc.update_lights(as_input(lights, src, "int32" if rebuild else "float32"), rebuild=rebuild)
    assert_outputs_equal(outputs(sc, o, d, lights), before)
    sc.close()


@pytest.mark.parametrize("rebuild", FORMS)
@pytest.mark.parametrize("src", INPUTS)
@pytest.mark.parametrize("name", UPDATE_ROWS)
def test_moved_lights_equal_a_fresh_scene(name, src, rebuild, lib, oracle):
    """Moved, rotated, rescaled and re-powered lights: the updated scene against a scene created with them, and its traces
    against the oracle's linear scan."""
    r = ROWS[name]
    sd, lights, sc = row_scene(name)
    moved = move_lights(lights, seed=len(lights) + 17 * int(rebuild))
    kind, pos, xa, ya, _ = light_arrays(moved)
    area = kind <= TRIANGLE
    if r.lightset:  # the generated sets stay inside the box, as test_light_sets_stay_inside_the_box requires
        corners = np.stack([pos, pos + xa, pos + ya, pos + xa + ya])[:, area]
        assert np.abs(corners).max() < 0.99
    fresh_sd = custom_scene(sd.name, lights=moved)
    fresh = capi.Scene(fresh_sd)
    o, d = rays_for(fresh_sd, oracle, moved, r.origins, r.region)
    sc.update_lights(as_input(moved, src), rebuild=rebuild)
    got, want = outputs(sc, o, d, moved), outputs(fresh, o, d, moved)
    assert_outputs_equal(got, want, refit=not rebuild and sc.dispatch()["n_light_bvh"] > 0)
    c = oracle.trace_batch(fresh_sd.ptr, o, d, use_bvh=0)
    for k in ("prim", "light", "outcome"):
        assert np.array_equal(got["trace"][k], c[k]), k
    assert np.array_equal(bits(got["trace"]["t"]), bits(c["t"])) and np.array_equal(bits(got["trace"]["light_pos"]), bits(c["light_pos"]))
    fresh.close(); sc.close()


@pytest.mark.parametrize("rebuild", FORMS)
@pytest.mark.parametrize("name", LIGHTSET_ROWS)
def test_moved_light_mixture_matches_oracle(name, rebuild, lib, oracle):
    """test_light_mixture_matches_oracle on the updated scene (device input): value() against the oracle at three points,
    sample() by the two-sample chi-square."""
    from scipy.stats import chi2 as chi2_dist

    from test_gpu_golden import histogram

    sd, lights, sc = row_scene(name)
    moved = move_lights(lights, seed=3)
    fresh_sd = custom_scene(sd.name, lights=moved)
    sc.update_lights(as_input(moved, "device"), rebuild=rebuild)
    rng = np.random.default_rng(5)
    for pt in LIGHT_POINTS:
        p = np.array(pt, np.float32)
        _, w = aimed_rays(moved, p[None], max_lights=200)
        v = rng.normal(size=(2000, 3))
        w = np.concatenate([w[::3], (v / np.linalg.norm(v, axis=1, keepdims=True))]).astype(np.float32)
        g = sc.light_ddf_value(p, w)
        c = oracle.light_ddf_value(fresh_sd.ptr, p, w)
        assert (c > 0).sum() > 100
        assert np.allclose(g, c, rtol=3e-4, atol=1e-6), pt
    p = np.array(LIGHT_POINTS[0], np.float32)
    n = 300000
    w = sc.light_ddf_sample(p, n, seed=4242)
    oracle.seed(271828)
    w_c = oracle.light_ddf_sample(fresh_sd.ptr, p, n)
    hg, rate_g = histogram(w)
    hc, rate_c = histogram(w_c)
    assert abs(rate_g - rate_c) < 5 * np.sqrt(0.25 / n) * np.sqrt(2), (rate_g, rate_c)
    use = (hg + hc) > 20
    dof = int(use.sum())
    chi2 = float(((hg[use] - hc[use]) ** 2 / (hg[use] + hc[use])).sum())
    assert dof >= 1 and chi2 < chi2_dist.ppf(0.9999, dof), (chi2, dof)
    sc.close()


@pytest.mark.parametrize("src", INPUTS)
def test_lights_inside_box_follows_the_light(src, lib, oracle):
    """The box scene's light moved to the B1 near-wall position and back: the wall skip goes off and on again, and each
    state renders like a fresh scene."""
    sd = capi.SceneDescription("box")
    home = copies(scene_lights(sd))
    sc = capi.Scene(sd)
    o, d = rays_for(sd, oracle, home, BOX_ORIGINS)
    assert sc.dispatch()["lights_inside_box"] == 1
    for lights, inside in (([box_light_moved(0.6995, 0.0)], 0), (home, 1)):
        sc.update_lights(as_input(lights, src))
        assert sc.dispatch()["lights_inside_box"] == inside
        fresh = capi.Scene(custom_scene("box", lights=lights))
        assert_outputs_equal(outputs(sc, o, d, lights), outputs(fresh, o, d, lights))
        fresh.close()
    sc.close()


@pytest.mark.parametrize("rebuild", FORMS)
@pytest.mark.parametrize("name", ["L1-diamonds", "B1-near-wall", "M1-lbvh"])
def test_plane_made_before_the_update_renders_like_a_fresh_scene(name, rebuild, lib):
    sd, lights, sc = row_scene(name)
    moved = move_lights(lights, seed=8)
    W = H = 48
    p = capi.default_params(width=W, height=H, pass_count=2, seed=77)
    plane = capi.Plane(sc, W, H)
    plane.render(p)
    before = plane.download()
    sc.update_lights(moved, rebuild=rebuild)
    for a, b in zip(plane.download(), before):  # the accumulators are the caller's: untouched
        assert a.tobytes() == b.tobytes()
    plane.clear()
    st = plane.render(p)
    s, q, cnt = plane.download()
    fresh = capi.Scene(custom_scene(sd.name, lights=moved))
    fplane = capi.Plane(fresh, W, H)
    fst = fplane.render(p)
    fs, fq, fcnt = fplane.download()
    assert np.array_equal(cnt, fcnt)
    a, b = st.as_dict(), fst.as_dict()
    refit = not rebuild and sc.dispatch()["n_light_bvh"] > 0
    for k in a:
        if k not in TIMINGS and not (refit and k in REFIT_FREE):
            assert a[k] == b[k], k
    assert np.allclose(s, fs, rtol=2e-5, atol=1e-7) and np.allclose(q, fq, rtol=5e-5, atol=1e-7)
    assert st.light_hits > 0 and not np.array_equal(s, before[0])
    fplane.close(); fresh.close(); plane.close(); sc.close()


@pytest.mark.parametrize("rebuild", FORMS)
def test_mesh_tree_and_triangle_materials_are_untouched(rebuild, lib, oracle):
    """M1-lbvh with per-triangle materials: a light update leaves the mesh tree byte for byte and renders like a fresh
    scene given the same materials."""
    sd, lights, sc = row_scene("M1-lbvh")
    mats = (np.arange(sd.desc.n_triangles) % sd.desc.n_materials).astype(np.uint32)[::-1].copy()
    sc.set_triangle_materials(mats)
    tree = [x.tobytes() for x in (*sc.bvh_export(), *sc.bvh_export_compact())]
    moved = move_lights(lights, seed=21)
    sc.update_lights(moved, rebuild=rebuild)
    assert [x.tobytes() for x in (*sc.bvh_export(), *sc.bvh_export_compact())] == tree
    fresh = capi.Scene(custom_scene(sd.name, lights=moved))
    fresh.set_triangle_materials(mats)
    o, d = rays_for(sd, oracle, moved, BOX_ORIGINS)
    assert_outputs_equal(outputs(sc, o, d, moved), outputs(fresh, o, d, moved), refit=not rebuild)
    fresh.close(); sc.close()


@pytest.mark.parametrize("src", INPUTS)
def test_repeated_refits_then_a_rebuild_equal_a_fresh_scene(src, lib, oracle):
    sd, lights, sc = row_scene("L1-diamonds")
    cur = lights
    for k in range(20):
        cur = move_lights(cur, seed=100 + k, amp=0.01)
        sc.update_lights(as_input(cur, src))
    sc.update_lights(as_input(cur, src), rebuild=True)
    fresh_sd = custom_scene("box", lights=cur)
    fresh = capi.Scene(fresh_sd)
    o, d = rays_for(fresh_sd, oracle, cur, BOX_ORIGINS)
    assert_outputs_equal(outputs(sc, o, d, cur), outputs(fresh, o, d, cur))
    fresh.close(); sc.close()


def test_thirty_thousand_diamonds_from_a_tensor(lib):
    """3 * 10^4 diamonds, updated from a CUDA tensor with a rebuild: traces on aimed rays and light_ddf_sample equal a fresh
    scene's bit for bit."""
    n = 30000
    lights = diamonds(np.random.default_rng(31), n, lo=(-0.9, -0.9, -0.9), hi=(0.9, 0.9, 0.9), size=(0.005, 0.02))
    moved = move_lights(lights, seed=32, amp=0.02)
    sc = capi.Scene(custom_scene("box", lights=lights))
    sc.update_lights(as_input(moved, "device"), rebuild=True)
    fresh = capi.Scene(custom_scene("box", lights=moved))
    o, d = aimed_rays(moved, BOX_ORIGINS, max_lights=2000)
    a, b = sc.trace_batch(o, d), fresh.trace_batch(o, d)
    for k in ("prim", "light", "outcome"):
        assert np.array_equal(a[k], b[k]), k
    assert np.array_equal(bits(a["t"]), bits(b["t"])) and np.array_equal(bits(a["light_pos"]), bits(b["light_pos"]))
    assert (a["light"] != capi.IPT_NO_HIT).mean() > 0.1
    for pt in LIGHT_POINTS:
        p = np.array(pt, np.float32)
        assert np.array_equal(bits(sc.light_ddf_sample(p, 50000, seed=5)), bits(fresh.light_ddf_sample(p, 50000, seed=5)))
    assert sc.dispatch() == fresh.dispatch()
    fresh.close(); sc.close()


def test_errors_leave_the_scene_as_it_was(lib, oracle):
    torch = pytest.importorskip("torch")
    sd, lights, sc = row_scene("L1-diamonds")
    box = capi.Scene(capi.SceneDescription("box"))
    o, d = rays_for(sd, oracle, lights, BOX_ORIGINS)
    ref = outputs(sc, o, d, lights)
    moved = move_lights(lights, seed=4)
    n = len(moved)
    host = (capi.Light * n)(*moved)
    hp = C.addressof(host)
    k = 57
    bad_kind = (capi.Light * n)(*copies(moved))
    bad_kind[k].kind = TRIANGLE
    rec = light_records(moved)
    on_gpu = torch.from_numpy(rec).to("cuda:0")
    bad_gpu = rec.copy()
    bad_gpu[k, 0] = TRIANGLE
    bad_gpu = torch.from_numpy(bad_gpu).to("cuda:0")
    cases = [
        (None, hp, n, 0, "null argument"),
        (sc.handle, None, n, 0, "null argument"),
        (sc.handle, hp, n, 4, "unknown flag bits"),
        (sc.handle, hp, n, capi.UPDATE_REBUILD | 8, "unknown flag bits"),
        (sc.handle, hp, n + 1, 0, f"{n + 1} lights given, the scene has {n}"),
        (box.handle, hp, n, 0, f"{n} lights given, the scene has 1"),
        (sc.handle, C.addressof(bad_kind), n, 0, f"lights[{k}].kind differs"),
        (sc.handle, bad_gpu.data_ptr(), n, capi.UPDATE_DEVICE_POINTER | capi.UPDATE_REBUILD, f"lights[{k}].kind differs"),
        (sc.handle, hp, n, capi.UPDATE_DEVICE_POINTER, "is not device or managed memory"),
        (sc.handle, on_gpu.data_ptr(), n, 0, "is device memory"),
        (sc.handle, on_gpu.data_ptr() + 2, n, capi.UPDATE_DEVICE_POINTER, "not aligned"),
    ]
    for handle, ptr, count, flags, msg in cases:
        assert lib.ipt_scene_dispatch(None, None) == capi.IPT_ERR_INVALID  # leaves another message behind
        rc = lib.ipt_scene_update_lights(handle, ptr, count, flags)
        assert rc == capi.IPT_ERR_INVALID, msg
        err = lib.ipt_last_error().decode()
        assert err.startswith("ipt_scene_update_lights") and msg in err, err
        assert_outputs_equal(outputs(sc, o, d, lights), ref)
    # the same through Python: the library's messages, or a Python error before the call
    bad = copies(moved)
    bad[k].kind = TRIANGLE
    for arg, msg in ((moved[:-1], f"{n - 1} lights given"), (bad, f"lights[{k}].kind differs"), (bad_gpu, f"lights[{k}].kind differs")):
        with pytest.raises(capi.IptError, match=msg.replace("[", r"\[").replace("]", r"\]")):
            sc.update_lights(arg)
    for arg, exc in ((rec, TypeError), ([1, 2], TypeError), (on_gpu.double(), TypeError), (on_gpu[:, :11].contiguous(), ValueError),
                     (on_gpu.t(), TypeError), (on_gpu.cpu(), ValueError), (on_gpu.reshape(-1), ValueError)):
        with pytest.raises(exc):
            sc.update_lights(arg)
    assert_outputs_equal(outputs(sc, o, d, lights), ref)
    box.close(); sc.close()
