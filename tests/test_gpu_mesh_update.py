"""GPU checks of ipt_scene_update_triangles (Scene.update_triangles): a refit keeps the tree's sorted order and topology and
recomputes every box byte for byte like the CPU restatement (test_oracle_mesh_refit.bvh_refit); a rebuild gives the tree a fresh scene of the new triangles
has; after either, traces are bit-identical to the oracle's linear scan over the new triangles and renders into a plane
made before the update equal those of a fresh scene. Deformations are seeded transforms of the sample meshes."""
import ctypes as C

import numpy as np
import pytest

from helpers import bits, custom_scene, ray_batch
from ipt_b200 import capi
from test_gpu_dispatch_matrix import smallpt_mesh
from test_oracle_mesh_refit import bvh_refit, carry_half, jitter

pytestmark = pytest.mark.gpu

DEFORMS = {"jitter": lambda t, seed: jitter(t, seed), "carry_half": lambda t, seed: carry_half(t, seed)}


def mesh_scene(n):
    sd = capi.SceneDescription(f"mesh:{n}")
    return sd, sd.triangles().copy(), capi.Scene(sd)


def trees(sc):
    nodes, order, keys = sc.bvh_export()
    qn, grid = sc.bvh_export_compact()
    return nodes, order, keys, qn, grid


def assert_same_trees(a, b):
    for x, y in zip(a, b):
        assert x.tobytes() == y.tobytes()


def rays_for(sd, oracle, tris, seed=3):
    """The ray_batch rays plus rays from random points of the box aimed at the centroids of (moved) triangles."""
    o, d, _ = ray_batch("box", lambda xy: oracle.camera_rays(sd.ptr, xy), n_cam_side=48, n_random=6000)
    rng = np.random.default_rng(seed)
    pick = rng.integers(0, len(tris), 4000)
    cen = tris[pick, 0:3] + (tris[pick, 3:6] + tris[pick, 6:9]) / np.float32(3)
    oo = rng.uniform(-0.95, 0.95, (len(pick), 3)).astype(np.float32)
    dd = (cen - oo).astype(np.float32)
    return np.concatenate([o, oo]), np.concatenate([d, dd])


def assert_traces_match_oracle(sc, oracle, tris, base="box"):
    """trace_batch of the updated scene == the oracle's linear scan over a description holding the new triangles."""
    sd = custom_scene(f"mesh:{len(tris)}" if base == "box" else base, triangles=tris)
    o, d = rays_for(sd, oracle, tris)
    g = sc.trace_batch(o, d)
    c = oracle.trace_batch(sd.ptr, o, d, use_bvh=1 if len(tris) > 2000 else 0)
    assert np.array_equal(g["prim"], c["prim"])
    assert np.array_equal(bits(g["t"]), bits(c["t"]))
    assert np.array_equal(g["outcome"], c["outcome"]) and np.array_equal(g["light"], c["light"])
    assert (c["prim"] >= sd.desc.n_prims).sum() > min(len(tris), 100)  # the moved triangles are actually hit
    return g


@pytest.mark.parametrize("deform", list(DEFORMS))
@pytest.mark.parametrize("n", [1, 2, 3, 4097, 300000])
def test_refit(n, deform, lib, oracle):
    sd, tris, sc = mesh_scene(n)
    dispatch = sc.dispatch()
    built = trees(sc)
    sc.update_triangles(tris)  # the build pose: a refit reproduces the built tree
    assert_same_trees(trees(sc), built)
    moved = DEFORMS[deform](tris, n)
    sc.update_triangles(moved)
    nodes, order, keys, qn, grid = after = trees(sc)
    assert np.array_equal(order, built[1]) and np.array_equal(keys, built[2]), "sorted order and keys are kept"
    want = bvh_refit(moved, built[0], built[1])
    assert nodes.tobytes() == want.tobytes(), "refitted boxes"
    cq, cgrid = oracle.bvh_compact(want)
    assert qn.tobytes() == cq.tobytes() and np.array_equal(bits(grid), bits(cgrid)), "32-byte nodes and grid"
    sc.update_triangles(moved)  # the same triangles again change no byte
    assert_same_trees(trees(sc), after)
    assert_traces_match_oracle(sc, oracle, moved)
    assert sc.dispatch() == dispatch
    sc.close()


@pytest.mark.parametrize("n", [1, 2, 3, 4097, 300000])
def test_rebuild(n, lib, oracle):
    sd, tris, sc = mesh_scene(n)
    dispatch = sc.dispatch()
    moved = carry_half(jitter(tris, n), n)
    sc.update_triangles(moved, rebuild=True)
    got = trees(sc)
    fresh = capi.Scene(custom_scene(f"mesh:{n}", triangles=moved))
    assert_same_trees(got, trees(fresh))
    cn, cids, ckeys = oracle.bvh_build(moved)
    cq, cgrid = oracle.bvh_compact(cn)
    assert_same_trees(got, (cn, cids, ckeys, cq, cgrid))
    assert_traces_match_oracle(sc, oracle, moved)
    assert sc.dispatch() == dispatch
    fresh.close()
    sc.close()


RENDER_SKIP = {"bvh_nodes_visited", "triangles_tested", "ms_total", "ms_generate", "ms_extend", "ms_shade", "ms_accumulate"}


@pytest.mark.parametrize("rebuild", [False, True], ids=["refit", "rebuild"])
@pytest.mark.parametrize("base", ["mesh:100000", "smallpt"])
def test_plane_made_before_the_update_renders_like_a_fresh_scene(base, rebuild, lib, oracle):
    if base == "smallpt":  # k_extend<smallpt, mesh>
        tris = smallpt_mesh()
        sd = custom_scene("smallpt", triangles=tris)
        moved = carry_half(jitter(tris, 1, scale=0.04), 2, centre=(50.0, 35.0, 70.0), size=40.0)
    else:
        sd = capi.SceneDescription(base)
        tris = sd.triangles().copy()
        moved = carry_half(jitter(tris, 1), 2)
    sc = capi.Scene(sd)
    W = H = 64
    p = capi.default_params(width=W, height=H, pass_count=2, seed=77)
    plane = capi.Plane(sc, W, H)
    plane.render(p)
    before = plane.download()
    sc.update_triangles(moved, rebuild=rebuild)
    for a, b in zip(plane.download(), before):  # the accumulators are the caller's: untouched
        assert a.tobytes() == b.tobytes()
    plane.clear()
    st = plane.render(p)
    s, q, cnt = plane.download()
    fresh = capi.Scene(custom_scene(base, triangles=moved))
    fplane = capi.Plane(fresh, W, H)
    fst = fplane.render(p)
    fs, fq, fcnt = fplane.download()
    assert np.array_equal(cnt, fcnt)
    a, b = st.as_dict(), fst.as_dict()
    for name in a:
        if name not in RENDER_SKIP:
            assert a[name] == b[name], name
    assert np.allclose(s, fs, rtol=2e-5, atol=1e-7) and np.allclose(q, fq, rtol=5e-5, atol=1e-7)
    assert st.light_hits > 0 and not np.array_equal(s, before[0])  # the update changed the image
    assert sc.dispatch() == fresh.dispatch()
    fplane.close(); fresh.close(); plane.close(); sc.close()


@pytest.mark.parametrize("rebuild", [False, True], ids=["refit", "rebuild"])
def test_device_input_equals_host_input(rebuild, lib, oracle):
    torch = pytest.importorskip("torch")
    n = 4097
    sd, tris, host = mesh_scene(n)
    dev = capi.Scene(capi.SceneDescription(f"mesh:{n}"))
    moved = carry_half(jitter(tris, 5), 6)
    host.update_triangles(moved, rebuild=rebuild)
    t = torch.from_numpy(moved.reshape(-1)).to("cuda:0")
    dev.update_triangles(t, rebuild=rebuild)
    assert_same_trees(trees(dev), trees(host))
    g = assert_traces_match_oracle(dev, oracle, moved)
    o, d = rays_for(custom_scene(f"mesh:{n}", triangles=moved), oracle, moved)
    h = host.trace_batch(o, d)
    assert np.array_equal(g["prim"], h["prim"]) and np.array_equal(bits(g["t"]), bits(h["t"]))
    dev.close(); host.close()


def test_errors_leave_the_scene_as_it_was(lib, oracle):
    torch = pytest.importorskip("torch")
    sd, tris, sc = mesh_scene(4097)
    box = capi.Scene(capi.SceneDescription("box"))
    o, d = rays_for(sd, oracle, tris)
    ref = sc.trace_batch(o, d)
    trees0 = trees(sc)
    moved = carry_half(tris, 9)
    on_gpu = torch.from_numpy(moved).to("cuda:0")
    hp = moved.ctypes.data
    cases = [
        (None, hp, len(tris), 0, "null argument"),
        (sc.handle, None, len(tris), 0, "null argument"),
        (sc.handle, hp, len(tris), 4, "unknown flag bits"),
        (sc.handle, hp, len(tris), capi.UPDATE_REBUILD | 8, "unknown flag bits"),
        (box.handle, hp, len(tris), 0, "no triangle mesh"),
        (sc.handle, hp, len(tris) + 1, 0, "4098 triangles given, the scene has 4097"),
        (sc.handle, hp, len(tris) - 1, capi.UPDATE_REBUILD, "4096 triangles given"),
        (sc.handle, hp, len(tris), capi.UPDATE_DEVICE_POINTER, "is not device or managed memory"),
        (sc.handle, on_gpu.data_ptr(), len(tris), 0, "is device memory"),
        (sc.handle, on_gpu.data_ptr() + 2, len(tris), capi.UPDATE_DEVICE_POINTER, "not aligned"),
    ]
    for handle, ptr, n, flags, msg in cases:
        assert lib.ipt_scene_dispatch(None, None) == capi.IPT_ERR_INVALID  # leaves another message behind
        rc = lib.ipt_scene_update_triangles(handle, ptr, C.c_uint64(n), flags)
        assert rc == capi.IPT_ERR_INVALID, msg
        err = lib.ipt_last_error().decode()
        assert err.startswith("ipt_scene_update_triangles") and msg in err, err
        g = sc.trace_batch(o, d)
        assert np.array_equal(g["prim"], ref["prim"]) and np.array_equal(bits(g["t"]), bits(ref["t"]))
    assert_same_trees(trees(sc), trees0)
    # the Python binding refuses what the C call cannot take, before calling it
    for bad, exc in ((moved.astype(np.float64), TypeError), (np.asfortranarray(moved), TypeError), (moved[:, :8].copy(), ValueError),
                     (moved.reshape(-1)[:-1].copy(), ValueError), (moved.tolist(), TypeError), (on_gpu.double(), TypeError),
                     (on_gpu.t(), TypeError), (on_gpu.cpu(), ValueError)):
        with pytest.raises(exc):
            sc.update_triangles(bad)
    assert_same_trees(trees(sc), trees0)
    box.close(); sc.close()
