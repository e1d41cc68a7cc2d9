"""GPU checks of per-triangle materials (ipt_scene_set_triangle_materials, Scene.set_triangle_materials) against the oracle
with the same array attached (ipt_oracle_set_triangle_materials): renders per pixel and with common random numbers, the
mixture at hits of every material, persistence through refit and rebuild, device input, SmallPt with a mesh, the state a
call leaves (dispatch, planes, trees) and every error case. Six materials past the scene's own, so that indices beyond
IPT_INLINE_MATS are used, assigned at random per triangle or by regions of the box."""
import ctypes as C

import numpy as np
import pytest

import oracle_lib
import oracle_tri_mats
from helpers import bits
from ipt_b200 import capi
from test_gpu_dispatch_matrix import _two_level, assert_accumulators_match, smallpt_mesh
from test_gpu_golden import histogram
from test_gpu_mesh_update import RENDER_SKIP, trees
from test_oracle_mesh_materials import halves_assignment, mesh_hits, random_assignment, with_six_materials
from test_oracle_mesh_refit import carry_half, jitter

pytestmark = pytest.mark.gpu

BASES = {"mesh:2000": 0, "mesh:100000": 1}  # scene -> oracle tracing (0: linear scan, 1: its LBVH)


@pytest.fixture(scope="module")
def oracle(lib):
    """The oracle that can attach per-triangle materials (tests/oracle_tri_mats.py) in place of the session's oracle."""
    return oracle_tri_mats.load()


def assignment(kind, tris, first):
    return random_assignment(len(tris), first, seed=len(tris)) if kind == "random" else halves_assignment(tris, first)


@pytest.fixture(scope="module")
def scenes(lib):
    """(description, scene, materials) per (base, assignment), with the materials set on the device."""
    cache = {}

    def get(base, kind):
        if (base, kind) not in cache:
            sd, first = with_six_materials(base)
            mats = assignment(kind, sd.triangles(), first)
            sc = capi.Scene(sd)
            sc.set_triangle_materials(mats)
            cache[base, kind] = (sd, sc, mats)
        return cache[base, kind]

    yield get
    for sd, sc, mats in cache.values():
        sc.close()


def assert_same_render_stats(a, b):
    """Counts and every counter but the node visits (which vary from run to run on mesh scenes) and the timings."""
    assert np.array_equal(a[2], b[2])
    x, y = a[3].as_dict(), b[3].as_dict()
    for name in x:
        if name not in RENDER_SKIP:
            assert x[name] == y[name], name


def assert_sums_close(a, b):
    """The fused-vs-queued tolerance: equal up to the order of the float atomics."""
    assert np.allclose(a[0], b[0], rtol=2e-5, atol=1e-7) and np.allclose(a[1], b[1], rtol=5e-5, atol=1e-7)


@pytest.mark.parametrize("kind", ["random", "halves"])
@pytest.mark.parametrize("base", list(BASES))
def test_two_level_render_per_pixel(base, kind, scenes, oracle):
    """depth 2, 16/8, same Philox numbers: counters and rays identical, sum and sumsq per pixel to float rounding."""
    sd, sc, mats = scenes(base, kind)
    with oracle.triangle_materials(sd.ptr, mats):
        s, q, cnt, st, o = _two_level(sd, sc, oracle, 48, BASES[base])
    assert np.array_equal(cnt.astype(np.uint64), o["counters"])
    assert [int(v) for v in st.rays_at_depth[:2]] == [int(v) for v in o["rays_at_depth"][:2]]
    assert st.rays == o["rays"]
    assert_accumulators_match(s, q, o, 4e-3, 1e-4)
    uniform = oracle.render(sd.ptr, capi.default_params(width=48, height=48, pass_count=2, depth_max=2, schedule=[16, 8],
                                                        flags=capi.FLAG_KEEP_ZERO_WEIGHT), oracle_lib.RNG_PHILOX, BASES[base])
    assert np.abs(uniform["sum"] - o["sum"]).max() > 0.01 * o["sum"].max()  # the materials change the image


@pytest.mark.parametrize("kind", ["random", "halves"])
@pytest.mark.parametrize("base", list(BASES))
def test_full_tree_render_with_common_random_numbers(base, kind, scenes, oracle):
    """16/8/4/2, same Philox numbers: most pixels identical, the rest unbiased, ray counts per depth within 1 % (the
    assertions of test_gpu_dispatch_matrix.py::test_full_tree_render_with_common_random_numbers)."""
    sd, sc, mats = scenes(base, kind)
    res = 48 if base == "mesh:2000" else 32
    p = capi.default_params(width=res, height=res, pass_count=2, flags=capi.FLAG_KEEP_ZERO_WEIGHT)
    s, q, cnt, st = sc.render_host(p)
    with oracle.triangle_materials(sd.ptr, mats):
        o = oracle.render(sd.ptr, p, oracle_lib.RNG_PHILOX, 1)
    ref = o["sum"]
    diff = s - ref
    same = np.abs(diff) / ref.max() <= 1e-5
    print(f"CRN_FULL_TREE {base} {kind} identical={same.mean():.4f}")
    assert same.mean() > 0.5
    d = diff[~same]
    if d.size > 20:
        assert abs(d.mean()) < 5 * d.std() / np.sqrt(d.size)
    assert abs(s.sum() - ref.sum()) < 0.01 * ref.sum()
    assert abs(int(st.rays) - int(o["rays"])) < 1e-2 * o["rays"]
    for k in range(4):
        assert abs(int(st.rays_at_depth[k]) - int(o["rays_at_depth"][k])) <= 1e-2 * o["rays_at_depth"][k] + 4


def test_mix_sample_at_hits_of_each_material(scenes, oracle):
    """ipt_mix_sample at a hit on a triangle of each material: mixture and sdf values at the sampled directions equal the
    oracle's mix_value to float rounding; the directions pass the two-sample chi-square against the oracle's samples."""
    from scipy.stats import chi2 as chi2_dist

    sd, sc, mats = scenes("mesh:2000", "random")
    o, d, k = mesh_hits(oracle, sd)
    n = 300000
    with oracle.triangle_materials(sd.ptr, mats):
        for m in np.unique(mats):
            i = int(np.flatnonzero(mats[k] == m)[0])
            w, mv, sv = sc.mix_sample(o[i], d[i], n, seed=777 + int(m))
            ok = np.any(w != 0, axis=1)
            mo, so, _ = oracle.mix_value(sd.ptr, o[i], d[i], w[ok][:5000])
            assert np.allclose(mv[ok][:5000], mo, rtol=3e-4, atol=1e-6) and np.allclose(sv[ok][:5000], so, rtol=3e-4, atol=1e-6), m
            oracle.seed(31337 + int(m))
            w_c, _, _ = oracle.mix_sample(sd.ptr, o[i], d[i], n)
            hg, rate_g = histogram(w)
            hc, rate_c = histogram(w_c)
            assert abs(rate_g - rate_c) < 5 * np.sqrt(0.25 / n) * np.sqrt(2), (m, rate_g, rate_c)
            use = (hg + hc) > 20
            dof = int(use.sum())
            chi2 = float(((hg[use] - hc[use]) ** 2 / (hg[use] + hc[use])).sum())
            assert dof >= 1 and chi2 < chi2_dist.ppf(0.9999, dof), (m, chi2, dof)


@pytest.mark.parametrize("base", ["mesh:100000", "smallpt"])
def test_uniform_array_equals_no_call(base, lib):
    """An array equal to triangle_material everywhere: the same render as the scene without the call."""
    tris = smallpt_mesh() if base == "smallpt" else None
    sd, first = with_six_materials(base, triangles=tris)
    a, b = capi.Scene(sd), capi.Scene(sd)
    b.set_triangle_materials(np.full(sd.desc.n_triangles, sd.desc.triangle_material, np.uint32))
    p = capi.default_params(width=64, height=64, pass_count=2, seed=5)
    ra, rb = a.render_host(p), b.render_host(p)
    assert_same_render_stats(ra, rb)
    assert_sums_close(ra, rb)
    assert a.dispatch() == b.dispatch()
    a.close(); b.close()


@pytest.mark.parametrize("source", ["host", "device"])
@pytest.mark.parametrize("rebuild", [False, True], ids=["refit", "rebuild"])
def test_materials_persist_through_updates(rebuild, source, lib, oracle):
    """After a refit or a rebuild (vertices from host or device memory) a render of the moved mesh matches the oracle on a
    description holding the moved triangles and the same array; the tree is the one a scene without materials has."""
    torch = pytest.importorskip("torch")
    sd, first = with_six_materials("mesh:100000")
    tris = sd.triangles().copy()
    mats = random_assignment(len(tris), first, seed=8)
    sc, twin = capi.Scene(sd), capi.Scene(sd)
    sc.set_triangle_materials(mats)
    for x, y in zip(trees(sc), trees(twin)):
        assert x.tobytes() == y.tobytes()
    moved = carry_half(jitter(tris, 1), 2)
    for s in (sc, twin):
        s.update_triangles(torch.from_numpy(moved).to("cuda:0") if source == "device" else moved, rebuild=rebuild)
    for x, y in zip(trees(sc), trees(twin)):
        assert x.tobytes() == y.tobytes()
    sdm, _ = with_six_materials("mesh:100000", triangles=moved)
    with oracle.triangle_materials(sdm.ptr, mats):
        s, q, cnt, st, o = _two_level(sdm, sc, oracle, 48, 1)
    assert np.array_equal(cnt.astype(np.uint64), o["counters"])
    assert [int(v) for v in st.rays_at_depth[:2]] == [int(v) for v in o["rays_at_depth"][:2]]
    assert st.rays == o["rays"]
    assert_accumulators_match(s, q, o, 4e-3, 1e-4)
    sc.close(); twin.close()


@pytest.mark.parametrize("dtype", ["int32", "uint32"])
def test_device_input_equals_host_input(dtype, scenes, oracle):
    torch = pytest.importorskip("torch")
    sd, host, mats = scenes("mesh:100000", "halves")
    dev = capi.Scene(sd)
    dev.set_triangle_materials(torch.from_numpy(mats.astype(dtype)).to("cuda:0"))
    p = capi.default_params(width=64, height=64, pass_count=2, seed=9)
    rh, rd = host.render_host(p), dev.render_host(p)
    assert_same_render_stats(rh, rd)
    assert_sums_close(rh, rd)
    o, d, _ = mesh_hits(oracle, sd)
    for a, b in zip(host.mix_sample(o[0], d[0], 4096, seed=3), dev.mix_sample(o[0], d[0], 4096, seed=3)):
        assert bits(a).tobytes() == bits(b).tobytes()
    dev.close()


def test_smallpt_with_a_mesh_two_level_per_pixel(lib, oracle):
    """SmallPt spheres and a mesh with per-triangle materials: k_extend<true, true> and k_shade<FUSE_NONE, true>."""
    sd, first = with_six_materials("smallpt", triangles=smallpt_mesh())
    mats = random_assignment(sd.desc.n_triangles, first, seed=4)
    sc = capi.Scene(sd)
    assert {k: v for k, v in sc.dispatch().items() if k in ("smallpt", "mesh")} == dict(smallpt=1, mesh=1)
    sc.set_triangle_materials(mats)
    with oracle.triangle_materials(sd.ptr, mats):
        s, q, cnt, st, o = _two_level(sd, sc, oracle, 48, 0)
    assert np.array_equal(cnt.astype(np.uint64), o["counters"])
    assert [int(v) for v in st.rays_at_depth[:2]] == [int(v) for v in o["rays_at_depth"][:2]]
    assert st.rays == o["rays"]
    assert_accumulators_match(s, q, o, 4e-3, 1e-4)
    sc.close()


def test_dispatch_and_planes_are_kept(lib):
    """The call changes no dispatch word; a plane made before it keeps its accumulators and then renders like a plane of a
    fresh scene with the same materials."""
    sd, first = with_six_materials("mesh:100000")
    mats = halves_assignment(sd.triangles(), first)
    sc = capi.Scene(sd)
    dispatch = sc.dispatch()
    W = H = 64
    p = capi.default_params(width=W, height=H, pass_count=2, seed=77)
    plane = capi.Plane(sc, W, H)
    plane.render(p)
    before = plane.download()
    sc.set_triangle_materials(mats)
    assert sc.dispatch() == dispatch
    for a, b in zip(plane.download(), before):
        assert a.tobytes() == b.tobytes()
    plane.clear()
    st = plane.render(p)
    got = plane.download()
    fresh = capi.Scene(sd)
    fresh.set_triangle_materials(mats)
    fplane = capi.Plane(fresh, W, H)
    fst = fplane.render(p)
    want = fplane.download()
    assert_same_render_stats((*got, st), (*want, fst))
    assert_sums_close(got, want)
    assert not np.allclose(got[0], before[0], rtol=1e-3)  # the materials changed the image
    fplane.close(); fresh.close(); plane.close(); sc.close()


def test_errors_leave_the_scene_as_it_was(lib):
    torch = pytest.importorskip("torch")
    sd, first = with_six_materials("mesh:4097")
    n = sd.desc.n_triangles
    sc = capi.Scene(sd)
    box = capi.Scene(capi.SceneDescription("box"))
    had = random_assignment(n, first, seed=1)
    sc.set_triangle_materials(had)
    p = capi.default_params(width=32, height=32, pass_count=2, seed=3)
    ref = sc.render_host(p)
    other = halves_assignment(sd.triangles(), first)
    on_gpu = torch.from_numpy(other).to("cuda:0")
    bad = other.copy()
    bad[n // 2] = sd.desc.n_materials
    bad_gpu = torch.from_numpy(bad.astype(np.int32)).to("cuda:0")
    negative = torch.from_numpy(other.astype(np.int32)).to("cuda:0")
    negative[3] = -1
    hp = other.ctypes.data
    cases = [
        (None, hp, n, 0, "null argument"),
        (sc.handle, None, n, 0, "null argument"),
        (sc.handle, hp, n, capi.UPDATE_REBUILD, "unknown flag bits"),
        (sc.handle, hp, n, capi.UPDATE_DEVICE_POINTER | 8, "unknown flag bits"),
        (box.handle, hp, n, 0, "no triangle mesh"),
        (sc.handle, hp, n + 1, 0, f"{n + 1} materials given, the scene has {n} triangles"),
        (sc.handle, hp, n - 1, capi.UPDATE_DEVICE_POINTER, f"{n - 1} materials given"),
        (sc.handle, hp, n, capi.UPDATE_DEVICE_POINTER, "is not device or managed memory"),
        (sc.handle, on_gpu.data_ptr(), n, 0, "is device memory"),
        (sc.handle, on_gpu.data_ptr() + 2, n, capi.UPDATE_DEVICE_POINTER, "not aligned to 4 bytes"),
        (sc.handle, hp + 2, n, 0, "not aligned to 4 bytes"),
        (sc.handle, bad.ctypes.data, n, 0, f"materials[{n // 2}] = {sd.desc.n_materials} is out of range"),
        (sc.handle, bad_gpu.data_ptr(), n, capi.UPDATE_DEVICE_POINTER, f"out of range (largest {sd.desc.n_materials})"),
        (sc.handle, negative.data_ptr(), n, capi.UPDATE_DEVICE_POINTER, "out of range (largest 4294967295)"),
    ]
    for handle, ptr, count, flags, msg in cases:
        assert lib.ipt_scene_dispatch(None, None) == capi.IPT_ERR_INVALID  # leaves another message behind
        rc = lib.ipt_scene_set_triangle_materials(handle, ptr, C.c_uint64(count), flags)
        assert rc == capi.IPT_ERR_INVALID, msg
        err = lib.ipt_last_error().decode()
        assert err.startswith("ipt_scene_set_triangle_materials") and msg in err, err
        got = sc.render_host(p)
        assert_same_render_stats(got, ref)
        assert_sums_close(got, ref)
    # the Python binding refuses what the C call cannot take, before calling it
    for bad_arg, exc in ((other.astype(np.int64), TypeError), (other.astype(np.float32), TypeError), (other.reshape(-1, 1), ValueError),
                         (np.repeat(other, 2)[::2], TypeError), (other.tolist(), TypeError), (on_gpu.float(), TypeError),
                         (on_gpu.reshape(-1, 1), ValueError), (on_gpu.cpu(), ValueError)):
        with pytest.raises(exc):
            sc.set_triangle_materials(bad_arg)
    with pytest.raises(capi.IptError):
        sc.set_triangle_materials(other[:-1].copy())
    got = sc.render_host(p)
    assert_same_render_stats(got, ref)
    assert_sums_close(got, ref)
    box.close(); sc.close()
