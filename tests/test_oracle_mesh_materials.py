"""CPU checks of the oracle with per-triangle materials (tests/oracle_tri_mats.c, ipt_oracle_set_triangle_materials):
without an attached array it is the oracle bit for bit, an attached array equal to the description's triangle_material
changes no bit of a render or of the mixture at a mesh hit, and under a mixed assignment a hit on triangle k is shaded
with materials[k]. The material set and the assignments are shared with test_gpu_mesh_materials.py. No GPU."""
import ctypes as C

import numpy as np
import pytest

import oracle_lib
import oracle_tri_mats
from helpers import bits, custom_scene
from ipt_b200 import capi

LAMBERT, GLOSSY = 0, 1


@pytest.fixture(scope="module")
def oracle(lib):
    """The oracle that can attach per-triangle materials (tests/oracle_tri_mats.py) in place of the session's oracle."""
    return oracle_tri_mats.load()


def material(ddf, albedo, kd=0.0, ks=0.0, exponent=0.0):
    m = capi.Material()
    m.ddf, m.albedo, m.kd, m.ks, m.exponent = ddf, albedo, kd, ks, exponent
    return m


def six_materials():
    """Lambert with albedo 0.3 and 0.9, glossy lobes with exponents 5 and 60, a glossy material that is half diffuse, and a
    black Lambert surface."""
    return [material(LAMBERT, 0.3), material(LAMBERT, 0.9), material(GLOSSY, 0.9, 0.1, 0.9, 5.0), material(GLOSSY, 0.9, 0.05, 0.95, 60.0),
            material(GLOSSY, 0.8, 0.5, 0.5, 20.0), material(LAMBERT, 0.0)]


def with_six_materials(base, **kw):
    """`base` (a sample scene name) with the six materials appended to its own: (description, index of the first of them).
    Indices past IPT_INLINE_MATS (4) are among them for every base."""
    sd = capi.SceneDescription(base)
    own = [capi.Material.from_buffer_copy(sd.desc.materials[i]) for i in range(sd.desc.n_materials)]
    return custom_scene(base, materials=own + six_materials(), **kw), len(own)


def random_assignment(n, first, seed=0):
    return (first + np.random.default_rng(seed).integers(0, 6, n)).astype(np.uint32)


def halves_assignment(tris, first):
    """Coherent regions: the material of a triangle follows the side of its centroid's median plane on each axis."""
    t = np.asarray(tris, np.float64).reshape(-1, 9)
    c = t[:, 0:3] + (t[:, 3:6] + t[:, 6:9]) / 3
    side = (c > np.median(c, axis=0)).astype(np.int64)
    return (first + (side[:, 0] + 2 * side[:, 1] + 4 * side[:, 2]) % 6).astype(np.uint32)


def mesh_hits(oracle, sd, n=1500, seed=0):
    """Rays from random points of the box aimed at the centroids of random triangles, those whose first hit is a
    triangle: (origins, unit directions as the renderer's rays have them, triangle index)."""
    rng = np.random.default_rng(seed)
    tris = sd.triangles()
    pick = rng.integers(0, len(tris), n)
    cen = tris[pick, 0:3] + (tris[pick, 3:6] + tris[pick, 6:9]) / np.float32(3)
    o = rng.uniform(-0.95, 0.95, (n, 3)).astype(np.float32)
    d = cen - o
    d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
    prim = oracle.trace_batch(sd.ptr, o, d, use_bvh=1)["prim"]
    hit = (prim != capi.IPT_NO_HIT) & (prim >= sd.desc.n_prims)
    return o[hit], d[hit], (prim[hit] - sd.desc.n_prims).astype(np.int64)


def render(oracle, sd, **kw):
    p = capi.default_params(**{**dict(width=16, height=16, pass_count=1, seed=11, flags=capi.FLAG_KEEP_ZERO_WEIGHT), **kw})
    return oracle.render(sd.ptr, p, oracle_lib.RNG_PHILOX, 1)


def assert_same_render(a, b):
    for k in ("sum", "sumsq", "counters", "pixels"):
        assert a[k].tobytes() == b[k].tobytes(), k
    assert a["rays"] == b["rays"] and a["rays_at_depth"] == b["rays_at_depth"]


@pytest.mark.parametrize("base", ["mesh:2000", "smallpt"])
def test_without_an_array_it_is_the_oracle(base, lib, oracle):
    """The hook changes nothing by itself: renders (tree and BVH tracing), traces and the mixture at mesh hits equal the
    session oracle's bit for bit."""
    from test_gpu_dispatch_matrix import smallpt_mesh

    plain = oracle_lib.load_oracle()
    sd, _ = with_six_materials(base, triangles=smallpt_mesh() if base == "smallpt" else None)
    for use_bvh in (0, 1):
        p = capi.default_params(width=16, height=16, pass_count=1, seed=11, depth_max=3, schedule=[8, 4, 2], flags=capi.FLAG_KEEP_ZERO_WEIGHT)
        assert_same_render(oracle.render(sd.ptr, p, oracle_lib.RNG_PHILOX, use_bvh), plain.render(sd.ptr, p, oracle_lib.RNG_PHILOX, use_bvh))
    if base == "smallpt":
        return
    o, d, _ = mesh_hits(oracle, sd)
    a, b = oracle.trace_batch(sd.ptr, o, d), plain.trace_batch(sd.ptr, o, d)
    for k in a:
        assert a[k].tobytes() == b[k].tobytes(), k
    for i in range(5):
        oracle.seed(7)
        x = oracle.mix_sample(sd.ptr, o[i], d[i], 200)
        plain.seed(7)
        y = plain.mix_sample(sd.ptr, o[i], d[i], 200)
        for u, v in zip(x, y):
            assert bits(u).tobytes() == bits(v).tobytes()


@pytest.mark.parametrize("index", [0, 5])
def test_uniform_array_reproduces_triangle_material(index, lib, oracle):
    """A description whose triangle_material is `index` against the same mesh with triangle_material 0 and an attached array
    of `index` everywhere: render (full 16/8/4/2 tree and the depth-8 one-child tree), mix_sample and mix_value at mesh
    hits, bit for bit."""
    sd, first = with_six_materials("mesh:2000", triangle_material=index)
    sd0, _ = with_six_materials("mesh:2000", triangle_material=0)
    n = sd.desc.n_triangles
    plain = [render(oracle, sd), render(oracle, sd, depth_max=8, schedule=[1] * 8, pass_count=4)]
    before0 = render(oracle, sd0)
    o, d, _ = mesh_hits(oracle, sd)
    assert len(o) > 50
    with oracle.triangle_materials(sd0.ptr, np.full(n, index, np.uint32)):
        attached = [render(oracle, sd0), render(oracle, sd0, depth_max=8, schedule=[1] * 8, pass_count=4)]
        for a, b in zip(attached, plain):
            assert_same_render(a, b)
        rng = np.random.default_rng(1)
        for i in rng.choice(len(o), 8, replace=False):
            oracle.seed(99)
            w, mv, sv = oracle.mix_sample(sd0.ptr, o[i], d[i], 200)
            oracle.seed(99)
            w2, mv2, sv2 = oracle.mix_sample(sd.ptr, o[i], d[i], 200)
            assert bits(w).tobytes() == bits(w2).tobytes() and bits(mv).tobytes() == bits(mv2).tobytes() and bits(sv).tobytes() == bits(sv2).tobytes()
            v = [oracle.mix_value(x.ptr, o[i], d[i], w) for x in (sd0, sd)]
            for x, y in zip(*v):
                assert bits(x).tobytes() == bits(y).tobytes()
    assert_same_render(render(oracle, sd0), before0)  # detached again


@pytest.mark.parametrize("assign", ["random", "halves"])
def test_hit_on_triangle_k_has_material_k(assign, lib, oracle):
    """Under a mixed assignment the mixture at a hit on triangle k equals, bit for bit, the mixture of the same mesh with
    triangle_material = materials[k] and nothing attached; the render differs from the uniform one."""
    sd, first = with_six_materials("mesh:2000")
    tris = sd.triangles()
    mats = random_assignment(len(tris), first, seed=3) if assign == "random" else halves_assignment(tris, first)
    assert set(np.unique(mats)) == set(range(first, first + 6))
    o, d, k = mesh_hits(oracle, sd)
    uniform = render(oracle, sd)
    by_index = {m: with_six_materials("mesh:2000", triangle_material=m)[0] for m in range(first, first + 6)}
    seen = set()
    with oracle.triangle_materials(sd.ptr, mats):
        mixed = render(oracle, sd)
        for i in np.random.default_rng(2).choice(len(o), 40, replace=False):
            want = by_index[int(mats[k[i]])]
            seen.add(int(mats[k[i]]))
            oracle.seed(5)
            got = oracle.mix_sample(sd.ptr, o[i], d[i], 100)
            oracle.seed(5)
            ref = oracle.mix_sample(want.ptr, o[i], d[i], 100)
            for x, y in zip(got, ref):
                assert bits(x).tobytes() == bits(y).tobytes()
            for x, y in zip(oracle.mix_value(sd.ptr, o[i], d[i], got[0]), oracle.mix_value(want.ptr, o[i], d[i], got[0])):
                assert bits(x).tobytes() == bits(y).tobytes()
    assert len(seen) >= 4
    assert np.array_equal(mixed["counters"], uniform["counters"])  # the same samples per cell ...
    assert not np.array_equal(mixed["sum"], uniform["sum"])  # ... shaded differently
    assert mixed["sum"].sum() < uniform["sum"].sum()  # the base material (albedo 1) is brighter than the mix on average


def test_out_of_range_index_is_refused(lib, oracle):
    sd, first = with_six_materials("mesh:100")
    n = sd.desc.n_triangles
    bad = np.zeros(n, np.uint32)
    bad[7] = sd.desc.n_materials
    assert oracle.lib.ipt_oracle_set_triangle_materials(sd.ptr, bad.ctypes.data_as(C.POINTER(C.c_uint32))) == 1
    before = render(oracle, sd, width=8, height=8)
    oracle.set_triangle_materials(sd.ptr, None)  # detaching what is not attached is a no-op
    assert_same_render(render(oracle, sd, width=8, height=8), before)
