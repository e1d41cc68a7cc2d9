"""Pin of the oracle against the compiled reference (oracle/_ref/libipt_ref.so): with libc drand48 seeded identically, a
whole render_sample pass of the restatement is BIT-IDENTICAL to the reference's, on every reference scene and on the C2
extension scene; so are its mixture, DDF and light-DDF samples. Where the reference is built it runs live (and the stored
copy of its outputs, tests/golden/pin_live.npz, must equal it); elsewhere the oracle is compared with that stored copy.

Each `*_record(side, chk, ...)` computes one comparison's arrays on either side: side "ref" with chk the compiled
reference, side "oracle" with chk the oracle. make_golden.py `pins` stores the reference side."""
import numpy as np
import pytest

import oracle_lib
from helpers import assert_same_record, bits, digest, reference_record
from ipt_b200 import capi

PASS_CASES = [("box", 4, 3), ("cornell", 4, 3), ("corner", 4, 3), ("square", 8, 4), ("smallpt", 2, 3), ("fractal", 4, 4),
              ("openspheres", 4, 3), ("box", 3, 4), ("mixedlights", 4, 3)]
MIX_SCENES = ["box", "cornell", "lightgrid:3x3", "fractal", "mixedlights"]
DDF_KINDS = [0, 1, 2, 40]
DDF_TOS = (None, [0.6, 0.0, 0.8], [0, 0, -1])
LIGHT_SCENES = ["box", "lightgrid:3x3", "corner", "fractal", "mixedlights"]
PASS_SAMPLE = np.sort(np.random.default_rng(0).choice(640 * 640, 4096, replace=False))  # stored pixels of a 640x640 pass


def _schedule(n, depth_max):
    out = []
    for _ in range(depth_max):
        out.append(n)
        n //= 2  # main.cpp:177 passes n_rays/2 down
    return out


def pass_record(side, chk, scene, n_rays, depth_max):
    """Verbatim src/main.cpp render_sample (640x640), srand48(4242): digests of pixels and counters, ray count, a pixel sample."""
    if side == "ref":
        h = chk.scene(scene)
        chk.set_tree(n_rays, depth_max)
        chk.seed(4242)
        r = chk.render(h, 1)
    else:
        sd = capi.SceneDescription(scene)
        p = capi.default_params(depth_max=depth_max, schedule=_schedule(n_rays, depth_max))
        chk.seed(4242)
        r = chk.render(sd.ptr, p, oracle_lib.RNG_DRAND48, 0)
    px = bits(r["pixels"])
    return dict(pixels=digest(px), counters=digest(r["counters"].astype(np.uint64)), rays=np.uint64(r["rays"]),
                sample=px.reshape(-1)[PASS_SAMPLE], max=np.float32(r["pixels"].max()))


def mix_record(side, chk, scene):
    """unite(light_ddf,1,sdf,1) at the surface hits of three camera rays (main.cpp:142-143): 400 sample() directions, and
    the mixture / sdf value() of the non-zero ones (value(vec3()) reads the racy Lighting::last_sample; the loop discards it)."""
    sd = capi.SceneDescription(scene)
    orc = oracle_lib.load_oracle()
    o0, d0 = orc.camera_rays(sd.ptr, np.array([[0.5, 0.3], [0.62, 0.45], [0.5, 0.5]], np.float32))
    out = {}
    for i, (o, d) in enumerate(zip(o0, d0)):
        if orc.trace_batch(sd.ptr, [o], [d])["prim"][0] == capi.IPT_NO_HIT:
            continue
        chk.seed(11)
        w, m, s = chk.mix_sample(chk.scene(scene) if side == "ref" else sd.ptr, o, d, 400)
        nz = np.any(w != 0, axis=1)
        out.update({f"w{i}": bits(w), f"m{i}": bits(m[nz]), f"s{i}": bits(s[nz])})
    return out


def ddf_record(side, chk, kind):
    out = {}
    for j, to in enumerate(DDF_TOS):
        chk.seed(5)
        out[f"to{j}"] = bits(chk.ddf_sample(kind, 300, to=to))
    return out


def light_record(side, chk, scene):
    """Lighting::distributionInPoint(pos) (CollectionLighting.cpp:12-21): value() on 300 directions, 200 sample()s."""
    rng = np.random.default_rng(2)
    w = rng.normal(size=(300, 3)).astype(np.float32)
    w /= np.linalg.norm(w, axis=1, keepdims=True).astype(np.float32)
    w[:, 2] = np.abs(w[:, 2])
    pos = np.array([0.1, -0.5, -1.0], np.float32)
    sd = capi.SceneDescription(scene)
    h = chk.scene(scene) if side == "ref" else sd.ptr
    value = bits(chk.light_ddf_value(h, pos, w))
    chk.seed(3)
    return dict(value=value, sample=bits(chk.light_ddf_sample(h, pos, 200)))


def pass_key(scene, n_rays, depth_max):
    return f"pass_{scene}_{n_rays}_{depth_max}"


@pytest.mark.parametrize("scene,n_rays,depth_max", PASS_CASES)
def test_whole_pass_bit_identical_to_reference(scene, n_rays, depth_max, lib, oracle, ref_or_none, pins):
    """Verbatim src/main.cpp render_sample (640x640) vs the oracle, same srand48 seed: pixels, counters and ray count."""
    want = reference_record(pins, ref_or_none, pass_key(scene, n_rays, depth_max), lambda r: pass_record("ref", r, scene, n_rays, depth_max))
    assert_same_record(pass_record("oracle", oracle, scene, n_rays, depth_max), want, scene)
    assert want["max"] > 0


def test_parametrised_loop_equals_verbatim_loop(ref):
    """oracle/ref_driver.cpp's W,H loop (used for non-640 goldens) is the reference loop at 640x640."""
    h = ref.scene("box")
    ref.set_tree(2, 3)
    ref.seed(7); a = ref.render(h, 1)
    ref.seed(7); b = ref.render(h, 1, 640, 640, verbatim=False)
    assert np.array_equal(bits(a["pixels"]), bits(b["pixels"])) and a["rays"] == b["rays"]


@pytest.mark.parametrize("scene", MIX_SCENES)
def test_mixture_samples_bit_identical(scene, lib, oracle, ref_or_none, pins):
    """unite(light_ddf,1,sdf,1) at a surface hit (main.cpp:142-143): sample(), value() and sdf value() sequences."""
    want = reference_record(pins, ref_or_none, f"mix_{scene}", lambda r: mix_record("ref", r, scene))
    assert_same_record(mix_record("oracle", oracle, scene), want, scene)
    assert len(want) > 0


@pytest.mark.parametrize("kind", DDF_KINDS)
def test_base_ddf_samples_bit_identical(kind, oracle, ref_or_none, pins):
    want = reference_record(pins, ref_or_none, f"ddf_{kind}", lambda r: ddf_record("ref", r, kind))
    assert_same_record(ddf_record("oracle", oracle, kind), want, kind)


def test_light_ddf_value_and_sample(lib, oracle, ref_or_none, pins):
    """Lighting::distributionInPoint(pos) (CollectionLighting.cpp:12-21): the iteratively renormalised weights."""
    for scene in LIGHT_SCENES:
        want = reference_record(pins, ref_or_none, f"light_{scene}", lambda r: light_record("ref", r, scene))
        assert_same_record(light_record("oracle", oracle, scene), want, scene)
