"""The light tables of a scene (ipt_light_tables_export: area, surface power, normal, mixture weight, cdf, guide) against
the oracle's prepare_light and prepare_weights, bit for bit: for created scenes of every light set of
test_gpu_light_update.py, of no lights, of one light of each kind, of 8 and 9 area lights (either side of the light LBVH),
of the L4 set with zero-power plateaus, and after ipt_scene_update_lights from host and device memory. The cdf is the
float32 running sum of the oracle's weights and guide[b] the first i with b / 4096 < cdf[i]."""
import numpy as np
import pytest

from helpers import bits, custom_scene, make_light
from ipt_b200 import capi
from test_gpu_dispatch_matrix import DIAMOND, POINT, ROWS, SPHERE, SPHERE_INVERTED, TRIANGLE, diamonds, lights_l4, scene_lights
from test_gpu_light_update import UPDATE_ROWS, as_input, copies, move_lights

pytestmark = pytest.mark.gpu

ONE_LIGHT = {
    "diamond": make_light(DIAMOND, (0.1, -0.9, -0.15), (0.2, 0.0, 0.0), (0.0, 0.2, 0.05), power=2.0),
    "triangle": make_light(TRIANGLE, (-0.3, 0.2, 0.6), (0.3, 0.1, -0.05), (-0.1, 0.25, 0.02), power=0.7),
    "sphere": make_light(SPHERE, (0.2, 0.3, 0.7), radius=0.1, power=4.0),
    "inverted-sphere": make_light(SPHERE_INVERTED, (0.0, 0.0, 0.0), radius=3.0, power=1.5),
    "point": make_light(POINT, (0.1, 0.2, 0.5), power=3.0),
}


def expected(oracle, sd):
    """The oracle's tables, with the cdf and guide built from its weights."""
    t = oracle.light_tables(sd.ptr, sd.desc.n_lights)
    cdf = np.zeros(len(t["weight"]), np.float32)
    acc = np.float32(0)
    for i, w in enumerate(t["weight"]):
        acc = np.float32(acc + w)
        cdf[i] = acc
    guide = np.zeros(capi.LIGHT_GUIDE_WORDS, np.uint32)
    i = 0
    for b in range(capi.LIGHT_GUIDE_WORDS):
        edge = np.float32(b) / np.float32(4096)
        while i < len(cdf) and not edge < cdf[i]:
            i += 1
        guide[b] = i
    return dict(t, cdf=cdf, guide=guide)


def assert_tables_match(sc, sd, oracle, nan_weights=False):
    got, want = sc.light_tables(), expected(oracle, sd)
    for k in ("area", "surface_power", "normal", "guide"):
        assert np.array_equal(bits(got[k]), bits(want[k])), k
    for k in ("weight", "cdf"):
        if nan_weights:  # 0/0: the host and the device give NaNs of different bit patterns
            assert np.array_equal(np.isnan(got[k]), np.isnan(want[k])), k
            ok = ~np.isnan(want[k])
            assert np.array_equal(bits(got[k][ok]), bits(want[k][ok])), k
        else:
            assert not np.isnan(want[k]).any(), k
            assert np.array_equal(bits(got[k]), bits(want[k])), k


def scene_of(lights):
    sd = custom_scene("box", lights=lights)
    return sd, capi.Scene(sd)


@pytest.mark.parametrize("name", UPDATE_ROWS)
def test_created_scene_tables_match_oracle(name, lib, oracle):
    sd = ROWS[name].build()
    sc = capi.Scene(sd)
    assert_tables_match(sc, sd, oracle)
    sc.close()


@pytest.mark.parametrize("kind", list(ONE_LIGHT))
def test_one_light_of_each_kind(kind, lib, oracle):
    sd, sc = scene_of([ONE_LIGHT[kind]])
    assert sc.dispatch()["light_inline"] == 1
    assert_tables_match(sc, sd, oracle)
    sc.close()


def test_no_lights(lib, oracle):
    sd, sc = scene_of([])
    t = sc.light_tables()
    assert not t["guide"].any() and t["weight"].size == 0
    assert_tables_match(sc, sd, oracle)
    sc.close()


@pytest.mark.parametrize("n", [8, 9])
def test_either_side_of_the_light_tree(n, lib, oracle):
    sd, sc = scene_of(diamonds(np.random.default_rng(40 + n), n))
    assert sc.dispatch()["n_light_bvh"] == (n if n > 8 else 0)
    assert_tables_match(sc, sd, oracle)
    sc.close()


def test_zero_power_plateaus(lib, oracle):
    sd, sc = scene_of(lights_l4())
    t = sc.light_tables()
    assert (np.diff(t["cdf"]) == 0).sum() >= 50 and np.bincount(t["guide"]).max() > 1
    assert_tables_match(sc, sd, oracle)
    sc.close()


def test_zero_power_first_light_gives_nan_weights(lib, oracle):
    """Light 0 of zero power: its weight is 0/0 and the cdf NaN from there on, on the host and on the device alike."""
    lights = diamonds(np.random.default_rng(46), 12)
    lights[0].power = 0.0
    sd, sc = scene_of(lights)
    t = sc.light_tables()
    assert np.isnan(t["weight"][0]) and np.isnan(t["cdf"]).all()
    assert_tables_match(sc, sd, oracle, nan_weights=True)
    sc.close()


@pytest.mark.parametrize("rebuild", [False, True], ids=["refit", "rebuild"])
@pytest.mark.parametrize("src", ["host", "device"])
@pytest.mark.parametrize("name", ["L1-diamonds", "L4-skewed", "L6-sphere", "S1-dome", "M1-mixedlights"])
def test_updated_scene_tables_match_oracle(name, src, rebuild, lib, oracle):
    sd = ROWS[name].build()
    sc = capi.Scene(sd)
    moved = move_lights(copies(scene_lights(sd)), seed=9)
    sc.update_lights(as_input(moved, src), rebuild=rebuild)
    assert_tables_match(sc, custom_scene(sd.name, lights=moved), oracle)
    sc.close()


def test_unknown_light_kind_is_refused(lib):
    lights = diamonds(np.random.default_rng(47), 3)
    lights[1].kind = POINT + 1
    with pytest.raises(capi.IptError, match="unknown light kind") as e:
        capi.Scene(custom_scene("box", lights=lights))
    assert e.value.code == capi.IPT_ERR_INVALID
