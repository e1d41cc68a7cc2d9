"""CPU checks of the LBVH refit restatement (bvh_refit below: what ipt_scene_update_triangles computes without
IPT_UPDATE_REBUILD, restated in numpy float32 in the device's operation order). Over unchanged triangles it reproduces the
tree the oracle builds (oracle/ipt_oracle_mesh.inc) byte for byte, and after a deformation it keeps the topology while every
box still bounds the padded triangles below it. No GPU."""
import numpy as np
import pytest

from ipt_b200 import capi

PAD = np.float32(7.62939453125e-06)  # ipt_lbvh.cuh: padded_box


def jitter(tris, seed, scale=1e-3):
    """Every vertex of every triangle moved by up to `scale` (v0 and both edges perturbed independently)."""
    rng = np.random.default_rng(seed)
    return (tris + rng.uniform(-scale, scale, tris.shape)).astype(np.float32)


def carry_half(tris, seed, centre=(0.0, 0.0, 0.0), size=1.0):
    """Half of the triangles, chosen at random, carried rigidly across the box of half-size `size` about `centre` (their
    first vertex mirrored through the centre, their edges kept)."""
    rng = np.random.default_rng(seed)
    out = tris.copy()
    pick = rng.random(len(tris)) < 0.5
    c = np.asarray(centre, np.float32)
    out[pick, 0:3] = (c - 0.9 * (out[pick, 0:3] - c) + size * rng.uniform(-0.05, 0.05, (int(pick.sum()), 3))).astype(np.float32)
    return out


def padded_boxes(tris):
    """The leaf boxes of the tree per original triangle (k_lbvh_bounds + padded_box): the tight box of (v0, v0+e1, v0+e2)
    widened by (1 + max |coordinate|) * 2^-17, every step one float32 operation rounded to nearest."""
    tris = np.ascontiguousarray(tris, np.float32).reshape(-1, 9)
    v0 = tris[:, 0:3]
    v = np.stack([v0, v0 + tris[:, 3:6], v0 + tris[:, 6:9]])
    lo, hi = v.min(0), v.max(0)
    m = np.maximum(np.abs(lo).max(1), np.abs(hi).max(1))
    pad = ((m + np.float32(1)) * PAD)[:, None]
    return lo - pad, hi + pad


def bvh_refit(tris, nodes, sorted_ids):
    """The boxes of an existing tree (64-byte nodes as ipt_bvh_export gives them, sorted ids) recomputed for new triangles:
    the topology (left, right, parent, pad) is kept; a leaf slot gets the padded box of its triangle, an internal slot the
    componentwise min / max of its child's two slots (k_lbvh_refit). Levels are filled from the deepest up."""
    out = np.array(nodes, copy=True)
    if len(out) == 0:
        return out
    lo, hi = padded_boxes(tris)
    ids = np.asarray(sorted_ids, np.int64)
    lo, hi = lo[ids], hi[ids]  # per sorted position
    kids = {"0": out["left"].astype(np.int64), "1": out["right"].astype(np.int64)}
    levels, level = [], np.array([0], np.int64)
    while level.size:
        levels.append(level)
        below = np.concatenate([kids["0"][level], kids["1"][level]])
        level = below[(below & 0x80000000) == 0]
    for level in reversed(levels):
        for slot, child in kids.items():
            c = child[level]
            leaf = (c & 0x80000000) != 0
            l = np.empty((len(level), 3), np.float32)
            h = np.empty((len(level), 3), np.float32)
            l[leaf], h[leaf] = lo[c[leaf] & 0x7FFFFFFF], hi[c[leaf] & 0x7FFFFFFF]
            inner = c[~leaf]
            l[~leaf] = np.minimum(out["lo0"][inner], out["lo1"][inner])
            h[~leaf] = np.maximum(out["hi0"][inner], out["hi1"][inner])
            out["lo" + slot][level], out["hi" + slot][level] = l, h
    return out


@pytest.mark.parametrize("n", [2, 3, 100, 4097])
def test_refit_of_unchanged_triangles_reproduces_the_build(n, lib, oracle):
    tris = capi.SceneDescription(f"mesh:{n}").triangles().copy()
    nodes, ids, _ = oracle.bvh_build(tris)
    scrambled = nodes.copy()
    for f in ("lo0", "hi0", "lo1", "hi1"):
        scrambled[f] = np.float32(123.0)  # every box must be recomputed, none carried over
    assert bvh_refit(tris, scrambled, ids).tobytes() == nodes.tobytes()


@pytest.mark.parametrize("deform", ["jitter", "carry_half"])
@pytest.mark.parametrize("n", [2, 3, 4097])
def test_refit_keeps_the_topology_and_bounds_the_moved_triangles(n, deform, lib, oracle):
    tris = capi.SceneDescription(f"mesh:{n}").triangles().copy()
    nodes, ids, _ = oracle.bvh_build(tris)
    moved = jitter(tris, n) if deform == "jitter" else carry_half(tris, n)
    refit = bvh_refit(moved, nodes, ids)
    for f in ("left", "right", "parent", "pad"):
        assert np.array_equal(refit[f], nodes[f]), f
    lo, hi = padded_boxes(moved)

    def below(child):  # sorted positions of the leaves under a child
        if child & 0x80000000:
            return [int(child & 0x7FFFFFFF)]
        nd = refit[child]
        return below(int(nd["left"])) + below(int(nd["right"]))

    for k, nd in enumerate(refit):
        for child, clo, chi in ((int(nd["left"]), nd["lo0"], nd["hi0"]), (int(nd["right"]), nd["lo1"], nd["hi1"])):
            leaves = ids[below(child)]
            assert (clo <= lo[leaves]).all() and (chi >= hi[leaves]).all(), (k, child)
            if child & 0x80000000:  # a leaf slot holds exactly the padded box
                assert np.array_equal(clo, lo[leaves[0]]) and np.array_equal(chi, hi[leaves[0]])
            else:  # an internal slot is the union of that child's two slots
                c = refit[child]
                assert np.array_equal(clo, np.minimum(c["lo0"], c["lo1"])) and np.array_equal(chi, np.maximum(c["hi0"], c["hi1"]))
    if deform == "carry_half" and n > 100:  # the move is large enough to change the boxes, not only their last bits
        assert not np.array_equal(refit["lo0"], nodes["lo0"])
