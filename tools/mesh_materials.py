"""tools/mesh_materials.py — what per-triangle materials cost in the render: the C3 scene (1 M triangles, 1920x1080) under
its own depth-8 one-child tree and under the reference's 16/8/4/2 tree, with no ipt_scene_set_triangle_materials call, with
an array equal to triangle_material everywhere, and with six materials assigned at random. The scene's material list is the
same in all three states (its own Lambert material plus six: Lambert 0.3 / 0.9, glossy exponents 5 / 60, a half-diffuse
glossy one, black), so only the per-hit lookup differs. Also times the call itself from host and from device memory.

    python tools/mesh_materials.py [--out DIR] [--rounds 3] [--steps 4] [--repeats 5]

One B200 run prints the card's name, power limit and max SM clock first, then one JSON line per measurement; the lines also
go to DIR/mesh_materials.jsonl. The three states are rendered by three scenes, alternated round by round. A rate is whole
ipt_render calls (host clock around synchronous calls) after one warm-up call: C3 calls render 16 passes, 16/8/4/2 calls one
pass. The summary lines give the median over the rounds and its ratio to the state without the call.
"""
from __future__ import annotations

import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))
sys.path.insert(0, str(ROOT / "tests"))

from ipt_b200 import capi  # noqa: E402
from mesh_update import card, emit, timed  # noqa: E402
from test_oracle_mesh_materials import random_assignment, with_six_materials  # noqa: E402

WORKLOADS = {
    "c3": dict(width=1920, height=1080, depth_max=8, schedule=[1] * 8, pass_count=16),
    "c3_16_8_4_2": dict(width=1920, height=1080, depth_max=4, schedule=[16, 8, 4, 2], pass_count=1),
}
STATES = ("none", "uniform", "random6")


def main():
    import argparse

    import torch

    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=".", help="directory of mesh_materials.jsonl")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=4, help="timed ipt_render calls per measurement")
    ap.add_argument("--repeats", type=int, default=5, help="timed calls of ipt_scene_set_triangle_materials")
    a = ap.parse_args()
    if capi.load().ipt_device_count() < 1:
        raise SystemExit("mesh_materials.py measures on a CUDA device: none found")
    out = Path(a.out)
    out.mkdir(parents=True, exist_ok=True)
    sd, first = with_six_materials("mesh:1000000")
    n = sd.desc.n_triangles
    arrays = {"uniform": np.full(n, sd.desc.triangle_material, np.uint32), "random6": random_assignment(n, first, seed=1)}
    scenes = {s: capi.Scene(sd) for s in STATES}
    for s, arr in arrays.items():
        scenes[s].set_triangle_materials(arr)
    with open(out / "mesh_materials.jsonl", "w") as sink:
        emit(dict(what="card", **card()), sink)
        on_gpu = torch.from_numpy(arrays["random6"]).to("cuda:0")
        torch.cuda.synchronize()
        for src, arr in (("host", arrays["random6"]), ("device", on_gpu)):
            emit(dict(what="ipt_scene_set_triangle_materials", input=src, triangles=n, **timed(lambda: scenes["random6"].set_triangle_materials(arr), a.repeats)), sink)
        rates = {(w, s): [] for w in WORKLOADS for s in STATES}
        for w, params in WORKLOADS.items():
            planes = {s: capi.Plane(sc, params["width"], params["height"]) for s, sc in scenes.items()}
            for r in range(a.rounds):
                for s in STATES:
                    plane = planes[s]
                    plane.clear()
                    plane.render(capi.default_params(**params))  # warm-up
                    paths = rays = 0
                    t0 = time.perf_counter()
                    for k in range(a.steps):
                        st = plane.render(capi.default_params(pass_begin=params["pass_count"] * (k + 1), **params))
                        paths += st.paths; rays += st.rays
                    dt = time.perf_counter() - t0
                    rates[w, s].append(paths / dt / 1e6)
                    emit(dict(what="render", workload=w, state=s, round=r, steps=a.steps, mpaths_per_s=paths / dt / 1e6,
                              mrays_per_s=rays / dt / 1e6), sink)
            for p in planes.values():
                p.close()
            base = float(np.median(rates[w, "none"]))
            for s in STATES:
                med = float(np.median(rates[w, s]))
                emit(dict(what="summary", workload=w, state=s, rounds=a.rounds, median_mpaths_per_s=med, vs_none=med / base,
                          all_mpaths_per_s=rates[w, s]), sink)
    for sc in scenes.values():
        sc.close()


if __name__ == "__main__":
    main()
