"""tools/mesh_update.py — what moving a mesh costs: ipt_scene_update_triangles (refit / rebuild, from host or device memory)
against creating the scene anew, and the C3 render (1920x1080, depth 8, one child per hit) after a refit under deformations
of growing size against the same vertices rebuilt.

    python tools/mesh_update.py [--out DIR] [--sizes 1000000,10000000] [--repeats 5] [--render-steps 4]

One B200 run prints the card's name, power limit and max SM clock first, then one JSON line per measurement; the lines also
go to DIR/mesh_update.jsonl. Times are a host clock around the synchronous call (the update returns once the tree is
complete), after one warm-up call, over `--repeats` calls: median and minimum. Render rates are whole ipt_render calls
(host clock, 16 passes each) after one warm-up call.
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from ipt_b200 import capi  # noqa: E402

C3 = dict(width=1920, height=1080, depth_max=8, schedule=[1] * 8, pass_count=16)


def card():
    q = "name,power.limit,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    line = r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown, unknown, unknown"
    return dict(zip(q.split(","), (v.strip() for v in line.split(","))))


def timed(fn, repeats):
    fn()  # warm-up
    ts = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return dict(median_ms=float(np.median(ts)), min_ms=float(np.min(ts)), repeats=repeats)


def move_triangles(tris, amplitude, seed=1):
    """Every triangle translated rigidly by a uniform random offset of up to `amplitude` per axis (edges kept)."""
    out = tris.copy()
    if amplitude:
        rng = np.random.default_rng(seed)
        out[:, 0:3] += rng.uniform(-amplitude, amplitude, (len(tris), 3)).astype(np.float32)
    return out


def emit(rec, sink):
    line = json.dumps(rec)
    print(line, flush=True)
    sink.write(line + "\n")


def update_costs(n, repeats, sink):
    import torch

    sd = capi.SceneDescription(f"mesh:{n}")
    tris = sd.triangles().copy()
    moved = move_triangles(tris, 0.01)
    on_gpu = torch.from_numpy(moved).to("cuda:0")
    torch.cuda.synchronize()
    create = timed(lambda: capi.Scene(sd).close(), repeats)
    emit(dict(what="ipt_scene_create", triangles=n, **create), sink)
    sc = capi.Scene(sd)
    for rebuild in (False, True):
        for src, arr in (("host", moved), ("device", on_gpu)):
            r = timed(lambda: sc.update_triangles(arr, rebuild=rebuild), repeats)
            emit(dict(what="ipt_scene_update_triangles", form="rebuild" if rebuild else "refit", input=src, triangles=n,
                      vs_create=r["median_ms"] / create["median_ms"], **r), sink)
    sc.close()


def render_after_update(amplitudes, steps, sink):
    sd = capi.SceneDescription("mesh:1000000")
    tris = sd.triangles().copy()
    sc = capi.Scene(sd)
    plane = capi.Plane(sc, C3["width"], C3["height"])
    for amp in amplitudes:
        moved = move_triangles(tris, amp)
        for form in ("refit", "rebuild"):
            # refit: the tree built over the original pose, boxes recomputed for the moved one; rebuild: built over the moved pose
            if form == "refit":
                sc.update_triangles(tris, rebuild=True)
            sc.update_triangles(moved, rebuild=form == "rebuild")
            plane.clear()
            plane.render(capi.default_params(**C3))  # warm-up
            paths = rays = nodes = 0
            t0 = time.perf_counter()
            for k in range(steps):
                st = plane.render(capi.default_params(pass_begin=16 * (k + 1), **C3))
                paths += st.paths; rays += st.rays; nodes += st.bvh_nodes_visited
            dt = time.perf_counter() - t0
            emit(dict(what="c3_render", form=form, amplitude=amp, steps=steps, mpaths_per_s=paths / dt / 1e6,
                      mrays_per_s=rays / dt / 1e6, bvh_nodes_per_ray=nodes / rays), sink)
    plane.close(); sc.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=".", help="directory of mesh_update.jsonl")
    ap.add_argument("--sizes", default="1000000,10000000")
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--render-steps", type=int, default=4)
    ap.add_argument("--amplitudes", default="0,0.001,0.003,0.01,0.03,0.1,0.3")
    a = ap.parse_args()
    lib = capi.load()
    if lib.ipt_device_count() < 1:
        raise SystemExit("mesh_update.py measures on a CUDA device: none found")
    out = Path(a.out)
    out.mkdir(parents=True, exist_ok=True)
    with open(out / "mesh_update.jsonl", "w") as sink:
        emit(dict(what="card", **card()), sink)
        for n in (int(v) for v in a.sizes.split(",")):
            update_costs(n, a.repeats, sink)
        render_after_update([float(v) for v in a.amplitudes.split(",")], a.render_steps, sink)


if __name__ == "__main__":
    main()
