"""tools/light_update.py — what moving lights costs: ipt_scene_update_lights (refit / rebuild, from host or device memory)
against creating the scene anew, and the C5 render (lightgrid:100x100, the `c5` entry of tools/run_configs.py) after every
light is moved by a seeded offset, refitted against rebuilt.

    python tools/light_update.py [--out DIR] [--scenes lightgrid:100x100,lightgrid:250x400] [--repeats 5] [--render-steps 2]

One run prints the card's name, power limit and max SM clock first, then one JSON line per measurement; the lines also go
to DIR/light_update.jsonl. Update and create times are a host clock around the synchronous call (the update returns once
the tables and the tree are complete), after one warm-up call, over `--repeats` calls: median and minimum. Render rates are
device time of whole ipt_render calls (CUDA events, ipt_render_stats::ms_total) after one warm-up pass.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from ipt_b200 import capi  # noqa: E402

C5 = dict(scene="lightgrid:100x100", width=2048, height=2048, depth_max=4, schedule=[16, 8, 4, 2], passes=16, tile=(768, 768, 512, 512))
MARGIN = 0.995  # moved corners stay inside [-MARGIN, MARGIN]^3


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


def records(sd):
    """The scene's lights as an (n, 12) int32 array of ipt_light records."""
    n = sd.desc.n_lights
    return np.ctypeslib.as_array(C.cast(sd.desc.lights, C.POINTER(C.c_int32)), shape=(n, 12)).copy()


def move(rec, amplitude, seed=1):
    """Every light translated by a uniform random offset of up to `amplitude` per axis, clamped so that its corners stay
    inside the box; axes and powers kept."""
    out = rec.copy()
    if not amplitude:
        return out
    f = out.view(np.float32)
    pos, xa, ya = f[:, 1:4], f[:, 4:7], f[:, 7:10]
    lo = np.minimum(0, xa) + np.minimum(0, ya)  # corner offsets relative to the position
    hi = np.maximum(0, xa) + np.maximum(0, ya)
    rng = np.random.default_rng(seed)
    moved = pos + rng.uniform(-amplitude, amplitude, pos.shape).astype(np.float32)
    f[:, 1:4] = np.clip(moved, -MARGIN - lo, MARGIN - hi)
    return out


def as_lights(rec):
    arr = (capi.Light * len(rec)).from_buffer_copy(np.ascontiguousarray(rec).tobytes())
    return list(arr)


def emit(rec, sink):
    line = json.dumps(rec)
    print(line, flush=True)
    sink.write(line + "\n")


def update_costs(scene, repeats, sink):
    import torch

    sd = capi.SceneDescription(scene)
    n = sd.desc.n_lights
    moved = move(records(sd), 0.01)
    host = as_lights(moved)
    on_gpu = torch.from_numpy(moved).to("cuda:0")
    torch.cuda.synchronize()
    create = timed(lambda: capi.Scene(sd).close(), repeats)
    emit(dict(what="ipt_scene_create", scene=scene, lights=n, **create), sink)
    sc = capi.Scene(sd)
    for rebuild in (False, True):
        for src, arr in (("host", host), ("device", on_gpu)):
            r = timed(lambda: sc.update_lights(arr, rebuild=rebuild), repeats)
            emit(dict(what="ipt_scene_update_lights", form="rebuild" if rebuild else "refit", input=src, scene=scene, lights=n,
                      vs_create=r["median_ms"] / create["median_ms"], **r), sink)
    sc.close()


def render_after_update(amplitudes, steps, sink):
    import torch

    sd = capi.SceneDescription(C5["scene"])
    base = records(sd)
    sc = capi.Scene(sd)
    plane = capi.Plane(sc, C5["width"], C5["height"])
    x0, y0, w, h = C5["tile"]
    kw = dict(width=C5["width"], height=C5["height"], depth_max=C5["depth_max"], schedule=C5["schedule"], tile_x0=x0, tile_y0=y0,
              tile_w=w, tile_h=h, flags=capi.FLAG_TIME_KERNELS)
    home = torch.from_numpy(base).to("cuda:0")
    for amp in amplitudes:
        moved = torch.from_numpy(move(base, amp)).to("cuda:0")
        for form in ("refit", "rebuild"):
            # refit: the tree built over the grid, boxes recomputed for the moved lights; rebuild: built over the moved lights
            if form == "refit":
                sc.update_lights(home, rebuild=True)
            sc.update_lights(moved, rebuild=form == "rebuild")
            plane.clear()
            plane.render(capi.default_params(pass_count=1, **kw))  # warm-up
            paths = rays = nodes = 0
            ms = 0.0
            for k in range(steps):
                st = plane.render(capi.default_params(pass_begin=1 + C5["passes"] * k, pass_count=C5["passes"], **kw))
                paths += st.paths; rays += st.rays; nodes += st.light_bvh_nodes_visited; ms += st.ms_total
            emit(dict(what="c5_render", form=form, amplitude=amp, steps=steps, passes=C5["passes"], mpaths_per_s=paths / ms / 1e3,
                      mrays_per_s=rays / ms / 1e3, light_nodes_per_ray=nodes / rays), sink)
    plane.close(); sc.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=".", help="directory of light_update.jsonl")
    ap.add_argument("--scenes", default="lightgrid:100x100,lightgrid:250x400")
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--render-steps", type=int, default=2)
    ap.add_argument("--amplitudes", default="0,0.003,0.01,0.03,0.1")
    a = ap.parse_args()
    lib = capi.load()
    if lib.ipt_device_count() < 1:
        raise SystemExit("light_update.py measures on a CUDA device: none found")
    out = Path(a.out)
    out.mkdir(parents=True, exist_ok=True)
    with open(out / "light_update.jsonl", "w") as sink:
        emit(dict(what="card", **card()), sink)
        for scene in a.scenes.split(","):
            update_costs(scene, a.repeats, sink)
        render_after_update([float(v) for v in a.amplitudes.split(",")], a.render_steps, sink)


if __name__ == "__main__":
    main()
