#!/usr/bin/env python
"""bench.py — the headline benchmark of BASELINE.json: path-tracing throughput (Mpaths/s, with Mrays/s beside it) of
the trace loop on BASELINE configs[1]: the Cornell-box-style scene ("cornell"), 1024x1024, diffuse+glossy DDFs,
split schedule 16/8/4/2, depth 4, 1024 spp for the whole job.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A *step* is one call of the hot path over one batch: `--passes-per-step` passes (default 8) of the full 1024x1024
frame = 8.4 M camera paths. The default K = 128 steps is the whole 1024-spp job. N GPUs: one process per GPU
(torchrun), every rank renders its own pass range (Philox counters make them disjoint), weak scaling; the only
collective is the all-reduce of the accumulators (sum, sumsq, count) at the end of the timed region.

Printed JSON keys are described in DESIGN.md §Measurement. `--impl reference` times the reference's own CPU
implementation (oracle/_ref, the unmodified dimalit/ipt sources + the C2 plug-in; else the oracle port) on all host
cores with forked single-threaded workers (drand48 is process-global, SURVEY.md §6).

`--dump-outputs DIR` writes, after the timed steps, the accumulators the timed path leaves in its plane after its last
step (what `ipt_plane_download` hands a caller) as DIR/sum.npy, DIR/sumsq.npy and DIR/count.npy (float32, H x W;
merged over the ranks for N > 1). The seed and the pass ranges depend only on the arguments, so two builds run with the
same arguments can be compared output for output. Frames above DUMP_LIMIT_BYTES are written as a fixed, seeded sample of
pixels (the same for all three arrays), with the sampled flat pixel indices in DIR/pixel_index.npy (float64).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import multiprocessing as mp
import os
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

# The bench line is BASELINE configs[1] ("c2"); the other configs are parity-test cases, selectable for the record.
WORKLOADS = {
    "c1": dict(config="configs[0]", scene="box", width=640, height=640, depth_max=4, schedule=[16, 8, 4, 2], spp_total=1024, passes_per_step=16,
               text="default scene of src/sample_scenes.cpp (make_scene_box: open unit box + sphere + one square light)"),
    "c2": dict(config="configs[1]", scene="cornell", width=1024, height=1024, depth_max=4, schedule=[16, 8, 4, 2], spp_total=1024, passes_per_step=8,
               text="Cornell-box-style scene 'cornell' (5 box planes, Lambert sphere, glossy sphere, ceiling area light)"),
    "c3": dict(config="configs[2]", scene="mesh:1000000", width=1920, height=1080, depth_max=8, schedule=[1] * 8, spp_total=256, passes_per_step=16,
               text="procedural 1M-triangle random mesh inside the open box, max depth 8"),
    "c4": dict(config="configs[3]", scene="mesh:10000000", width=3840, height=2160, depth_max=8, schedule=[1] * 8, spp_total=4096, passes_per_step=4,
               text="10M-triangle synthetic mesh, sample-sharded across the GPUs"),
    "c5": dict(config="configs[4]", scene="lightgrid:100x100", width=2048, height=2048, depth_max=4, schedule=[16, 8, 4, 2], spp_total=16, passes_per_step=16,
               tile=(768, 768, 512, 512), text="many-light CollectionLighting scene (10k emitters), 512x512 crop of the 2048x2048 frame per step"),
}
WORKLOAD = dict(WORKLOADS["c2"])
CPU_SAMPLE = dict(width=128, height=128)  # the CPU legs render the same view/estimator at this frame size


def measured_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
        except Exception:
            pass
    return 6650.0, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"


# ---------------------------------------------------------------------------------------------------------------
# CPU legs (the only place bench.py executes anything under oracle/)
# ---------------------------------------------------------------------------------------------------------------
_worker_state = {}


def _cpu_worker_init(kind, counter):
    import oracle_lib

    with counter.get_lock():
        rank = counter.value
        counter.value += 1
    W, H = CPU_SAMPLE["width"], CPU_SAMPLE["height"]
    if kind == "reference":
        ref = oracle_lib.load_ref()
        h = ref.scene(WORKLOAD["scene"])
        ref.set_tree(WORKLOAD["schedule"][0], WORKLOAD["depth_max"])
        ref.seed(1000 + rank)
        _worker_state.update(kind=kind, ref=ref, scene=h, W=W, H=H)
    else:
        from ipt_b200 import capi

        orc = oracle_lib.load_oracle()
        sd = capi.SceneDescription(WORKLOAD["scene"])
        orc.seed(1000 + rank)
        p = capi.default_params(width=W, height=H, depth_max=WORKLOAD["depth_max"], schedule=WORKLOAD["schedule"], pass_count=1)
        _worker_state.update(kind=kind, orc=orc, sd=sd, p=p, W=W, H=H)


def _cpu_worker_pass(_):
    st = _worker_state
    if st["kind"] == "reference":
        r = st["ref"].render(st["scene"], 1, st["W"], st["H"], verbatim=False)
        return st["W"] * st["H"], int(r["rays"])
    import oracle_lib

    r = st["orc"].render(st["sd"].ptr, st["p"], oracle_lib.RNG_DRAND48, 0)
    return st["W"] * st["H"], int(r["rays"])


class CpuPool:
    """nproc forked single-threaded workers, each with its own drand48 stream (srand48(1000+rank))."""

    def __init__(self):
        import oracle_lib

        self.kind = "reference" if oracle_lib.build_ref() is not None else "port"
        if self.kind == "port":
            oracle_lib.build_oracle()
        self.cores = os.cpu_count() or 1
        try:
            self.cores = len(os.sched_getaffinity(0))
        except Exception:
            pass
        ctx = mp.get_context("fork")
        counter = ctx.Value("i", 0)
        devnull = os.open(os.devnull, os.O_WRONLY)
        saved = os.dup(1)
        os.dup2(devnull, 1)  # the reference prints "NEW POOL ..." from its allocator (ddf.cpp:28)
        try:
            self.pool = ctx.Pool(self.cores, initializer=_cpu_worker_init, initargs=(self.kind, counter))
            self.pool.map(_cpu_worker_pass, range(self.cores))  # warm every worker (allocator pools, page-in)
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(devnull)
            os.close(saved)

    def step(self, passes_per_worker=1):
        """One bounded sample: every worker renders `passes_per_worker` passes of the CPU_SAMPLE frame."""
        t0 = time.perf_counter()
        out = self.pool.map(_cpu_worker_pass, range(self.cores * passes_per_worker), chunksize=passes_per_worker)
        dt = time.perf_counter() - t0
        return sum(o[0] for o in out), sum(o[1] for o in out), dt

    def close(self):
        self.pool.close()
        self.pool.join()

    def sample_text(self, steps, passes_per_worker=1):
        return (f"{WORKLOAD['scene']} view at {CPU_SAMPLE['width']}x{CPU_SAMPLE['height']}, same estimator (16/8/4/2, depth 4), "
                f"{steps} x {passes_per_worker} pass(es) on each of {self.cores} forked single-threaded processes, libc drand48")


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # each step is a bounded sample (one pass of the CPU_SAMPLE frame per host core); shrink the frame for long runs so
    # that `--steps K --warmup W` still ends within a few minutes (the rate does not depend on the frame size)
    total = args.steps + args.warmup
    side = 128 if total <= 20 else (96 if total <= 48 else 64)
    CPU_SAMPLE.update(width=side, height=side)
    pool = CpuPool()
    for _ in range(args.warmup):
        pool.step()
    paths = rays = 0
    t0 = time.perf_counter()
    for _ in range(args.steps):
        p, r, _ = pool.step()
        paths += p
        rays += r
    dt = time.perf_counter() - t0
    value = paths / dt / 1e6
    line = {
        "impl": "reference", "metric": "path-tracing throughput", "value": value, "unit": "Mpaths/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": cpu_config(pool),
        "mrays_per_s": rays / dt / 1e6, "rays_per_path": rays / max(paths, 1),
        "cpu_baseline": {"value": value, "unit": "Mpaths/s", "cores": pool.cores, "kind": pool.kind, "sample": pool.sample_text(args.steps),
                         "cpu": cpu_model()},
        "e2e": {"value": value, "unit": "Mpaths/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    pool.close()
    print(json.dumps(line), flush=True)


def cpu_config(pool):
    """What the CPU legs really render: the workload's view and estimator on a small sample frame (a rate in paths/s does
    not depend on the frame size or the pass count; a 1024x1024x1024-spp job would take the 16 host cores about an hour)."""
    w = WORKLOAD
    return {"workload": workload_text() + f" -- CPU leg: the same scene, view and estimator on a {CPU_SAMPLE['width']}x{CPU_SAMPLE['height']} sample frame",
            "sample_width": CPU_SAMPLE["width"], "sample_height": CPU_SAMPLE["height"], "sample_passes_per_step_per_core": 1,
            "job_width": w["width"], "job_height": w["height"], "same_config": False,
            "parallelism": f"{pool.cores} host processes"}


def workload_text():
    w = WORKLOAD
    return (f"BASELINE {w['config']}: {w['text']}, {w['width']}x{w['height']}, {w['spp_total']} spp job, "
            f"split schedule {'/'.join(map(str, w['schedule']))}, depth {w['depth_max']}")


# ---------------------------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap", 0x80: "hw_power_brake"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), threading.Event(), None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        while not self.stop_flag.is_set():
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                r = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, name in self.REASONS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.1)

    def result(self):
        self.stop_flag.set()
        if self.nv is None or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


# ---------------------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------------------
class Dist:
    """torch.distributed plumbing of one process per GPU (N = 1: everything is a no-op)."""

    def __init__(self):
        import torch

        self.torch = torch
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        self.dist = None
        self.comm = None
        if not torch.cuda.is_available():
            raise RuntimeError("bench.py needs a CUDA device: the product has no CPU fallback")
        torch.cuda.set_device(self.local)
        if self.world > 1:
            import torch.distributed as dist

            from ipt_b200 import nccl_comm

            dist.init_process_group("nccl", device_id=torch.device(f"cuda:{self.local}"))
            self.dist = dist
            # the ncclComm_t handed to the product's collective (ipt_plane_allreduce); torch only ships the unique id
            self.comm = nccl_comm.NcclComm(dist, self.rank, self.world)

    def sync(self):
        self.torch.cuda.synchronize()
        if self.dist is not None:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def reduce(self, values, op="sum"):
        """Scalars over all ranks (bookkeeping, outside the timed regions)."""
        if self.dist is None:
            return [float(v) for v in values]
        t = self.torch.tensor(list(values), dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op={"sum": self.dist.ReduceOp.SUM, "max": self.dist.ReduceOp.MAX, "min": self.dist.ReduceOp.MIN}[op])
        return [float(x) for x in t.tolist()]

    def close(self):
        if self.comm is not None:
            self.comm.close()
        if self.dist is not None:
            self.dist.destroy_process_group()


AGG_KEYS = ("paths", "rays", "kernel_launches", "ms_total", "ms_extend", "ms_shade", "ms_generate", "ms_accumulate", "n_extend", "n_shade",
            "surface_hits", "light_hits", "queue_bytes", "rays_resolved_in_shade", "bvh_nodes_visited", "triangles_tested", "lights_tested",
            "light_bvh_nodes_visited")


def measure(D, w, steps, warmup, pps, args, ranks_active=None, e2e_steps=0):
    """Times `steps` steps of workload `w` on every active rank (default: all) and returns the measurements of the line.
    A step = `pps` passes of the frame (or of its tile). Device-resident part: scene and accumulators stay in HBM, the
    accumulators of all ranks are merged once at the end by the product's collective. End-to-end part: every step goes
    through the C ABI with the camera coming from the host and the merged accumulators going back to pinned host memory."""
    import torch

    from ipt_b200 import capi

    lib = capi.load()
    active = ranks_active is None or D.rank in ranks_active
    n_active = D.world if ranks_active is None else len(ranks_active)
    W, H = w["width"], w["height"]
    tile = w.get("tile")
    paths_per_pass = (tile[2] * tile[3]) if tile else W * H
    out = dict(n_active=n_active, paths_per_pass=paths_per_pass)
    sd = sc = plane = None
    if active:
        t0 = time.perf_counter()
        sd = capi.SceneDescription(w["scene"])
        sc = capi.Scene(sd, D.local)
        plane = capi.Plane(sc, W, H)  # library-owned accumulators: one packed block sum | sumsq | count
        out["scene_setup_s"] = time.perf_counter() - t0
    first_pass = D.rank * (warmup + steps + e2e_steps + 1) * pps  # disjoint pass ranges per rank

    def params(step, flags=capi.FLAG_TIME_KERNELS):
        kw = dict(tile_x0=tile[0], tile_y0=tile[1], tile_w=tile[2], tile_h=tile[3]) if tile else {}
        return capi.default_params(width=W, height=H, depth_max=w["depth_max"], schedule=w["schedule"], seed=args.seed,
                                   pass_begin=first_pass + step * pps, pass_count=pps, flags=flags, batch_paths=args.batch_paths, **kw)

    use_comm = D.comm is not None and ranks_active is None
    agg = {k: 0.0 for k in AGG_KEYS}
    coll_ms = 0.0
    if active:
        for s_ in range(warmup):
            plane.render(params(s_))
        if use_comm:
            plane.allreduce(D.comm.comm)  # full-size warm-up of the collective: ring / NVLS set-up is not part of the job
        plane.clear()
    sampler = ClockSampler(D.local)
    sampler.start()
    D.sync()
    t0 = time.perf_counter()
    if active:
        for s_ in range(steps):
            st = plane.render(params(warmup + s_))
            for k in AGG_KEYS:
                agg[k] += getattr(st, k)
        if use_comm:  # the only collective of the path: merge the accumulators over NVLink (ipt_plane_allreduce)
            coll_ms = plane.allreduce(D.comm.comm)
    D.sync()
    elapsed = time.perf_counter() - t0
    out["clocks"] = sampler.result()
    out["elapsed"] = D.reduce([elapsed], "max")[0]
    tot = D.reduce([agg["paths"], agg["rays"], agg["kernel_launches"]])
    out["paths_all"], out["rays_all"], out["launches_all"] = tot
    dev_ms = agg["ms_total"] / max(steps, 1) if active else 0.0
    out["device_ms_per_step_max"] = D.reduce([dev_ms], "max")[0]
    out["device_ms_per_step_min"] = D.reduce([dev_ms if active else 1e30], "min")[0]
    out["collective_ms"] = D.reduce([coll_ms], "max")[0]
    out["agg"] = agg
    if active and D.rank == 0:
        s_, q_, c_ = plane.download()
        out["image_mean"] = float(s_.sum(dtype=np.float64) / max(int(c_.sum(dtype=np.uint64)), 1))
        out["accumulators"] = {"sum": s_, "sumsq": q_, "count": c_}

    # ---- end to end through the C ABI with HOST buffers --------------------------------------------------------------
    if e2e_steps:
        cam = sd.desc.camera if active else None
        host_out = None
        if active and D.rank == 0 or (active and not use_comm):
            host_out = (torch.empty(H * W, dtype=torch.float32).pin_memory().numpy(), torch.empty(H * W, dtype=torch.float32).pin_memory().numpy(),
                        torch.empty(H * W, dtype=torch.int32).pin_memory().numpy().view(np.uint32))

        def e2e_step(step):
            capi.check(lib.ipt_scene_set_camera(sc.handle, C.byref(cam)))  # this step's input: the camera, from the host
            if not use_comm:
                hs, hq, hc, st = sc.render_host(params(step, flags=0), out=host_out)  # clear + render + download
                return st.paths, float(hs.reshape(-1)[0])
            plane.clear()
            st = plane.render(params(step, flags=0))
            plane.allreduce(D.comm.comm)  # merged on the device over NVLink ...
            v = 0.0
            if D.rank == 0:  # ... and read where the user reads the image
                plane.download_into(*host_out)
                v = float(host_out[0][0])
            return st.paths, v

        if active:
            e2e_step(warmup + steps)  # warm the staging path
        D.sync()
        t0 = time.perf_counter()
        e2e_paths = 0
        if active:
            for s_ in range(e2e_steps):
                p_, _ = e2e_step(warmup + steps + 1 + s_)
                e2e_paths += p_
        D.sync()
        e2e_elapsed = D.reduce([time.perf_counter() - t0], "max")[0]
        out["e2e_value"] = D.reduce([e2e_paths])[0] / e2e_elapsed / 1e6
        out["e2e_steps"] = e2e_steps
        out["h2d_bytes_per_step"] = C.sizeof(capi.Camera) + C.sizeof(capi.RenderParams)
        out["d2h_bytes_per_step"] = 12 * W * H
    if active:
        plane.close()
        sc.close()
    return out


def roofline_block(m, w, args):
    """The dominant kernel against the HBM roofline of SURVEY.md 8d, and what really binds it.

    `achieved` = ALGORITHMIC bytes / CUDA-event time of the dominant kernel: the wavefront model of SURVEY 8d (every ray a
    36 B record written once and read once, every queued hit a 32 B record written once and read once, plus 64 B per BVH
    node visit and per triangle / light record fetched). The fused shade kernels never queue the rays they trace, so the
    bytes they really move (`implemented_bytes_per_launch`, and ncu's `traffic`) are far below the model and the kernel is
    bound by instruction issue, not by HBM: `binding` says so and `issue_frac` is ncu's issue-slot utilisation."""
    agg = m["agg"]
    peak, peak_src = measured_peak()
    children = agg["rays"] - agg["paths"]
    queued = (agg["queue_bytes"] - 72 * agg["rays"] - 8 * agg["paths"]) // 64
    fused = agg["rays_resolved_in_shade"]
    nodes, tris = agg["bvh_nodes_visited"], agg["triangles_tested"]
    lnodes = agg["light_bvh_nodes_visited"]
    lrecs = agg["lights_tested"] if lnodes else 0  # inline / linear light lists live in the constant bank or L1
    scene_bytes = 64 * (nodes + tris) + 64 * lnodes + 128 * lrecs
    hits_by_shade = max(queued - agg["paths"], 0) if fused == children and fused else 0  # all but the camera rays' hits
    bytes_ext = 36 * (agg["rays"] - fused) + 32 * (queued - hits_by_shade) + 8 * agg["light_hits"] * (0 if fused else 1) + 64 * (nodes + tris)
    bytes_shade = 32 * queued + 36 * children + 36 * fused + 32 * hits_by_shade + 8 * agg["light_hits"] * (1 if fused else 0)
    bytes_shade_impl = 32 * queued + 36 * (children - fused) + 32 * hits_by_shade + 8 * agg["light_hits"] * (1 if fused else 0)
    if fused:
        bytes_shade += 64 * lnodes + 128 * lrecs
        bytes_shade_impl += 64 * lnodes + 128 * lrecs
    else:
        bytes_ext += 64 * lnodes + 128 * lrecs
    dom = "shade" if agg["ms_shade"] >= agg["ms_extend"] else "extend"
    dom_ms = agg["ms_shade"] if dom == "shade" else agg["ms_extend"]
    dom_n = agg["n_shade"] if dom == "shade" else agg["n_extend"]
    dom_bytes = bytes_shade if dom == "shade" else bytes_ext
    achieved = dom_bytes / (dom_ms * 1e-3) / 1e9 if dom_ms > 0 else 0.0
    avg_ms = dom_ms / max(dom_n, 1)
    # SURVEY 8d's own per-ray figures (96 B per ray, 32 B per node, 36 B per triangle, 24 B per path), whole pipeline
    survey_bytes = 96 * agg["rays"] + 32 * nodes + 36 * tris + 48 * (agg["lights_tested"] if lnodes else 0) + 32 * lnodes + 24 * agg["paths"]
    whole_bytes = agg["queue_bytes"] + scene_bytes
    block = {"bound": "hbm", "kernel": ("k_extend_mesh" if dom == "extend" and w["scene"].startswith("mesh") else f"k_{dom}"),
             "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
             "launches": int(dom_n), "avg_launch_ms": avg_ms, "algorithmic_bytes_per_launch": dom_bytes / max(dom_n, 1),
             "implemented_bytes_per_launch": (bytes_shade_impl if dom == "shade" else bytes_ext) / max(dom_n, 1),
             "model": "SURVEY 8d wavefront queue model: 36 B ray record written + read per ray, 32 B hit record written + read per queued hit, "
                      "64 B per BVH node visit / triangle record, 128 B per light record of a light LBVH",
             "whole_pipeline": {"bytes": whole_bytes, "achieved_gbs": whole_bytes / (agg["ms_total"] * 1e-3) / 1e9,
                                "frac": whole_bytes / (agg["ms_total"] * 1e-3) / 1e9 / peak},
             "survey_8d": {"formula": "96 R + 32 V + 36 T + 48 L + 32 V_L + 24 P", "bytes": survey_bytes,
                           "achieved_gbs": survey_bytes / (agg["ms_total"] * 1e-3) / 1e9, "frac": survey_bytes / (agg["ms_total"] * 1e-3) / 1e9 / peak},
             "kernel_ms": {"generate": agg["ms_generate"], "extend": agg["ms_extend"], "shade": agg["ms_shade"], "accumulate": agg["ms_accumulate"]},
             "per_ray": {"bvh_nodes": nodes / max(agg["rays"], 1), "triangles": tris / max(agg["rays"], 1),
                         "light_bvh_nodes": lnodes / max(agg["rays"], 1), "lights": agg["lights_tested"] / max(agg["rays"], 1)}}
    # profile-time evidence (ncu cannot run inside the timed region): DRAM bytes per launch and issue-slot utilisation
    # of the dominant kernel from the committed capture, with the source hash it was taken on
    prof = ROOT / "profiles" / "roofline_latest.json"
    if prof.exists() and not args.batch_paths:
        try:
            pj = json.loads(prof.read_text())
            rec = pj.get("workloads", {}).get(args.workload, {}).get(dom)
            if rec:
                block["traffic"] = rec.get("dram_bytes_per_launch")
                block["traffic_source"] = f"profile-time: ncu capture {pj.get('source', '')}; kernel sources then {pj.get('source_sha16')}, now {source_sha16()}"
                if block["traffic"]:
                    block["dram_gbs"] = block["traffic"] / (avg_ms * 1e-3) / 1e9
                    block["dram_frac"] = block["dram_gbs"] / peak
                if rec.get("issue_active_pct") is not None:
                    block["issue_frac"] = rec["issue_active_pct"] / 100.0
                    block["active_lanes_per_instruction"] = rec.get("lanes_per_inst")
        except Exception:
            pass
    traffic = block["traffic"]
    if traffic is not None and traffic < 0.5 * block["algorithmic_bytes_per_launch"]:
        # the model's bytes are credited, not moved through HBM: ncu's DRAM traffic is far below them
        block["binding"] = ("instruction issue (the fused shade kernels trace the rays they spawn: the ray queue the model credits is never written)"
                            if dom == "shade" and fused else
                            "instruction issue + dependent L2 loads (the BVH / light records the model credits are L2-resident, not HBM traffic)")
    else:
        block["binding"] = "hbm / L2 latency (no profile-time traffic figure for this workload)" if traffic is None else "hbm / L2 latency"
    return block


def source_sha16():
    import hashlib

    h = hashlib.sha256()
    for p in sorted((ROOT / "ipt_b200" / "csrc").glob("*.cu*")):
        h.update(p.read_bytes())
    return h.hexdigest()[:16]


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(directory, accumulators):
    """The plane's accumulators as float32 .npy files; a seeded pixel sample when the whole frame exceeds the limit."""
    out = Path(directory)
    out.mkdir(parents=True, exist_ok=True)
    arrays = {k: np.asarray(v, np.float32) for k, v in accumulators.items()}
    n = next(iter(arrays.values())).size
    per_pixel = sum(a.itemsize for a in arrays.values())
    if n * per_pixel > DUMP_LIMIT_BYTES:
        k = (DUMP_LIMIT_BYTES - 4096) // (per_pixel + 8)  # 8 B per sampled index; 4 KB for the .npy headers
        idx = np.sort(np.random.default_rng(0).choice(n, size=k, replace=False))
        arrays = {name: a.reshape(-1)[idx] for name, a in arrays.items()}
        arrays["pixel_index"] = idx.astype(np.float64)
    for name, a in arrays.items():
        np.save(out / f"{name}.npy", a)


def run_ours(args):
    from ipt_b200 import build, capi

    D = Dist()
    build.build()
    capi.load()
    w = WORKLOAD
    pps = args.passes_per_step
    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    m = measure(D, w, args.steps, args.warmup, pps, args, e2e_steps=e2e_steps)
    if args.dump_outputs and D.rank == 0:
        dump_outputs(args.dump_outputs, m["accumulators"])
    elapsed = m["elapsed"]
    line = None
    if D.rank == 0:
        line = {
            "metric": "path-tracing throughput", "value": m["paths_all"] / elapsed / 1e6, "unit": "Mpaths/s", "n_gpus": D.world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": elapsed / args.steps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_text(), "passes_per_step": pps, "paths_per_step_per_gpu": m["paths_per_pass"] * pps,
                       "parallelism": f"pass-sharded x{D.world}, accumulators merged once by ipt_plane_allreduce (NCCL)" if D.world > 1 else "single GPU",
                       "l2": "per-step ray/hit queue working set (>1 GB) exceeds the 126 MB L2; no flush needed",
                       "batch_paths": args.batch_paths or "library default"},
            "mrays_per_s": m["rays_all"] / elapsed / 1e6, "rays_per_path": m["rays_all"] / max(m["paths_all"], 1), "image_mean": m.get("image_mean"),
            "device_ms_per_step": m["agg"]["ms_total"] / args.steps,
            "device_ms_per_step_ranks": {"min": m["device_ms_per_step_min"], "max": m["device_ms_per_step_max"]},
            "collective_ms": m["collective_ms"],
            "host_overhead_ms_per_step": elapsed / args.steps * 1e3 - m["device_ms_per_step_max"] - m["collective_ms"] / args.steps,
            "clocks": m["clocks"],
            "e2e": {"value": m["e2e_value"], "unit": "Mpaths/s", "h2d_bytes_per_step": m["h2d_bytes_per_step"],
                    "d2h_bytes_per_step": m["d2h_bytes_per_step"], "steps": m["e2e_steps"],
                    "call": ("ipt_scene_set_camera + ipt_render_host (host sum/sumsq/count buffers)" if D.world == 1 else
                             "per step: ipt_scene_set_camera + ipt_plane_clear + ipt_render + ipt_plane_allreduce on every rank, ipt_plane_download to pinned host memory on rank 0")},
            "gpu_launches": int(m["launches_all"]),
            "roofline": roofline_block(m, w, args),
        }
    # BASELINE configs[3] (the multi-GPU config) rides along on N > 1: same invocation, its own sub-record
    if (D.world > 1 or args.with_c4) and args.workload == "c2" and not args.no_c4:
        c4 = dict(WORKLOADS["c4"])
        k4, w4, p4 = args.c4_steps, 2, c4["passes_per_step"]
        one = measure(D, c4, k4, w4, p4, args, ranks_active=[0]) if D.world > 1 else None  # rank 0 alone: the 1-GPU denominator, same box
        alln = measure(D, c4, k4, w4, p4, args, e2e_steps=min(k4, 4))
        if D.rank == 0:
            rec = {"workload": f"BASELINE {c4['config']}: {c4['text']}, {c4['width']}x{c4['height']}, depth {c4['depth_max']}, split schedule 1x8",
                   "n_gpus": D.world, "steps": k4, "warmup": w4, "passes_per_step": p4,
                   "value": alln["paths_all"] / alln["elapsed"] / 1e6, "unit": "Mpaths/s", "mrays_per_s": alln["rays_all"] / alln["elapsed"] / 1e6,
                   "ms_per_step": alln["elapsed"] / k4 * 1e3, "device_ms_per_step_ranks": {"min": alln["device_ms_per_step_min"], "max": alln["device_ms_per_step_max"]},
                   "collective_ms": alln["collective_ms"], "e2e": {"value": alln["e2e_value"], "unit": "Mpaths/s", "d2h_bytes_per_step": alln["d2h_bytes_per_step"]},
                   "scene_setup_s": alln.get("scene_setup_s"), "image_mean": alln.get("image_mean"), "roofline": roofline_block(alln, c4, args)}
            if one is not None:
                v1 = one["paths_all"] / one["elapsed"] / 1e6
                rec["one_gpu_same_box"] = {"value": v1, "unit": "Mpaths/s", "ms_per_step": one["elapsed"] / k4 * 1e3}
                rec["speedup_vs_one_gpu"] = rec["value"] / v1
            line["c4"] = rec
    if D.rank == 0:
        if D.world == 1 and not args.no_cpu_baseline and w["scene"] not in ("box", "cornell"):
            line["cpu_baseline"] = {"value": None, "unit": "Mpaths/s", "cores": 0, "kind": "port",
                                    "sample": "not run: the reference has no mesh / 10k-light scene; see the c1/c2 workloads"}
        elif D.world == 1 and not args.no_cpu_baseline:
            pool = CpuPool()
            paths = rays = 0
            t0 = time.perf_counter()
            reps = 0
            while time.perf_counter() - t0 < args.cpu_seconds or reps < 2:
                p, r, _ = pool.step()
                paths += p; rays += r; reps += 1
            dt = time.perf_counter() - t0
            line["cpu_baseline"] = {"value": paths / dt / 1e6, "unit": "Mpaths/s", "cores": pool.cores, "kind": pool.kind,
                                    "sample": pool.sample_text(reps), "mrays_per_s": rays / dt / 1e6, "cpu": cpu_model(),
                                    "config": cpu_config(pool)}
            pool.close()
        print(json.dumps(line), flush=True)
    D.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default: 128, the whole job; 8 for --impl reference)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS), help="c2 = BASELINE configs[1], the bench line")
    ap.add_argument("--passes-per-step", type=int, default=0)
    ap.add_argument("--batch-paths", type=int, default=0)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--e2e-steps", type=int, default=16)
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--with-c4", action="store_true", help="add the BASELINE configs[3] sub-record on one GPU too (always on for N > 1)")
    ap.add_argument("--no-c4", action="store_true")
    ap.add_argument("--c4-steps", type=int, default=6)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the accumulators of the timed path after its last step to DIR/*.npy")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl ours (the reference arm only counts paths)")
    WORKLOAD.clear()
    WORKLOAD.update(WORKLOADS[args.workload])
    if args.passes_per_step <= 0:
        args.passes_per_step = WORKLOAD["passes_per_step"]
    if args.impl == "reference":
        if args.steps is None:
            args.steps = 8  # each step is a bounded sample: keep the default run within minutes
        run_reference_arm(args)
    else:
        if args.steps is None:
            args.steps = 128
        if args.warmup < 3:
            args.warmup = 3  # timing rule: at least 3 warm-up steps
        run_ours(args)


if __name__ == "__main__":
    main()
