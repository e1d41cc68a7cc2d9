"""Round-2 A/B of the fused shade kernels: builds -D variants of the same sources (here, on CPU) and benches each on the GPU box.

    python tools/ab_r02.py build [names]     # in the container (cross-compiles)
    python tools/ab_r02.py run [names] [workloads]   # on the GPU box: two interleaved repetitions per variant
"""
import json, os, subprocess, sys
sys.path.insert(0, '.')
VARIANTS = {
    "base": [],
    "nofast": ["IPT_FAST_SECONDARY=0"],
    "u24": ["IPT_U01_BITS=24"],
    "r10": ["IPT_PHILOX_ROUNDS=10"],
    "b4": ["IPT_SHADE_FUSED_MIN_BLOCKS=4", "IPT_SHADE_NEXT_MIN_BLOCKS=4"],
    "nearr1": ["IPT_FAST_SECONDARY=0", "IPT_U01_BITS=24", "IPT_PHILOX_ROUNDS=10", "IPT_BVH_WIDE_NODES=1", "IPT_LIGHT_TWO_QUEUES=0"],
    "wide": ["IPT_BVH_WIDE_NODES=1"],      # mesh traversal over the 64-byte float nodes
    "oneq": ["IPT_LIGHT_TWO_QUEUES=0"],    # many-light scenes: a single park queue at the non-last depths
    "lightq": ["IPT_LIGHT_QNODES=1"],      # light LBVH through its 32-byte quantised nodes (measured: no gain)
    "nosamp": ["IPT_LIGHT_SAMP_RECORDS=0"], # light sampling from the 112-byte records
    "walls": ["IPT_SHADOW_SKIP_WALLS=0"],  # shadow rays of box scenes test the wall planes too
    "m_s8": ["IPT_TRAV_STEPS=8"], "m_s32": ["IPT_TRAV_STEPS=32"], "m_l16": ["IPT_LEAF_BATCH=16"], "m_b5": ["IPT_MESH_MIN_BLOCKS=5"],
    "m_l4": ["IPT_LEAF_BATCH=4"], "m_l8": ["IPT_LEAF_BATCH=8"], "m_l10": ["IPT_LEAF_BATCH=10"], "m_r2": ["IPT_REFILL_MIN=2"], "m_r8": ["IPT_REFILL_MIN=8"], "m_v1": ["IPT_VISITS_PER_ROUND=1"],  # mesh kernel sweeps
    "m_st8": ["IPT_STACK_SHORT=8"], "m_st16": ["IPT_STACK_SHORT=16"], "m_st20": ["IPT_STACK_SHORT=20"], "m_st24": ["IPT_STACK_SHORT=24"], "m_st32": ["IPT_STACK_SHORT=32"], "m_b3": ["IPT_MESH_MIN_BLOCKS=3"], "m_s24": ["IPT_TRAV_STEPS=24"],
    "nopq": ["IPT_PAIR_QUEUE=0"],          # mesh kernel: every lane tests its own postponed leaf
    "bounds": ["IPT_DEBUG_BOUNDS"],        # every queue append checked against its capacity (compute-sanitizer is closed on this pool)
}
if __name__ == "__main__":
    what = sys.argv[1]
    names = sys.argv[2].split(",") if len(sys.argv) > 2 and sys.argv[2] != "all" else list(VARIANTS)
    if what == "build":
        from ipt_b200 import build
        for n in names:
            print(n, build.build_variant(n, VARIANTS[n]), flush=True)
    elif what == "configs":  # tools/run_configs.py per variant: python tools/ab_r02.py configs base,wide c3,c3_tree
        for rep in range(2):
            for n in names:
                env = dict(os.environ, IPT_B200_LIB=f"ipt_b200/lib/variants/{n}.so")
                r = subprocess.run([sys.executable, "tools/run_configs.py", sys.argv[3]], env=env, capture_output=True, text=True)
                for l in r.stdout.strip().splitlines():
                    try:
                        d = json.loads(l)
                        print(f"{n:8s} {d['config']:8s} {d['mpaths_per_s']:8.1f} Mpaths/s {d['mrays_per_s']:9.1f} Mrays/s  extend {d['ms_extend']:8.2f} shade {d['ms_shade']:8.2f} ms  "
                              f"nodes/ray {d['bvh_nodes_per_ray']:.2f} tris/ray {d['tris_per_ray']:.2f} lnodes/ray {d.get('light_nodes_per_ray', 0):.2f} lights/ray {d.get('lights_per_ray', 0):.2f} mean {d['image_mean']:.6f}", flush=True)
                    except Exception:
                        print(n, "?", l[:300], r.stderr[-300:], flush=True)
    else:
        workloads = sys.argv[3].split(",") if len(sys.argv) > 3 else ["c2"]
        for rep in range(2):
            for n in names:
                for w in workloads:
                    env = dict(os.environ, IPT_B200_LIB=f"ipt_b200/lib/variants/{n}.so")
                    r = subprocess.run([sys.executable, "bench.py", "--workload", w, "--steps", "12", "--warmup", "3", "--no-cpu-baseline", "--e2e-steps", "1", "--no-c4"],
                                       env=env, capture_output=True, text=True)
                    try:
                        d = json.loads(r.stdout.strip().splitlines()[-1])
                        k = d["roofline"]["kernel_ms"]
                        print(f"{n:10s} {w}  {d['value']:7.1f} Mpaths/s  extend {k['extend']:7.1f}  shade {k['shade']:7.1f}  rays/path {d['rays_per_path']:.3f} mean {d['image_mean']:.6f} sm {d['clocks']['sm_mhz']}", flush=True)
                    except Exception as e:
                        print(n, w, "failed", r.stderr[-600:], flush=True)
