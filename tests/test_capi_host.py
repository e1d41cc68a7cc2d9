"""Host-side checks that need no GPU: the C-ABI library loads and exports every symbol include/ipt_b200.h declares,
argument validation, the no-CPU-fallback contract, scene descriptions, the mesh generator."""
import ctypes as C
import re
from pathlib import Path

import numpy as np
import pytest

from ipt_b200 import capi

ROOT = Path(__file__).resolve().parent.parent


def test_library_exports_every_declared_symbol(lib):
    header = (ROOT / "include" / "ipt_b200.h").read_text()
    declared = set(re.findall(r"\b(ipt_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 25
    for name in declared:
        assert hasattr(lib, name), f"{name} is declared in include/ipt_b200.h but not exported"
    assert declared == set(capi.SIGNATURES), "ctypes binding and header disagree"
    assert lib.ipt_abi_version() == 3


def test_struct_layouts_match_the_header(lib):
    # sizes a C compiler gives the structs of include/ipt_b200.h (checked once with a C program: see oracle build)
    assert C.sizeof(capi.Prim) == 32 and C.sizeof(capi.Light) == 48 and C.sizeof(capi.Material) == 20
    assert C.sizeof(capi.Camera) == 48 and C.sizeof(capi.BvhNode) == 64
    p = capi.default_params()
    assert (p.width, p.height, p.depth_max, list(p.schedule)[:4], p.plane_mode) == (640, 640, 4, [16, 8, 4, 2], capi.PLANE_GRID)


def test_enum_values_and_struct_sizes_against_a_c_compiler(lib, tmp_path):
    """The numeric constants and struct sizes of the ctypes mirror against what gcc sees in include/ipt_b200.h."""
    import subprocess

    names = ["IPT_FLAG_TIME_KERNELS", "IPT_FLAG_KEEP_ZERO_WEIGHT", "IPT_FLAG_DEBUG_PRINT", "IPT_FLAG_RESOLVE_LAST_LEVEL",
             "IPT_FLAG_NO_FUSED_LAST_LEVEL", "IPT_FLAG_NO_FUSED_TRACE", "IPT_PLANE_GRID", "IPT_PLANE_GUI", "IPT_PLANE_LINEAR",
             "IPT_KEY_LEFT", "IPT_KEY_RIGHT", "IPT_KEY_DOWN", "IPT_KEY_UP", "IPT_ERR_INVALID", "IPT_ERR_NO_DEVICE", "IPT_MAX_DEPTH", "IPT_DISPATCH_WORDS"]
    structs = ["ipt_material", "ipt_prim", "ipt_light", "ipt_camera", "ipt_scene_desc", "ipt_render_params", "ipt_render_stats", "ipt_bvh_node"]
    src = tmp_path / "probe.c"
    src.write_text('#include <stdio.h>\n#include "ipt_b200.h"\nint main(void) {\n'
                   + "".join(f'  printf("{n} %lld\\n", (long long){n});\n' for n in names)
                   + "".join(f'  printf("sizeof_{t} %zu\\n", sizeof({t}));\n' for t in structs) + "  return 0;\n}\n")
    exe = tmp_path / "probe"
    subprocess.run(["gcc", "-std=c11", f"-I{ROOT / 'include'}", "-o", str(exe), str(src)], check=True)
    got = dict(line.split() for line in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    got = {k: int(v) for k, v in got.items()}
    want = {"IPT_FLAG_TIME_KERNELS": capi.FLAG_TIME_KERNELS, "IPT_FLAG_KEEP_ZERO_WEIGHT": capi.FLAG_KEEP_ZERO_WEIGHT,
            "IPT_FLAG_DEBUG_PRINT": capi.FLAG_DEBUG_PRINT, "IPT_FLAG_RESOLVE_LAST_LEVEL": capi.FLAG_RESOLVE_LAST_LEVEL,
            "IPT_FLAG_NO_FUSED_LAST_LEVEL": capi.FLAG_NO_FUSED_LAST_LEVEL, "IPT_FLAG_NO_FUSED_TRACE": capi.FLAG_NO_FUSED_TRACE,
            "IPT_PLANE_GRID": capi.PLANE_GRID, "IPT_PLANE_GUI": capi.PLANE_GUI, "IPT_PLANE_LINEAR": capi.PLANE_LINEAR,
            "IPT_KEY_LEFT": 0, "IPT_KEY_RIGHT": 1, "IPT_KEY_DOWN": 2, "IPT_KEY_UP": 3,
            "IPT_ERR_INVALID": capi.IPT_ERR_INVALID, "IPT_ERR_NO_DEVICE": capi.IPT_ERR_NO_DEVICE, "IPT_MAX_DEPTH": capi.IPT_MAX_DEPTH,
            "IPT_DISPATCH_WORDS": capi.DISPATCH_WORDS,
            "sizeof_ipt_material": C.sizeof(capi.Material), "sizeof_ipt_prim": C.sizeof(capi.Prim), "sizeof_ipt_light": C.sizeof(capi.Light),
            "sizeof_ipt_camera": C.sizeof(capi.Camera), "sizeof_ipt_scene_desc": C.sizeof(capi.SceneDesc),
            "sizeof_ipt_render_params": C.sizeof(capi.RenderParams), "sizeof_ipt_render_stats": C.sizeof(capi.RenderStats),
            "sizeof_ipt_bvh_node": C.sizeof(capi.BvhNode)}
    assert got == want


def test_no_cpu_fallback(lib, has_gpu):
    """Without a CUDA device every compute entry point fails loudly with IPT_ERR_NO_DEVICE."""
    if has_gpu:
        pytest.skip("a GPU is present")
    sd = capi.SceneDescription("box")
    with pytest.raises(capi.IptError) as e:
        capi.Scene(sd)
    assert e.value.code == capi.IPT_ERR_NO_DEVICE and "no CPU fallback" in str(e.value)


def test_sample_scene_names_and_errors(lib):
    for name, prims, lights in [("box", 6, 1), ("smallpt", 7, 1), ("square", 1, 1), ("corner", 3, 1), ("openspheres", 4, 1),
                                ("cornell", 7, 1), ("lightgrid:10x10", 6, 100)]:
        sd = capi.SceneDescription(name)
        assert (sd.desc.n_prims, sd.desc.n_lights) == (prims, lights), name
    assert capi.SceneDescription("fractal").desc.n_prims == 7  # FractalSpheres prints 7 spheres (r >= 0.001)
    for bad in ["nope", "mesh:0", "lightgrid:0x3", "lightgrid:abc"]:
        with pytest.raises(capi.IptError, match=bad):
            capi.SceneDescription(bad)
    out = C.POINTER(capi.SceneDesc)()
    # the message is this call's own, not one left on the thread by an earlier failure
    assert lib.ipt_sample_scene(None, C.byref(out)) != 0 and b"ipt_sample_scene" in lib.ipt_last_error()


def test_generated_mesh_is_integer_defined(lib):
    a = np.empty((1000, 9), np.float32); b = np.empty((1000, 9), np.float32)
    assert lib.ipt_generate_mesh(1000, 1, a.ctypes.data_as(capi.f32p)) == 0
    assert lib.ipt_generate_mesh(1000, 1, b.ctypes.data_as(capi.f32p)) == 0
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    assert np.abs(a[:, :3]).max() <= 0.9 and np.abs(a[:, 3:]).max() <= 0.02
    sd = capi.SceneDescription("mesh:1000")
    assert np.array_equal(sd.triangles().view(np.uint32), a.view(np.uint32))
    # every value is k/2^24 scaled once: reproducible from the integer hash in numpy
    def splitmix(x):
        x = (x + 0x9E3779B97F4A7C15) & 0xFFFFFFFFFFFFFFFF
        x = ((x ^ (x >> 30)) * 0xBF58476D1CE4E5B9) & 0xFFFFFFFFFFFFFFFF
        x = ((x ^ (x >> 27)) * 0x94D049BB133111EB) & 0xFFFFFFFFFFFFFFFF
        return x ^ (x >> 31)
    for k, j in [(0, 0), (17, 4), (999, 8)]:
        h = splitmix((1 * 0x100000001B3 + k * 9 + j) & 0xFFFFFFFFFFFFFFFF)
        u = np.float32(h >> 40) * np.float32(1 / 16777216)
        sym = u * np.float32(2) - np.float32(1)
        assert a[k, j] == sym * np.float32(0.9 if j < 3 else 0.02)


def test_camera_look_matches_simplecamera(lib):
    cam = capi.Camera()
    pos = (C.c_float * 3)(0, -3, 0.1); d = (C.c_float * 3)(0.0, 0.9642, -0.2652); up = (C.c_float * 3)(0, 0, 1)
    assert lib.ipt_camera_look(pos, d, up, C.byref(cam)) == 0
    r = np.array(list(cam.right)); u = np.array(list(cam.up)); dd = np.array(list(cam.direction))
    assert abs(np.linalg.norm(r) - 1) < 1e-6 and abs(np.linalg.norm(u) - 1) < 1e-6
    assert abs(r @ dd) < 1e-6 and abs(u @ dd) < 1e-6 and abs(r @ u) < 1e-6
