"""ctypes binding of include/ipt_b200.h — test / bench harness glue only (the product is the C ABI).

Mirrors the C structs one to one. `load()` raises if the CUDA library has not been built: there is no
CPU fallback anywhere in this package.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

IPT_MAX_DEPTH = 16
IPT_NO_HIT = 0xFFFFFFFF
PLANE_GRID, PLANE_GUI, PLANE_LINEAR = 0, 1, 2
FLAG_TIME_KERNELS, FLAG_KEEP_ZERO_WEIGHT, FLAG_DEBUG_PRINT, FLAG_RESOLVE_LAST_LEVEL, FLAG_NO_FUSED_LAST_LEVEL, FLAG_NO_FUSED_TRACE = 1, 2, 4, 8, 16, 32
STATUS = {0: "IPT_OK", 1: "IPT_ERR_INVALID", 2: "IPT_ERR_CUDA", 3: "IPT_ERR_NO_DEVICE", 4: "IPT_ERR_UNSUPPORTED", 5: "IPT_ERR_OVERFLOW"}
IPT_ERR_INVALID = 1
IPT_ERR_NO_DEVICE = 3
# ipt_scene_dispatch: out[0] names the shade spec, the other words are flags / counts
SPEC_FEW_LIGHTS, SPEC_LIGHT_BVH, SPEC_RUNTIME, SPEC_ONE_LIGHT, SPEC_ONE_AREA_LIGHT, SPEC_BOX_SCENE, SPEC_LAMBERT_BOX = range(7)
DISPATCH_FIELDS = ("spec", "smallpt", "mesh", "mesh_box_scene", "lights_inside_box", "light_inline", "n_light_bvh")
DISPATCH_WORDS = len(DISPATCH_FIELDS)
UPDATE_DEVICE_POINTER, UPDATE_REBUILD = 1, 2  # ipt_update_flags

import os

# IPT_B200_LIB selects another build of the SAME sources (kernel tuning experiments); never a different implementation
LIB_PATH = Path(os.environ.get("IPT_B200_LIB") or Path(__file__).resolve().parent / "lib" / "libipt_b200.so")

f32p = C.POINTER(C.c_float)
u32p = C.POINTER(C.c_uint32)
u64p = C.POINTER(C.c_uint64)
u8p = C.POINTER(C.c_uint8)


class Material(C.Structure):
    _fields_ = [("ddf", C.c_uint32), ("albedo", C.c_float), ("kd", C.c_float), ("ks", C.c_float), ("exponent", C.c_float)]


class Prim(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("material", C.c_uint32), ("p", C.c_float * 3), ("radius", C.c_float),
                ("flip_normal", C.c_uint32), ("curvature", C.c_float)]


class Light(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("position", C.c_float * 3), ("x_axis", C.c_float * 3), ("y_axis", C.c_float * 3),
                ("radius", C.c_float), ("power", C.c_float)]


class Camera(C.Structure):
    _fields_ = [("position", C.c_float * 3), ("direction", C.c_float * 3), ("right", C.c_float * 3), ("up", C.c_float * 3)]


class SceneDesc(C.Structure):
    _fields_ = [("n_prims", C.c_uint32), ("prims", C.POINTER(Prim)), ("n_materials", C.c_uint32), ("materials", C.POINTER(Material)),
                ("n_lights", C.c_uint32), ("lights", C.POINTER(Light)), ("n_triangles", C.c_uint64), ("triangles", f32p),
                ("triangle_material", C.c_uint32), ("camera", Camera)]


class RenderParams(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("depth_max", C.c_uint32), ("schedule", C.c_uint32 * IPT_MAX_DEPTH),
                ("seed", C.c_uint64), ("pass_begin", C.c_uint32), ("pass_count", C.c_uint32),
                ("tile_x0", C.c_uint32), ("tile_y0", C.c_uint32), ("tile_w", C.c_uint32), ("tile_h", C.c_uint32),
                ("plane_mode", C.c_uint32), ("flags", C.c_uint32), ("batch_paths", C.c_uint32)]


class RenderStats(C.Structure):
    _fields_ = [("paths", C.c_uint64), ("rays", C.c_uint64), ("rays_at_depth", C.c_uint64 * IPT_MAX_DEPTH),
                ("surface_hits", C.c_uint64), ("light_hits", C.c_uint64), ("misses", C.c_uint64),
                ("failed_samples", C.c_uint64), ("zero_weight_pruned", C.c_uint64), ("nonfinite_dropped", C.c_uint64),
                ("bvh_nodes_visited", C.c_uint64), ("triangles_tested", C.c_uint64), ("lights_tested", C.c_uint64), ("light_bvh_nodes_visited", C.c_uint64),
                ("batches", C.c_uint32), ("kernel_launches", C.c_uint32), ("ms_total", C.c_float),
                ("ms_generate", C.c_float), ("ms_extend", C.c_float), ("ms_shade", C.c_float), ("ms_accumulate", C.c_float),
                ("n_extend", C.c_uint32), ("n_shade", C.c_uint32), ("queue_bytes", C.c_uint64),
                ("rays_resolved_in_shade", C.c_uint64)]

    def as_dict(self):
        d = {}
        for name, _ in self._fields_:
            v = getattr(self, name)
            d[name] = list(v) if hasattr(v, "__len__") else v
        return d


class BvhNode(C.Structure):
    _fields_ = [("lo0", C.c_float * 3), ("left", C.c_uint32), ("hi0", C.c_float * 3), ("right", C.c_uint32),
                ("lo1", C.c_float * 3), ("parent", C.c_uint32), ("hi1", C.c_float * 3), ("pad", C.c_uint32)]


BVH_NODE_DTYPE = np.dtype([("lo0", "<f4", 3), ("left", "<u4"), ("hi0", "<f4", 3), ("right", "<u4"),
                           ("lo1", "<f4", 3), ("parent", "<u4"), ("hi1", "<f4", 3), ("pad", "<u4")])

# every symbol include/ipt_b200.h declares: name -> (restype, argtypes)
_vp = C.c_void_p
SIGNATURES = {
    "ipt_abi_version": (C.c_int, []),
    "ipt_last_error": (C.c_char_p, []),
    "ipt_device_count": (C.c_int, []),
    "ipt_scene_create": (C.c_int, [C.POINTER(SceneDesc), C.c_int, C.POINTER(_vp)]),
    "ipt_scene_destroy": (C.c_int, [_vp]),
    "ipt_scene_set_camera": (C.c_int, [_vp, C.POINTER(Camera)]),
    "ipt_scene_dispatch": (C.c_int, [_vp, u32p]),
    "ipt_scene_update_triangles": (C.c_int, [_vp, _vp, C.c_uint64, C.c_uint32]),
    "ipt_scene_set_triangle_materials": (C.c_int, [_vp, _vp, C.c_uint64, C.c_uint32]),
    "ipt_scene_update_lights": (C.c_int, [_vp, _vp, C.c_uint32, C.c_uint32]),
    "ipt_sample_scene": (C.c_int, [C.c_char_p, C.POINTER(C.POINTER(SceneDesc))]),
    "ipt_scene_desc_free": (C.c_int, [C.POINTER(SceneDesc)]),
    "ipt_light_derived": (C.c_int, [C.POINTER(Light), f32p, f32p, f32p]),
    "ipt_camera_look": (C.c_int, [f32p, f32p, f32p, C.POINTER(Camera)]),
    "ipt_trace_batch": (C.c_int, [_vp, f32p, f32p, C.c_size_t, u32p, f32p, u32p, f32p, u32p]),
    "ipt_preview_batch": (C.c_int, [_vp, f32p, f32p, C.c_size_t, f32p]),
    "ipt_camera_rays": (C.c_int, [_vp, f32p, C.c_size_t, f32p, f32p]),
    "ipt_ddf_value": (C.c_int, [_vp, C.c_int, f32p, f32p, C.c_size_t, f32p]),
    "ipt_ddf_sample": (C.c_int, [_vp, C.c_int, f32p, C.c_uint64, C.c_size_t, f32p]),
    "ipt_mix_sample": (C.c_int, [_vp, f32p, f32p, C.c_uint64, C.c_size_t, f32p, f32p, f32p]),
    "ipt_light_ddf_value": (C.c_int, [_vp, f32p, f32p, C.c_size_t, f32p]),
    "ipt_light_ddf_sample": (C.c_int, [_vp, f32p, C.c_uint64, C.c_size_t, f32p]),
    "ipt_philox_batch": (C.c_int, [C.c_int, u32p, C.c_size_t, C.c_uint64, u32p, f32p]),
    "ipt_bvh_export": (C.c_int, [_vp, C.POINTER(BvhNode), u32p, u64p, u64p]),
    "ipt_bvh_export_compact": (C.c_int, [_vp, u32p, f32p, u64p]),
    "ipt_plane_create": (C.c_int, [_vp, C.c_uint32, C.c_uint32, C.POINTER(_vp)]),
    "ipt_plane_wrap": (C.c_int, [_vp, C.c_uint32, C.c_uint32, _vp, _vp, _vp, C.POINTER(_vp)]),
    "ipt_plane_clear": (C.c_int, [_vp]),
    "ipt_plane_add_rays": (C.c_int, [_vp, C.c_uint32, C.c_size_t, f32p, f32p, f32p]),
    "ipt_plane_destroy": (C.c_int, [_vp]),
    "ipt_plane_download": (C.c_int, [_vp, f32p, f32p, u32p]),
    "ipt_plane_upload": (C.c_int, [_vp, f32p, f32p, u32p]),
    "ipt_plane_device_ptrs": (C.c_int, [_vp, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp)]),
    "ipt_plane_allreduce": (C.c_int, [_vp, _vp, f32p]),
    "ipt_plane_merge": (C.c_int, [_vp, _vp]),
    "ipt_plane_resolve": (C.c_int, [_vp, f32p, u64p, f32p]),
    "ipt_image_glare": (C.c_int, [C.c_int, f32p, C.c_uint32, C.c_uint32, C.c_float, f32p, u32p]),
    "ipt_image_normalize": (C.c_int, [C.c_int, f32p, C.c_uint32, C.c_uint32, f32p]),
    "ipt_image_save_bytes": (C.c_int, [C.c_int, f32p, C.c_uint32, C.c_uint32, u8p]),
    "ipt_plane_display": (C.c_int, [_vp, C.c_float, f32p, f32p]),
    "ipt_plane_save_bytes": (C.c_int, [_vp, u8p]),
    "ipt_plane_save_png": (C.c_int, [_vp, C.c_char_p]),
    "ipt_write_png_gray8": (C.c_int, [C.c_char_p, u8p, C.c_uint32, C.c_uint32]),
    "ipt_camera_orbit": (C.c_int, [C.POINTER(Camera), C.c_int]),
    "ipt_render": (C.c_int, [_vp, _vp, C.POINTER(RenderParams), C.POINTER(RenderStats)]),
    "ipt_render_host": (C.c_int, [_vp, C.POINTER(RenderParams), f32p, f32p, u32p, C.POINTER(RenderStats)]),
    "ipt_render_params_default": (None, [C.POINTER(RenderParams)]),
    "ipt_generate_mesh": (C.c_int, [C.c_uint64, C.c_uint64, f32p]),
}

_lib = None


def load() -> C.CDLL:
    """dlopen the built CUDA library; never falls back to anything else."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise RuntimeError(f"{LIB_PATH} is missing: run `python -m ipt_b200.build` (nvcc, sm_100a). There is no CPU fallback.")
        lib = C.CDLL(str(LIB_PATH))
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


class IptError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"{STATUS.get(code, code)}: {msg}")
        self.code = code


def check(code: int):
    if code != 0:
        raise IptError(code, load().ipt_last_error().decode())


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _ptr(a, t):
    return a.ctypes.data_as(t) if a is not None else None


def image_glare(image, cutoff: float, device: int = 0):
    """glare(image, cutoff) of gui.cpp:38-52 on the device; returns (filtered image, number of halo sources)."""
    img = _f32(image); h, w = img.shape
    out = np.empty_like(img); nb = C.c_uint32(0)
    check(load().ipt_image_glare(device, _ptr(img, f32p), w, h, cutoff, _ptr(out, f32p), C.byref(nb)))
    return out, nb.value


def image_normalize(image, device: int = 0):
    img = _f32(image); h, w = img.shape
    out = np.empty_like(img)
    check(load().ipt_image_normalize(device, _ptr(img, f32p), w, h, _ptr(out, f32p)))
    return out


def image_save_bytes(image, device: int = 0):
    img = _f32(image); h, w = img.shape
    out = np.empty((h, w), np.uint8)
    check(load().ipt_image_save_bytes(device, _ptr(img, f32p), w, h, _ptr(out, u8p)))
    return out


def write_png_gray8(path, image_u8):
    a = np.ascontiguousarray(image_u8, np.uint8); h, w = a.shape
    check(load().ipt_write_png_gray8(str(path).encode(), _ptr(a, u8p), w, h))


def philox_batch(counters, seed: int = 0, device: int = 0):
    """ipt_philox_batch: (blocks uint32[n,4], uniforms float32[n,4]) of the render's Philox stream for uint32[n,4] counters."""
    c = np.ascontiguousarray(counters, dtype=np.uint32).reshape(-1, 4)
    blocks = np.empty_like(c)
    uni = np.empty(c.shape, np.float32)
    check(load().ipt_philox_batch(device, _ptr(c, u32p), c.shape[0], seed, _ptr(blocks, u32p), _ptr(uni, f32p)))
    return blocks, uni


def camera_orbit(camera: Camera, key: int) -> Camera:
    check(load().ipt_camera_orbit(C.byref(camera), key))
    return camera


def default_params(**kw) -> RenderParams:
    p = RenderParams()
    load().ipt_render_params_default(C.byref(p))
    for k, v in kw.items():
        if k == "schedule":
            for i in range(IPT_MAX_DEPTH):
                p.schedule[i] = v[i] if i < len(v) else 0
        else:
            setattr(p, k, v)
    return p


class SceneDescription:
    """A scene description owned by the library (ipt_sample_scene)."""

    def __init__(self, name: str):
        self.name = name
        self.ptr = C.POINTER(SceneDesc)()
        check(load().ipt_sample_scene(name.encode(), C.byref(self.ptr)))

    @property
    def desc(self) -> SceneDesc:
        return self.ptr.contents

    def triangles(self) -> np.ndarray:
        n = self.desc.n_triangles
        if n == 0:
            return np.zeros((0, 9), np.float32)
        return np.ctypeslib.as_array(self.desc.triangles, shape=(n, 9))

    def close(self):
        if self.ptr:
            load().ipt_scene_desc_free(self.ptr)
            self.ptr = C.POINTER(SceneDesc)()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Scene:
    """Device copy of a scene (ipt_scene_create) + the calls of the hot path."""

    def __init__(self, description: SceneDescription, device: int = 0):
        self.description = description
        self.device = device
        self.handle = _vp()
        check(load().ipt_scene_create(description.ptr, device, C.byref(self.handle)))

    def set_camera(self, camera: Camera):
        """Replace the camera of the device scene (what Gui::work does after an arrow key, gui.cpp:129-133)."""
        check(load().ipt_scene_set_camera(self.handle, C.byref(camera)))

    def close(self):
        if self.handle:
            load().ipt_scene_destroy(self.handle)
            self.handle = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def dispatch(self) -> dict:
        """ipt_scene_dispatch: the kernel instantiations ipt_scene_create chose (see include/ipt_b200.h)."""
        out = np.zeros(DISPATCH_WORDS, np.uint32)
        check(load().ipt_scene_dispatch(self.handle, _ptr(out, u32p)))
        return dict(zip(DISPATCH_FIELDS, (int(v) for v in out)))

    def update_triangles(self, triangles, rebuild: bool = False):
        """ipt_scene_update_triangles: new vertices for the scene's mesh, same triangle count. `triangles` is a C-contiguous
        float32 numpy array of shape (n, 9) or (9n,) (host input), or a contiguous float32 CUDA tensor of either shape on the
        scene's device (device input: torch's current stream on that device is synchronised first). rebuild=False refits
        the existing tree, rebuild=True builds it anew over the new vertices."""
        flags = UPDATE_REBUILD if rebuild else 0
        if isinstance(triangles, np.ndarray):
            if triangles.dtype != np.float32 or not triangles.flags.c_contiguous:
                raise TypeError("triangles: a C-contiguous float32 array is required")
            shape, ptr = triangles.shape, triangles.ctypes.data
        else:
            import torch  # the only torch use of this module: device input

            if not isinstance(triangles, torch.Tensor):
                raise TypeError(f"triangles: a numpy array or a CUDA tensor is required, not {type(triangles).__name__}")
            if triangles.dtype != torch.float32 or not triangles.is_contiguous():
                raise TypeError("triangles: a contiguous float32 tensor is required")
            if triangles.device.type != "cuda" or triangles.device.index != self.device:
                raise ValueError(f"triangles: a tensor on cuda:{self.device} (the scene's device) is required, not on {triangles.device}")
            torch.cuda.current_stream(triangles.device).synchronize()
            shape, ptr = tuple(triangles.shape), triangles.data_ptr()
            flags |= UPDATE_DEVICE_POINTER
        if not (len(shape) == 2 and shape[1] == 9 or len(shape) == 1 and shape[0] % 9 == 0):
            raise ValueError(f"triangles: shape (n, 9) or (9n,) required, got {shape}")
        n = shape[0] if len(shape) == 2 else shape[0] // 9
        check(load().ipt_scene_update_triangles(self.handle, ptr, n, flags))

    def set_triangle_materials(self, materials):
        """ipt_scene_set_triangle_materials: materials[k] (an index into the scene's material list) for triangle k of the
        mesh. `materials` is a C-contiguous uint32 numpy array of length n (host input), or a contiguous int32 or uint32
        CUDA tensor of length n on the scene's device (device input: torch's current stream on that device is synchronised
        first). Kept through update_triangles; a later call replaces the whole array."""
        flags = 0
        if isinstance(materials, np.ndarray):
            if materials.dtype != np.uint32 or not materials.flags.c_contiguous:
                raise TypeError("materials: a C-contiguous uint32 array is required")
            shape, ptr = materials.shape, materials.ctypes.data
        else:
            import torch  # device input, as in update_triangles

            if not isinstance(materials, torch.Tensor):
                raise TypeError(f"materials: a numpy array or a CUDA tensor is required, not {type(materials).__name__}")
            if materials.dtype not in (torch.int32, torch.uint32) or not materials.is_contiguous():
                raise TypeError("materials: a contiguous int32 or uint32 tensor is required")
            if materials.device.type != "cuda" or materials.device.index != self.device:
                raise ValueError(f"materials: a tensor on cuda:{self.device} (the scene's device) is required, not on {materials.device}")
            torch.cuda.current_stream(materials.device).synchronize()
            shape, ptr = tuple(materials.shape), materials.data_ptr()
            flags |= UPDATE_DEVICE_POINTER
        if len(shape) != 1:
            raise ValueError(f"materials: shape (n,) required, got {shape}")
        check(load().ipt_scene_set_triangle_materials(self.handle, ptr, shape[0], flags))

    def update_lights(self, lights, rebuild: bool = False):
        """ipt_scene_update_lights: new positions, axes, radii and powers for the scene's lights, same count and kinds.
        `lights` is a sequence of Light (host input), or a contiguous float32 or int32 CUDA tensor of shape (n, 12) on the
        scene's device laid out as ipt_light records, column 0 holding the kind's bit pattern (device input: torch's current
        stream on that device is synchronised first). rebuild=False refits the light LBVH, rebuild=True builds it anew."""
        flags = UPDATE_REBUILD if rebuild else 0
        if isinstance(lights, (list, tuple)):
            if not all(isinstance(l, Light) for l in lights):
                raise TypeError("lights: a sequence of capi.Light is required")
            arr = (Light * len(lights))(*lights)
            n, ptr = len(lights), C.addressof(arr)
        else:
            import torch  # device input, as in update_triangles

            if not isinstance(lights, torch.Tensor):
                raise TypeError(f"lights: a sequence of capi.Light or a CUDA tensor is required, not {type(lights).__name__}")
            if lights.dtype not in (torch.float32, torch.int32) or not lights.is_contiguous():
                raise TypeError("lights: a contiguous float32 or int32 tensor is required")
            if lights.device.type != "cuda" or lights.device.index != self.device:
                raise ValueError(f"lights: a tensor on cuda:{self.device} (the scene's device) is required, not on {lights.device}")
            if lights.dim() != 2 or lights.shape[1] != C.sizeof(Light) // 4:
                raise ValueError(f"lights: shape (n, {C.sizeof(Light) // 4}) required, got {tuple(lights.shape)}")
            torch.cuda.current_stream(lights.device).synchronize()
            n, ptr = lights.shape[0], lights.data_ptr()
            flags |= UPDATE_DEVICE_POINTER
        check(load().ipt_scene_update_lights(self.handle, ptr, n, flags))

    def trace_batch(self, origins, directions):
        o, d = _f32(origins).reshape(-1, 3), _f32(directions).reshape(-1, 3)
        n = o.shape[0]
        prim = np.empty(n, np.uint32); t = np.empty(n, np.float32); light = np.empty(n, np.uint32)
        lpos = np.empty((n, 3), np.float32); outcome = np.empty(n, np.uint32)
        check(load().ipt_trace_batch(self.handle, _ptr(o, f32p), _ptr(d, f32p), n, _ptr(prim, u32p), _ptr(t, f32p),
                                     _ptr(light, u32p), _ptr(lpos, f32p), _ptr(outcome, u32p)))
        return dict(prim=prim, t=t, light=light, light_pos=lpos, outcome=outcome)

    def preview_batch(self, origins, directions):
        o, d = _f32(origins).reshape(-1, 3), _f32(directions).reshape(-1, 3)
        v = np.empty(o.shape[0], np.float32)
        check(load().ipt_preview_batch(self.handle, _ptr(o, f32p), _ptr(d, f32p), o.shape[0], _ptr(v, f32p)))
        return v

    def camera_rays(self, xy):
        xy = _f32(xy).reshape(-1, 2)
        n = xy.shape[0]
        o = np.empty((n, 3), np.float32); d = np.empty((n, 3), np.float32)
        check(load().ipt_camera_rays(self.handle, _ptr(xy, f32p), n, _ptr(o, f32p), _ptr(d, f32p)))
        return o, d

    def ddf_value(self, kind, dirs, to=None):
        w = _f32(dirs).reshape(-1, 3)
        out = np.empty(w.shape[0], np.float32)
        tt = _f32(to) if to is not None else None
        check(load().ipt_ddf_value(self.handle, kind, _ptr(tt, f32p), _ptr(w, f32p), w.shape[0], _ptr(out, f32p)))
        return out

    def ddf_sample(self, kind, n, seed=0, to=None):
        w = np.empty((n, 3), np.float32)
        tt = _f32(to) if to is not None else None
        check(load().ipt_ddf_sample(self.handle, kind, _ptr(tt, f32p), seed, n, _ptr(w, f32p)))
        return w

    def mix_sample(self, origin, direction, n, seed=0):
        o, d = _f32(origin), _f32(direction)
        w = np.empty((n, 3), np.float32); mv = np.empty(n, np.float32); sv = np.empty(n, np.float32)
        check(load().ipt_mix_sample(self.handle, _ptr(o, f32p), _ptr(d, f32p), seed, n, _ptr(w, f32p), _ptr(mv, f32p), _ptr(sv, f32p)))
        return w, mv, sv

    def light_ddf_value(self, pos, dirs):
        p, w = _f32(pos), _f32(dirs).reshape(-1, 3)
        out = np.empty(w.shape[0], np.float32)
        check(load().ipt_light_ddf_value(self.handle, _ptr(p, f32p), _ptr(w, f32p), w.shape[0], _ptr(out, f32p)))
        return out

    def light_ddf_sample(self, pos, n, seed=0):
        p = _f32(pos)
        w = np.empty((n, 3), np.float32)
        check(load().ipt_light_ddf_sample(self.handle, _ptr(p, f32p), seed, n, _ptr(w, f32p)))
        return w

    def bvh_export(self):
        n_nodes = C.c_uint64(0)
        check(load().ipt_bvh_export(self.handle, None, None, None, C.byref(n_nodes)))
        n = n_nodes.value
        ntri = self.description.desc.n_triangles
        nodes = np.zeros(n, BVH_NODE_DTYPE); order = np.empty(ntri, np.uint32); keys = np.empty(ntri, np.uint64)
        check(load().ipt_bvh_export(self.handle, nodes.ctypes.data_as(C.POINTER(BvhNode)), _ptr(order, u32p), _ptr(keys, u64p), C.byref(n_nodes)))
        return nodes, order, keys

    def bvh_export_compact(self):
        """(nodes uint32[n-1, 8], grid float32[6]): the 32-byte traversal nodes and their world -> grid map."""
        n = C.c_uint64(0)
        check(load().ipt_bvh_export_compact(self.handle, None, None, C.byref(n)))
        nodes = np.zeros((n.value, 8), np.uint32); grid = np.zeros(6, np.float32)
        check(load().ipt_bvh_export_compact(self.handle, _ptr(nodes, u32p), _ptr(grid, f32p), C.byref(n)))
        return nodes, grid

    def render_host(self, params: RenderParams, out=None):
        """The end-to-end call: host buffers in, host buffers out. `out` = (sum, sumsq, count) arrays to reuse."""
        n = params.width * params.height
        if out is None:
            s = np.empty(n, np.float32); q = np.empty(n, np.float32); c = np.empty(n, np.uint32)
        else:
            s, q, c = (a.reshape(-1) for a in out)
        st = RenderStats()
        check(load().ipt_render_host(self.handle, C.byref(params), _ptr(s, f32p), _ptr(q, f32p), _ptr(c, u32p), C.byref(st)))
        shape = (params.height, params.width)
        return s.reshape(shape), q.reshape(shape), c.reshape(shape), st


class Plane:
    """Device accumulators (sum, sumsq, count) == what RenderPlane::addRay accumulates."""

    def __init__(self, scene: Scene, width: int, height: int, wrap=None):
        self.scene, self.width, self.height = scene, width, height
        self.handle = _vp()
        if wrap is None:
            check(load().ipt_plane_create(scene.handle, width, height, C.byref(self.handle)))
        else:
            d_sum, d_sumsq, d_count = wrap
            check(load().ipt_plane_wrap(scene.handle, width, height, d_sum, d_sumsq, d_count, C.byref(self.handle)))

    def clear(self):
        check(load().ipt_plane_clear(self.handle))

    def render(self, params: RenderParams) -> RenderStats:
        st = RenderStats()
        check(load().ipt_render(self.scene.handle, self.handle, C.byref(params), C.byref(st)))
        return st

    def add_rays(self, x, y, v, mode=PLANE_GRID):
        x, y, v = _f32(x), _f32(y), _f32(v)
        check(load().ipt_plane_add_rays(self.handle, mode, len(x), _ptr(x, f32p), _ptr(y, f32p), _ptr(v, f32p)))

    def download(self):
        n = self.width * self.height
        s = np.empty(n, np.float32); q = np.empty(n, np.float32); c = np.empty(n, np.uint32)
        check(load().ipt_plane_download(self.handle, _ptr(s, f32p), _ptr(q, f32p), _ptr(c, u32p)))
        shape = (self.height, self.width)
        return s.reshape(shape), q.reshape(shape), c.reshape(shape)

    def upload(self, s, q, c):
        s, q = _f32(s).ravel(), _f32(q).ravel()
        c = np.ascontiguousarray(c, np.uint32).ravel()
        check(load().ipt_plane_upload(self.handle, _ptr(s, f32p), _ptr(q, f32p), _ptr(c, u32p)))

    def allreduce(self, nccl_comm) -> float:
        """ipt_plane_allreduce with an ncclComm_t (integer / c_void_p) of the calling process; returns its device time in ms."""
        ms = C.c_float(0)
        check(load().ipt_plane_allreduce(self.handle, nccl_comm, C.byref(ms)))
        return ms.value

    def merge(self, other: "Plane"):
        """ipt_plane_merge: self += other (the planes may live on different devices of this process)."""
        check(load().ipt_plane_merge(self.handle, other.handle))

    def download_into(self, s, q, c):
        """ipt_plane_download into caller-owned (e.g. pinned) host arrays."""
        check(load().ipt_plane_download(self.handle, _ptr(s, f32p), _ptr(q, f32p), _ptr(c, u32p)))

    def resolve(self):
        n = self.width * self.height
        pix = np.empty(n, np.float32); cnt = np.empty(n, np.uint64); mx = C.c_float(0)
        check(load().ipt_plane_resolve(self.handle, _ptr(pix, f32p), _ptr(cnt, u64p), C.byref(mx)))
        shape = (self.height, self.width)
        return pix.reshape(shape), cnt.reshape(shape), mx.value

    def display(self, glare_cutoff: float = 1.01):
        """What Gui::updateDisplay shows: normalize(glare(image, cutoff)) (gui.cpp:83-87); returns (image, device ms)."""
        out = np.empty((self.height, self.width), np.float32); ms = C.c_float(0)
        check(load().ipt_plane_display(self.handle, glare_cutoff, _ptr(out, f32p), C.byref(ms)))
        return out, ms.value

    def save_bytes(self):
        """The pixel bytes of Gui::save (gui.cpp:192-194)."""
        out = np.empty((self.height, self.width), np.uint8)
        check(load().ipt_plane_save_bytes(self.handle, _ptr(out, u8p)))
        return out

    def save_png(self, path: str):
        check(load().ipt_plane_save_png(self.handle, str(path).encode()))

    def close(self):
        if self.handle:
            load().ipt_plane_destroy(self.handle)
            self.handle = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
