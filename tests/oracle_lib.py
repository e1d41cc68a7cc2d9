"""ctypes access to the two CPU checkers — TEST INFRASTRUCTURE, importable from tests/, smoke() and bench.py only.

* oracle/libipt_oracle.so — our plain-C restatement (oracle/ipt_oracle.c), built with `make -C oracle oracle`.
* oracle/_ref/libipt_ref.so — the unmodified reference compiled from the dimalit/ipt checkout that IPT_REFERENCE names
  (`make -C oracle ref REF=...`); where none is given, a prebuilt file is used if present.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
ORACLE_SO = ROOT / "oracle" / "libipt_oracle.so"
REF_SO = ROOT / "oracle" / "_ref" / "libipt_ref.so"
REF_SRC = Path(os.environ["IPT_REFERENCE"]) if os.environ.get("IPT_REFERENCE") else None  # not part of this repository

f32p = C.POINTER(C.c_float)
f64p = C.POINTER(C.c_double)
u32p = C.POINTER(C.c_uint32)
i32p = C.POINTER(C.c_int32)
u64p = C.POINTER(C.c_uint64)
u8p = C.POINTER(C.c_uint8)
RNG_DRAND48, RNG_PHILOX = 0, 1


def _stale(target: Path, deps) -> bool:
    if not target.exists():
        return True
    t = target.stat().st_mtime
    return any(p.exists() and p.stat().st_mtime > t for p in deps)


def build_oracle():
    deps = [ROOT / "oracle" / "ipt_oracle.c", ROOT / "oracle" / "ipt_oracle_mesh.inc", ROOT / "oracle" / "ipt_oracle_output.inc",
            ROOT / "include" / "ipt_b200.h"]
    if _stale(ORACLE_SO, deps):
        subprocess.run(["make", "-C", str(ROOT / "oracle"), "oracle"], check=True, capture_output=True)
    return ORACLE_SO


def build_ref():
    """Compiles the reference where it lies; returns None if it is neither built nor buildable here."""
    if REF_SRC is not None and REF_SRC.exists():
        if _stale(REF_SO, [ROOT / "oracle" / "ref_driver.cpp", ROOT / "oracle" / "ref_gui_driver.cpp"]):
            subprocess.run(["make", "-C", str(ROOT / "oracle"), "ref", f"REF={REF_SRC}"], check=True, capture_output=True)
    return REF_SO if REF_SO.exists() else None


DROPIN = ROOT / "oracle" / "_ref" / "ab_dropin"


def build_dropin():
    """oracle/_ref/ab_dropin (ipt_b200's host classes compiled against the reference's headers + the reference's own
    estimator): built where the reference sources exist, else the prebuilt binary if it travelled with the snapshot."""
    if REF_SRC is not None and REF_SRC.exists() and (ROOT / "ipt_b200" / "lib" / "libipt_b200.so").exists():
        deps = [ROOT / "oracle" / "ab_dropin.cpp", ROOT / "ipt_b200" / "host" / "device_plugins.cpp", ROOT / "ipt_b200" / "host" / "device_plugins.hpp", REF_SO]
        if _stale(DROPIN, deps):
            subprocess.run(["make", "-C", str(ROOT / "oracle"), "ref", "dropin", f"REF={REF_SRC}"], check=True, capture_output=True)
    return DROPIN if DROPIN.exists() else None


def _p(a, t):
    return a.ctypes.data_as(t) if a is not None else None


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


class _OutputStage:
    """The output stage (src/gui.cpp) behind either checker: prefix 'ipt_oracle_' (restatement) or 'iptref_' (reference)."""
    _prefix = ""

    def _fn(self, name):
        return getattr(self.lib, self._prefix + name)

    def image_normalize(self, image):
        img = _f32(image); h, w = img.shape
        out = np.empty_like(img)
        assert self._fn("image_normalize")(_p(img, f32p), C.c_uint32(w), C.c_uint32(h), _p(out, f32p)) == 0
        return out

    def image_glare(self, image, cutoff):
        img = _f32(image); h, w = img.shape
        out = np.empty_like(img)
        assert self._fn("image_glare")(_p(img, f32p), C.c_uint32(w), C.c_uint32(h), C.c_float(cutoff), _p(out, f32p)) == 0
        return out

    def image_save_bytes(self, image):
        img = _f32(image); h, w = img.shape
        out = np.empty((h, w), np.uint8)
        assert self._fn("image_save_bytes")(_p(img, f32p), C.c_uint32(w), C.c_uint32(h), _p(out, u8p)) == 0
        return out

    def camera_orbit(self, position, direction, key):
        """Returns a (4,3) float32 array: position, direction, right, up after the key."""
        cam = np.zeros((4, 3), np.float32)
        cam[0], cam[1] = position, direction
        if self._prefix == "iptref_":
            assert self.lib.iptref_camera_orbit(_p(cam[0:1], f32p), C.cast(cam[1:2].ctypes.data, f32p), C.cast(cam[2:3].ctypes.data, f32p),
                                                C.cast(cam[3:4].ctypes.data, f32p), key) == 0
        else:
            assert self.lib.ipt_oracle_camera_orbit(C.c_void_p(cam.ctypes.data), key) == 0  # ipt_camera == 12 floats
        return cam


class Oracle(_OutputStage):
    _prefix = "ipt_oracle_"

    def __init__(self, lib):
        self.lib = lib
        lib.ipt_oracle_threads.restype = C.c_int
        lib.ipt_oracle_seed.argtypes = [C.c_long]

    def threads(self):
        return self.lib.ipt_oracle_threads()

    def seed(self, s):
        self.lib.ipt_oracle_seed(s)

    def render(self, desc_ptr, params, rng_mode=RNG_PHILOX, use_bvh=1):
        """Returns dict(pixels, counters, sum, sumsq, rays, rays_at_depth) for params.pass_count passes."""
        W, H = params.width, params.height
        n = W * H
        pixels = np.zeros(n, np.float32); counters = np.zeros(n, np.uint64)
        s = np.zeros(n, np.float64); q = np.zeros(n, np.float64)
        rays = C.c_uint64(0); rad = (C.c_uint64 * 16)()
        rc = self.lib.ipt_oracle_render(desc_ptr, C.byref(params), rng_mode, use_bvh, _p(pixels, f32p), _p(counters, u64p),
                                        _p(s, f64p), _p(q, f64p), C.byref(rays), rad)
        assert rc == 0
        return dict(pixels=pixels.reshape(H, W), counters=counters.reshape(H, W), sum=s.reshape(H, W), sumsq=q.reshape(H, W),
                    rays=rays.value, rays_at_depth=list(rad))

    def trace_batch(self, desc_ptr, o, d, use_bvh=0):
        o, d = _f32(o).reshape(-1, 3), _f32(d).reshape(-1, 3)
        n = o.shape[0]
        prim = np.empty(n, np.uint32); t = np.empty(n, np.float32); pos = np.empty((n, 3), np.float32)
        normal = np.empty((n, 3), np.float32); light = np.empty(n, np.uint32); lpos = np.empty((n, 3), np.float32)
        outcome = np.empty(n, np.uint32)
        rc = self.lib.ipt_oracle_trace_batch(desc_ptr, _p(o, f32p), _p(d, f32p), C.c_size_t(n), use_bvh, _p(prim, u32p), _p(t, f32p),
                                             _p(pos, f32p), _p(normal, f32p), _p(light, u32p), _p(lpos, f32p), _p(outcome, u32p))
        assert rc == 0
        return dict(prim=prim, t=t, pos=pos, normal=normal, light=light, light_pos=lpos, outcome=outcome)

    def preview_batch(self, desc_ptr, o, d, use_bvh=0):
        o, d = _f32(o).reshape(-1, 3), _f32(d).reshape(-1, 3)
        v = np.empty(o.shape[0], np.float32)
        self.lib.ipt_oracle_preview_batch(desc_ptr, _p(o, f32p), _p(d, f32p), C.c_size_t(o.shape[0]), use_bvh, _p(v, f32p))
        return v

    def camera_rays(self, desc_ptr, xy):
        xy = _f32(xy).reshape(-1, 2)
        n = xy.shape[0]
        o = np.empty((n, 3), np.float32); d = np.empty((n, 3), np.float32)
        self.lib.ipt_oracle_camera_rays(desc_ptr, _p(xy, f32p), C.c_size_t(n), _p(o, f32p), _p(d, f32p))
        return o, d

    def ddf_value(self, kind, w, to=None):
        w = _f32(w).reshape(-1, 3)
        out = np.empty(w.shape[0], np.float32)
        tt = _f32(to) if to is not None else None
        self.lib.ipt_oracle_ddf_value(kind, _p(tt, f32p), _p(w, f32p), C.c_size_t(w.shape[0]), _p(out, f32p))
        return out

    def ddf_sample(self, kind, n, to=None):
        w = np.empty((n, 3), np.float32)
        tt = _f32(to) if to is not None else None
        self.lib.ipt_oracle_ddf_sample(kind, _p(tt, f32p), C.c_size_t(n), _p(w, f32p))
        return w

    def mix_sample(self, desc_ptr, o, d, n):
        o, d = _f32(o), _f32(d)
        w = np.empty((n, 3), np.float32); mv = np.empty(n, np.float32); sv = np.empty(n, np.float32)
        rc = self.lib.ipt_oracle_mix_sample(desc_ptr, _p(o, f32p), _p(d, f32p), C.c_size_t(n), _p(w, f32p), _p(mv, f32p), _p(sv, f32p))
        assert rc == 0
        return w, mv, sv

    def mix_value(self, desc_ptr, o, d, w):
        o, d, w = _f32(o), _f32(d), _f32(w).reshape(-1, 3)
        n = w.shape[0]
        mv = np.empty(n, np.float32); sv = np.empty(n, np.float32); lv = np.empty(n, np.float32)
        rc = self.lib.ipt_oracle_mix_value(desc_ptr, _p(o, f32p), _p(d, f32p), C.c_size_t(n), _p(w, f32p), _p(mv, f32p), _p(sv, f32p), _p(lv, f32p))
        assert rc == 0
        return mv, sv, lv

    def light_ddf_value(self, desc_ptr, pos, w):
        pos, w = _f32(pos), _f32(w).reshape(-1, 3)
        out = np.empty(w.shape[0], np.float32)
        self.lib.ipt_oracle_light_ddf_value(desc_ptr, _p(pos, f32p), _p(w, f32p), C.c_size_t(w.shape[0]), _p(out, f32p))
        return out

    def light_ddf_sample(self, desc_ptr, pos, n):
        pos = _f32(pos)
        w = np.empty((n, 3), np.float32)
        self.lib.ipt_oracle_light_ddf_sample(desc_ptr, _p(pos, f32p), C.c_size_t(n), _p(w, f32p))
        return w

    def arealight(self, origin, xa, ya, power, triangle, ro, rd):
        area = C.c_float(); hit = C.c_int32(); sp = C.c_float()
        a = [_f32(v) for v in (origin, xa, ya, ro, rd)]
        self.lib.ipt_oracle_arealight(_p(a[0], f32p), _p(a[1], f32p), _p(a[2], f32p), C.c_float(power), int(triangle),
                                      _p(a[3], f32p), _p(a[4], f32p), C.byref(area), C.byref(hit), C.byref(sp))
        return area.value, bool(hit.value), sp.value

    def light_fields(self, desc_ptr, i):
        out = np.empty(5, np.float32)
        self.lib.ipt_oracle_light_fields(desc_ptr, C.c_uint32(i), _p(out, f32p))
        return out

    def light_tables(self, desc_ptr, n_lights):
        """Per light the area, surface power, normal (n, 3) and mixture weight the oracle derives, as float32 arrays."""
        area, sp, w = (np.empty(n_lights, np.float32) for _ in range(3))
        normal = np.empty((n_lights, 3), np.float32)
        assert self.lib.ipt_oracle_light_tables(desc_ptr, _p(area, f32p), _p(sp, f32p), _p(normal, f32p), _p(w, f32p)) == 0
        return dict(area=area, surface_power=sp, normal=normal, weight=w)

    def bvh_build(self, triangles):
        """The LBVH exactly as ipt_b200/csrc/ipt_lbvh.cuh builds it: (nodes, sorted ids, sorted Morton keys)."""
        from ipt_b200.capi import BVH_NODE_DTYPE

        t = _f32(triangles).reshape(-1, 9)
        n = t.shape[0]
        nodes = np.zeros(max(n - 1, 0), BVH_NODE_DTYPE); ids = np.empty(n, np.uint32); keys = np.empty(n, np.uint64)
        self.lib.ipt_oracle_bvh_build(_p(t, f32p), C.c_uint64(n), nodes.ctypes.data_as(C.c_void_p), _p(ids, u32p), _p(keys, u64p))
        return nodes, ids, keys

    def bvh_compact(self, nodes):
        """The 32-byte traversal nodes derived from the 64-byte ones (k_lbvh_compact): (uint32[n, 8], grid float32[6])."""
        out = np.zeros((len(nodes), 8), np.uint32); grid = np.zeros(6, np.float32)
        self.lib.ipt_oracle_bvh_compact(nodes.ctypes.data_as(C.c_void_p), C.c_uint64(len(nodes)), _p(out, u32p), _p(grid, f32p))
        return out, grid

    def bvh_trace_counts(self, triangles, o, d, compact):
        """Closest triangle per ray over the float nodes (compact=0) or the quantised nodes (compact=1), with the node visits and
        triangle tests it took: dict(prim, t, nodes, tris)."""
        t = _f32(triangles).reshape(-1, 9); o, d = _f32(o).reshape(-1, 3), _f32(d).reshape(-1, 3)
        n = o.shape[0]
        prim = np.empty(n, np.uint32); tt = np.empty(n, np.float32); nodes = np.empty(n, np.uint32); tris = np.empty(n, np.uint32)
        rc = self.lib.ipt_oracle_bvh_trace_counts(_p(t, f32p), C.c_uint64(t.shape[0]), _p(o, f32p), _p(d, f32p), C.c_uint64(n), int(compact),
                                                  _p(prim, u32p), _p(tt, f32p), _p(nodes, u32p), _p(tris, u32p))
        assert rc == 0
        return dict(prim=prim, t=tt, nodes=nodes, tris=tris)

    def philox_rounds(self, rounds, c, k):
        out = (C.c_uint32 * 4)()
        self.lib.ipt_oracle_philox_rounds(rounds, *[C.c_uint32(v) for v in c], *[C.c_uint32(v) for v in k], out)
        return list(out)

    def philox(self, c, k):
        out = (C.c_uint32 * 4)()
        self.lib.ipt_oracle_philox(*[C.c_uint32(v) for v in c], *[C.c_uint32(v) for v in k], out)
        return list(out)


class Ref(_OutputStage):
    """The compiled reference behind oracle/ref_driver.cpp (main.cpp) and oracle/ref_gui_driver.cpp (gui.cpp)."""
    _prefix = "iptref_"

    def __init__(self, lib):
        self.lib = lib
        lib.iptref_scene_create.argtypes = [C.c_char_p]
        lib.iptref_seed.argtypes = [C.c_long]
        lib.iptref_render.restype = C.c_uint64
        lib.iptref_render_wh.restype = C.c_uint64
        lib.iptref_rays_traced.restype = C.c_uint64
        lib.iptref_ray_power.restype = C.c_float
        self._scenes = {}

    def scene(self, name: str) -> int:
        if name not in self._scenes:
            if name.startswith("lightgrid:"):
                r, c = name[10:].split("x")
                h = self.lib.iptref_scene_create(b"box")
                self.lib.iptref_scene_set_light_grid(h, int(r), int(c), C.c_float(0.01), C.c_float(0.99), C.c_float(1.0))
            elif name == "mixedlights":
                h = self.lib.iptref_scene_create(b"box")
                self.lib.iptref_scene_set_mixed_lights(h)
            else:
                h = self.lib.iptref_scene_create(name.encode())
            assert h >= 0, name
            self._scenes[name] = h
        return self._scenes[name]

    def set_tree(self, n_rays, depth_max):
        self.lib.iptref_set_tree(n_rays, depth_max)

    def seed(self, s):
        self.lib.iptref_seed(s)

    def camera_fields(self, scene):
        out = np.empty(12, np.float32)
        self.lib.iptref_camera_fields(scene, _p(out, f32p))
        return out.reshape(4, 3)

    def camera_rays(self, scene, xy):
        xy = _f32(xy).reshape(-1, 2)
        n = xy.shape[0]
        o = np.empty((n, 3), np.float32); d = np.empty((n, 3), np.float32)
        self.lib.iptref_camera_rays(scene, C.c_size_t(n), _p(xy, f32p), _p(o, f32p), _p(d, f32p))
        return o, d

    def trace_geometry(self, scene, o, d):
        o, d = _f32(o).reshape(-1, 3), _f32(d).reshape(-1, 3)
        n = o.shape[0]
        hit = np.empty(n, np.int32); pos = np.empty((n, 3), np.float32); normal = np.empty((n, 3), np.float32); curv = np.empty(n, np.float32)
        self.lib.iptref_trace_geometry(scene, C.c_size_t(n), _p(o, f32p), _p(d, f32p), _p(hit, i32p), _p(pos, f32p), _p(normal, f32p), _p(curv, f32p))
        return dict(hit=hit.astype(bool), pos=pos, normal=normal, curvature=curv)

    def trace_light(self, scene, o, d):
        o, d = _f32(o).reshape(-1, 3), _f32(d).reshape(-1, 3)
        n = o.shape[0]
        hit = np.empty(n, np.int32); pos = np.empty((n, 3), np.float32); normal = np.empty((n, 3), np.float32); power = np.empty(n, np.float32)
        self.lib.iptref_trace_light(scene, C.c_size_t(n), _p(o, f32p), _p(d, f32p), _p(hit, i32p), _p(pos, f32p), _p(normal, f32p), _p(power, f32p))
        return dict(hit=hit.astype(bool), pos=pos, normal=normal, power=power)

    def light_count(self, scene):
        return self.lib.iptref_light_count(scene)

    def light_fields(self, scene, i):
        out = np.empty(5, np.float32)
        self.lib.iptref_light_fields(scene, i, _p(out, f32p))
        return out

    def sdf_value(self, scene, o, d, w):
        o, d, w = _f32(o), _f32(d), _f32(w).reshape(-1, 3)
        out = np.empty(w.shape[0], np.float32)
        ok = self.lib.iptref_sdf_value(scene, _p(o, f32p), _p(d, f32p), C.c_size_t(w.shape[0]), _p(w, f32p), _p(out, f32p))
        assert ok
        return out

    def sdf_sample(self, scene, o, d, n):
        o, d = _f32(o), _f32(d)
        w = np.empty((n, 3), np.float32)
        ok = self.lib.iptref_sdf_sample(scene, _p(o, f32p), _p(d, f32p), C.c_size_t(n), _p(w, f32p))
        assert ok
        return w

    def light_ddf_value(self, scene, pos, w):
        pos, w = _f32(pos), _f32(w).reshape(-1, 3)
        out = np.empty(w.shape[0], np.float32)
        self.lib.iptref_light_ddf_value(scene, _p(pos, f32p), C.c_size_t(w.shape[0]), _p(w, f32p), _p(out, f32p))
        return out

    def light_ddf_sample(self, scene, pos, n):
        pos = _f32(pos)
        w = np.empty((n, 3), np.float32)
        self.lib.iptref_light_ddf_sample(scene, _p(pos, f32p), C.c_size_t(n), _p(w, f32p))
        return w

    def mix_sample(self, scene, o, d, n):
        o, d = _f32(o), _f32(d)
        w = np.empty((n, 3), np.float32); mv = np.empty(n, np.float32); sv = np.empty(n, np.float32)
        ok = self.lib.iptref_mix_sample(scene, _p(o, f32p), _p(d, f32p), C.c_size_t(n), _p(w, f32p), _p(mv, f32p), _p(sv, f32p))
        assert ok
        return w, mv, sv

    def ddf_value(self, kind, w, to=None):
        w = _f32(w).reshape(-1, 3)
        out = np.empty(w.shape[0], np.float32)
        tt = _f32(to) if to is not None else None
        self.lib.iptref_ddf_value(kind, _p(tt, f32p), C.c_size_t(w.shape[0]), _p(w, f32p), _p(out, f32p))
        return out

    def ddf_sample(self, kind, n, to=None):
        w = np.empty((n, 3), np.float32)
        tt = _f32(to) if to is not None else None
        self.lib.iptref_ddf_sample(kind, _p(tt, f32p), C.c_size_t(n), _p(w, f32p))
        return w

    def arealight(self, origin, xa, ya, power, triangle, ro, rd):
        area = C.c_float(); hit = C.c_int32(); sp = C.c_float()
        a = [_f32(v) for v in (origin, xa, ya, ro, rd)]
        self.lib.iptref_arealight(_p(a[0], f32p), _p(a[1], f32p), _p(a[2], f32p), C.c_float(power), int(triangle),
                                  _p(a[3], f32p), _p(a[4], f32p), C.byref(area), C.byref(hit), C.byref(sp))
        return area.value, bool(hit.value), sp.value

    def preview_batch(self, scene, o, d):
        o, d = _f32(o).reshape(-1, 3), _f32(d).reshape(-1, 3)
        v = np.empty(o.shape[0], np.float32)
        self.lib.iptref_preview_batch(scene, C.c_size_t(o.shape[0]), _p(o, f32p), _p(d, f32p), _p(v, f32p))
        return v

    def ray_power(self, scene, o, d, depth, n):
        o, d = _f32(o), _f32(d)
        return self.lib.iptref_ray_power(scene, _p(o, f32p), _p(d, f32p), depth, n)

    def render(self, scene, passes, W=640, H=640, verbatim=True):
        """verbatim=True: the reference's own render_sample (640x640 only). Else the W,H-parametrised loop of the driver."""
        n = W * H
        pixels = np.zeros(n, np.float32); counters = np.zeros(n, np.uint64); s = np.zeros(n, np.float64); q = np.zeros(n, np.float64)
        if verbatim:
            assert (W, H) == (640, 640)
            rays = self.lib.iptref_render(scene, passes, _p(pixels, f32p), _p(counters, u64p), _p(s, f64p), _p(q, f64p))
        else:
            rays = self.lib.iptref_render_wh(scene, passes, C.c_size_t(W), C.c_size_t(H), _p(pixels, f32p), _p(counters, u64p), _p(s, f64p), _p(q, f64p))
        return dict(pixels=pixels.reshape(H, W), counters=counters.reshape(H, W), sum=s.reshape(H, W), sumsq=q.reshape(H, W), rays=rays)

    def plane_addray(self, W, H, x, y, v):
        x, y, v = _f32(x), _f32(y), _f32(v)
        pixels = np.zeros(W * H, np.float32); counters = np.zeros(W * H, np.uint64); mx = C.c_float()
        self.lib.iptref_plane_addray(C.c_size_t(W), C.c_size_t(H), C.c_size_t(len(x)), _p(x, f32p), _p(y, f32p), _p(v, f32p),
                                     _p(pixels, f32p), _p(counters, u64p), C.byref(mx))
        return pixels.reshape(H, W), counters.reshape(H, W), mx.value


_oracle = None
_ref = None


def load_oracle() -> Oracle:
    global _oracle
    if _oracle is None:
        _oracle = Oracle(C.CDLL(str(build_oracle())))
    return _oracle


def load_ref():
    global _ref
    if _ref is None:
        so = build_ref()
        if so is None:
            return None
        _ref = Ref(C.CDLL(str(so)))
    return _ref
