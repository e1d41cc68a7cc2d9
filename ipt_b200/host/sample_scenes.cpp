// sample_scenes.cpp — the reference's scene factory as plain scene descriptions.
//
// The reference builds its scenes by constructing Geometry/Lighting/Camera objects whose data is
// private or literal inside traceRay() (SURVEY.md S12), so the device cannot introspect them. This file
// states the same scenes as ipt_scene_desc data:
//   make_scene_box                  src/sample_scenes.cpp:20-41   + GeometrySphereInBox.cpp:11-21
//   make_scene_fractal              src/sample_scenes.cpp:43-54   + FractalSpheres.cpp:18-64
//   make_scene_smallpt              src/sample_scenes.cpp:56-75   + GeometrySmallPt.cpp:25-34
//   make_scene_square_lit_by_square src/sample_scenes.cpp:78-90   + GeometryFloor.cpp:11
//   make_scene_lit_corner           src/sample_scenes.cpp:92-108  + GeometryCorner.cpp:11-13
//   (GeometryOpenSpheres.cpp:13-33 is reachable from no factory; offered as "openspheres")
// plus the benchmark scenes BASELINE.json names: "cornell" (configs[1]), "mesh:<n>" (configs[2..3]),
// "lightgrid:<r>x<c>" (configs[4]). tests/test_scene_desc.py checks every derived float against the
// compiled reference.
#include "ipt_b200.h"
#include "glm_order.hpp"

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <string>
#include <vector>

using namespace ipt_host;

namespace {

struct SceneHolder {
    ipt_scene_desc desc; // must stay the first member: ipt_scene_desc_free casts back
    std::vector<ipt_prim> prims;
    std::vector<ipt_material> materials;
    std::vector<ipt_light> lights;
    std::vector<float> triangles;
    void finish() {
        desc.n_prims = (uint32_t)prims.size();
        desc.prims = prims.data();
        desc.n_materials = (uint32_t)materials.size();
        desc.materials = materials.data();
        desc.n_lights = (uint32_t)lights.size();
        desc.lights = lights.data();
        desc.n_triangles = triangles.size() / 9;
        desc.triangles = triangles.empty() ? nullptr : triangles.data();
    }
};

ipt_material lambert() { return ipt_material{IPT_DDF_COSINE, 1.0f, 1.0f, 0.0f, 0.0f}; }

ipt_prim box_plane(float x, float y, float z, uint32_t material = 0) {
    ipt_prim p{};
    p.kind = IPT_PRIM_BOX_PLANE;
    p.material = material;
    p.p[0] = x; p.p[1] = y; p.p[2] = z;
    p.curvature = 0.0f;
    return p;
}
ipt_prim sphere(f3 c, float r, float curvature, uint32_t material = 0) {
    ipt_prim p{};
    p.kind = IPT_PRIM_SPHERE;
    p.material = material;
    put(p.p, c);
    p.radius = r;
    p.curvature = curvature;
    return p;
}

// CollectionLighting::addSquareLight (src/CollectionLighting.cpp:42-46): y_side = cross(normal, x_side)
ipt_light square_light(f3 corner, f3 normal, f3 x_side, float power = 1.0f) {
    ipt_light l{};
    l.kind = IPT_LIGHT_AREA_DIAMOND;
    put(l.position, corner);
    put(l.x_axis, x_side);
    put(l.y_axis, cross(normal, x_side));
    l.power = power;
    return l;
}
// CollectionLighting::addTriangleLight (src/CollectionLighting.cpp:47-50)
ipt_light triangle_light(f3 corner, f3 x_side, f3 y_side, float power = 1.0f) {
    ipt_light l{};
    l.kind = IPT_LIGHT_AREA_TRIANGLE;
    put(l.position, corner);
    put(l.x_axis, x_side);
    put(l.y_axis, y_side);
    l.power = power;
    return l;
}
// CollectionLighting::addSphereLight (src/CollectionLighting.cpp:39-41)
ipt_light sphere_light(f3 position, float radius, float power = 1.0f) {
    ipt_light l{};
    l.kind = IPT_LIGHT_SPHERE;
    put(l.position, position);
    l.radius = radius;
    l.power = power;
    return l;
}

// SimpleCamera::SimpleCamera (src/SimpleCamera.cpp:8-13)
ipt_camera look(f3 position, f3 direction, f3 up_hint = mk(0, 0, 1)) {
    ipt_camera c{};
    put(c.position, position);
    put(c.direction, direction);
    f3 right = normalize(cross(direction, up_hint));
    f3 up = normalize(cross(right, direction));
    put(c.right, right);
    put(c.up, up);
    return c;
}

void add_sphere_in_box_planes(SceneHolder& s) {
    // GeometrySphereInBox.cpp:11-17: +x, +y, +z, -x, -z (open towards -y)
    s.prims.push_back(box_plane(1, 0, 0));
    s.prims.push_back(box_plane(0, 1, 0));
    s.prims.push_back(box_plane(0, 0, 1));
    s.prims.push_back(box_plane(-1, 0, 0));
    s.prims.push_back(box_plane(0, 0, -1));
}

void scene_box(SceneHolder& s) {
    s.materials.push_back(lambert());
    add_sphere_in_box_planes(s);
    s.prims.push_back(sphere(mk(0, 0, 0), 0.5f, 2.0f)); // GeometrySphereInBox.cpp:31,55
    s.lights.push_back(square_light(mk(+0.1f, -0.8f - 0.1f, -0.15f), mk(0.0f, 0.0f, -1.0f), mk(0.0f, 0.2f, 0.0f), 1.0f));
    f3 camera_pos = mk(0.0f, -3.0f, 0.1f);
    f3 camera_dir = normalize(mk(0.0f, 1.0f, -1.0f) - camera_pos);
    s.desc.camera = look(camera_pos, camera_dir);
}

// generate_spheres (src/geometry/FractalSpheres.cpp:16-46) + the constructor (:48-64)
void fractal_generate(float r1, f3 c1, float r2, f3 c2, bool light_from_left, const std::function<bool(float, f3)>& cb) {
    float L = length(c1 - c2) - r1 - r2;
    if (L < 0.01) return;
    float sin_alpha = r1 / (r1 + L);
    float alpha = asinf(sin_alpha);
    float sin_beta = r2 / (r2 + L);
    float beta = asinf(sin_beta);
    const float pi32 = 3.141592653589793238462643383279502884f; // M_PIf32
    float gamma = pi32 - alpha - beta;
    float A = L * sin_alpha / sinf(gamma);
    float x = A * sinf(gamma / 2) / sinf(pi32 - beta - gamma / 2);
    f3 c3 = c1 + normalize(c2 - c1) * (x + r1);
    float r3 = x * sin_beta;
    if (cb(r3, c3)) return;
    if (light_from_left) fractal_generate(r1, c1, r3, c3, !light_from_left, cb);
    else fractal_generate(r3, c3, r2, c2, !light_from_left, cb);
}
void scene_fractal(SceneHolder& s) {
    s.materials.push_back(lambert());
    auto add = [&s](float r, f3 c) -> bool {
        if (r < 0.001) return true;
        s.prims.push_back(sphere(c, r, 1.0f / r)); // FractalSpheres.cpp:93
        return false;
    };
    float r1 = 0.5f, r2 = 0.5f;
    f3 c1 = mk(-2, 0, 0), c2 = mk(2, 0, 0);
    add(r1, c1);
    add(r2, c2);
    fractal_generate(r1, c1, r2, c2, true, add);
    s.lights.push_back(sphere_light(mk(-5.5f, 0, 0), 1.0f));
    s.desc.camera = look(mk(0.0f, -4.0f, 0.0f), mk(0, 1, 0));
}

void scene_smallpt(SceneHolder& s) {
    s.materials.push_back(lambert());
    struct S { double rad; f3 p; };
    // GeometrySmallPt.cpp:25-34 (vec3 is float: the double literals round once)
    const S spheres[] = {
        {1e3, mk((float)(1e3 + 1), (float)40.8, (float)81.6)},  {1e3, mk((float)(-1e3 + 99), (float)40.8, (float)81.6)},
        {1e3, mk(50, (float)40.8, (float)1e3)},                 {1e3, mk(50, (float)1e3, (float)81.6)},
        {1e3, mk(50, (float)(-1e3 + 81.6), (float)81.6)},       {16.5, mk(27, (float)16.5, 47)},
        {16.5, mk(73, (float)16.5, 78)},
    };
    for (const S& sp : spheres) {
        ipt_prim p{};
        p.kind = IPT_PRIM_SPHERE_SMALLPT;
        put(p.p, sp.p);
        p.radius = (float)sp.rad;             // 1e3 and 16.5 are exact in float; widened back to double on use
        p.flip_normal = sp.rad < 100 ? 0 : 1; // GeometrySmallPt.cpp:53
        p.curvature = (float)(-1.0 / sp.rad);
        s.prims.push_back(p);
    }
    f3 lc = mk(50, (float)(81.6 - 16.5), (float)81.6);
    s.lights.push_back(square_light(lc - mk(4.0f, 0, 4.0f), mk(0, -1, 0), mk(8.0f, 0, 0)));
    f3 camera_pos = mk(50.0f, 52.0f, 295.6f);
    f3 camera_dir = normalize(mk(0.0f, -0.042612f, -1.0f));
    s.desc.camera = look(camera_pos, camera_dir * 2.0f, mk(0, 1, 0));
}

void scene_square(SceneHolder& s) {
    s.materials.push_back(lambert());
    s.prims.push_back(box_plane(0, 0, -1)); // GeometryFloor.cpp:11
    s.lights.push_back(square_light(mk(-0.05f, -0.05f, -0.9f), mk(0, 0, -1), mk(0, 0.1f, 0)));
    f3 camera_pos = mk(0, -5.0f, 0);
    f3 camera_dir = normalize(mk(0, 0, -1.0f) - camera_pos);
    s.desc.camera = look(camera_pos, camera_dir * 2.0f, mk(0, 1, 0));
}

void scene_corner(SceneHolder& s) {
    s.materials.push_back(lambert());
    s.prims.push_back(box_plane(-1, 0, 0)); // GeometryCorner.cpp:11-13
    s.prims.push_back(box_plane(0, -1, 0));
    s.prims.push_back(box_plane(0, 0, -1));
    f3 out = mk(1, 1, 1);
    f3 cx = mk(-0.5f, -1.0f, -1.0f) + 0.5f * out;
    f3 cy = mk(-1.0f, -0.5f, -1.0f) + 0.5f * out;
    f3 cz = mk(-1.0f, -1.0f, -0.5f) + 0.5f * out;
    s.lights.push_back(triangle_light(cx, cz - cx, cy - cx));
    f3 camera_pos = mk(4.0f, 1.0f, 1.0f);
    f3 camera_dir = normalize(mk(0, 0, 0.0f) - camera_pos);
    s.desc.camera = look(camera_pos, camera_dir);
}

void scene_openspheres(SceneHolder& s) {
    s.materials.push_back(lambert());
    // GeometryOpenSpheres.cpp:13-33: three spheres first, then the floor plane
    s.prims.push_back(sphere(mk(-0.2f, -0.2f, -0.8f), 0.2f, (float)(1.0 / 0.2f)));
    s.prims.push_back(sphere(mk(+0.2f, -0.2f, -0.8f), 0.2f, (float)(1.0 / 0.2f)));
    s.prims.push_back(sphere(mk(0.0f, +0.2f, -0.8f), 0.2f, (float)(1.0 / 0.2f)));
    s.prims.push_back(box_plane(0, 0, -1));
    s.lights.push_back(square_light(mk(-0.05f, -0.05f, -0.2f), mk(0, 0, -1), mk(0, 0.1f, 0)));
    f3 camera_pos = mk(0, -5.0f, 0);
    f3 camera_dir = normalize(mk(0, 0, -1.0f) - camera_pos);
    s.desc.camera = look(camera_pos, camera_dir * 2.0f, mk(0, 0, 1));
}

// BASELINE.json configs[1] ("C2"): same literals as GeometryCornell in oracle/ref_driver.cpp
void scene_cornell(SceneHolder& s) {
    s.materials.push_back(lambert());
    s.materials.push_back(ipt_material{IPT_DDF_GLOSSY, 1.0f, 0.3f, 0.7f, 40.0f});
    add_sphere_in_box_planes(s);
    s.prims.push_back(sphere(mk(-0.45f, 0.25f, -0.65f), 0.35f, 1.0f / 0.35f, 0));
    s.prims.push_back(sphere(mk(+0.45f, -0.2f, -0.65f), 0.35f, 1.0f / 0.35f, 1));
    s.lights.push_back(square_light(mk(-0.25f, -0.25f, 0.98f), mk(0.0f, 0.0f, -1.0f), mk(0.0f, 0.5f, 0.0f), 4.0f));
    s.desc.camera = look(mk(0.0f, -3.2f, 0.0f), normalize(mk(0.0f, 1.0f, 0.0f)));
}

// One of every Light class over the default geometry (lighting.h:16-73 through CollectionLighting.cpp:36-55):
// same literals as iptref_scene_set_mixed_lights in oracle/ref_driver.cpp
void scene_mixedlights(SceneHolder& s) {
    scene_box(s);
    s.lights.clear();
    s.lights.push_back(square_light(mk(+0.1f, -0.8f - 0.1f, -0.15f), mk(0.0f, 0.0f, -1.0f), mk(0.0f, 0.2f, 0.0f), 1.0f));
    s.lights.push_back(triangle_light(mk(-0.8f, -0.2f, 0.6f), mk(0.3f, 0.0f, 0.0f), mk(0.0f, 0.0f, -0.3f), 0.5f));
    s.lights.push_back(sphere_light(mk(-0.7f, -0.5f, -0.8f), 0.1f, 0.7f));
    ipt_light outer = sphere_light(mk(0, 0, 0), 10.0f, 20.0f); // addOuterLight: InvertedSphereLight at the origin
    outer.kind = IPT_LIGHT_SPHERE_INVERTED;
    s.lights.push_back(outer);
    ipt_light point = sphere_light(mk(0.9f, 0.0f, -0.8f), 0.0f, 1.0f); // addPointLight (virtual_radius is unused)
    point.kind = IPT_LIGHT_POINT;
    s.lights.push_back(point);
}

// BASELINE.json configs[4] ("C5"): rows x cols square emitters under the ceiling over the C1 geometry
void scene_lightgrid(SceneHolder& s, int rows, int cols) {
    scene_box(s);
    s.lights.clear();
    const float side = 0.01f, z = 0.99f, power = 1.0f;
    for (int r = 0; r < rows; ++r)
        for (int c = 0; c < cols; ++c) {
            float cx = -1.0f + (2.0f * (c + 0.5f)) / cols - 0.5f * side;
            float cy = -1.0f + (2.0f * (r + 0.5f)) / rows - 0.5f * side;
            s.lights.push_back(square_light(mk(cx, cy, z), mk(0.0f, 0.0f, -1.0f), mk(0.0f, side, 0.0f), power));
        }
}

// BASELINE.json configs[2..3] ("C3"/"C4"): n generated triangles inside the open box, big ceiling light
void scene_mesh(SceneHolder& s, uint64_t n) {
    s.materials.push_back(lambert());
    add_sphere_in_box_planes(s);
    s.triangles.resize(n * 9);
    ipt_generate_mesh(n, 1, s.triangles.data());
    s.desc.triangle_material = 0;
    s.lights.push_back(square_light(mk(-0.4f, -0.4f, 0.98f), mk(0.0f, 0.0f, -1.0f), mk(0.0f, 0.8f, 0.0f), 4.0f));
    f3 camera_pos = mk(0.0f, -3.0f, 0.1f);
    f3 camera_dir = normalize(mk(0.0f, 1.0f, -1.0f) - camera_pos);
    s.desc.camera = look(camera_pos, camera_dir);
}

inline uint64_t splitmix64(uint64_t x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

} // namespace

int ipt_host_fail(int code, const char* msg); // ipt_capi.cu: sets the calling thread's ipt_last_error()

extern "C" {

// Integer-defined mesh: every float is built from a 24-bit integer so that host, oracle and device inputs
// are byte-identical (SURVEY.md §8d C3). Centre uniform in [-0.9,0.9]^3, edges uniform in [-0.02,0.02]^3.
int ipt_generate_mesh(uint64_t n, uint64_t seed, float* triangles) {
    if (!triangles) return IPT_ERR_INVALID;
    for (uint64_t k = 0; k < n; ++k) {
        for (int j = 0; j < 9; ++j) {
            uint64_t h = splitmix64(seed * 0x100000001B3ull + k * 9 + j);
            float u = (float)(uint32_t)(h >> 40) * (1.0f / 16777216.0f); // 24 bits, exact
            float sym = u * 2.0f - 1.0f;                                  // exact
            triangles[k * 9 + j] = j < 3 ? sym * 0.9f : sym * 0.02f;
        }
    }
    return IPT_OK;
}

int ipt_camera_look(const float position[3], const float direction[3], const float up_hint[3], ipt_camera* out) {
    if (!position || !direction || !up_hint || !out) return IPT_ERR_INVALID;
    *out = look(mk(position), mk(direction), mk(up_hint));
    return IPT_OK;
}

// The arrow keys of Gui::work (src/gui.cpp:105-134): orbit about the z axis by pi/12, dolly by 1.1, then re-derive
// right/up with the fixed up hint (0,0,1) (gui.cpp:130-131).
int ipt_camera_orbit(ipt_camera* camera, int key) {
    if (!camera) return IPT_ERR_INVALID;
    f3 pos = mk(camera->position), dir = mk(camera->direction);
    if (key == IPT_KEY_LEFT || key == IPT_KEY_RIGHT) {
        float angle = key == IPT_KEY_LEFT ? (float)-M_PI / 12 : (float)+M_PI / 12; // gui.cpp:108,114
        ipt_host::f33 mat = ipt_host::rotation(angle, mk(0, 0, 1));
        pos = mat * pos;
        dir = mat * dir;
    } else if (key == IPT_KEY_DOWN) {
        float f = static_cast<float>(1.1); // vec3 *= double casts the scalar first (type_vec3.inl:284-290)
        pos = mk(pos.x * f, pos.y * f, pos.z * f);
    } else if (key == IPT_KEY_UP) {
        float f = static_cast<float>(1.1);
        pos = mk(pos.x / f, pos.y / f, pos.z / f);
    } else return IPT_ERR_INVALID;
    f3 right = normalize(cross(dir, mk(0, 0, 1)));
    f3 up = normalize(cross(right, dir));
    put(camera->position, pos);
    put(camera->direction, dir);
    put(camera->right, right);
    put(camera->up, up);
    return IPT_OK;
}

int ipt_sample_scene(const char* name, ipt_scene_desc** out) {
    if (!name || !out) return ipt_host_fail(IPT_ERR_INVALID, "ipt_sample_scene: name and out must not be null");
    std::string n(name);
    SceneHolder* s = new SceneHolder();
    std::memset(&s->desc, 0, sizeof(s->desc));
    if (n == "box") scene_box(*s);
    else if (n == "fractal") scene_fractal(*s);
    else if (n == "smallpt") scene_smallpt(*s);
    else if (n == "square") scene_square(*s);
    else if (n == "corner") scene_corner(*s);
    else if (n == "openspheres") scene_openspheres(*s);
    else if (n == "cornell") scene_cornell(*s);
    else if (n == "mixedlights") scene_mixedlights(*s);
    else if (n.rfind("lightgrid:", 0) == 0) {
        int r = 0, c = 0;
        if (std::sscanf(n.c_str() + 10, "%dx%d", &r, &c) != 2 || r <= 0 || c <= 0) { delete s; return ipt_host_fail(IPT_ERR_INVALID, ("ipt_sample_scene: expected lightgrid:<rows>x<cols>, got " + n).c_str()); }
        scene_lightgrid(*s, r, c);
    } else if (n.rfind("mesh:", 0) == 0) {
        long long cnt = std::atoll(n.c_str() + 5);
        if (cnt <= 0) { delete s; return ipt_host_fail(IPT_ERR_INVALID, ("ipt_sample_scene: expected mesh:<triangles>, got " + n).c_str()); }
        scene_mesh(*s, (uint64_t)cnt);
    } else {
        delete s;
        return ipt_host_fail(IPT_ERR_INVALID, ("ipt_sample_scene: unknown scene " + n).c_str());
    }
    s->finish();
    *out = &s->desc;
    return IPT_OK;
}

int ipt_scene_desc_free(ipt_scene_desc* desc) {
    if (!desc) return IPT_ERR_INVALID;
    delete reinterpret_cast<SceneHolder*>(desc);
    return IPT_OK;
}

} // extern "C"
