/*
 * oracle/ipt_oracle.c — CPU restatement of dimalit/ipt's path-tracing hot path.
 *
 * TEST INFRASTRUCTURE ONLY. This file is the checker for the CUDA path; it is never shipped and never
 * measured as the product. Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
 * `--impl reference` legs may load liboracle. Nothing under ipt_b200/ includes or links it.
 *
 * Parity status: PINNED. With rng_mode = IPT_ORACLE_RNG_DRAND48 every function below consumes libc
 * drand48() in exactly the order the reference does, so one whole render_sample pass is BIT-IDENTICAL
 * to the reference compiled from /root/reference (oracle/_ref/libipt_ref.so); tests/test_oracle_pin.py
 * checks that on the five reference scenes + the C2 extension scene, plus the reference's own
 * known-answer tests (src/libddf/test_ddf.cpp:181-223, src/lighting/test_lighting.cpp:130-144).
 * With rng_mode = IPT_ORACLE_RNG_PHILOX the same code draws from the counter-based Philox4x32-10
 * stream the CUDA kernels use, which makes GPU-vs-oracle comparisons per pixel instead of statistical.
 *
 * Every function cites the reference lines it follows. Float arithmetic follows the reference's op
 * order literally (glm 0.9.9.7 scalar path: dot = (x*x + y*y) + z*z, normalize = v * (1/sqrt(dot)),
 * see SURVEY.md Appendix A); build with -O2 -ffp-contract=off and no -march (oracle/Makefile).
 */
#define _GNU_SOURCE
#include "ipt_b200.h"

#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <stdio.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define IPT_ORACLE_RNG_DRAND48 0
#define IPT_ORACLE_RNG_PHILOX 1

typedef struct { float x, y, z; } v3;
typedef struct { v3 c[3]; } m3; /* column-major like glm: c[col] */

/* ---- glm 0.9.9.7 scalar arithmetic, literally (include/glm/detail/func_geometric.inl:48-110) ------ */
static inline v3 V(float x, float y, float z) { v3 r = {x, y, z}; return r; }
static inline v3 vadd(v3 a, v3 b) { return V(a.x + b.x, a.y + b.y, a.z + b.z); }
static inline v3 vsub(v3 a, v3 b) { return V(a.x - b.x, a.y - b.y, a.z - b.z); }
static inline v3 vscale(v3 a, float s) { return V(a.x * s, a.y * s, a.z * s); }
static inline v3 vneg(v3 a) { return V(-a.x, -a.y, -a.z); }
static inline float vdot(v3 a, v3 b) { float tx = a.x * b.x, ty = a.y * b.y, tz = a.z * b.z; return tx + ty + tz; }
static inline v3 vcross(v3 x, v3 y) {
    return V(x.y * y.z - y.y * x.z, x.z * y.x - y.z * x.x, x.x * y.y - y.x * x.y);
}
static inline float vlength(v3 a) { return sqrtf(vdot(a, a)); }
static inline v3 vnormalize(v3 a) { return vscale(a, 1.0f / sqrtf(vdot(a, a))); }
static inline int vis_zero(v3 a) { return a.x == 0.0f && a.y == 0.0f && a.z == 0.0f; }
/* glm::reflect: I - N * dot(N, I) * 2 */
static inline v3 vreflect(v3 I, v3 N) { return vsub(I, vscale(vscale(N, vdot(N, I)), 2.0f)); }
/* mat3 * vec3 (include/glm/detail/type_mat3x3.inl:468-474) */
static inline v3 mmul(const m3* m, v3 v) {
    return V(m->c[0].x * v.x + m->c[1].x * v.y + m->c[2].x * v.z,
             m->c[0].y * v.x + m->c[1].y * v.y + m->c[2].y * v.z,
             m->c[0].z * v.x + m->c[1].z * v.y + m->c[2].z * v.z);
}
/* glm::inverse(mat3) (include/glm/detail/func_matrix.inl:269-291); m[i][j] = column i, row j */
static m3 minverse(const m3* mm) {
#define M(i, j) (((const float*)&mm->c[i])[j])
    float ood = 1.0f / (+M(0, 0) * (M(1, 1) * M(2, 2) - M(2, 1) * M(1, 2)) - M(1, 0) * (M(0, 1) * M(2, 2) - M(2, 1) * M(0, 2)) +
                        M(2, 0) * (M(0, 1) * M(1, 2) - M(1, 1) * M(0, 2)));
    m3 r;
    r.c[0].x = +(M(1, 1) * M(2, 2) - M(2, 1) * M(1, 2)) * ood;
    r.c[1].x = -(M(1, 0) * M(2, 2) - M(2, 0) * M(1, 2)) * ood;
    r.c[2].x = +(M(1, 0) * M(2, 1) - M(2, 0) * M(1, 1)) * ood;
    r.c[0].y = -(M(0, 1) * M(2, 2) - M(2, 1) * M(0, 2)) * ood;
    r.c[1].y = +(M(0, 0) * M(2, 2) - M(2, 0) * M(0, 2)) * ood;
    r.c[2].y = -(M(0, 0) * M(2, 1) - M(2, 0) * M(0, 1)) * ood;
    r.c[0].z = +(M(0, 1) * M(1, 2) - M(1, 1) * M(0, 2)) * ood;
    r.c[1].z = -(M(0, 0) * M(1, 2) - M(1, 0) * M(0, 2)) * ood;
    r.c[2].z = +(M(0, 0) * M(1, 1) - M(1, 0) * M(0, 1)) * ood;
#undef M
    return r;
}

/* ---- RNG: libc drand48 (include/randf.h:6-11) or Philox4x32-10 keyed like the CUDA kernels --------- */
static float randf_drand48(void) {
    float res = (float)drand48();
    while (res == 1.0f) res = (float)drand48();
    return res;
}

/* Philox4x32-R (Salmon, Moraes, Dror, Shaw: "Parallel random numbers: as easy as 1, 2, 3", SC11), the published algorithm */
static void philox4x32_r(int rounds, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t out[4]) {
    for (int r = 0; r < rounds; ++r) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c0;
        uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
        uint32_t n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        uint32_t n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
static void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t out[4]) {
    philox4x32_r(IPT_PHILOX_ROUNDS, c0, c1, c2, c3, k0, k1, out); /* the render's stream (name kept from the 10-round default) */
}
static inline float u01(uint32_t x) { return (float)(x >> (32 - IPT_U01_BITS)) * (1.0f / (float)(1u << IPT_U01_BITS)); }

/* One tree node's draws. DRAND48: sequential. PHILOX: out[role] of counter (pixel, pass, node, depth). */
typedef struct {
    int mode;
    float u[4];
} draws;
enum { ROLE_SELECT = 0, ROLE_U1 = 1, ROLE_U2 = 2, ROLE_LOBE = 3 };
static inline float draw(const draws* d, int role) { return d->mode == IPT_ORACLE_RNG_DRAND48 ? randf_drand48() : d->u[role]; }

typedef struct {
    int mode;
    uint32_t pixel, pass;
    uint32_t k0, k1;
} rng_ctx;
static draws node_draws(const rng_ctx* r, uint32_t node, uint32_t depth) {
    draws d;
    d.mode = r->mode;
    if (r->mode == IPT_ORACLE_RNG_PHILOX) {
        uint32_t o[4];
        philox4x32_10(r->pixel, r->pass, node, depth, r->k0, r->k1, o);
        for (int i = 0; i < 4; ++i) d.u[i] = u01(o[i]);
    }
    return d;
}

/* ---- prepared scene -------------------------------------------------------------------------------- */
typedef struct {
    ipt_light l;
    float area;
    v3 normal; /* area lights: normalize(cross(x,y)) */
    m3 inverse_matrix;
    float surface_power;
} olight;

typedef struct {
    const ipt_scene_desc* d;
    olight* lights;
    float* light_w; /* mixture weights inside unite(light_ddf,1,sdf,1): CollectionLighting.cpp:12-21 then *0.5 */
    float sdf_w;
    /* mesh acceleration (oracle_mesh section) */
    struct obvh* bvh;
    uint64_t stat_rays;
} oscene;

static v3 A3(const float* p) { return V(p[0], p[1], p[2]); }

/* AreaLight::AreaLight (src/lighting/lighting.cpp:79-90), SphereLight ctor (lighting.h:46-53), PointLight (lighting.h:35-39) */
static void prepare_light(olight* o, const ipt_light* l) {
    o->l = *l;
    memset(&o->inverse_matrix, 0, sizeof(m3));
    o->normal = V(0, 0, 0);
    if (l->kind == IPT_LIGHT_AREA_DIAMOND || l->kind == IPT_LIGHT_AREA_TRIANGLE) {
        v3 xa = A3(l->x_axis), ya = A3(l->y_axis);
        float full_area = vlength(vcross(xa, ya));
        o->area = l->kind == IPT_LIGHT_AREA_DIAMOND ? full_area : full_area / 2.0f;
        m3 m;
        m.c[0] = xa; m.c[1] = ya; m.c[2] = vcross(xa, ya);
        o->inverse_matrix = minverse(&m);
        o->normal = vnormalize(vcross(xa, ya));
        o->surface_power = l->power / o->area;
    } else if (l->kind == IPT_LIGHT_SPHERE || l->kind == IPT_LIGHT_SPHERE_INVERTED) {
        o->area = (float)(4.0 * M_PI * l->radius * l->radius);
        o->surface_power = l->power / o->area;
    } else {
        o->area = 0.0f;
        o->surface_power = NAN;
    }
}

/* CollectionLighting::distributionInPoint (src/CollectionLighting.cpp:12-21) through unite()'s
 * union+simple branch (src/libddf/ddf.cpp:207-223), then main.cpp:143 unite(light,1,sdf,1). */
static void prepare_weights(oscene* s) {
    uint32_t n = s->d->n_lights;
    s->light_w = (float*)malloc(sizeof(float) * (n ? n : 1));
    float acc_power = 0.0f;
    for (uint32_t j = 0; j < n; ++j) {
        float ka = acc_power, kb = s->d->lights[j].power;
        float f = ka / (ka + kb);
        for (uint32_t i = 0; i < j; ++i) s->light_w[i] *= f;
        s->light_w[j] = kb / (ka + kb);
        acc_power += kb;
    }
    if (n == 0) {
        s->sdf_w = 1.0f; /* ddf.cpp:209-210 -> unite(nullptr,0,b,kb): weight kb/(0+kb) */
    } else {
        float f = 1.0f / (1.0f + 1.0f);
        for (uint32_t i = 0; i < n; ++i) s->light_w[i] *= f;
        s->sdf_w = 1.0f / (1.0f + 1.0f);
    }
}

struct obvh;
static struct obvh* obvh_build(const float* tris, uint64_t n);
static void obvh_free(struct obvh*);

static oscene* oscene_prepare(const ipt_scene_desc* d) {
    oscene* s = (oscene*)calloc(1, sizeof(oscene));
    s->d = d;
    s->lights = (olight*)malloc(sizeof(olight) * (d->n_lights ? d->n_lights : 1));
    for (uint32_t i = 0; i < d->n_lights; ++i) prepare_light(&s->lights[i], &d->lights[i]);
    prepare_weights(s);
    s->bvh = d->n_triangles ? obvh_build(d->triangles, d->n_triangles) : NULL;
    return s;
}
static void oscene_free(oscene* s) {
    if (s->bvh) obvh_free(s->bvh);
    free(s->lights); free(s->light_w); free(s);
}

/* ---- geometry ------------------------------------------------------------------------------------- */
/* intersection_with_box_plane (src/geometry/geometric_utils.cpp:8-26) */
static float isect_box_plane(v3 plane, v3 origin, v3 direction) {
    float dir_plane = vdot(direction, plane);
    if (fabsf(dir_plane) < 1e-6) return INFINITY;
    float t = (1.0f - vdot(origin, plane)) / dir_plane;
    v3 point = vadd(origin, vscale(direction, t));
    if (fabsf(point.x) > 1.0f || fabsf(point.y) > 1.0f || fabsf(point.z) > 1.0f) return INFINITY;
    if (vdot(direction, plane) < 0.0f) return INFINITY;
    if (t < 1e-6) return INFINITY;
    return t;
}
/* intersection_with_sphere (src/geometry/geometric_utils.cpp:28-55); pow(x,2.0f) is x*x at -O2 (SURVEY App. A) */
static float isect_sphere(float radius, v3 origin, v3 direction) {
    float origin_x_dir = vdot(origin, direction);
    float desc = 4.0f * (origin_x_dir * origin_x_dir) - 4.0f * (vdot(origin, origin) - radius * radius);
    if (desc < 0.0f) return INFINITY;
    float sqrt_desc = sqrtf(desc);
    float t1 = (float)((-2.0 * origin_x_dir - sqrt_desc) / 2.0);
    float t2 = (float)((-2.0 * origin_x_dir + sqrt_desc) / 2.0);
    if (t1 < 1e-6) t1 = INFINITY;
    if (t2 < 1e-6) t2 = INFINITY;
    float t = t2 < t1 ? t2 : t1; /* std::min(t1,t2) */
    v3 pos = vadd(origin, vscale(direction, t));
    if (vdot(pos, vsub(origin, pos)) <= 0.0f) return INFINITY;
    return t;
}
/* Sphere::intersect (src/geometry/GeometrySmallPt.cpp:17-22), double, 0 = no hit */
static double isect_sphere_smallpt(double rad, v3 p, v3 ro, v3 rd) {
    v3 op = vsub(p, ro);
    double t, eps = 1e-4, b = vdot(op, rd), det = b * b - vdot(op, op) + rad * rad;
    if (det < 0) return 0;
    det = sqrt(det);
    return (t = b - det) > eps ? t : ((t = b + det) > eps ? t : 0);
}

/* The triangle / parallelogram test of AreaLight::traceRay (src/lighting/lighting.cpp:107-144).
 * Returns t or +inf; rel = origin + direction*t - corner. */
static float isect_parallelogram(v3 corner, v3 n, const m3* inv, int triangle, v3 origin, v3 direction, v3* rel_out) {
    float n_dir = vdot(n, direction);
    if (fabsf(n_dir) < 1e-6 || n_dir > 0.0f) return INFINITY;
    float t = vdot(n, vsub(corner, origin)) / n_dir;
    if (t < 1e-6) return INFINITY;
    v3 rel = vsub(vadd(origin, vscale(direction, t)), corner);
    v3 coord = mmul(inv, rel);
    int hit;
    if (!triangle) hit = coord.x >= 0.0f && coord.x <= 1.0f && coord.y >= 0.0f && coord.y <= 1.0f;
    else hit = coord.x >= 0.0f && coord.y >= 0.0 && coord.x + coord.y <= 1.0f;
    if (!hit) return INFINITY;
    if (rel_out) *rel_out = rel;
    return t;
}

/* mesh triangle k: derived quantities exactly as AreaLight's ctor derives them (lighting.cpp:79-90) */
static float isect_mesh_triangle(const float* tri, v3 origin, v3 direction) {
    v3 v0 = A3(tri), e1 = A3(tri + 3), e2 = A3(tri + 6);
    v3 cr = vcross(e1, e2);
    m3 m; m.c[0] = e1; m.c[1] = e2; m.c[2] = cr;
    m3 inv = minverse(&m);
    v3 n = vnormalize(cr);
    return isect_parallelogram(v0, n, &inv, 1, origin, direction, NULL);
}

static int obvh_closest(const struct obvh* b, const float* tris, v3 o, v3 d, double* dist, uint32_t* best);

typedef struct {
    int hit;
    uint32_t prim;
    float t;
    v3 position, normal;
    float curvature;
    uint32_t material;
} osurf;

/* Geometry::traceRay of every reference geometry as one ordered list (GeometrySphereInBox.cpp:10-81,
 * GeometryFloor.cpp:10-23, GeometryCorner.cpp:10-39, GeometryOpenSpheres.cpp:12-68, FractalSpheres.cpp:66-97,
 * GeometrySmallPt.cpp:36-61). `dist` is double only so that smallpt spheres compare in double like
 * GeometrySmallPt.cpp:41-44; float candidates widen exactly. use_bvh=0 -> brute-force mesh scan. */
static osurf trace_geometry(const oscene* s, v3 origin, v3 direction, int use_bvh) {
    const ipt_scene_desc* d = s->d;
    double dist = INFINITY;
    uint32_t best = IPT_NO_HIT;
    for (uint32_t i = 0; i < d->n_prims; ++i) {
        const ipt_prim* p = &d->prims[i];
        if (p->kind == IPT_PRIM_BOX_PLANE) {
            float t = isect_box_plane(A3(p->p), origin, direction);
            if (t < dist) { dist = t; best = i; }
        } else if (p->kind == IPT_PRIM_SPHERE) {
            float t = isect_sphere(p->radius, vsub(origin, A3(p->p)), direction);
            if (t < dist) { dist = t; best = i; }
        } else {
            double t = isect_sphere_smallpt((double)p->radius, A3(p->p), origin, direction);
            if (t != 0.0 && t < dist) { dist = t; best = i; }
        }
    }
    if (d->n_triangles) {
        if (use_bvh && s->bvh) {
            obvh_closest(s->bvh, d->triangles, origin, direction, &dist, &best);
            if (best != IPT_NO_HIT && best >= 0x80000000u) best = d->n_prims + (best & 0x7FFFFFFFu);
        } else {
            for (uint64_t k = 0; k < d->n_triangles; ++k) {
                float t = isect_mesh_triangle(d->triangles + 9 * k, origin, direction);
                if (t < dist) { dist = t; best = (uint32_t)(d->n_prims + k); }
            }
        }
    }
    osurf r;
    memset(&r, 0, sizeof r);
    r.prim = best;
    r.t = INFINITY;
    if (best == IPT_NO_HIT) return r;
    r.hit = 1;
    r.t = (float)dist;
    r.position = vadd(origin, vscale(direction, r.t));
    if (best >= d->n_prims) {
        const float* tri = d->triangles + 9 * (uint64_t)(best - d->n_prims);
        r.normal = vnormalize(vcross(A3(tri + 3), A3(tri + 6)));
        r.curvature = 0.0f;
        r.material = d->triangle_material;
        return r;
    }
    const ipt_prim* p = &d->prims[best];
    r.material = p->material;
    r.curvature = p->curvature;
    if (p->kind == IPT_PRIM_BOX_PLANE) {
        r.normal = vneg(A3(p->p));
    } else {
        v3 nn = vnormalize(vsub(r.position, A3(p->p)));
        r.normal = p->flip_normal ? vneg(nn) : nn;
    }
    return r;
}

/* ---- lights --------------------------------------------------------------------------------------- */
typedef struct { int hit; v3 position, normal; float surface_power; } olhit;

/* lighting.cpp's private intersection_with_sphere for non-unit directions (src/lighting/lighting.cpp:11-36) */
static float isect_light_sphere(float radius, v3 origin, v3 direction) {
    float od = vdot(origin, direction);
    float desc = 4.0f * (od * od) - 4.0f * vdot(direction, direction) * (vdot(origin, origin) - radius * radius);
    if (desc < 0.0f) return INFINITY;
    float t1 = (float)((-2.0 * vdot(origin, direction) - sqrtf(desc)) / 2.0 / vdot(direction, direction));
    float t2 = (float)((-2.0 * vdot(origin, direction) + sqrtf(desc)) / 2.0 / vdot(direction, direction));
    if (t1 < 1e-6) t1 = INFINITY;
    if (t2 < 1e-6) t2 = INFINITY;
    float t = t2 < t1 ? t2 : t1;
    v3 pos = vadd(origin, vscale(direction, t));
    v3 outer_normal = vnormalize(pos);
    float direction_sign = vdot(outer_normal, vsub(origin, pos));
    float position_sign = vlength(origin) - radius;
    if (direction_sign * position_sign <= 0.0f) return INFINITY;
    return t;
}

/* Light::traceRay: AreaLight (lighting.cpp:107-144), SphereLight (:158-169), InvertedSphereLight (lighting.h:61-66),
 * PointLight (lighting.h:41-43) */
static olhit light_trace(const olight* L, v3 origin, v3 direction) {
    olhit r;
    memset(&r, 0, sizeof r);
    const ipt_light* l = &L->l;
    if (l->kind == IPT_LIGHT_AREA_DIAMOND || l->kind == IPT_LIGHT_AREA_TRIANGLE) {
        v3 rel;
        float t = isect_parallelogram(A3(l->position), L->normal, &L->inverse_matrix, l->kind == IPT_LIGHT_AREA_TRIANGLE,
                                      origin, direction, &rel);
        if (t == INFINITY) return r;
        r.hit = 1;
        r.position = vadd(A3(l->position), rel);
        r.normal = L->normal;
        r.surface_power = L->surface_power;
    } else if (l->kind == IPT_LIGHT_SPHERE || l->kind == IPT_LIGHT_SPHERE_INVERTED) {
        float t = isect_light_sphere(l->radius, vsub(origin, A3(l->position)), direction);
        if (t == INFINITY) return r;
        r.hit = 1;
        r.position = vadd(origin, vscale(direction, t));
        r.normal = vnormalize(vsub(r.position, A3(l->position)));
        if (l->kind == IPT_LIGHT_SPHERE_INVERTED) r.normal = vneg(r.normal);
        r.surface_power = L->surface_power;
    }
    return r;
}

/* CollectionLighting::traceRayToLight (src/CollectionLighting.cpp:23-34) */
static olhit lighting_trace(const oscene* s, v3 origin, v3 direction, uint32_t* which) {
    olhit res;
    memset(&res, 0, sizeof res);
    for (uint32_t i = 0; i < s->d->n_lights; ++i) {
        olhit e = light_trace(&s->lights[i], origin, direction);
        if (!e.hit) continue;
        if (!res.hit || vlength(vsub(res.position, origin)) > vlength(vsub(e.position, origin))) {
            res = e;
            if (which) *which = i;
        }
    }
    return res;
}

/* Light::sample: AreaLight (lighting.cpp:93-104), SphereLight (:172-190), PointLight (:193-207) */
static olhit light_sample(const olight* L, const draws* dr) {
    olhit r;
    memset(&r, 0, sizeof r);
    r.hit = 1;
    const ipt_light* l = &L->l;
    if (l->kind == IPT_LIGHT_AREA_DIAMOND || l->kind == IPT_LIGHT_AREA_TRIANGLE) {
        float u1 = draw(dr, ROLE_U1);
        float u2 = draw(dr, ROLE_U2) * (l->kind == IPT_LIGHT_AREA_TRIANGLE ? 1.0f - u1 : 1.0f);
        v3 pos = vadd(vscale(A3(l->x_axis), u1), vscale(A3(l->y_axis), u2));
        r.position = vadd(pos, A3(l->position));
        r.normal = L->normal;
        r.surface_power = L->surface_power;
    } else {
        float u1 = draw(dr, ROLE_U1) * 2.0f - 1.0f;
        float u2 = draw(dr, ROLE_U2);
        float alpha = acosf(u1);
        float phi = (float)(2 * M_PI * u2);
        if (l->kind == IPT_LIGHT_POINT) {
            float rr = sinf(alpha);
            r.position = A3(l->position);
            r.normal = V(rr * cosf(phi), rr * sinf(phi), u1);
            r.surface_power = NAN;
        } else {
            float rr = l->radius * sinf(alpha);
            v3 pos = V(rr * cosf(phi), rr * sinf(phi), l->radius * u1);
            r.position = vadd(pos, A3(l->position));
            r.normal = vnormalize(pos);
            if (l->kind == IPT_LIGHT_SPHERE_INVERTED) r.normal = vneg(r.normal);
            r.surface_power = L->surface_power;
        }
    }
    return r;
}

/* DdfFromLight::sample (src/lighting/lighting.cpp:50-59): zero vector == failed sample */
static v3 light_ddf_sample(const olight* L, v3 origin, const draws* dr) {
    olhit inter = light_sample(L, dr);
    v3 dir = vnormalize(vsub(inter.position, origin));
    float cosinus = vdot(inter.normal, vneg(dir));
    if (cosinus < 1e-5f) return V(0, 0, 0);
    return dir;
}
/* DdfFromLight::value (src/lighting/lighting.cpp:61-73). The `direction==vec3()` branch reads the racy static
 * Lighting::last_sample; its result is discarded by main.cpp:161-163, so it is not restated. */
static float light_ddf_value(const olight* L, v3 origin, v3 direction) {
    olhit inter = light_trace(L, origin, direction);
    if (!inter.hit) return 0.0f;
    v3 dir = vnormalize(vsub(inter.position, origin));
    float cosinus = vdot(inter.normal, vneg(dir));
    if (cosinus < 0.0f) return 0.0f;
    v3 dp = vsub(inter.position, origin);
    float decay = vdot(dp, dp);
    return decay / cosinus / L->area;
}

/* ---- surface DDFs ----------------------------------------------------------------------------------- */
/* RotateDdf::RotateDdf (src/libddf/ddf_detail.h:72-85) with glm::rotate(identity, angle, axis)
 * (include/glm/ext/matrix_transform.inl:18-46): acos is the DOUBLE libm call at this site, cos/sin float. */
typedef struct { m3 transformation, inverse; } orot;
static orot make_rotation(v3 to) {
    v3 z = V(0.0f, 0.0f, 1.0f);
    v3 axis = vcross(z, to);
    if (vlength(axis) < 1e-6) axis = V(1.0f, 0.0f, 0.0f);
    float cosinus = vdot(z, to);
    float a = (float)acos((double)cosinus);
    float c = cosf(a), s = sinf(a);
    v3 ax = vnormalize(axis);
    v3 temp = vscale(ax, 1.0f - c);
    float R[3][3];
    R[0][0] = c + temp.x * ax.x;
    R[0][1] = temp.x * ax.y + s * ax.z;
    R[0][2] = temp.x * ax.z - s * ax.y;
    R[1][0] = temp.y * ax.x - s * ax.z;
    R[1][1] = c + temp.y * ax.y;
    R[1][2] = temp.y * ax.z + s * ax.x;
    R[2][0] = temp.z * ax.x + s * ax.y;
    R[2][1] = temp.z * ax.y - s * ax.x;
    R[2][2] = c + temp.z * ax.z;
    /* Result[i] = m[0]*R[i][0] + m[1]*R[i][1] + m[2]*R[i][2] with m = identity (vec4 arithmetic, xyz kept) */
    orot o;
    for (int i = 0; i < 3; ++i) {
        v3 col;
        col.x = 1.0f * R[i][0] + 0.0f * R[i][1] + 0.0f * R[i][2];
        col.y = 0.0f * R[i][0] + 1.0f * R[i][1] + 0.0f * R[i][2];
        col.z = 0.0f * R[i][0] + 0.0f * R[i][1] + 1.0f * R[i][2];
        o.transformation.c[i] = col;
    }
    o.inverse = minverse(&o.transformation);
    return o;
}

/* CosineDdf (src/libddf/ddf.cpp:91-108), UpperHalfDdf (:74-89), SphericalDdf (:58-72), PowerCosine (oracle/ref_driver.cpp) */
static v3 base_sample(int kind, const draws* dr) {
    float u1 = draw(dr, ROLE_U1);
    float u2 = draw(dr, ROLE_U2);
    float zc;
    if (kind == 0) { u1 = u1 * 2.0f - 1.0f; zc = u1; }
    else if (kind == 1) zc = u1;
    else if (kind == 2) zc = sqrtf(u1);
    else zc = powf(u1, 1.0f / ((float)kind + 1.0f));
    float alpha = acosf(zc);
    float phi = (float)(2 * M_PI * u2);
    float r = sinf(alpha);
    return V(r * cosf(phi), r * sinf(phi), zc);
}
static float base_value(int kind, v3 arg) {
    if (kind == 0) return (float)(0.25 / M_PI);
    if (arg.z < 0.0f) return 0.0f;
    if (kind == 1) return (float)(0.5f / M_PI);
    if (kind == 2) return (float)(arg.z / M_PI);
    return (float)(((float)kind + 1.0f) * powf(arg.z, (float)kind) / (2 * M_PI));
}

/* the sdf attached to a hit */
typedef struct {
    uint32_t ddf;
    orot rot;      /* about the normal */
    orot rot_lobe; /* glossy: about reflect(d, n) */
    v3 normal;
    float wd, ws;
    int exponent;
} osdf;

static osdf make_sdf(const ipt_material* m, v3 normal, v3 direction) {
    osdf s;
    memset(&s, 0, sizeof s);
    s.ddf = m->ddf;
    s.normal = normal;
    s.rot = make_rotation(normal);
    if (m->ddf == IPT_DDF_GLOSSY) {
        s.rot_lobe = make_rotation(vreflect(direction, normal));
        s.wd = m->kd / (m->kd + m->ks);
        s.ws = m->ks / (m->kd + m->ks);
        s.exponent = (int)m->exponent;
    }
    return s;
}
/* TransformDdf::sample / value (src/libddf/ddf_detail.h:26-33) */
static v3 sdf_sample(const osdf* s, const draws* dr) {
    if (s->ddf == IPT_DDF_COSINE) return mmul(&s->rot.transformation, base_sample(2, dr));
    float r = draw(dr, ROLE_LOBE);
    v3 w = r < s->wd ? mmul(&s->rot.transformation, base_sample(2, dr)) : mmul(&s->rot_lobe.transformation, base_sample(s->exponent, dr));
    if (vdot(s->normal, w) < 0.0f) return V(0, 0, 0);
    return w;
}
static float sdf_value(const osdf* s, v3 arg) {
    if (s->ddf == IPT_DDF_COSINE) return base_value(2, mmul(&s->rot.inverse, arg));
    if (vdot(s->normal, arg) < 0.0f) return 0.0f;
    return s->wd * base_value(2, mmul(&s->rot.inverse, arg)) + s->ws * base_value(s->exponent, mmul(&s->rot_lobe.inverse, arg));
}

/* UnionDdf::sample over [lights..., sdf] (src/libddf/ddf.cpp:138-154). If r >= sum of weights the reference
 * returns an uninitialised vector (UB); restated as a failed sample. */
static v3 mix_sample(const oscene* s, const osdf* sdf, v3 pos, const draws* dr) {
    float r = draw(dr, ROLE_SELECT);
    float acc = 0.0f;
    for (uint32_t i = 0; i < s->d->n_lights; ++i) {
        acc += s->light_w[i];
        if (r < acc) return light_ddf_sample(&s->lights[i], pos, dr);
    }
    acc += s->sdf_w;
    if (r < acc) return sdf_sample(sdf, dr);
    return V(0, 0, 0);
}
/* UnionDdf::value (src/libddf/ddf.cpp:156-162) */
static float mix_value(const oscene* s, const osdf* sdf, v3 pos, v3 arg) {
    float res = 0.0f;
    for (uint32_t i = 0; i < s->d->n_lights; ++i) res += s->light_w[i] * light_ddf_value(&s->lights[i], pos, arg);
    res += s->sdf_w * sdf_value(sdf, arg);
    return res;
}

/* ---- the estimator: ray_power_recursive (src/main.cpp:98-184) ------------------------------------- */
typedef struct {
    oscene* s;
    const ipt_render_params* p;
    rng_ctx rng;
    uint64_t rays;
    uint64_t rays_at_depth[IPT_MAX_DEPTH];
    int use_bvh;
} octx;

static float ray_power(octx* c, v3 origin, v3 direction, uint32_t depth, uint32_t node) {
    if (depth == c->p->depth_max) return 0.0f;
    c->rays++;
    if (depth < IPT_MAX_DEPTH) c->rays_at_depth[depth]++;
    osurf si = trace_geometry(c->s, origin, direction, c->use_bvh);
    olhit li = lighting_trace(c->s, origin, direction, NULL);
    if (c->p->flags & 4u)
        printf("CPU extend d=%u node=%u o=(%.9g %.9g %.9g) d=(%.9g %.9g %.9g) si=%d li=%d prim=%u t=%.9g\n", depth, node, origin.x, origin.y,
               origin.z, direction.x, direction.y, direction.z, si.hit, li.hit, si.prim, si.t);
    if (li.hit) {
        if (!si.hit || vlength(vsub(si.position, origin)) > vlength(vsub(li.position, origin)))
            return isfinite(li.surface_power) ? li.surface_power : 1.0f;
    }
    if (!si.hit) return 0.0f;

    const ipt_material* mat = &c->s->d->materials[si.material];
    osdf sdf = make_sdf(mat, si.normal, direction);
    uint32_t n_rays = c->p->schedule[depth];
    /* A node with n_rays == 0 (reference: n_rays/2 reaching 0, main.cpp:177) evaluates 0.0f/0 = NaN at main.cpp:181,
     * which poisons its parent to 0 -- reachable only with non-default command-line arguments. The DRAND48 mode keeps
     * that behaviour (it is pinned bit-exactly to the reference); the PHILOX mode, which checks the CUDA path, uses the
     * defined extension "a split count of 0 spawns nothing and contributes 0" (include/ipt_b200.h, DESIGN.md). */
    if (n_rays == 0 && c->rng.mode == IPT_ORACLE_RNG_PHILOX) return 0.0f;
    float res = 0.0f;
    for (uint32_t i = 0; i < n_rays; ++i) {
        uint32_t child = node * n_rays + i;
        draws dr = node_draws(&c->rng, child, depth + 1);
        v3 nd = mix_sample(c->s, &sdf, si.position, &dr);
        if (vis_zero(nd)) {
            if (c->p->flags & 4u) printf("CPU shade d=%u child=%u u=(%.9g %.9g %.9g) FAILED\n", depth, child, dr.u[0], dr.u[1], dr.u[2]);
            continue; /* mix value is computed first in the reference but has no side effect */
        }
        float mix_val = mix_value(c->s, &sdf, si.position, nd);
        float sdf_val = sdf_value(&sdf, nd);
        if (c->p->flags & 4u)
            printf("CPU shade d=%u child=%u u=(%.9g %.9g %.9g) w=(%.9g %.9g %.9g) sv=%.9g mv=%.9g\n", depth, child, dr.u[0], dr.u[1], dr.u[2], nd.x, nd.y,
                   nd.z, sdf_val, mix_val);
        float multiplier = sdf_val / mix_val;
        res += multiplier * mat->albedo * ray_power(c, si.position, nd, depth + 1, child);
    }
    res = isfinite(res) ? res / n_rays : 0.0f;
    return res;
}

/* SimpleCamera::sampleRay (src/SimpleCamera.cpp:15-21) */
static void camera_ray(const ipt_camera* cam, float x, float y, v3* o, v3* d) {
    x -= 0.5f;
    y -= 0.5f;
    v3 ray = vadd(vadd(vscale(A3(cam->right), x), vscale(A3(cam->up), y)), A3(cam->direction));
    *o = A3(cam->position);
    *d = vnormalize(ray);
}

/* accumulator cell of a sample: GridRenderPlane::addRay (src/GridRenderPlane.cpp:66-67) / Gui::addRay (src/gui.cpp:168-172) */
static size_t plane_cell(uint32_t mode, uint32_t W, uint32_t H, float x, float y, uint32_t ix, uint32_t iy) {
    if (mode == IPT_PLANE_LINEAR) return (size_t)iy * W + ix;
    size_t xi = (size_t)(x * W);
    size_t yi;
    if (mode == IPT_PLANE_GRID) {
        yi = (size_t)(int64_t)(H - y * H - 1); /* x86 cvttss2si of a value in (-1,0) is 0 */
    } else {
        yi = (size_t)(H - y * H);
        if (xi > W - 1) xi = W - 1;
        if (yi > H - 1) yi = H - 1;
    }
    return yi * W + xi;
}

/* ==== exported API ================================================================================== */

/* render_sample (src/main.cpp:186-223) x pass_count into a GridRenderPlane-like accumulator:
 * pixels (float running mean, GridRenderPlane.cpp:68-72), counters, double sum / sumsq per cell.
 * rng_mode DRAND48: call srand48 yourself first (ipt_oracle_seed); single-threaded, reference draw order.
 * rng_mode PHILOX: OpenMP over pixels; values are applied to the plane in loop order afterwards. */
int ipt_oracle_render(const ipt_scene_desc* desc, const ipt_render_params* p, int rng_mode, int use_bvh, float* pixels,
                      uint64_t* counters, double* sum, double* sumsq, uint64_t* rays_out, uint64_t* rays_at_depth) {
    oscene* s = oscene_prepare(desc);
    uint32_t W = p->width, H = p->height;
    uint32_t x0 = p->tile_w ? p->tile_x0 : 0, y0 = p->tile_w ? p->tile_y0 : 0;
    uint32_t tw = p->tile_w ? p->tile_w : W, th = p->tile_w ? p->tile_h : H;
    size_t np = (size_t)tw * th;
    float* vals = (float*)malloc(sizeof(float) * np);
    float* xs = (float*)malloc(sizeof(float) * np);
    float* ys = (float*)malloc(sizeof(float) * np);
    uint64_t rays = 0;
    uint64_t rad[IPT_MAX_DEPTH];
    memset(rad, 0, sizeof rad);
    for (uint32_t pass = p->pass_begin; pass < p->pass_begin + p->pass_count; ++pass) {
#pragma omp parallel for schedule(dynamic, 64) reduction(+ : rays) reduction(+ : rad[:IPT_MAX_DEPTH]) if (rng_mode == IPT_ORACLE_RNG_PHILOX)
        for (size_t k = 0; k < np; ++k) {
            uint32_t iy = y0 + (uint32_t)(k / tw), ix = x0 + (uint32_t)(k % tw);
            octx c;
            memset(&c, 0, sizeof c);
            c.s = s; c.p = p; c.use_bvh = use_bvh;
            c.rng.mode = rng_mode;
            c.rng.pixel = iy * W + ix;
            c.rng.pass = pass;
            c.rng.k0 = (uint32_t)p->seed;
            c.rng.k1 = (uint32_t)(p->seed >> 32);
            draws dr = node_draws(&c.rng, 0, 0);
            float x = ((float)ix + draw(&dr, 0)) / (float)W;
            float y = ((float)iy + draw(&dr, 1)) / (float)H;
            if (x == 1.0f) x = nextafterf(x, 0.0f);
            if (y == 1.0f) y = nextafterf(y, 0.0f);
            v3 o, d;
            camera_ray(&desc->camera, x, y, &o, &d);
            float value = ray_power(&c, o, d, 0, 0);
            value = value >= 0.0f ? value : 0.0f;
            if (!isfinite(value)) value = 0.0f; /* reference asserts (main.cpp:215); unreachable in practice */
            vals[k] = value; xs[k] = x; ys[k] = y;
            rays += c.rays;
            for (int q = 0; q < IPT_MAX_DEPTH; ++q) rad[q] += c.rays_at_depth[q];
        }
        for (size_t k = 0; k < np; ++k) {
            uint32_t iy = y0 + (uint32_t)(k / tw), ix = x0 + (uint32_t)(k % tw);
            size_t cell = plane_cell(p->plane_mode, W, H, xs[k], ys[k], ix, iy);
            if (pixels && counters) {
                pixels[cell] = (pixels[cell] * counters[cell] + vals[k]) / (counters[cell] + 1);
                ++counters[cell];
            }
            if (sum) sum[cell] += vals[k];
            if (sumsq) sumsq[cell] += (double)vals[k] * vals[k];
        }
    }
    if (rays_out) *rays_out = rays;
    if (rays_at_depth) memcpy(rays_at_depth, rad, sizeof rad);
    free(vals); free(xs); free(ys);
    oscene_free(s);
    return 0;
}

void ipt_oracle_seed(long seed) { srand48(seed); }
int ipt_oracle_threads(void) {
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}

/* Geometry::traceRay + Lighting::traceRayToLight + the decision of main.cpp:111-128 for n rays. */
int ipt_oracle_trace_batch(const ipt_scene_desc* desc, const float* o, const float* d, size_t n, int use_bvh,
                           uint32_t* prim_id, float* t, float* pos, float* normal, uint32_t* light_id, float* light_pos,
                           uint32_t* outcome) {
    oscene* s = oscene_prepare(desc);
#pragma omp parallel for schedule(dynamic, 256)
    for (size_t i = 0; i < n; ++i) {
        v3 oo = A3(o + 3 * i), dd = A3(d + 3 * i);
        osurf si = trace_geometry(s, oo, dd, use_bvh);
        uint32_t which = IPT_NO_HIT;
        olhit li = lighting_trace(s, oo, dd, &which);
        if (prim_id) prim_id[i] = si.prim;
        if (t) t[i] = si.t;
        if (pos) { pos[3 * i] = si.position.x; pos[3 * i + 1] = si.position.y; pos[3 * i + 2] = si.position.z; }
        if (normal) { normal[3 * i] = si.normal.x; normal[3 * i + 1] = si.normal.y; normal[3 * i + 2] = si.normal.z; }
        if (light_id) light_id[i] = li.hit ? which : IPT_NO_HIT;
        if (light_pos) { light_pos[3 * i] = li.position.x; light_pos[3 * i + 1] = li.position.y; light_pos[3 * i + 2] = li.position.z; }
        if (outcome) {
            uint32_t oc = 0;
            if (li.hit && (!si.hit || vlength(vsub(si.position, oo)) > vlength(vsub(li.position, oo)))) oc = 2;
            else if (si.hit) oc = 1;
            outcome[i] = oc;
        }
    }
    oscene_free(s);
    return 0;
}

/* ray_power_preview (src/main.cpp:55-92) */
int ipt_oracle_preview_batch(const ipt_scene_desc* desc, const float* o, const float* d, size_t n, int use_bvh, float* value) {
    oscene* s = oscene_prepare(desc);
    for (size_t i = 0; i < n; ++i) {
        v3 oo = A3(o + 3 * i), dd = A3(d + 3 * i);
        osurf si = trace_geometry(s, oo, dd, use_bvh);
        olhit li = lighting_trace(s, oo, dd, NULL);
        float v;
        if (li.hit && (!si.hit || vlength(vsub(si.position, oo)) > vlength(vsub(li.position, oo)))) v = 1.0f;
        else if (!si.hit) v = 0.0f;
        else v = vdot(si.normal, vneg(dd)) / vlength(dd);
        value[i] = v;
    }
    oscene_free(s);
    return 0;
}

int ipt_oracle_camera_rays(const ipt_scene_desc* desc, const float* xy, size_t n, float* o, float* d) {
    for (size_t i = 0; i < n; ++i) {
        v3 oo, dd;
        camera_ray(&desc->camera, xy[2 * i], xy[2 * i + 1], &oo, &dd);
        o[3 * i] = oo.x; o[3 * i + 1] = oo.y; o[3 * i + 2] = oo.z;
        d[3 * i] = dd.x; d[3 * i + 1] = dd.y; d[3 * i + 2] = dd.z;
    }
    return 0;
}

/* SimpleCamera::SimpleCamera (src/SimpleCamera.cpp:8-13) */
int ipt_oracle_camera_look(const float* position, const float* direction, const float* up_hint, ipt_camera* out) {
    v3 dir = A3(direction);
    v3 right = vnormalize(vcross(dir, A3(up_hint)));
    v3 up = vnormalize(vcross(right, dir));
    memcpy(out->position, position, 12);
    memcpy(out->direction, direction, 12);
    out->right[0] = right.x; out->right[1] = right.y; out->right[2] = right.z;
    out->up[0] = up.x; out->up[1] = up.y; out->up[2] = up.z;
    return 0;
}

/* Ddf::value / Ddf::sample of the base DDFs, optionally rotated to `to` (drand48 draws) */
int ipt_oracle_ddf_value(int kind, const float* to, const float* w, size_t n, float* out) {
    orot r;
    if (to) r = make_rotation(A3(to));
    for (size_t i = 0; i < n; ++i) {
        v3 a = A3(w + 3 * i);
        out[i] = base_value(kind, to ? mmul(&r.inverse, a) : a);
    }
    return 0;
}
int ipt_oracle_ddf_sample(int kind, const float* to, size_t n, float* w) {
    orot r;
    if (to) r = make_rotation(A3(to));
    draws dr;
    dr.mode = IPT_ORACLE_RNG_DRAND48;
    for (size_t i = 0; i < n; ++i) {
        v3 x = base_sample(kind, &dr);
        if (to) x = mmul(&r.transformation, x);
        w[3 * i] = x.x; w[3 * i + 1] = x.y; w[3 * i + 2] = x.z;
    }
    return 0;
}

/* The mixture of main.cpp:142-143 at the hit of ray (o,d): n drand48 samples with mixture / sdf values. */
int ipt_oracle_mix_sample(const ipt_scene_desc* desc, const float* o, const float* d, size_t n, float* w, float* mixv,
                          float* sdfv) {
    oscene* s = oscene_prepare(desc);
    osurf si = trace_geometry(s, A3(o), A3(d), 0);
    if (!si.hit) { oscene_free(s); return 1; }
    osdf sdf = make_sdf(&desc->materials[si.material], si.normal, A3(d));
    draws dr;
    dr.mode = IPT_ORACLE_RNG_DRAND48;
    for (size_t i = 0; i < n; ++i) {
        v3 x = mix_sample(s, &sdf, si.position, &dr);
        w[3 * i] = x.x; w[3 * i + 1] = x.y; w[3 * i + 2] = x.z;
        /* the reference evaluates value(vec3()) through Lighting::last_sample; skip zero vectors */
        mixv[i] = vis_zero(x) ? 0.0f : mix_value(s, &sdf, si.position, x);
        sdfv[i] = vis_zero(x) ? 0.0f : sdf_value(&sdf, x);
    }
    oscene_free(s);
    return 0;
}
int ipt_oracle_mix_value(const ipt_scene_desc* desc, const float* o, const float* d, size_t n, const float* w, float* mixv,
                         float* sdfv, float* lightv) {
    oscene* s = oscene_prepare(desc);
    osurf si = trace_geometry(s, A3(o), A3(d), 0);
    if (!si.hit) { oscene_free(s); return 1; }
    osdf sdf = make_sdf(&desc->materials[si.material], si.normal, A3(d));
    for (size_t i = 0; i < n; ++i) {
        v3 x = A3(w + 3 * i);
        if (mixv) mixv[i] = mix_value(s, &sdf, si.position, x);
        if (sdfv) sdfv[i] = sdf_value(&sdf, x);
        if (lightv) {
            /* Lighting::distributionInPoint(pos)->value(w): weights without the final 1:1 unite */
            float res = 0.0f;
            for (uint32_t k = 0; k < desc->n_lights; ++k)
                res += (s->light_w[k] * 2.0f) * light_ddf_value(&s->lights[k], si.position, x);
            lightv[i] = res;
        }
    }
    oscene_free(s);
    return 0;
}
/* Lighting::distributionInPoint(pos)->value(dir) */
int ipt_oracle_light_ddf_value(const ipt_scene_desc* desc, const float* pos, const float* w, size_t n, float* out) {
    oscene* s = oscene_prepare(desc);
    for (size_t i = 0; i < n; ++i) {
        float res = 0.0f;
        for (uint32_t k = 0; k < desc->n_lights; ++k)
            res += (s->light_w[k] * 2.0f) * light_ddf_value(&s->lights[k], A3(pos), A3(w + 3 * i));
        out[i] = res;
    }
    oscene_free(s);
    return 0;
}
int ipt_oracle_light_ddf_sample(const ipt_scene_desc* desc, const float* pos, size_t n, float* w) {
    oscene* s = oscene_prepare(desc);
    draws dr;
    dr.mode = IPT_ORACLE_RNG_DRAND48;
    for (size_t i = 0; i < n; ++i) {
        float r = draw(&dr, ROLE_SELECT), acc = 0.0f;
        v3 x = V(0, 0, 0);
        for (uint32_t k = 0; k < desc->n_lights; ++k) {
            acc += s->light_w[k] * 2.0f;
            if (r < acc) { x = light_ddf_sample(&s->lights[k], A3(pos), &dr); break; }
        }
        w[3 * i] = x.x; w[3 * i + 1] = x.y; w[3 * i + 2] = x.z;
    }
    oscene_free(s);
    return 0;
}

/* AreaLight ctor + traceRay for the known-answer test of src/lighting/test_lighting.cpp:130-144 */
int ipt_oracle_arealight(const float* origin, const float* xa, const float* ya, float power, int triangle, const float* ro,
                         const float* rd, float* area, int32_t* hit, float* surface_power) {
    ipt_light l;
    memset(&l, 0, sizeof l);
    l.kind = triangle ? IPT_LIGHT_AREA_TRIANGLE : IPT_LIGHT_AREA_DIAMOND;
    memcpy(l.position, origin, 12); memcpy(l.x_axis, xa, 12); memcpy(l.y_axis, ya, 12);
    l.power = power;
    olight L;
    prepare_light(&L, &l);
    *area = L.area;
    olhit h = light_trace(&L, A3(ro), A3(rd));
    *hit = h.hit;
    *surface_power = h.hit ? h.surface_power : 0.0f;
    return 0;
}

/* light derived fields for scene-builder checks: power, area, position */
int ipt_oracle_light_fields(const ipt_scene_desc* desc, uint32_t i, float* out5) {
    olight L;
    prepare_light(&L, &desc->lights[i]);
    out5[0] = desc->lights[i].power; out5[1] = L.area;
    memcpy(out5 + 2, desc->lights[i].position, 12);
    return 0;
}

/* the light tables a scene's lights make: per light prepare_light's area, surface power and normal (3 floats) and
 * prepare_weights' mixture weight */
int ipt_oracle_light_tables(const ipt_scene_desc* desc, float* area, float* surface_power, float* normal, float* weight) {
    oscene s;
    memset(&s, 0, sizeof s);
    s.d = desc;
    prepare_weights(&s);
    for (uint32_t i = 0; i < desc->n_lights; ++i) {
        olight L;
        prepare_light(&L, &desc->lights[i]);
        area[i] = L.area;
        surface_power[i] = L.surface_power;
        normal[3 * i] = L.normal.x; normal[3 * i + 1] = L.normal.y; normal[3 * i + 2] = L.normal.z;
        weight[i] = s.light_w[i];
    }
    free(s.light_w);
    return 0;
}

/* Philox known-answer access for tests */
void ipt_oracle_philox_rounds(int rounds, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t* out) {
    philox4x32_r(rounds, c0, c1, c2, c3, k0, k1, out);
}
void ipt_oracle_philox(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t* out) {
    philox4x32_10(c0, c1, c2, c3, k0, k1, out);
}

#include "ipt_oracle_mesh.inc"
#include "ipt_oracle_output.inc"
