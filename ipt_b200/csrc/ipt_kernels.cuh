// ipt_kernels.cuh — the wavefront pipeline: generate -> [extend -> shade] x depth -> accumulate.
//
// It replaces the recursive per-pixel loop render_sample -> ray_power_recursive (src/main.cpp:98-223).
// The estimator is linear in the leaf emissions (each surface hit divides by its child count and multiplies
// by sdf/mix * albedo, main.cpp:172-181), so every ray simply carries the product of those factors
// ("throughput") and a light hit adds throughput * emission to its path; no tree reduction is needed.
//
// Queues (SoA, one 128-bit load/store per field and thread, coalesced):
//   ray  : float4 (origin.xyz, K)  float4 (direction.xyz, tag)  float sv                         36 B
//          the ray's weight is K * sv / mix(direction) and the mixture density needs the light hits along the ray,
//          which whoever traces the ray computes anyway -> the weight is resolved there (sv < 0: weight = K)
//   hit  : float4 (position.xyz, throughput) uint4 (tag, prim, octahedral incoming direction) 32 B
//   tag  = path slot in the batch | node index within its tree level << slot_bits
// Live-path compaction: a ray that misses or reaches a light writes nothing; survivors are appended with a
// warp ballot + one atomicAdd per warp (warp-aggregated stream compaction).
// The rays of the LAST traced depth of analytic scenes are never queued: k_shade<FUSE_LAST> resolves them itself.
// All kernels are persistent grid-stride loops over a device-side element count, so no host round trip
// separates the stages.
#pragma once
#include "ipt_shading.cuh"
#ifndef IPT_SHADE_MIN_BLOCKS
#define IPT_SHADE_MIN_BLOCKS 2
#endif
#ifndef IPT_SHADE_FUSED_MIN_BLOCKS
#define IPT_SHADE_FUSED_MIN_BLOCKS 3 // 80 registers, 156 B of spills: still 4 % faster than 2 blocks (profiles/tuning_r01.md)
#endif
#ifndef IPT_SHADE_NEXT_MIN_BLOCKS
#define IPT_SHADE_NEXT_MIN_BLOCKS 3
#endif
#ifndef IPT_EXTEND_MIN_BLOCKS
#define IPT_EXTEND_MIN_BLOCKS 3
#endif
#include <cstdio>
// -DIPT_DEBUG_BOUNDS: every queue append checks its slot against the capacity the host allocated and every park-queue
// write against IPT_PARK; violations are counted (ST_OVERFLOW) instead of written, and ipt_render returns IPT_ERR_OVERFLOW.
// compute-sanitizer is not available on this pool, so this build (tools/ab_r02.py variant "bounds") is what checks that the
// worst-case queue sizing really is the worst case.
#ifdef IPT_DEBUG_BOUNDS
#define IPT_BOUNDS_OK(index, capacity, stats) ((index) < (capacity) ? true : (atomicAdd(&(stats)[ST_OVERFLOW], 1ull), false))
#else
#define IPT_BOUNDS_OK(index, capacity, stats) true
#endif
#ifndef IPT_SHADOW_SKIP_WALLS
#define IPT_SHADOW_SKIP_WALLS 1 // 0: shadow rays of box scenes intersect the wall planes too (tuning A/B only)
#endif
#ifndef IPT_LIGHT_TWO_QUEUES
#define IPT_LIGHT_TWO_QUEUES 1 // 0: one park queue for every child of a many-light scene (tuning A/B only)
#endif
#ifndef IPT_FAST_SECONDARY
#define IPT_FAST_SECONDARY 1 // rays of depth >= 1 use the contracted arithmetic (tdot3 / tpoint<false>), see DESIGN.md section 2
#endif

namespace iptd {

enum LightQuery { LQ_PDF = 0, LQ_NEAREST = 1, LQ_BOTH = 2 };

enum StatSlot {
    ST_SURFACE = 0, ST_LIGHT, ST_MISS, ST_FAILED, ST_PRUNED, ST_DROPPED, ST_NODES, ST_TRIS, ST_LIGHTS, ST_PATHS, ST_QUEUED, ST_FUSED, ST_LIGHT_NODES, ST_OVERFLOW,
    ST_RAYS_AT_DEPTH = 16, // + depth
    ST_COUNT = 16 + IPT_MAX_DEPTH
};

struct RenderCtx {
    // queues
    float4* ray_o;
    float4* ray_d;
    float* ray_x;              // sdf value of the sampled direction (weight resolution is deferred to k_extend), or -1
    float4* hit_a[2];          // hits of depth d live in set d & 1: the fused shade kernel reads one set while it fills the other
    uint4* hit_b[2];           // (the two sets alias where extend and shade are separate launches)
    float* pathval;
    uint32_t* cnt;             // [2*d] rays at depth d, [2*d+1] surface hits at depth d
    uint32_t* fetch;           // [d] next unfetched ray of depth d (persistent mesh kernel)
    unsigned long long* stats; // StatSlot
    // accumulators
    float* sum;
    float* sumsq;
    uint32_t* count;
    // frame / batch
    uint32_t width, height;
    uint32_t tile_x0, tile_y0, tile_w, tile_h, tile_pixels;
    uint32_t pass_begin;
    unsigned long long g0; // first global path index of the batch
    uint32_t batch;        // paths in this batch
    uint32_t ray_cap, hit_cap; // allocated records per ray queue / hit set (checked by -DIPT_DEBUG_BOUNDS builds)
    uint32_t slot_bits, slot_mask;
    uint32_t depth_max;
    uint32_t schedule[IPT_MAX_DEPTH];
    PhiloxKeys keys;   // Philox round keys of the seed
    uint32_t plane_mode, flags;
    // slot -> (pass, loop pixel): g0 = pass0 * tile_pixels + rem0 (host), divisions by launch-constant divisors
    uint32_t pass0, rem0;
    FastDiv div_tile_pixels, div_tile_w;
};

__device__ __forceinline__ f3 ld3(const float* p) { return mk3(p[0], p[1], p[2]); }

// Octahedral map of a unit vector to two floats (full float precision, ~1e-7): lets the 32-byte hit record carry
// the incoming direction, which only the glossy lobe (reflect(d, n)) needs. The parent ray record cannot be re-read
// at shading time: the shade kernel is already overwriting the ray queue with the next depth.
__device__ __forceinline__ float2 oct_encode(f3 d) {
    float inv = frcp(__fadd_rn(__fadd_rn(fabsf(d.x), fabsf(d.y)), fabsf(d.z))); // 1 ulp: the decoder re-normalises
    float px = pmul(d.x, inv), py = pmul(d.y, inv);
    if (d.z < 0.0f) {
        float tx = copysignf(__fsub_rn(1.0f, fabsf(py)), px);
        py = copysignf(__fsub_rn(1.0f, fabsf(px)), py);
        px = tx;
    }
    return make_float2(px, py);
}
__device__ __forceinline__ f3 oct_decode(float ex, float ey) {
    float z = __fsub_rn(__fsub_rn(1.0f, fabsf(ex)), fabsf(ey));
    float x = ex, y = ey;
    if (z < 0.0f) {
        x = copysignf(__fsub_rn(1.0f, fabsf(ey)), ex);
        y = copysignf(__fsub_rn(1.0f, fabsf(ex)), ey);
    }
    float inv = rsqrtf(dot3(mk3(x, y, z), mk3(x, y, z)));
    return mk3(pmul(x, inv), pmul(y, inv), pmul(z, inv));
}

// slot -> loop pixel and pass (render_sample's iy/ix loops, main.cpp:189-190)
__device__ __forceinline__ void slot_to_pixel(const RenderCtx& C, uint32_t slot, uint32_t& ix, uint32_t& iy, uint32_t& pass) {
    uint32_t g = C.rem0 + slot; // < 2^32: ipt_render bounds tile_pixels + batch
    uint32_t p = fastdiv(g, C.div_tile_pixels);
    uint32_t pl = g - p * C.tile_pixels;
    uint32_t ty = fastdiv(pl, C.div_tile_w);
    ix = C.tile_x0 + (pl - ty * C.tile_w);
    iy = C.tile_y0 + ty;
    pass = C.pass0 + p;
}

// jittered sample position (main.cpp:192-198), exact float ops
__device__ __forceinline__ void jitter_xy(const RenderCtx& C, uint32_t ix, uint32_t iy, uint32_t pass, float& x, float& y) {
    uint4 r = philox4x32(iy * C.width + ix, pass, 0u, 0u, C.keys);
    x = xdiv(xadd((float)ix, u01(r.x)), (float)C.width);
    y = xdiv(xadd((float)iy, u01(r.y)), (float)C.height);
    if (x == 1.0f) x = __uint_as_float(0x3F7FFFFFu); // nextafter(1.0f, 0.0f)
    if (y == 1.0f) y = __uint_as_float(0x3F7FFFFFu);
}

// SimpleCamera::sampleRay (src/SimpleCamera.cpp:15-21), exact
__device__ __forceinline__ void camera_ray(const DevCamera& cam, float x, float y, f3& o, f3& d) {
    x = xsub(x, 0.5f);
    y = xsub(y, 0.5f);
    f3 ray = xadd3(xadd3(xscale3(ld3(cam.right), x), xscale3(ld3(cam.up), y)), ld3(cam.dir));
    o = ld3(cam.pos);
    d = xnormalize3(ray);
}

// K1 generate: one thread per path of the batch.
__global__ void __launch_bounds__(256) k_generate(const __grid_constant__ DevScene S, const __grid_constant__ RenderCtx C) {
    uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x; slot < C.batch; slot += stride) {
        uint32_t ix, iy, pass;
        slot_to_pixel(C, slot, ix, iy, pass);
        float x, y;
        jitter_xy(C, ix, iy, pass, x, y);
        f3 o, d;
        camera_ray(S.cam, x, y, o, d);
        C.ray_o[slot] = make_float4(o.x, o.y, o.z, 1.0f);
        C.ray_d[slot] = make_float4(d.x, d.y, d.z, __uint_as_float(slot));
        C.ray_x[slot] = -1.0f;
        C.pathval[slot] = 0.0f;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) C.cnt[0] = C.batch;
}

// ---- closest hit over the whole scene (Geometry::traceRay) ------------------------------------------

template <bool SMALLPT, bool MESH, bool GFAST = false, bool X = true>
__device__ __forceinline__ SurfHit trace_geometry(const DevScene& S, f3 o, f3 d, TraceCounters& tc, bool skip_planes = false);

// ---- nearest light (CollectionLighting::traceRayToLight, src/CollectionLighting.cpp:23-34) -----------
template <bool PDF, bool AREA = false, bool X = true, class LightRef>
__device__ __forceinline__ void trace_one_light(const LightRef& L, uint32_t i, f3 o, f3 d, bool& any, float& best_len, uint32_t& which, f3& lpos,
                                                float& lpdf) {
    LightHit e = light_trace<AREA, X>(L, o, d);
    if (!e.hit) return;
    // X = false: the rays are unit length, so the distance along the ray orders the lights like length(pos - origin) does
    float len = X ? xlength3(xsub3(e.position, o)) : e.t;
    if (!any || best_len > len) {
        any = true;
        best_len = len;
        which = i;
        lpos = e.position;
    }
    if (PDF) lpdf = pfma(L.weight, light_pdf_at<AREA>(L, o, e.position), lpdf);
}
// conservative ray/box test for the light LBVH (see slab() in ipt_trace.cuh); limit = farthest useful entry distance
__device__ __forceinline__ bool light_box(const f8& a, int base, f3 o, f3 inv, float limit) {
    float t0x = (a.v[base] - o.x) * inv.x, t1x = (a.v[base + 4] - o.x) * inv.x;
    float t0y = (a.v[base + 1] - o.y) * inv.y, t1y = (a.v[base + 5] - o.y) * inv.y;
    float t0z = (a.v[base + 2] - o.z) * inv.z, t1z = (a.v[base + 6] - o.z) * inv.z;
    float tn = fmaxf(fmaxf(fminf(t0x, t1x), fminf(t0y, t1y)), fmaxf(fminf(t0z, t1z), 0.0f));
    float tf = fminf(fminf(fmaxf(t0x, t1x), fmaxf(t0y, t1y)), fmaxf(t0z, t1z));
    return tn <= tf * 1.0000003f && tn <= limit;
}

// ---- the light LBVH through its 32-byte quantised nodes (BvhNodeQ, see ipt_device.cuh) -----------------------------------------
// Same node format and grid space as the mesh traversal (ipt_trace.cuh), but a ray towards the lights starts anywhere in the
// scene, possibly many box extents away from the (often flat) root box of the lights, where the float error of the mapped
// origin o' is no longer small against a grid cell. The test therefore carries a per-axis slack s = |o'| |1/d'| 2^-20 — twice
// the bound on the accumulated rounding error of t = g / d' - o' / d' that grows with |o'|; the part that does not is covered
// by the full cell every quantised box is padded with — folded into the two constants of the fused multiply-adds: the
// entry distance of an axis is g_near / d' + (c - s), the exit distance g_far / d' + (c + s), with the near / far plane
// chosen by the sign of the direction (a select instead of the min / max of the symmetric form). Conservative for any
// origin; a direction component of 0 gets 1/d' = +-1e37 as in grid_ray.
#ifndef IPT_LIGHT_QNODES
#define IPT_LIGHT_QNODES 0 // 1: traverse the light LBVH through its 32-byte nodes. Measured (profiles/tuning_r02.md): same node visits, C5 unchanged, 100 emitters -12 % (the walk waits on dependent loads, not on L1 sectors, and the decode costs issue slots): off
#endif
struct LightGridRay {
    f3 inv, cn, cf;
    bool nx, ny, nz; // direction component negative: the box's upper plane is the near one
};
__device__ __forceinline__ LightGridRay light_grid_ray(const GridMap& G, f3 o, f3 d) {
    LightGridRay r;
    float ox = __fmaf_rn(__fsub_rn(o.x, G.lo[0]), G.scale[0], IPT_GRID_BASE), oy = __fmaf_rn(__fsub_rn(o.y, G.lo[1]), G.scale[1], IPT_GRID_BASE),
          oz = __fmaf_rn(__fsub_rn(o.z, G.lo[2]), G.scale[2], IPT_GRID_BASE);
    float dx = d.x * G.scale[0], dy = d.y * G.scale[1], dz = d.z * G.scale[2];
    r.inv = mk3(copysignf(fminf(fabsf(1.0f / dx), 1e37f), dx), copysignf(fminf(fabsf(1.0f / dy), 1e37f), dy), copysignf(fminf(fabsf(1.0f / dz), 1e37f), dz));
    float cx = -ox * r.inv.x, cy = -oy * r.inv.y, cz = -oz * r.inv.z;
    const float k = 9.5367431640625e-07f; // 2^-20
    float sx = fabsf(cx) * k, sy = fabsf(cy) * k, sz = fabsf(cz) * k; // |c| = |o'| |1/d'|
    r.cn = mk3(cx - sx, cy - sy, cz - sz);
    r.cf = mk3(cx + sx, cy + sy, cz + sz);
    r.nx = r.inv.x < 0.0f; r.ny = r.inv.y < 0.0f; r.nz = r.inv.z < 0.0f;
    return r;
}
// one child box of a BvhNodeQ: wa = lo.x | lo.y, wb = lo.z | hi.x, wc = hi.y | hi.z; true = the ray may hit it before `limit`
__device__ __forceinline__ bool light_box_q(uint32_t wa, uint32_t wb, uint32_t wc, const LightGridRay& R, float limit) {
    float lox = grid_lo16(wa), loy = grid_hi16(wa), loz = grid_lo16(wb), hix = grid_hi16(wb), hiy = grid_lo16(wc), hiz = grid_hi16(wc);
    float tnx = __fmaf_rn(R.nx ? hix : lox, R.inv.x, R.cn.x), tfx = __fmaf_rn(R.nx ? lox : hix, R.inv.x, R.cf.x);
    float tny = __fmaf_rn(R.ny ? hiy : loy, R.inv.y, R.cn.y), tfy = __fmaf_rn(R.ny ? loy : hiy, R.inv.y, R.cf.y);
    float tnz = __fmaf_rn(R.nz ? hiz : loz, R.inv.z, R.cn.z), tfz = __fmaf_rn(R.nz ? loz : hiz, R.inv.z, R.cf.z);
    float tn = fmaxf(fmaxf(tnx, tny), fmaxf(tnz, 0.0f));
    float tf = fminf(fminf(tfx, tfy), tfz);
    return tn <= tf * 1.0000003f && tn <= limit;
}

// One stack traversal of the light LBVH serving both queries of CollectionLighting:
//   LQ_NEAREST: traceRayToLight (CollectionLighting.cpp:23-34): nearest hit by length(pos - origin), earliest index on ties
//   LQ_PDF:     the mixture density sum_i w_i * DdfFromLight_i::value(d) over ALL lights the ray hits (ddf.cpp:156-162)
//   LQ_BOTH:    both from one traversal (returns the density; the nearest hit in which / lpos) — what a traced child ray
//               needs: its own traceRayToLight and the density of the mixture it was sampled from
// An LBVH is at most 63 key bits + 32 tie-breaking index bits deep, and the walk pushes one sibling per level.
#define IPT_LBVH_MAX_HEIGHT 96
template <int MODE, bool X>
__device__ __forceinline__ float light_bvh_query(const DevScene& S, f3 o, f3 d, uint32_t& which, f3& lpos, float& best_len, TraceCounters& tc) {
    constexpr bool NEAREST = MODE != LQ_PDF, PDF = MODE != LQ_NEAREST;
    float pdf_sum = 0.0f;
    best_len = IPT_INF;
    which = IPT_NO_HIT;
#if IPT_LIGHT_QNODES
    const LightGridRay R = light_grid_ray(S.light_grid, o, d);
#else
    f3 inv = mk3(1.0f / d.x, 1.0f / d.y, 1.0f / d.z);
#endif
    float dlen = sqrtf(d.x * d.x + d.y * d.y + d.z * d.z);
    uint32_t stack[IPT_LBVH_MAX_HEIGHT];
    int sp = 0;
    uint32_t node = S.n_light_bvh > 1 ? 0u : 0x80000000u; // a single light is a lone leaf
    while (true) {
        if (node & 0x80000000u) {
            uint32_t pos = node & 0x7FFFFFFFu;
            f8 r0 = ldg256(&S.light_recs[4 * (size_t)pos]);
            f8 r1 = ldg256(&S.light_recs[4 * (size_t)pos + 2]);
            ++tc.lights;
            f3 corner = mk3(r0.v[0], r0.v[1], r0.v[2]), n = mk3(r0.v[3], r0.v[4], r0.v[5]), rel;
            float t = isect_parallelogram<X>(corner, n, mk3(r0.v[6], r0.v[7], r1.v[0]), mk3(r1.v[1], r1.v[2], r1.v[3]), r1.v[5] != 0.0f, o, d, &rel);
            if (t != IPT_INF) {
                f3 hp = xadd3(corner, rel);
                uint32_t orig = __float_as_uint(r1.v[4]);
                if (NEAREST) {
                    float len = X ? xlength3(xsub3(hp, o)) : t; // unit direction: see trace_one_light
                    if (len < best_len || (len == best_len && orig < which)) { best_len = len; which = orig; lpos = hp; }
                }
                if (PDF) {
                    f3 dp = mk3(__fsub_rn(hp.x, o.x), __fsub_rn(hp.y, o.y), __fsub_rn(hp.z, o.z));
                    float decay = dot3(dp, dp);
                    float cosinus = pmul(-dot3(n, dp), rsqrtf(decay));
                    if (cosinus >= 0.0f) pdf_sum = pfma(r1.v[7], __fdividef(decay, pmul(cosinus, r1.v[6])), pdf_sum);
                }
            }
            node = IPT_NO_HIT;
        } else {
            ++tc.light_nodes;
            // entry distances are in units of t; a hit at length L has t = L / |d|
            float limit = MODE == LQ_NEAREST ? (best_len / dlen) * 1.0001f + 1e-6f : IPT_INF;
#if IPT_LIGHT_QNODES
            u8x32 q = ldg256u(&S.light_qnodes[node]);
            bool h0 = light_box_q(q.v[0], q.v[1], q.v[2], R, limit), h1 = light_box_q(q.v[3], q.v[4], q.v[5], R, limit);
            uint32_t left = q.v[6], right = q.v[7];
#else
            f8 n0 = ldg256(&S.light_nodes[node]);
            f8 n1 = ldg256(reinterpret_cast<const char*>(&S.light_nodes[node]) + 32);
            bool h0 = light_box(n0, 0, o, inv, limit), h1 = light_box(n1, 0, o, inv, limit);
            uint32_t left = __float_as_uint(n0.v[3]), right = __float_as_uint(n0.v[7]);
#endif
            node = IPT_NO_HIT;
            if (h0 && h1) { node = left; stack[sp++] = right; }
            else if (h0) node = left;
            else if (h1) node = right;
        }
        if (node == IPT_NO_HIT) {
            if (sp == 0) break;
            node = stack[--sp];
        }
    }
    return pdf_sum;
}

// nearest light, scanning in list order with strict `>` (CollectionLighting.cpp:23-34); `lpdf` receives the light part
// of the mixture density along the same ray, sum_i w_i * DdfFromLight_i::value(d) (lighting.cpp:61-73, ddf.cpp:156-162),
// which needs exactly the intersections this scan performs (PDF = false: nearest light only)
// SPEC: what the fused shade kernels know about the scene at COMPILE time, so that each instantiation carries only the
// light and geometry code its scenes can run (the generic kernel was 10 360 SASS instructions, the box-scene one is 2944):
//   SPEC_RUNTIME          nothing: every decision is taken from the scene (k_extend, the mesh path, SmallPt scenes)
//   SPEC_LIGHT_BVH        the lights sit in the light LBVH (> 8 lights)
//   SPEC_FEW_LIGHTS       no LBVH; inline or linear scan decided at run time
//   SPEC_ONE_LIGHT        no LBVH and at most IPT_INLINE_LIGHTS lights, i.e. the constant-bank copies
//   SPEC_ONE_AREA_LIGHT   ... and that light is an area light (no sphere-light code at all)
//   SPEC_BOX_SCENE        ... and the geometry is grouped box planes + inline spheres (GFAST in ipt_trace.cuh): every
//                         Lambert / glossy box scene of the reference and BASELINE configs[0..1]
//   SPEC_LAMBERT_BOX      ... and every material is the cosine DDF (the reference's own box scenes, BASELINE configs[0])
enum SceneSpec { SPEC_FEW_LIGHTS = 0, SPEC_LIGHT_BVH = 1, SPEC_RUNTIME = 2, SPEC_ONE_LIGHT = 3, SPEC_ONE_AREA_LIGHT = 4, SPEC_BOX_SCENE = 5, SPEC_LAMBERT_BOX = 6 };
#define IPT_SPEC_INLINE_LIGHTS(SPEC) ((SPEC) == SPEC_ONE_LIGHT || (SPEC) == SPEC_ONE_AREA_LIGHT || (SPEC) == SPEC_BOX_SCENE || (SPEC) == SPEC_LAMBERT_BOX)
#define IPT_SPEC_AREA_LIGHTS(SPEC) ((SPEC) == SPEC_ONE_AREA_LIGHT || (SPEC) == SPEC_BOX_SCENE || (SPEC) == SPEC_LAMBERT_BOX)
#define IPT_SPEC_FAST_GEOMETRY(SPEC) ((SPEC) == SPEC_BOX_SCENE || (SPEC) == SPEC_LAMBERT_BOX)
template <int SPEC>
__device__ __forceinline__ bool has_light_bvh(const DevScene& S) { return SPEC == SPEC_RUNTIME ? S.n_light_bvh != 0 : SPEC == SPEC_LIGHT_BVH; }
template <int SPEC>
__device__ __forceinline__ bool lights_inline(const DevScene& S) { return IPT_SPEC_INLINE_LIGHTS(SPEC) ? true : SPEC == SPEC_LIGHT_BVH ? false : S.light_inline != 0; }
template <int SPEC>
__device__ __forceinline__ float light_power(const DevScene& S, uint32_t i) {
    float power = lights_inline<SPEC>(S) ? S.lights[i].surface_power : S.lights_g[i].surface_power;
    return isfinite(power) ? power : 1.0f; // main.cpp:123 point-light hack
}
// `ldist` receives the nearest light's distance: length(pos - origin) as CollectionLighting.cpp:27 computes it, or — for
// the contracted secondary-ray form (X = false) of the inline / linear scans — the distance along the unit direction.
template <bool PDF = true, int SPEC = SPEC_RUNTIME, bool X = true>
__device__ __forceinline__ bool trace_lights(const DevScene& S, f3 o, f3 d, uint32_t& which, f3& lpos, float& lpdf, float& ldist, TraceCounters& tc) {
    bool any = false;
    ldist = 0.0f;
    lpdf = 0.0f;
    if (has_light_bvh<SPEC>(S)) {
        if (PDF) lpdf = light_bvh_query<LQ_BOTH, X>(S, o, d, which, lpos, ldist, tc);
        else light_bvh_query<LQ_NEAREST, X>(S, o, d, which, lpos, ldist, tc);
        return which != IPT_NO_HIT;
    }
    if (SPEC == SPEC_LIGHT_BVH) return false; // unreachable: the LBVH branch above always returns
    if (lights_inline<SPEC>(S)) {
#pragma unroll
        for (int i = 0; i < IPT_INLINE_LIGHTS; ++i) // static indices: light constants become immediate constant-bank operands
            if (i < (int)S.n_lights) trace_one_light<PDF, IPT_SPEC_AREA_LIGHTS(SPEC), X>(S.lights[i], i, o, d, any, ldist, which, lpos, lpdf);
        tc.lights += min(S.n_lights, (uint32_t)IPT_INLINE_LIGHTS);
    } else if (!IPT_SPEC_INLINE_LIGHTS(SPEC)) {
        for (uint32_t i = 0; i < S.n_lights; ++i) trace_one_light<PDF, false, X>(S.lights_g[i], i, o, d, any, ldist, which, lpos, lpdf);
        tc.lights += S.n_lights;
    }
    return any;
}

struct Outcome {
    uint32_t kind; // 0 miss, 1 surface, 2 light
    SurfHit surf;
    uint32_t light;
    f3 light_pos;
    float light_pdf; // light part of the mixture density along the ray (see trace_lights)
};

// main.cpp:113: the light wins if there is no surface hit or the surface point is farther than the light's
template <bool X>
__device__ __forceinline__ bool light_nearer(const SurfHit& sh, f3 o, f3 d, float ldist) {
    if (sh.prim == IPT_NO_HIT) return true;
    if (!X) return sh.t > ldist; // unit direction: the distances along the ray compare like the lengths
    return xlength3(xsub3(xpoint(o, d, sh.t), o)) > ldist;
}

// Geometry::traceRay + Lighting::traceRayToLight + the decision of main.cpp:111-128
template <bool SMALLPT, bool MESH, int SPEC = SPEC_RUNTIME, bool X = true>
__device__ __forceinline__ Outcome trace_scene(const DevScene& S, f3 o, f3 d, TraceCounters& tc) {
    Outcome r;
    r.surf = trace_geometry<SMALLPT, MESH, IPT_SPEC_FAST_GEOMETRY(SPEC), X>(S, o, d, tc);
    r.light = IPT_NO_HIT;
    r.light_pos = mk3(0, 0, 0);
    float ldist;
    bool lh = trace_lights<true, SPEC, X>(S, o, d, r.light, r.light_pos, r.light_pdf, ldist, tc);
    r.kind = r.surf.prim != IPT_NO_HIT ? 1u : 0u;
    if (lh && light_nearer<X>(r.surf, o, d, ldist)) r.kind = 2;
    return r;
}

// Last traced depth: children of this level are never traced (main.cpp:100-101), so the ray matters only if it reaches
// a light before any surface. Lights are tested first and the geometry only for rays that hit one ("shadow ray"):
// the decision is the same expression as in trace_scene, evaluated for fewer rays. kind 3 = no light along the ray
// (surface or miss, not resolved).
template <bool SMALLPT, bool MESH, int SPEC = SPEC_RUNTIME, bool X = true>
__device__ __forceinline__ Outcome trace_scene_last(const DevScene& S, f3 o, f3 d, TraceCounters& tc) {
    Outcome r;
    r.light = IPT_NO_HIT;
    r.light_pos = mk3(0, 0, 0);
    r.surf.prim = IPT_NO_HIT; r.surf.t = IPT_INF; r.surf.tri_pos = IPT_NO_HIT;
    float ldist;
    bool lh = trace_lights<true, SPEC, X>(S, o, d, r.light, r.light_pos, r.light_pdf, ldist, tc);
    r.kind = 3;
    if (!lh) return r;
    r.surf = trace_geometry<SMALLPT, MESH, IPT_SPEC_FAST_GEOMETRY(SPEC), X>(S, o, d, tc);
    r.kind = light_nearer<X>(r.surf, o, d, ldist) ? 2u : 1u;
    return r;
}

// Resolves a ray's weight (see the queue description above): K * sv / (sum_i w_i * pdf_light_i(dir) + w_sdf * sv), the
// `sdf/mix` multiplier of main.cpp:172-173 with UnionDdf::value (ddf.cpp:156-162); `lpdf` comes from trace_lights.
__device__ __forceinline__ float resolve_weight(const DevScene& S, float K, float sv, float lpdf) {
    if (sv < 0.0f) return K;
    return pmul(K, __fdividef(sv, pfma(S.sdf_weight, sv, lpdf)));
}

__device__ __forceinline__ void flush_stat(unsigned long long* stats, int slot, uint32_t v) {
    // warp reduce, then one atomic per warp
    for (int off = 16; off > 0; off >>= 1) v += __shfl_down_sync(0xffffffffu, v, off);
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(&stats[slot], (unsigned long long)v);
}

// K2 extend: one thread per ray of depth `depth`. Light hits are accumulated here (the emission is the leaf
// of the estimator tree); surface hits are compacted into the hit queue unless this is the last traced depth.
// X: exact arithmetic (the camera rays, depth 0) or the contracted secondary-ray form (depth > 0; never with MESH)
template <bool SMALLPT, bool MESH, bool LAST, bool X = true>
__global__ void __launch_bounds__(256, IPT_EXTEND_MIN_BLOCKS) k_extend(const __grid_constant__ DevScene S, const __grid_constant__ RenderCtx C, uint32_t depth) {
    const uint32_t n = C.cnt[2 * depth];
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
    const uint32_t gwarp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    uint32_t n_surface = 0, n_light = 0, n_miss = 0, n_dropped = 0;
    TraceCounters tc{0, 0, 0, 0};
    for (uint32_t base = gwarp * 32; base < n; base += warps * 32) {
        uint32_t i = base + lane;
        bool active = i < n;
        bool emit = false;
        float4 ro, rd;
        Outcome oc;
        if (active) {
            ro = C.ray_o[i];
            rd = C.ray_d[i];
            float sv = C.ray_x[i];
            f3 o = mk3(ro.x, ro.y, ro.z), d = mk3(rd.x, rd.y, rd.z);
            if (LAST && !(C.flags & IPT_FLAG_RESOLVE_LAST_LEVEL)) oc = trace_scene_last<SMALLPT, MESH, SPEC_RUNTIME, X>(S, o, d, tc);
            else oc = trace_scene<SMALLPT, MESH, SPEC_RUNTIME, X>(S, o, d, tc);
            ro.w = resolve_weight(S, ro.w, sv, oc.light_pdf);
            if (!isfinite(ro.w)) { ++n_dropped; oc.kind = 4; } // non-finite multiplier (main.cpp:175): drop this sample
#ifdef IPT_DEBUG_PRINT
            if (C.flags & IPT_FLAG_DEBUG_PRINT)
                printf("GPU extend d=%u node=%u o=(%.9g %.9g %.9g) d=(%.9g %.9g %.9g) thr=%.9g kind=%u prim=%u t=%.9g\n", depth,
                       C.slot_bits == 32 ? 0u : (__float_as_uint(rd.w) >> C.slot_bits), o.x, o.y, o.z, d.x, d.y, d.z, ro.w, oc.kind, oc.surf.prim, oc.surf.t);
#endif
            if (oc.kind == 2) {
                ++n_light;
                float power = S.light_inline ? S.lights[oc.light].surface_power : S.lights_g[oc.light].surface_power;
                if (!isfinite(power)) power = 1.0f; // main.cpp:123 point-light hack
                uint32_t slot = __float_as_uint(rd.w) & C.slot_mask;
                atomicAdd(&C.pathval[slot], ro.w * power);
            } else if (oc.kind == 1) {
                ++n_surface;
                emit = !LAST;
            } else if (oc.kind == 0) {
                ++n_miss;
            }
        }
        if (!LAST) {
            // warp-aggregated append: one atomicAdd per warp reserves the slots of all its emitting lanes
            uint32_t ballot = __ballot_sync(0xffffffffu, emit);
            if (ballot) {
                uint32_t basepos = 0;
                if (lane == 0) basepos = atomicAdd(&C.cnt[2 * depth + 1], (uint32_t)__popc(ballot));
                basepos = __shfl_sync(0xffffffffu, basepos, 0);
                if (emit) {
                    uint32_t j = basepos + __popc(ballot & ((1u << lane) - 1u));
                    f3 p = xpoint(mk3(ro.x, ro.y, ro.z), mk3(rd.x, rd.y, rd.z), oc.surf.t);
                    uint32_t iprim = oc.surf.tri_pos != IPT_NO_HIT ? S.n_prims + oc.surf.tri_pos : oc.surf.prim;
                    float2 oct = oct_encode(mk3(rd.x, rd.y, rd.z));
                    if (IPT_BOUNDS_OK(j, C.hit_cap, C.stats)) {
                        C.hit_a[depth & 1][j] = make_float4(p.x, p.y, p.z, ro.w);
                        C.hit_b[depth & 1][j] = make_uint4(__float_as_uint(rd.w), iprim, __float_as_uint(oct.x), __float_as_uint(oct.y));
                    }
                }
            }
        }
    }
    flush_stat(C.stats, ST_SURFACE, n_surface);
    flush_stat(C.stats, ST_LIGHT, n_light);
    flush_stat(C.stats, ST_MISS, n_miss);
    flush_stat(C.stats, ST_DROPPED, n_dropped);
    if (MESH) {
        flush_stat(C.stats, ST_NODES, tc.nodes);
        flush_stat(C.stats, ST_TRIS, tc.tris);
    }
    flush_stat(C.stats, ST_LIGHTS, tc.lights);
    flush_stat(C.stats, ST_LIGHT_NODES, tc.light_nodes);
}

// geometric normal + material of a hit primitive (GeometrySphereInBox.cpp:43-56 and the other geometries).
// TRI_MATS = false for kernels that never shade a mesh hit (the fused shade kernels: mesh scenes run the unfused loop).
template <bool TRI_MATS = true>
__device__ __forceinline__ void surface_frame(const DevScene& S, uint32_t prim, f3 pos, f3& normal, uint32_t& material) {
    if (prim >= S.n_prims) {
        uint32_t k = prim - S.n_prims; // sorted triangle position
        float4 a = __ldg(&S.tris[4 * (size_t)k]);
        float4 b = __ldg(&S.tris[4 * (size_t)k + 1]);
        normal = mk3(a.w, b.x, b.y);
        // a uniform branch: the pointer is a kernel parameter
        material = TRI_MATS && S.tri_mats ? __ldg(S.tri_mats + k) : S.tri_material;
        return;
    }
    // the index differs per lane: a constant-bank read would serialise, a global (L1-cached) read does not
    const float4* pp = reinterpret_cast<const float4*>(&S.prims_g[prim]);
    float4 p0 = __ldg(pp), p1 = __ldg(pp + 1);
    DevPrim p;
    p.px = p0.x; p.py = p0.y; p.pz = p0.z; p.radius = p0.w;
    p.kind = __float_as_uint(p1.x); p.material = __float_as_uint(p1.y); p.flags = __float_as_uint(p1.z); p.r2 = p1.w;
    material = p.material;
    if (p.kind == IPT_PRIM_BOX_PLANE) {
        normal = mk3(-p.px, -p.py, -p.pz);
    } else {
        f3 nn = xnormalize3(xsub3(pos, mk3(p.px, p.py, p.pz)));
        normal = (p.flags & 8u) ? neg3(nn) : nn;
    }
}

#ifndef IPT_PARK
#define IPT_PARK 64 // entries per warp: fewer than 32 are parked when up to 32 more arrive
#endif
// Second half of trace_scene_last for a parked ray that reached a light at `lpos`: Geometry::traceRay and the
// light-vs-surface decision of main.cpp:113; the light's contribution is added if nothing is nearer.
template <bool SMALLPT, int SPEC, bool X>
__device__ __forceinline__ void resolve_parked(const DevScene& S, const RenderCtx& C, const float* dq, uint32_t k, TraceCounters& tc,
                                               uint32_t& n_light, uint32_t& n_surface) {
    f3 o = mk3(dq[0 * IPT_PARK + k], dq[1 * IPT_PARK + k], dq[2 * IPT_PARK + k]);
    f3 d = mk3(dq[3 * IPT_PARK + k], dq[4 * IPT_PARK + k], dq[5 * IPT_PARK + k]);
    float ldist = dq[6 * IPT_PARK + k];
    // the ray reached a light: only what can lie between the origin and that light has to be intersected
    SurfHit sh = trace_geometry<SMALLPT, false, IPT_SPEC_FAST_GEOMETRY(SPEC), X>(S, o, d, tc, IPT_SHADOW_SKIP_WALLS && IPT_SPEC_FAST_GEOMETRY(SPEC) && S.lights_inside_box != 0);
    if (light_nearer<X>(sh, o, d, ldist)) {
        ++n_light;
        atomicAdd(&C.pathval[__float_as_uint(dq[8 * IPT_PARK + k])], dq[7 * IPT_PARK + k]);
    } else ++n_surface;
}

// First node visit of the light LBVH: false = the ray misses both root boxes, i.e. there is no light along it.
__device__ __forceinline__ bool light_root_hit(const DevScene& S, f3 o, f3 d, TraceCounters& tc) {
    ++tc.light_nodes;
#if IPT_LIGHT_QNODES
    const LightGridRay R = light_grid_ray(S.light_grid, o, d);
    u8x32 q = ldg256u(&S.light_qnodes[0]);
    return light_box_q(q.v[0], q.v[1], q.v[2], R, IPT_INF) || light_box_q(q.v[3], q.v[4], q.v[5], R, IPT_INF);
#else
    f3 inv = mk3(1.0f / d.x, 1.0f / d.y, 1.0f / d.z);
    f8 n0 = ldg256(&S.light_nodes[0]);
    f8 n1 = ldg256(reinterpret_cast<const char*>(&S.light_nodes[0]) + 32);
    return light_box(n0, 0, o, inv, IPT_INF) || light_box(n1, 0, o, inv, IPT_INF);
#endif
}
// Many-light scenes, last traced depth: the whole of trace_scene_last for a parked ray (light LBVH walk, weight, and the
// occlusion test if a light was reached). Parked are only rays that passed light_root_hit, so the lanes of a pop walk
// the LBVH together instead of idling next to the rays that leave at the root.
template <bool SMALLPT, bool X>
__device__ __forceinline__ void last_parked(const DevScene& S, const RenderCtx& C, const float* dq, uint32_t k, TraceCounters& tc,
                                            uint32_t& n_light, uint32_t& n_surface, uint32_t& n_dropped) {
    f3 o = mk3(dq[0 * IPT_PARK + k], dq[1 * IPT_PARK + k], dq[2 * IPT_PARK + k]);
    f3 d = mk3(dq[3 * IPT_PARK + k], dq[4 * IPT_PARK + k], dq[5 * IPT_PARK + k]);
    Outcome oc = trace_scene_last<SMALLPT, false, SPEC_LIGHT_BVH, X>(S, o, d, tc);
    float wr = resolve_weight(S, dq[6 * IPT_PARK + k], dq[7 * IPT_PARK + k], oc.light_pdf);
    if (!isfinite(wr)) ++n_dropped;
    else if (oc.kind == 2) {
        ++n_light;
        atomicAdd(&C.pathval[__float_as_uint(dq[8 * IPT_PARK + k])], wr * light_power<SPEC_LIGHT_BVH>(S, oc.light));
    } else if (oc.kind == 1) ++n_surface;
}

struct ExtendCounters {
    uint32_t surface, light, miss, dropped;
};
// The body of k_extend<.., LAST = false> for one parked child ray of depth `depth` (entry k of the warp's queue; all 32
// lanes call this, `valid` masks the drain): trace_scene, weight resolution, emission, and the warp-aggregated append
// of the surface hits to the hit set of `depth`.
// LIGHTS = false: the caller has established that no light lies along the ray (it misses the root boxes of the light LBVH),
// so only Geometry::traceRay runs; the light part of the mixture density is 0 and the ray cannot end on a light.
template <bool SMALLPT, int SPEC, bool X, bool LIGHTS = true>
__device__ __forceinline__ void extend_parked(const DevScene& S, const RenderCtx& C, const float* dq, uint32_t k, bool valid, uint32_t depth,
                                              TraceCounters& tc, ExtendCounters& ec) {
    const uint32_t lane = threadIdx.x & 31;
    bool emit = false;
    f3 o = mk3(0, 0, 0), d = mk3(0, 0, 1);
    float wr = 0.0f;
    uint32_t ctag = 0;
    Outcome oc;
    if (valid) {
        o = mk3(dq[0 * IPT_PARK + k], dq[1 * IPT_PARK + k], dq[2 * IPT_PARK + k]);
        d = mk3(dq[3 * IPT_PARK + k], dq[4 * IPT_PARK + k], dq[5 * IPT_PARK + k]);
        ctag = __float_as_uint(dq[8 * IPT_PARK + k]);
        if (LIGHTS) oc = trace_scene<SMALLPT, false, SPEC, X>(S, o, d, tc);
        else {
            oc.surf = trace_geometry<SMALLPT, false, IPT_SPEC_FAST_GEOMETRY(SPEC), X>(S, o, d, tc);
            oc.kind = oc.surf.prim != IPT_NO_HIT ? 1u : 0u;
            oc.light = IPT_NO_HIT;
            oc.light_pdf = 0.0f;
        }
        wr = resolve_weight(S, dq[6 * IPT_PARK + k], dq[7 * IPT_PARK + k], oc.light_pdf);
        if (!isfinite(wr)) ++ec.dropped; // non-finite multiplier (main.cpp:175): drop this sample
        else if (oc.kind == 2) {
            ++ec.light;
            atomicAdd(&C.pathval[ctag & C.slot_mask], wr * light_power<SPEC>(S, oc.light));
        } else if (oc.kind == 1) {
            ++ec.surface;
            emit = true;
        } else ++ec.miss;
    }
    uint32_t ballot = __ballot_sync(0xffffffffu, emit);
    if (ballot) {
        uint32_t basepos = 0;
        if (lane == 0) basepos = atomicAdd(&C.cnt[2 * depth + 1], (uint32_t)__popc(ballot));
        basepos = __shfl_sync(0xffffffffu, basepos, 0);
        if (emit) {
            uint32_t j = basepos + __popc(ballot & ((1u << lane) - 1u));
            f3 p = xpoint(o, d, oc.surf.t);
            float2 oct = oct_encode(d);
            if (IPT_BOUNDS_OK(j, C.hit_cap, C.stats)) {
                C.hit_a[depth & 1][j] = make_float4(p.x, p.y, p.z, wr);
                C.hit_b[depth & 1][j] = make_uint4(ctag, oc.surf.prim, __float_as_uint(oct.x), __float_as_uint(oct.y));
            }
        }
    }
}

// K3 shade: one thread per surface hit; spawns schedule[depth] children from the 1:1 mixture of the light DDF
// and the surface DDF (main.cpp:142-177).
//   FUSE_NONE  the survivors are appended to the ray queue of depth+1 (mesh scenes: k_extend_mesh traces them).
//   FUSE_NEXT  (analytic scenes) the children are traced HERE: each one is parked in a per-warp shared-memory queue and
//              whenever 32 are waiting the warp runs the body of k_extend for them (extend_parked) — full warps, no ray
//              record written or read, no k_extend launch; surface hits go to the other hit set (depth+1).
//   FUSE_LAST  (analytic scenes, children are the last traced depth) the children are "shadow rays" (trace_scene_last):
//              light test at once, and only the rays that reach a light are parked for the occlusion test.
// Same functions, same operands, same counters as the separate kernels.
enum ShadeFusion { FUSE_NONE = 0, FUSE_NEXT = 1, FUSE_LAST = 2 };
template <int FUSE, bool SMALLPT, int SPEC = SPEC_RUNTIME>
__global__ void __launch_bounds__(256, FUSE == FUSE_LAST ? IPT_SHADE_FUSED_MIN_BLOCKS : FUSE == FUSE_NEXT ? IPT_SHADE_NEXT_MIN_BLOCKS : IPT_SHADE_MIN_BLOCKS) k_shade(const __grid_constant__ DevScene S, const __grid_constant__ RenderCtx C, uint32_t depth) {
    const uint32_t n = C.cnt[2 * depth + 1];
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
    const uint32_t gwarp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t n_children = C.schedule[depth];
    const float inv_n = 1.0f / (float)n_children;
    const bool keep_zero = (C.flags & IPT_FLAG_KEEP_ZERO_WEIGHT) != 0;
    uint32_t n_failed = 0, n_pruned = 0, n_dropped = 0;
    uint32_t n_fused = 0, n_light = 0, n_surface = 0;
    ExtendCounters ec{0, 0, 0, 0};
    TraceCounters tc{0, 0, 0, 0};
    // every ray traced here is downstream of a random number (depth >= 1): the contracted secondary-ray arithmetic, the
    // same k_extend<.., X = false> uses for queued rays of depth > 0
    constexpr bool X = !IPT_FAST_SECONDARY;
    constexpr int PARK_WORDS = 9;
    // many-light scenes, non-last depths: children are regrouped by whether they can see a light at all (the root boxes of
    // the light LBVH): the ones that can walk the LBVH 32 at a time, the others only intersect the geometry
    constexpr bool TWO_Q = FUSE == FUSE_NEXT && SPEC == SPEC_LIGHT_BVH && IPT_LIGHT_TWO_QUEUES;
    constexpr int QUEUES = TWO_Q ? 2 : 1;
    __shared__ float dq_all[FUSE != FUSE_NONE ? (256 / 32) * PARK_WORDS * IPT_PARK * QUEUES : 1];
    float* dq = dq_all + (FUSE != FUSE_NONE ? (threadIdx.x >> 5) * PARK_WORDS * IPT_PARK * QUEUES : 0); // this warp's parked rays
    float* dq2 = dq + (TWO_Q ? PARK_WORDS * IPT_PARK : 0);
    uint32_t qn = 0, qn2 = 0;                                                   // warp-uniform
    uint32_t* out_count = &C.cnt[2 * (depth + 1)];
    for (uint32_t base = gwarp * 32; base < n; base += warps * 32) {
        uint32_t i = base + lane;
        bool active = i < n;
        f3 pos = mk3(0, 0, 0);
        float thr = 0.0f;
        uint32_t tag = 0, node = 0, pixel = 0, pass = 0;
        Sdf sdf;
        Basis bn, bl;
        float albedo = 1.0f;
        if (active) {
            float4 a = C.hit_a[depth & 1][i];
            uint4 b = C.hit_b[depth & 1][i];
            pos = mk3(a.x, a.y, a.z);
            thr = a.w;
            tag = b.x;
            node = tag >> C.slot_bits;
            if (C.slot_bits == 32) node = 0;
            uint32_t ix, iy;
            slot_to_pixel(C, tag & C.slot_mask, ix, iy, pass);
            pixel = iy * C.width + ix;
            f3 normal;
            uint32_t material;
            surface_frame<FUSE == FUSE_NONE>(S, b.y, pos, normal, material);
            const float4* mp = reinterpret_cast<const float4*>(&S.mats_g[material]);
            float4 m0 = __ldg(mp), m1 = __ldg(mp + 1);
            DevMaterial m;
            m.ddf = __float_as_uint(m0.x); m.albedo = m0.y; m.wd = m0.z; m.ws = m0.w; m.exponent = m1.x; m.inv_np1 = m1.y; m.lobe_norm = m1.z;
            albedo = m.albedo;
            f3 din = mk3(0, 0, 0);
            if (SPEC != SPEC_LAMBERT_BOX && m.ddf == IPT_DDF_GLOSSY) din = oct_decode(__uint_as_float(b.z), __uint_as_float(b.w)); // only the glossy lobe needs it
            sdf = make_sdf(m, normal, din);
            // SmallPt scenes: the reference's own operation sequence for the rotation and the samples (ipt_shading.cuh)
            bn = SMALLPT ? make_basis_exact(normal) : make_basis(normal);
            bl = (SPEC != SPEC_LAMBERT_BOX && m.ddf == IPT_DDF_GLOSSY) ? (SMALLPT ? make_basis_exact(sdf.refl) : make_basis(sdf.refl)) : bn;
        }
        const float hit_k = pmul(pmul(thr, albedo), inv_n);
        for (uint32_t c = 0; c < n_children; ++c) {
            bool emit = false;
            f3 w = mk3(0, 0, 0);
            float wgt = 0.0f, child_sv = -1.0f;
            uint32_t child = node * n_children + c;
            if (active) {
                uint4 r = philox4x32(pixel, pass, child, depth + 1, C.keys);
                w = mix_sample<IPT_SPEC_INLINE_LIGHTS(SPEC), IPT_SPEC_AREA_LIGHTS(SPEC), SPEC == SPEC_LAMBERT_BOX, SMALLPT>(S, sdf, bn, bl, pos, u01(r.x), u01(r.y), u01(r.z), u01(r.w));
                if (w.x == 0.0f && w.y == 0.0f && w.z == 0.0f) {
#ifdef IPT_DEBUG_PRINT
                    if (FUSE == FUSE_NONE && (C.flags & IPT_FLAG_DEBUG_PRINT)) printf("GPU shade d=%u child=%u u=(%.9g %.9g %.9g) FAILED\n", depth, child, u01(r.x), u01(r.y), u01(r.z));
#endif
                    ++n_failed; // still counted in the 1/n divisor (main.cpp:161-163,181)
                } else {
                    float sv = sdf_value<SPEC == SPEC_LAMBERT_BOX>(sdf, w);
                    // the ray's own light intersection (k_extend, or the fused block below) also yields the light part of
                    // the mixture density, so the weight K*sv/mix is resolved there; sv == 0 already means weight 0
                    wgt = hit_k; // throughput * albedo / n of this hit
                    child_sv = sv;
                    // sv and wgt are >= 0 or non-finite: their sum is finite iff both are, their minimum is 0 iff one is
                    if (!(__fadd_rn(sv, wgt) < IPT_INF)) ++n_dropped;
                    else if (fminf(sv, wgt) == 0.0f && !keep_zero) ++n_pruned;
                    else emit = true;
                }
            }
            if (FUSE == FUSE_NEXT) {
                if (emit) ++n_fused;
                const uint32_t ctag = (tag & C.slot_mask) | (C.slot_bits == 32 ? 0u : (child << C.slot_bits));
                bool to_lights = emit, plain = false;
                if (TWO_Q) {
                    to_lights = emit && light_root_hit(S, pos, w, tc);
                    plain = emit && !to_lights;
                }
                uint32_t pb = __ballot_sync(0xffffffffu, to_lights);
                if (pb) {
                    if (to_lights) {
                        uint32_t k = qn + __popc(pb & ((1u << lane) - 1u));
                        if (!IPT_BOUNDS_OK(k, (uint32_t)IPT_PARK, C.stats)) k = IPT_PARK - 1;
                        dq[0 * IPT_PARK + k] = pos.x; dq[1 * IPT_PARK + k] = pos.y; dq[2 * IPT_PARK + k] = pos.z;
                        dq[3 * IPT_PARK + k] = w.x; dq[4 * IPT_PARK + k] = w.y; dq[5 * IPT_PARK + k] = w.z;
                        dq[6 * IPT_PARK + k] = wgt; dq[7 * IPT_PARK + k] = child_sv; dq[8 * IPT_PARK + k] = __uint_as_float(ctag);
                    }
                    qn += __popc(pb);
                    __syncwarp();
                    if (qn >= 32) {
                        qn -= 32;
                        extend_parked<SMALLPT, SPEC, X>(S, C, dq, qn + lane, true, depth + 1, tc, ec);
                        __syncwarp();
                    }
                }
                if (TWO_Q) {
                    uint32_t pb2 = __ballot_sync(0xffffffffu, plain);
                    if (pb2) {
                        if (plain) {
                            uint32_t k = qn2 + __popc(pb2 & ((1u << lane) - 1u));
                            if (!IPT_BOUNDS_OK(k, (uint32_t)IPT_PARK, C.stats)) k = IPT_PARK - 1;
                            dq2[0 * IPT_PARK + k] = pos.x; dq2[1 * IPT_PARK + k] = pos.y; dq2[2 * IPT_PARK + k] = pos.z;
                            dq2[3 * IPT_PARK + k] = w.x; dq2[4 * IPT_PARK + k] = w.y; dq2[5 * IPT_PARK + k] = w.z;
                            dq2[6 * IPT_PARK + k] = wgt; dq2[7 * IPT_PARK + k] = child_sv; dq2[8 * IPT_PARK + k] = __uint_as_float(ctag);
                        }
                        qn2 += __popc(pb2);
                        __syncwarp();
                        if (qn2 >= 32) {
                            qn2 -= 32;
                            extend_parked<SMALLPT, SPEC, X, false>(S, C, dq2, qn2 + lane, true, depth + 1, tc, ec);
                            __syncwarp();
                        }
                    }
                }
                continue;
            }
            if (FUSE == FUSE_LAST) {
                // the body of k_extend<LAST> for this ray, in two steps: the light test now; the occlusion test of the
                // rays that did reach a light (about a third) is parked in a per-warp shared-memory queue and run 32 at a
                // time, so the geometry intersection is issued for full warps instead of for the third of the lanes
                if (has_light_bvh<SPEC>(S)) {
                    // many lights: regroup BEFORE the light-LBVH walk. A ray that misses the root boxes sees no light and,
                    // at the last traced depth, is done; the others are parked and walk the LBVH 32 at a time.
                    bool parkb = false;
                    if (emit) {
                        ++n_fused;
                        parkb = light_root_hit(S, pos, w, tc);
                    }
                    uint32_t pbb = __ballot_sync(0xffffffffu, parkb);
                    if (pbb) {
                        if (parkb) {
                            uint32_t k = qn + __popc(pbb & ((1u << lane) - 1u));
                            if (!IPT_BOUNDS_OK(k, (uint32_t)IPT_PARK, C.stats)) k = IPT_PARK - 1;
                            dq[0 * IPT_PARK + k] = pos.x; dq[1 * IPT_PARK + k] = pos.y; dq[2 * IPT_PARK + k] = pos.z;
                            dq[3 * IPT_PARK + k] = w.x; dq[4 * IPT_PARK + k] = w.y; dq[5 * IPT_PARK + k] = w.z;
                            dq[6 * IPT_PARK + k] = wgt; dq[7 * IPT_PARK + k] = child_sv;
                            dq[8 * IPT_PARK + k] = __uint_as_float(tag & C.slot_mask);
                        }
                        qn += __popc(pbb);
                        __syncwarp();
                        if (qn >= 32) {
                            qn -= 32;
                            last_parked<SMALLPT, X>(S, C, dq, qn + lane, tc, n_light, n_surface, n_dropped);
                            __syncwarp();
                        }
                    }
                    continue;
                }
                bool park = false;
                float contrib = 0.0f, ldist = 0.0f;
                if (emit) {
                    ++n_fused;
                    uint32_t li = IPT_NO_HIT;
                    float lpdf;
                    f3 lpos;
                    bool lh = trace_lights<true, SPEC == SPEC_LIGHT_BVH ? SPEC_FEW_LIGHTS : SPEC, X>(S, pos, w, li, lpos, lpdf, ldist, tc);
                    float wr = resolve_weight(S, wgt, child_sv, lpdf);
                    if (!isfinite(wr)) ++n_dropped;
                    else if (lh) {
                        contrib = wr * light_power<SPEC>(S, li);
                        park = true;
                    }
                }
                uint32_t pb = __ballot_sync(0xffffffffu, park);
                if (pb) {
                    if (park) {
                        uint32_t k = qn + __popc(pb & ((1u << lane) - 1u));
                        if (!IPT_BOUNDS_OK(k, (uint32_t)IPT_PARK, C.stats)) k = IPT_PARK - 1;
                        dq[0 * IPT_PARK + k] = pos.x; dq[1 * IPT_PARK + k] = pos.y; dq[2 * IPT_PARK + k] = pos.z;
                        dq[3 * IPT_PARK + k] = w.x; dq[4 * IPT_PARK + k] = w.y; dq[5 * IPT_PARK + k] = w.z;
                        dq[6 * IPT_PARK + k] = ldist; dq[7 * IPT_PARK + k] = contrib; dq[8 * IPT_PARK + k] = __uint_as_float(tag & C.slot_mask);
                    }
                    qn += __popc(pb);
                    __syncwarp();
                    if (qn >= 32) {
                        qn -= 32;
                        resolve_parked<SMALLPT, SPEC, X>(S, C, dq, qn + lane, tc, n_light, n_surface);
                        __syncwarp();
                    }
                }
                continue;
            }
            // warp-aggregated append (see k_extend)
            uint32_t ballot = __ballot_sync(0xffffffffu, emit);
            if (ballot) {
                uint32_t basepos = 0;
                if (lane == 0) basepos = atomicAdd(out_count, (uint32_t)__popc(ballot));
                basepos = __shfl_sync(0xffffffffu, basepos, 0);
                if (emit) {
                    uint32_t j = basepos + __popc(ballot & ((1u << lane) - 1u));
                    uint32_t ctag = (tag & C.slot_mask) | (C.slot_bits == 32 ? 0u : (child << C.slot_bits));
                    if (IPT_BOUNDS_OK(j, C.ray_cap, C.stats)) {
                        C.ray_o[j] = make_float4(pos.x, pos.y, pos.z, wgt);
                        C.ray_d[j] = make_float4(w.x, w.y, w.z, __uint_as_float(ctag));
                        C.ray_x[j] = child_sv;
                    }
                }
            }
        }
    }
    if (FUSE == FUSE_LAST && lane < qn) { // drain
        if (has_light_bvh<SPEC>(S)) last_parked<SMALLPT, X>(S, C, dq, lane, tc, n_light, n_surface, n_dropped);
        else resolve_parked<SMALLPT, SPEC, X>(S, C, dq, lane, tc, n_light, n_surface);
    }
    if (FUSE == FUSE_NEXT && qn) extend_parked<SMALLPT, SPEC, X>(S, C, dq, lane, lane < qn, depth + 1, tc, ec); // drain (warp-uniform qn)
    if (TWO_Q && qn2) extend_parked<SMALLPT, SPEC, X, false>(S, C, dq2, lane, lane < qn2, depth + 1, tc, ec);
    n_light += ec.light; n_surface += ec.surface; n_dropped += ec.dropped;
    flush_stat(C.stats, ST_FAILED, n_failed);
    flush_stat(C.stats, ST_PRUNED, n_pruned);
    flush_stat(C.stats, ST_DROPPED, n_dropped);
    if (FUSE != FUSE_NONE) {
        flush_stat(C.stats, ST_LIGHT, n_light);
        flush_stat(C.stats, ST_SURFACE, n_surface);
        flush_stat(C.stats, ST_MISS, ec.miss);
        flush_stat(C.stats, ST_LIGHTS, tc.lights);
        flush_stat(C.stats, ST_LIGHT_NODES, tc.light_nodes);
        // rays of depth+1 that were traced without being queued: k_accumulate folds cnt[] into the per-depth ray counts
        for (int off = 16; off > 0; off >>= 1) n_fused += __shfl_down_sync(0xffffffffu, n_fused, off);
        if (lane == 0 && n_fused) {
            atomicAdd(out_count, n_fused);
            atomicAdd(&C.stats[ST_FUSED], (unsigned long long)n_fused);
        }
    }
}

// accumulator cell of a sample: GridRenderPlane::addRay (src/GridRenderPlane.cpp:66-67), Gui::addRay (gui.cpp:168-172)
__device__ __forceinline__ uint32_t plane_cell(const RenderCtx& C, float x, float y, uint32_t ix, uint32_t iy) {
    if (C.plane_mode == IPT_PLANE_LINEAR) return iy * C.width + ix;
    float W = (float)C.width, H = (float)C.height;
    int xi = (int)xmul(x, W); // size_t xi = x*width (truncation)
    int yi;
    if (C.plane_mode == IPT_PLANE_GRID) yi = (int)xsub(xsub(H, xmul(y, H)), 1.0f); // height - y*height - 1; (-1,0) truncates to 0
    else yi = (int)xsub(H, xmul(y, H));
    xi = min(max(xi, 0), (int)C.width - 1); // the reference would write out of bounds; unreachable for x,y in [0,1)
    yi = min(max(yi, 0), (int)C.height - 1);
    return (uint32_t)yi * C.width + (uint32_t)xi;
}

// K6 accumulate: one thread per path; RenderPlane::addRay for the path's value (main.cpp:213-216).
__global__ void __launch_bounds__(256) k_accumulate(const __grid_constant__ RenderCtx C) {
    uint32_t stride = gridDim.x * blockDim.x;
    uint32_t dropped = 0;
    for (uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x; slot < C.batch; slot += stride) {
        float v = C.pathval[slot];
        if (!isfinite(v)) { v = 0.0f; ++dropped; }
        v = v >= 0.0f ? v : 0.0f;
        uint32_t ix, iy, pass;
        slot_to_pixel(C, slot, ix, iy, pass);
        float x, y;
        jitter_xy(C, ix, iy, pass, x, y);
        uint32_t cell = plane_cell(C, x, y, ix, iy);
        atomicAdd(&C.sum[cell], v);
        atomicAdd(&C.sumsq[cell], v * v);
        atomicAdd(&C.count[cell], 1u);
    }
    flush_stat(C.stats, ST_DROPPED, dropped);
    // fold this batch's per-depth ray counts into the running statistics
    if (blockIdx.x == 0 && threadIdx.x < IPT_MAX_DEPTH) {
        uint32_t r = C.cnt[2 * threadIdx.x], h = C.cnt[2 * threadIdx.x + 1];
        if (r) atomicAdd(&C.stats[ST_RAYS_AT_DEPTH + threadIdx.x], (unsigned long long)r);
        if (h) atomicAdd(&C.stats[ST_QUEUED], (unsigned long long)h);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&C.stats[ST_PATHS], (unsigned long long)C.batch);
}

} // namespace iptd
