/*
 * ipt_b200.h — C ABI of the B200-native trace loop for dimalit/ipt.
 *
 * Everything the reference's hot path (`render_sample` -> `ray_power_recursive`, src/main.cpp:98-223)
 * consumes arrives through the abstract interfaces of src/tracer_interfaces.h:26-54. Those virtuals
 * cannot run on a GPU and the reference's concrete classes hide their data (SURVEY.md S12), so this
 * boundary takes the same information as plain C structs ("scene description") and returns what
 * `RenderPlane::addRay` would have accumulated. Plain pointers and sizes only; no C++ or torch types.
 *
 * Each entry point names the reference interface it replaces (file:line relative to the reference
 * repository root). The C++ host classes that derive from the reference's interfaces and marshal to
 * this ABI are in ipt_b200/host/; INTEGRATION.md shows the binding a maintainer of ipt would add.
 *
 * All functions return IPT_OK (0) or an error code; ipt_last_error() gives the message of the last
 * failure on the calling thread. No function ever falls back to a CPU path: without a CUDA device
 * every compute entry point returns IPT_ERR_NO_DEVICE.
 */
#ifndef IPT_B200_H
#define IPT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IPT_B200_ABI_VERSION 3
#define IPT_MAX_DEPTH 16
/* The random numbers of a render: Philox4x32 (Salmon et al. 2011) with IPT_PHILOX_ROUNDS rounds, key = seed, counter =
 * (loop pixel, pass, node index within its tree level, depth); the four 32-bit outputs become uniforms in [0,1) with
 * IPT_U01_BITS bits: (x >> (32 - bits)) * 2^-bits. Shared by the device code and the CPU oracle so that both draw the
 * same numbers. */
#ifndef IPT_PHILOX_ROUNDS
#define IPT_PHILOX_ROUNDS 7 /* Philox4x32-7: the smallest round count that passes BigCrush (Salmon et al., table 2); -10 costs 3 % */
#endif
#ifndef IPT_U01_BITS
#define IPT_U01_BITS 23
#endif
#define IPT_NO_HIT 0xFFFFFFFFu

enum ipt_status {
    IPT_OK = 0,
    IPT_ERR_INVALID = 1,     /* bad argument / inconsistent description */
    IPT_ERR_CUDA = 2,        /* a CUDA runtime call failed */
    IPT_ERR_NO_DEVICE = 3,   /* no CUDA device: there is no CPU fallback */
    IPT_ERR_UNSUPPORTED = 4, /* feature outside the hot path */
    IPT_ERR_OVERFLOW = 5     /* a queue capacity was exceeded */
};

/* ---- scene description (host memory, copied by ipt_scene_create) ------------------------------- */

/* Analytic primitives. The list is ORDERED: like every reference Geometry::traceRay, primitives are
 * tested in list order and a later one wins only if strictly nearer (GeometrySphereInBox.cpp:23-36). */
enum ipt_prim_kind {
    IPT_PRIM_BOX_PLANE = 0,     /* intersection_with_box_plane, src/geometry/geometric_utils.cpp:8-26 */
    IPT_PRIM_SPHERE = 1,        /* intersection_with_sphere,    src/geometry/geometric_utils.cpp:28-55 */
    IPT_PRIM_SPHERE_SMALLPT = 2 /* Sphere::intersect (double),  src/geometry/GeometrySmallPt.cpp:17-22 */
};

/* Surface DDF ("sdf") a geometry attaches to a hit (tracer_interfaces.h:16-20). */
enum ipt_ddf_kind {
    IPT_DDF_COSINE = 0, /* RotateDdf(CosineDdf, normal): ddf.cpp:91-108, ddf_detail.h:72-85 */
    IPT_DDF_GLOSSY = 1  /* extension (BASELINE configs[1]): kd*Lambert + ks*PowerCosine(exponent) about reflect(d,n) */
};

typedef struct ipt_material {
    uint32_t ddf;   /* ipt_ddf_kind */
    float albedo;   /* surface_intersection::albedo, tracer_interfaces.h:19 */
    float kd, ks;   /* IPT_DDF_GLOSSY mixture weights (normalised by kd+ks) */
    float exponent; /* IPT_DDF_GLOSSY lobe exponent */
} ipt_material;

typedef struct ipt_prim {
    uint32_t kind;        /* ipt_prim_kind */
    uint32_t material;    /* index into ipt_scene_desc::materials */
    float p[3];           /* plane: the axis-aligned unit `plane` vector (surface normal is -p); sphere: centre */
    float radius;         /* spheres */
    uint32_t flip_normal; /* sphere: inward normal (GeometrySmallPt.cpp:53) */
    float curvature;      /* surface_intersection::curvature, reported only */
} ipt_prim;

enum ipt_light_kind {
    IPT_LIGHT_AREA_DIAMOND = 0,    /* AreaLight TYPE_DIAMOND,  src/lighting/lighting.cpp:79-144 */
    IPT_LIGHT_AREA_TRIANGLE = 1,   /* AreaLight TYPE_TRIANLE */
    IPT_LIGHT_SPHERE = 2,          /* SphereLight,             src/lighting/lighting.cpp:158-190 */
    IPT_LIGHT_SPHERE_INVERTED = 3, /* InvertedSphereLight,     src/lighting/lighting.h:58-73 */
    IPT_LIGHT_POINT = 4            /* PointLight (never hit),  src/lighting/lighting.h:33-44 */
};

typedef struct ipt_light {
    uint32_t kind;     /* ipt_light_kind */
    float position[3]; /* Light::position (area light: corner) */
    float x_axis[3];   /* area lights */
    float y_axis[3];
    float radius;      /* sphere lights */
    float power;       /* Light::power */
} ipt_light;

/* SimpleCamera's public fields (src/SimpleCamera.h:11-13); `direction` is NOT normalised. */
typedef struct ipt_camera {
    float position[3];
    float direction[3];
    float right[3];
    float up[3];
} ipt_camera;

typedef struct ipt_scene_desc {
    uint32_t n_prims;
    const ipt_prim* prims;
    uint32_t n_materials;
    const ipt_material* materials;
    uint32_t n_lights;
    const ipt_light* lights; /* CollectionLighting::lights, src/CollectionLighting.h:11 */
    /* Triangle mesh (extension, BASELINE configs[2..3]): 9 floats per triangle = v0, e1, e2. Tested after
     * the analytic list with the arithmetic of AreaLight::traceRay TYPE_TRIANLE (lighting.cpp:107-144);
     * primitive id of triangle k is n_prims + k. */
    uint64_t n_triangles;
    const float* triangles;
    uint32_t triangle_material;
    ipt_camera camera;
} ipt_scene_desc;

/* ---- render parameters --------------------------------------------------------------------------- */

/* How a sample at (x,y) in [0,1)^2 is mapped to an accumulator cell. */
enum ipt_plane_mode {
    IPT_PLANE_GRID = 0,  /* GridRenderPlane::addRay: xi=x*W, yi=H-y*H-1   (src/GridRenderPlane.cpp:66-67) */
    IPT_PLANE_GUI = 1,   /* Gui::addRay:             xi=x*W, yi=H-y*H, clamped (src/gui.cpp:168-172) */
    IPT_PLANE_LINEAR = 2 /* the loop pixel (ix,iy) itself */
};

enum ipt_render_flags {
    IPT_FLAG_TIME_KERNELS = 1u, /* bracket every kernel with CUDA events on the render stream -> ipt_render_stats::ms_* */
    IPT_FLAG_KEEP_ZERO_WEIGHT = 2u, /* trace children whose weight is exactly 0 (the reference does, main.cpp:177) */
    IPT_FLAG_DEBUG_PRINT = 4u,      /* device printf of every ray / sample (single-path debugging); only in a library built with
                                     * -DIPT_DEBUG_PRINT, else IPT_ERR_UNSUPPORTED: the production kernels carry no printf */
    /* At the last traced depth a ray only matters if it reaches a light, so by default the geometry is intersected
     * only for rays that hit a light ("shadow ray"); with this flag every last-level ray is resolved into
     * surface hit / miss as well, which only affects ipt_render_stats::surface_hits / misses. */
    IPT_FLAG_RESOLVE_LAST_LEVEL = 8u,
    /* Analytic scenes resolve the last traced depth inside the shade kernel that spawns it (the rays of the widest
     * tree level are never queued). This flag keeps them on the queue + k_extend<LAST> path; results are the same up to
     * the order of the float atomics. */
    IPT_FLAG_NO_FUSED_LAST_LEVEL = 16u,
    /* Analytic scenes: the shade kernel of every depth traces the children it spawns (no ray queue, no extend launch
     * after depth 0). This flag puts the children of all but the last shading level back on the ray queue +
     * k_extend path (IPT_FLAG_NO_FUSED_LAST_LEVEL implies it). Same results up to the order of the float atomics. */
    IPT_FLAG_NO_FUSED_TRACE = 32u
};

typedef struct ipt_render_params {
    uint32_t width, height;            /* frame the jitter/camera loop runs over (reference: 640x640, main.cpp:189-193) */
    uint32_t depth_max;                /* main.cpp:95; rays exist at depths 0..depth_max-1 */
    uint32_t schedule[IPT_MAX_DEPTH];  /* children spawned by a surface hit at depth d (reference: 16,8,4,2: main.cpp:94,177) */
    uint64_t seed;                     /* Philox key */
    uint32_t pass_begin, pass_count;   /* passes == calls of render_sample; Philox counters make them disjoint */
    uint32_t tile_x0, tile_y0, tile_w, tile_h; /* loop-pixel rectangle; tile_w==0 means the full frame */
    uint32_t plane_mode;               /* ipt_plane_mode */
    uint32_t flags;                    /* ipt_render_flags */
    uint32_t batch_paths;              /* paths per wavefront batch; 0 = library default */
} ipt_render_params;

typedef struct ipt_render_stats {
    uint64_t paths;                    /* camera samples == addRay calls (SURVEY.md §8d) */
    uint64_t rays;                     /* traced segments (Geometry::traceRay + Lighting::traceRayToLight pairs) */
    uint64_t rays_at_depth[IPT_MAX_DEPTH];
    uint64_t surface_hits, light_hits, misses; /* last-level rays without a light along them are in neither (see flags) */
    uint64_t failed_samples;           /* zero-vector samples (lighting.cpp:55-56); still in the 1/n divisor */
    uint64_t zero_weight_pruned;       /* children with weight exactly 0 that were not traced */
    uint64_t nonfinite_dropped;        /* non-finite weights/values dropped (main.cpp:175,181,215) */
    uint64_t bvh_nodes_visited, triangles_tested; /* mesh LBVH (device counters) */
    uint64_t lights_tested;            /* Light::traceRay evaluations of traced rays (device counter, any light container) */
    uint64_t light_bvh_nodes_visited;  /* node visits of the light LBVH (many-light scenes; device counter) */
    uint32_t batches;
    uint32_t kernel_launches;          /* kernels of this library launched by the call */
    float ms_total;                    /* device time of the whole call (CUDA events) */
    float ms_generate, ms_extend, ms_shade, ms_accumulate; /* with IPT_FLAG_TIME_KERNELS */
    uint32_t n_extend, n_shade;        /* launches summed into ms_extend / ms_shade */
    uint64_t queue_bytes;              /* queue traffic of the wavefront MODEL (SURVEY.md 8d): 72 B per ray (36 B record written
                                        * + read), 64 B per queued surface hit, 8 B per path */
    uint64_t rays_resolved_in_shade;   /* rays of the last traced depth that the fused shade kernel resolved without queueing
                                        * them: the implementation moves queue_bytes - 72 * this */
} ipt_render_stats;

typedef struct ipt_scene ipt_scene; /* opaque: device copy of the scene (+ LBVH) */
typedef struct ipt_plane ipt_plane; /* opaque: device accumulators sum / sumsq / count */

/* ---- library ------------------------------------------------------------------------------------- */
int ipt_abi_version(void);
const char* ipt_last_error(void);
int ipt_device_count(void);

/* ---- scenes: replaces constructing Geometry/Lighting/Camera objects (sample_scenes.cpp:20-108) ---- */
int ipt_scene_create(const ipt_scene_desc* desc, int device, ipt_scene** out);
int ipt_scene_destroy(ipt_scene* scene);
/* SimpleCamera can be orbited by the caller (gui.cpp:107-137): replace the camera without a rebuild. */
int ipt_scene_set_camera(ipt_scene* scene, const ipt_camera* camera);
/* Which kernel instantiations ipt_scene_create chose for the scene (read-only; renders do not depend on it):
 *   out[0] spec of the fused shade kernels: 0 FEW_LIGHTS (no light LBVH; the lights are scanned from global memory),
 *          1 LIGHT_BVH (more than 8 lights, all of them area lights), 2 RUNTIME (SmallPt scenes: decided per call),
 *          3 ONE_LIGHT (one light, not an area light), 4 ONE_AREA_LIGHT (one area light), 5 BOX_SCENE (... and the
 *          geometry is grouped box planes + inline spheres), 6 LAMBERT_BOX (... and every material is the cosine DDF)
 *   out[1] SmallPt spheres present, out[2] triangle mesh present: together they select k_extend<smallpt, mesh>
 *   out[3] mesh scene traced by the box-scene mesh kernel (k_extend_mesh<., BOX_SCENE>) instead of the generic one
 *   out[4] shadow rays skip the box walls (every sphere inside the box, every area-light corner 1e-3 from the walls)
 *   out[5] the lights are held in kernel parameters (a single light)
 *   out[6] number of lights in the light LBVH (0: none) */
#define IPT_DISPATCH_WORDS 7
int ipt_scene_dispatch(ipt_scene* scene, uint32_t out[IPT_DISPATCH_WORDS]);

/* Moving a mesh or the lights without recreating the scene (its stream, workspace and planes stay). */
enum ipt_update_flags {
    IPT_UPDATE_DEVICE_POINTER = 1u, /* the input is device memory on the scene's device (e.g. a CUDA tensor) */
    IPT_UPDATE_REBUILD = 2u         /* full LBVH build over the new vertices or lights; default: refit the existing tree */
};
/* Replace the vertices of the scene's triangle mesh (9 floats per triangle, v0 e1 e2, as in ipt_scene_desc).
 * n_triangles must equal the scene's count; a different count needs a new scene. Lights are not moved.
 *   Result: afterwards every result (traces, renders, ipt_scene_dispatch) equals that of a scene created from the new
 *     triangles. The exception is the tree itself after a refit: it keeps the topology, Morton keys and sorted order of
 *     its last build and only recomputes every box, so its node boxes differ, and so do the node-visit counters of renders
 *     (bvh_nodes_visited, triangles_tested). A refit is cheap; the tree's quality degrades as the mesh moves away from the
 *     pose it was built in, and IPT_UPDATE_REBUILD restores it.
 *   Synchronisation: takes the scene's mutex and runs on the scene's stream, after the work already enqueued there. It
 *     returns once the update is complete: the caller may then free or overwrite its buffer. With
 *     IPT_UPDATE_DEVICE_POINTER the caller must have finished writing the buffer on its own stream before the call; the
 *     library waits on no other stream.
 *   Planes made on the scene stay valid, and their accumulators are not touched: clearing them is the caller's decision,
 *     as after ipt_scene_set_camera.
 *   Errors (IPT_ERR_INVALID): a null argument, unknown flag bits, a scene without a mesh, a count that differs from the
 *     scene's, and a pointer whose kind does not match the flag (by cudaPointerGetAttributes: with
 *     IPT_UPDATE_DEVICE_POINTER it must be device or managed memory on the scene's device, without it it must not be
 *     device memory), or that is not aligned to a float.
 *   Atomicity: if an allocation fails (IPT_ERR_CUDA), the scene keeps its previous triangles and tree.
 *   Per-triangle materials set by ipt_scene_set_triangle_materials stay with their triangles, after a refit and a rebuild. */
int ipt_scene_update_triangles(ipt_scene* scene, const float* triangles, uint64_t n_triangles, uint32_t flags);

/* Give each triangle of the scene's mesh its own material. materials[k] indexes the material list the scene was created
 * with, for triangle k in the order of ipt_scene_desc::triangles (the triangle whose primitive id is n_prims + k).
 * n_triangles must equal the scene's count.
 *   Flags: only IPT_UPDATE_DEVICE_POINTER: `materials` is then device or managed memory on the scene's device (e.g. a CUDA
 *     tensor of int32 or uint32).
 *   Result: afterwards every render and ipt_mix_sample equals what a scene whose triangle k has material materials[k] would
 *     give. ipt_trace_batch, ipt_preview_batch, ipt_bvh_export* and ipt_scene_dispatch do not change. Until the first call,
 *     every triangle has ipt_scene_desc::triangle_material.
 *   Persistence: a material belongs to its original triangle index and is kept through ipt_scene_update_triangles, refit
 *     and rebuild alike. A later call replaces the whole array.
 *   Synchronisation: as ipt_scene_update_triangles: takes the scene's mutex, runs on the scene's stream after the work
 *     already enqueued there and returns once the call is complete. With IPT_UPDATE_DEVICE_POINTER the caller must have
 *     finished writing the buffer on its own stream before the call.
 *   Planes made on the scene stay valid, and their accumulators are not touched.
 *   Errors (IPT_ERR_INVALID): a null argument, unknown flag bits, a scene without a mesh, a count that differs from the
 *     scene's, a pointer whose kind does not match the flag (as for ipt_scene_update_triangles) or that is not 4-byte
 *     aligned, and any index >= the scene's n_materials (device input is checked on the device before anything changes).
 *   Atomicity: on any error, including a failed allocation (IPT_ERR_CUDA), the scene keeps the materials it had. */
int ipt_scene_set_triangle_materials(ipt_scene* scene, const uint32_t* materials, uint64_t n_triangles, uint32_t flags);

/* Move and re-power the scene's lights without recreating the scene: each light's position, axes, radius and power may
 * change. n_lights must equal the scene's count, and lights[i].kind the kind of the scene's light i: count and kinds decide
 * the kernels ipt_scene_create chose, so a change of either needs a new scene.
 *   Flags: IPT_UPDATE_DEVICE_POINTER: `lights` is device or managed memory on the scene's device (e.g. a CUDA tensor of
 *     48-byte ipt_light records). IPT_UPDATE_REBUILD: build the light LBVH anew; by default the existing tree is refitted.
 *     A scene without a light LBVH accepts IPT_UPDATE_REBUILD and has nothing to rebuild.
 *   Result: afterwards every result (traces, ipt_light_ddf_*, ipt_mix_sample, renders, ipt_scene_dispatch) equals that of
 *     a scene created from the same description with the new lights; after a rebuild bit for bit. A refit keeps the light
 *     tree's topology and sorted order and only recomputes every box and record, so two things may differ from a fresh
 *     scene: the light tree's traversal counters of renders (light_bvh_nodes_visited, and lights_tested, which counts the
 *     tree's leaves reached), and the order in which the all-hits mixture density is summed over the lights a
 *     direction crosses, so the density (ipt_light_ddf_value, the mixture value of ipt_mix_sample, the child weights of a
 *     render) may differ in the last bits where a direction crosses more than one light. The nearest light is exact (ties
 *     go to the lower original index). Of ipt_scene_dispatch only out[4] (lights_inside_box) can change.
 *   Synchronisation: as ipt_scene_update_triangles: takes the scene's mutex, runs on the scene's stream after the work
 *     already enqueued there and returns once the update is complete. With IPT_UPDATE_DEVICE_POINTER the caller must have
 *     finished writing the buffer on its own stream before the call.
 *   Planes made on the scene stay valid, and their accumulators are not touched. The mesh and per-triangle materials are
 *     not touched.
 *   Errors (IPT_ERR_INVALID): a null argument, unknown flag bits, a count that differs from the scene's, a kind that
 *     differs from the scene's (the message names the first such index; device input is checked on the device before
 *     anything changes), and a pointer whose kind does not match the flag (as for ipt_scene_update_triangles) or that is
 *     not 4-byte aligned. Values are not range-checked, as ipt_scene_create does not check them.
 *   Atomicity: on any error, including a failed allocation (IPT_ERR_CUDA), the scene keeps the lights, tables and light
 *     tree it had. */
int ipt_scene_update_lights(ipt_scene* scene, const ipt_light* lights, uint32_t n_lights, uint32_t flags);

/* The reference's five scenes + this repo's benchmark scenes as descriptions:
 * "box" (make_scene_box, the default), "fractal", "smallpt", "square", "corner", "openspheres", "cornell" (C2),
 * "mixedlights" (one of every Light class over the default geometry),
 * "lightgrid:<rows>x<cols>" (C5), "mesh:<n>" (C3/C4: `n` generated triangles inside the C1 box).
 * The returned description and its arrays are owned by the library until ipt_scene_desc_free. */
int ipt_sample_scene(const char* name, ipt_scene_desc** out);
int ipt_scene_desc_free(ipt_scene_desc* desc);
/* What the Light constructors derive (AreaLight::AreaLight lighting.cpp:79-90, SphereLight lighting.h:46-53):
 * Light::area, power/area, and for area lights normalize(cross(x,y)). Host arithmetic in glm operation order. */
int ipt_light_derived(const ipt_light* light, float* area, float* surface_power, float normal[3]);
/* SimpleCamera::SimpleCamera (src/SimpleCamera.cpp:8-13) */
/* The arrow keys of Gui::work (src/gui.cpp:105-134): LEFT/RIGHT orbit position and direction about the z axis by
 * -/+ pi/12, DOWN/UP scale the position by 1.1 / (1/1.1); right and up are re-derived with the up hint (0,0,1).
 * Host arithmetic in glm's operation order: bit-exact. */
enum { IPT_KEY_LEFT = 0, IPT_KEY_RIGHT = 1, IPT_KEY_DOWN = 2, IPT_KEY_UP = 3 };
int ipt_camera_orbit(ipt_camera* camera, int key);
int ipt_camera_look(const float position[3], const float direction[3], const float up_hint[3], ipt_camera* out);

/* ---- parity entry: Geometry::traceRay + Lighting::traceRayToLight + the light-vs-surface decision ---
 * (tracer_interfaces.h:28,35; main.cpp:107-128) for n rays given as xyz triples in HOST memory.
 * Outputs (host, any may be NULL): prim_id (IPT_NO_HIT on miss), t (+inf on miss), light_id, light_pos
 * (xyz of light_intersection::position), outcome: 0 miss, 1 surface, 2 light. */
int ipt_trace_batch(ipt_scene* scene, const float* origins, const float* directions, size_t n, uint32_t* prim_id,
                    float* t, uint32_t* light_id, float* light_pos, uint32_t* outcome);

/* ray_power_preview (src/main.cpp:55-92), the reference's alternative `ray_power` (main.cpp:53): 1 if a light is
 * reached first, 0 on a miss, else dot(normal, -direction) / length(direction) at the first surface hit. n rays in
 * HOST memory, one float each out. Deterministic, so it is compared bit for bit. */
int ipt_preview_batch(ipt_scene* scene, const float* origins, const float* directions, size_t n, float* value);

/* Camera::sampleRay (tracer_interfaces.h:42) for n (x,y) pairs. */
int ipt_camera_rays(ipt_scene* scene, const float* xy, size_t n, float* origins, float* directions);

/* DDF parity entries (Ddf::sample / Ddf::value, src/libddf/ddf.h:14-17), evaluated ON THE DEVICE.
 * `kind`: 0 Spherical, 1 UpperHalf, 2 Cosine, >=3 PowerCosine(kind); `to` (may be NULL) rotates it.
 * Samples use Philox stream (seed, index). */
int ipt_ddf_value(ipt_scene* scene, int kind, const float* to, const float* dirs, size_t n, float* out);
int ipt_ddf_sample(ipt_scene* scene, int kind, const float* to, uint64_t seed, size_t n, float* dirs);
/* The mixture of main.cpp:142-143 at the surface hit of ray (o,d): n samples with mixture and sdf values. */
int ipt_mix_sample(ipt_scene* scene, const float origin[3], const float direction[3], uint64_t seed, size_t n,
                   float* dirs, float* mix_value, float* sdf_value);
/* Lighting::distributionInPoint(pos)->value(dir) (CollectionLighting.cpp:12-21, lighting.cpp:61-73). */
int ipt_light_ddf_value(ipt_scene* scene, const float pos[3], const float* dirs, size_t n, float* out);
/* Lighting::distributionInPoint(pos)->sample(): n directions (zero vector = failed sample), Philox stream (seed, index). */
int ipt_light_ddf_sample(ipt_scene* scene, const float pos[3], uint64_t seed, size_t n, float* dirs);

/* randf (include/randf.h:6-11) on the device: the render's random stream. For each of n counters (4 x uint32: loop pixel,
 * pass, node, depth) the Philox4x32-IPT_PHILOX_ROUNDS block keyed by `seed` (4 x uint32) and its four uniforms
 * (4 x float, see IPT_U01_BITS). HOST arrays; either output may be NULL. */
int ipt_philox_batch(int device, const uint32_t* counters, size_t n, uint64_t seed, uint32_t* blocks, float* uniforms);

/* LBVH over the triangle mesh, as built on the device: n_triangles-1 internal nodes of 64 bytes (root = 0), each
 * holding BOTH children's boxes; the sorted primitive order; the sorted 63-bit Morton keys. */
typedef struct ipt_bvh_node {
    float lo0[3];
    uint32_t left;   /* child index; bit31 set = leaf (low bits: sorted position) */
    float hi0[3];
    uint32_t right;
    float lo1[3];
    uint32_t parent; /* IPT_NO_HIT for the root */
    float hi1[3];
    uint32_t pad;
} ipt_bvh_node;
int ipt_bvh_export(ipt_scene* scene, ipt_bvh_node* nodes, uint32_t* sorted_prims, uint64_t* morton, uint64_t* n_nodes);
/* The same tree in the form the traversal kernels read: 32 bytes per node = both children's boxes on a 16-bit grid over
 * the root box (rounded outwards by one extra cell: conservative) + the two child ids. 8 uint32 per node:
 * lo0.x|lo0.y<<16, lo0.z|hi0.x<<16, hi0.y|hi0.z<<16, lo1.x|lo1.y<<16, lo1.z|hi1.x<<16, hi1.y|hi1.z<<16, left, right.
 * grid[0..2] = lower corner of the root box, grid[3..5] = (1 - 2^-13) / extent: a world coordinate x sits at grid
 * coordinate (x - lo) * scale * 65536 + 4. Integer work + three float steps: byte-identical to the CPU restatement. */
int ipt_bvh_export_compact(ipt_scene* scene, uint32_t* nodes32, float grid[6], uint64_t* n_nodes);

/* The scene's light tables as the render kernels read them, for the scene's n_lights lights in description order: Light::area,
 * power / area (NaN for point lights), the normal of an area light (3 floats per light, zero for the other kinds), the
 * weight of the light in the mixture of main.cpp:142-143 (CollectionLighting.cpp:12-21 weights, halved) and the running
 * float sum of those weights (cdf); and the light-selection guide: guide[b] = the first i with b / 4096 < cdf[i]
 * (n_lights if none), b = 0 .. IPT_LIGHT_GUIDE_WORDS - 1. HOST arrays; any output may be NULL. */
#define IPT_LIGHT_GUIDE_WORDS 4098
int ipt_light_tables_export(ipt_scene* scene, float* area, float* surface_power, float* normal, float* weight, float* cdf,
                            uint32_t guide[IPT_LIGHT_GUIDE_WORDS]);

/* ---- render plane: replaces RenderPlane::addRay accumulation (tracer_interfaces.h:51-54) --------- */
int ipt_plane_create(ipt_scene* scene, uint32_t width, uint32_t height, ipt_plane** out);
/* Accumulate into caller-owned DEVICE arrays (e.g. torch tensors that NCCL will all-reduce). */
int ipt_plane_wrap(ipt_scene* scene, uint32_t width, uint32_t height, float* d_sum, float* d_sumsq, uint32_t* d_count,
                   ipt_plane** out);
int ipt_plane_clear(ipt_plane* plane);
/* RenderPlane::addRay itself (tracer_interfaces.h:53) for n samples given in HOST memory: cell mapping per plane_mode. */
int ipt_plane_add_rays(ipt_plane* plane, uint32_t plane_mode, size_t n, const float* x, const float* y, const float* value);
int ipt_plane_destroy(ipt_plane* plane);
int ipt_plane_download(ipt_plane* plane, float* sum, float* sumsq, uint32_t* count);     /* device -> host */
int ipt_plane_upload(ipt_plane* plane, const float* sum, const float* sumsq, const uint32_t* count); /* resume */
int ipt_plane_device_ptrs(ipt_plane* plane, float** d_sum, float** d_sumsq, uint32_t** d_count);
/* The path's ONLY collective: element-wise sum of sum / sumsq / count over all ranks of an NCCL communicator (one
 * process or thread per GPU, each rendering its own pass range; replaces the mutex-guarded running mean that merges the
 * reference's four threads, src/gui.cpp:165-182). `nccl_comm` is an ncclComm_t owned by the host application. The
 * library links against no NCCL: it resolves ncclAllReduce from the NCCL already loaded in the process (libnccl.so.2).
 * One grouped launch (ncclGroupStart/End): the two float arrays as one message when they are contiguous (they are in a
 * plane made by ipt_plane_create: one packed block sum | sumsq | count), then the counters. */
int ipt_plane_allreduce(ipt_plane* plane, void* nccl_comm, float* ms /* device time of the collective, may be NULL */);
/* dst += src, element-wise over sum / sumsq / count. The two planes may belong to scenes on DIFFERENT devices of this
 * process (src is fetched with a peer copy over NVLink, or staged by the driver where peer access is unavailable): how a
 * single-process, one-thread-per-GPU host (the shape of the reference's own driver, src/main.cpp:258-277) merges its
 * per-GPU pass ranges without NCCL. Same frame size required; src is left unchanged. */
int ipt_plane_merge(ipt_plane* dst, ipt_plane* src);
/* GridRenderPlane state after the same samples: pixels = sum/count, pixel_counters, max_value (GridRenderPlane.h:9-12). */
int ipt_plane_resolve(ipt_plane* plane, float* pixels, uint64_t* pixel_counters, float* max_value);

/* ---- the output stage: what Gui does with the accumulated image (src/gui.cpp) -------------------------
 * All of it runs on the device; there is no CPU fallback (IPT_ERR_NO_DEVICE without a GPU). Images are row-major
 * float32, `width*height` values, as CImg<float> stores them. */
/* glare(image, cutoff), src/gui.cpp:38-52 with draw_halo :28-36 — the filter Gui::updateDisplay applies (:84): every
 * pixel brighter than `cutoff` adds the halo 0.1*val/(0.25+r)^2 to every pixel; the sum is cut to [0, cutoff].
 * Bit-exact. `n_bright` (may be NULL) receives the number of halo sources. */
int ipt_image_glare(int device, const float* image, uint32_t width, uint32_t height, float cutoff, float* out, uint32_t* n_bright);
/* normalize(image), src/gui.cpp:11-16: (image/max)^(1/2.2) cut to [0,1]. Within 1 ulp of the reference's powf. */
int ipt_image_normalize(int device, const float* image, uint32_t width, uint32_t height, float* out);
/* The pixel bytes of Gui::save (src/gui.cpp:192-194): normalize(image).normalize(0,255) truncated to 8 bits (CImg
 * without libpng saves through an 8-bit PGM, include/CImg.h:60650-60667,59204-59209). Bit-exact. */
int ipt_image_save_bytes(int device, const float* image, uint32_t width, uint32_t height, uint8_t* out);
/* The same on a plane's accumulators (image = sum/count), without leaving the device:
 * ipt_plane_display = what Gui::updateDisplay shows, normalize(glare(image, glare_cutoff)) (gui.cpp:83-87, no text overlay;
 * Gui's default cutoff is 1.01, gui.h:24); `ms` (may be NULL) receives the device time of the filter chain.
 * ipt_plane_save_bytes / ipt_plane_save_png = Gui::save. */
int ipt_plane_display(ipt_plane* plane, float glare_cutoff, float* out, float* ms);
int ipt_plane_save_bytes(ipt_plane* plane, uint8_t* out);
int ipt_plane_save_png(ipt_plane* plane, const char* path);
/* 8-bit greyscale PNG writer (host only; stored deflate blocks, no zlib dependency). */
int ipt_write_png_gray8(const char* path, const uint8_t* bytes, uint32_t width, uint32_t height);

/* ---- the hot path: replaces pass_count calls of render_sample (main.cpp:186-223) ------------------ */
int ipt_render(ipt_scene* scene, ipt_plane* plane, const ipt_render_params* params, ipt_render_stats* stats);
/* Same through HOST buffers: clears a plane, renders, copies sum/sumsq/count back (the end-to-end call). */
int ipt_render_host(ipt_scene* scene, const ipt_render_params* params, float* sum, float* sumsq, uint32_t* count,
                    ipt_render_stats* stats);
/* Fills params with the reference defaults: 640x640, depth 4, schedule 16/8/4/2, GRID plane. */
void ipt_render_params_default(ipt_render_params* params);

/* Deterministic synthetic mesh (C3/C4): n triangles, 9 floats each, from integer hashes of (seed, index). */
int ipt_generate_mesh(uint64_t n, uint64_t seed, float* triangles);

#ifdef __cplusplus
}
#endif
#endif /* IPT_B200_H */
