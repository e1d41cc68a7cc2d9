// ipt_capi.cu — the C ABI of include/ipt_b200.h: scene flattening, workspace management, the per-batch
// kernel sequence of the wavefront pipeline, and the parity entry points.
//
// The scene's light tables are derived on the device (k_light_derive and the kernels after it), for ipt_scene_create
// and ipt_scene_update_lights alike. Host-side float work (ipt_light_derived) follows the reference's constructors in glm
// operation order (ipt_b200/host/glm_order.hpp) so it gives the same bits.
#include "ipt_b200.h"

#include "../host/glm_order.hpp"
#include "ipt_lbvh.cuh"
#include "ipt_trace.cuh"

#include <dlfcn.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <type_traits>
#include <vector>

using namespace iptd;

#define IPT_LIGHT_BVH_MIN 8 // light sets larger than this get an LBVH
#define IPT_CNT_WORDS (3 * IPT_MAX_DEPTH + 2) // ray counts, hit counts, persistent-kernel fetch cursors

// ---------------------------------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------------------------------
static thread_local std::string g_last_error;
static int fail(int code, const std::string& msg) {
    g_last_error = msg;
    return code;
}
// the same for the entry points defined in host/sample_scenes.cpp
int ipt_host_fail(int code, const char* msg) { return fail(code, msg); }
#define CUDA_TRY(expr)                                                                                           \
    do {                                                                                                         \
        cudaError_t e__ = (expr);                                                                                \
        if (e__ != cudaSuccess)                                                                                  \
            return fail(IPT_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e__) + " (" __FILE__ ":" + \
                                          std::to_string(__LINE__) + ")");                                      \
    } while (0)

static bool check_eps_constants() {
    // ipt_device.cuh: (double)x < 1e-6  <=>  x <= (float)1e-6
    float f;
    uint32_t bits = IPT_EPS6_BITS;
    std::memcpy(&f, &bits, 4);
    return f == (float)1e-6 && (double)f < 1e-6 && (double)std::nextafterf(f, 1.0f) > 1e-6;
}

// ---------------------------------------------------------------------------------------------------
// opaque handles
// ---------------------------------------------------------------------------------------------------
struct Workspace {
    float4* ray_o = nullptr;
    float4* ray_d = nullptr;
    float* ray_x = nullptr;
    float4* hit_a = nullptr;
    uint4* hit_b = nullptr;
    float4* hit_a2 = nullptr; // second hit set, only when the shade kernels trace their own children
    uint4* hit_b2 = nullptr;
    float* pathval = nullptr;
    size_t ray_cap = 0, hit_cap = 0, path_cap = 0;
    bool two_hit_sets = false;
    // the batch the last render settled on for a (requested batch, queue widths, budget) combination: cudaMemGetInfo takes
    // milliseconds on a 180 GB device, so the free-memory clamp is only re-evaluated when the question changes
    uint64_t choice_key[5] = {0, 0, 0, 0, 0};
    uint64_t choice_batch = 0;
};

// grow-only device scratch of the output stage (ipt_output.cuh): cudaMalloc/cudaFree per call would cost more than the
// filters themselves
struct GrowBuf {
    void* p = nullptr;
    size_t cap = 0;
    ~GrowBuf() { cudaFree(p); }
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        cudaFree(p);
        p = nullptr; cap = 0;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e == cudaSuccess) cap = bytes;
        return e;
    }
    template <typename T> T* as() const { return static_cast<T*>(p); }
};
struct OutputScratch {
    GrowBuf mean, glare, shown, bytes, rows, bright, small;
};

// One kernel of ipt_render's depth loop (k_extend, k_extend_mesh or k_shade), the grid its own occupancy allows and its
// dynamic shared memory
struct RenderKernel {
    using Fn = void (*)(DevScene, RenderCtx, uint32_t);
    Fn kernel = nullptr;
    int grid = 0;
    size_t smem = 0;
};

struct ipt_scene {
    // The reference calls render_sample from four threads on one Scene (main.cpp:258-277). One scene owns one stream and
    // one workspace, so every entry point that touches them takes this lock: concurrent callers are serialised.
    std::recursive_mutex mu;
    int device = 0;
    cudaStream_t stream = nullptr;
    int sm_count = 0;
    DevScene dev{};
    DevPrim* d_prims = nullptr;
    DevLight* d_lights = nullptr;
    float* d_light_cdf = nullptr;
    uint32_t* d_light_guide = nullptr;
    float* d_light_samp = nullptr;
    DevMaterial* d_mats = nullptr;
    LbvhDevice bvh{};
    // per-triangle materials, null until ipt_scene_set_triangle_materials: the caller's array (by original triangle index)
    // and its gather into the tree's sorted order (DevScene::tri_mats), redone by every rebuild
    uint32_t* d_tri_mats_orig = nullptr;
    uint32_t* d_tri_mats = nullptr;
    LbvhDevice light_bvh{};
    bool smallpt = false, mesh = false;
    SceneSpec shade_spec = SPEC_RUNTIME; // k_shade<FUSE_NEXT / FUSE_LAST, ., shade_spec>
    SceneSpec mesh_spec = SPEC_RUNTIME;  // k_extend_mesh<., mesh_spec> (mesh scenes without SmallPt)
    // the kernels of ipt_render's depth loop, chosen once by ipt_scene_create; extend[last depth][exact arithmetic]
    RenderKernel extend[2][2], shade, shade_next, shade_last;
    Workspace ws;
    uint32_t* d_cnt = nullptr;
    unsigned long long* d_stats = nullptr;
    std::vector<cudaEvent_t> events;
    cudaEvent_t ev_begin = nullptr, ev_end = nullptr;
    ipt_plane* host_plane = nullptr; // for ipt_render_host
    float* pinned = nullptr;         // staging for ipt_render_host
    size_t pinned_bytes = 0;
    int grid_generate = 0, grid_accumulate = 0;
    OutputScratch out;
};

struct ipt_plane {
    ipt_scene* scene = nullptr;
    uint32_t width = 0, height = 0;
    float* sum = nullptr;
    float* sumsq = nullptr;
    uint32_t* count = nullptr;
    bool owned = false;
};

// ---------------------------------------------------------------------------------------------------
// parity / utility kernels
// ---------------------------------------------------------------------------------------------------
template <bool SMALLPT, bool MESH>
__global__ void __launch_bounds__(IPT_BLOCK) k_trace_batch(const __grid_constant__ DevScene S, const float* __restrict__ o,
                                                           const float* __restrict__ d, size_t n, uint32_t* prim, float* t,
                                                           uint32_t* light, float* lpos, uint32_t* outcome) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    TraceCounters tc{0, 0};
    Outcome oc = trace_scene<SMALLPT, MESH>(S, mk3(o[3 * i], o[3 * i + 1], o[3 * i + 2]), mk3(d[3 * i], d[3 * i + 1], d[3 * i + 2]), tc);
    if (prim) prim[i] = oc.surf.prim;
    if (t) t[i] = oc.surf.prim == IPT_NO_HIT ? IPT_INF : oc.surf.t;
    if (light) light[i] = oc.light;
    if (lpos) { lpos[3 * i] = oc.light_pos.x; lpos[3 * i + 1] = oc.light_pos.y; lpos[3 * i + 2] = oc.light_pos.z; }
    if (outcome) outcome[i] = oc.kind;
}

// ray_power_preview (src/main.cpp:55-92)
template <bool SMALLPT, bool MESH>
__global__ void __launch_bounds__(IPT_BLOCK) k_preview_batch(const __grid_constant__ DevScene S, const float* __restrict__ o, const float* __restrict__ d,
                                                             size_t n, float* value) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    TraceCounters tc{0, 0};
    f3 oo = mk3(o[3 * i], o[3 * i + 1], o[3 * i + 2]), dd = mk3(d[3 * i], d[3 * i + 1], d[3 * i + 2]);
    Outcome oc = trace_scene<SMALLPT, MESH>(S, oo, dd, tc);
    float v = 0.0f;
    if (oc.kind == 2) v = 1.0f;
    else if (oc.kind == 1) {
        f3 pos = xpoint(oo, dd, oc.surf.t), normal;
        uint32_t material;
        surface_frame(S, oc.surf.tri_pos != IPT_NO_HIT ? S.n_prims + oc.surf.tri_pos : oc.surf.prim, pos, normal, material);
        v = xdiv(xdot3(normal, neg3(dd)), xlength3(dd));
    }
    value[i] = v;
}

__global__ void k_camera_rays(const __grid_constant__ DevScene S, const float* __restrict__ xy, size_t n, float* o, float* d) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    f3 oo, dd;
    camera_ray(S.cam, xy[2 * i], xy[2 * i + 1], oo, dd);
    o[3 * i] = oo.x; o[3 * i + 1] = oo.y; o[3 * i + 2] = oo.z;
    d[3 * i] = dd.x; d[3 * i + 1] = dd.y; d[3 * i + 2] = dd.z;
}

__global__ void k_ddf_value(int kind, bool rotated, f3 to, const float* __restrict__ w, size_t n, float* out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    f3 a = mk3(w[3 * i], w[3 * i + 1], w[3 * i + 2]);
    out[i] = base_value(kind, rotated ? dot3(to, a) : a.z);
}
__global__ void k_ddf_sample(int kind, bool rotated, f3 to, uint32_t k0, uint32_t k1, size_t n, float* w) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint4 r = philox4x32_10((uint32_t)i, (uint32_t)(i >> 32), 0u, 0xDDF0u, k0, k1);
    f3 x = base_sample(kind, u01(r.y), u01(r.z));
    if (rotated) x = rotate(make_basis(to), x);
    w[3 * i] = x.x; w[3 * i + 1] = x.y; w[3 * i + 2] = x.z;
}
template <bool SMALLPT, bool MESH>
__global__ void __launch_bounds__(IPT_BLOCK) k_mix_sample(const __grid_constant__ DevScene S, f3 o, f3 d, uint32_t k0, uint32_t k1, size_t n,
                                                          float* w, float* mixv, float* sdfv, int* hit_flag) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    TraceCounters tc{0, 0};
    SurfHit sh = trace_geometry<SMALLPT, MESH>(S, o, d, tc);
    if (sh.prim == IPT_NO_HIT) { if (i == 0) *hit_flag = 0; return; }
    if (i == 0) *hit_flag = 1;
    if (i >= n) return;
    f3 pos = xpoint(o, d, sh.t), normal;
    uint32_t material;
    surface_frame(S, sh.tri_pos != IPT_NO_HIT ? S.n_prims + sh.tri_pos : sh.prim, pos, normal, material);
    DevMaterial m = material < IPT_INLINE_MATS ? S.mats[material] : S.mats_g[material];
    Sdf sdf = make_sdf(m, normal, d);
    Basis bn = make_basis(normal);
    Basis bl = make_basis(sdf.refl);
    uint4 r = philox4x32_10((uint32_t)i, (uint32_t)(i >> 32), 1u, 0xDDF1u, k0, k1);
    f3 x = mix_sample(S, sdf, bn, bl, pos, u01(r.x), u01(r.y), u01(r.z), u01(r.w));
    w[3 * i] = x.x; w[3 * i + 1] = x.y; w[3 * i + 2] = x.z;
    bool zero = x.x == 0.0f && x.y == 0.0f && x.z == 0.0f;
    float sv = zero ? 0.0f : sdf_value(sdf, x);
    sdfv[i] = sv;
    mixv[i] = zero ? 0.0f : mix_value(S, sdf, pos, x, sv);
}
__global__ void k_light_ddf_value(const __grid_constant__ DevScene S, f3 pos, const float* __restrict__ w, size_t n, float* out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    f3 a = mk3(w[3 * i], w[3 * i + 1], w[3 * i + 2]);
    Sdf dummy{};
    // Lighting::distributionInPoint(pos)->value(w): the light weights before main.cpp:143 halves them
    float v = mix_value(S, dummy, pos, a, 0.0f);
    out[i] = S.n_lights ? v / (1.0f - S.sdf_weight) : 0.0f;
}

__global__ void k_light_ddf_sample(const __grid_constant__ DevScene S, f3 pos, uint32_t k0, uint32_t k1, size_t n, float* w) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint4 r = philox4x32_10((uint32_t)i, (uint32_t)(i >> 32), 2u, 0xDDF2u, k0, k1);
    // UnionDdf::sample over the lights alone: the draw is scaled into the light half of the 1:1 mixture's cdf
    float us = u01(r.x) * (1.0f - S.sdf_weight);
    Sdf dummy{};
    Basis bn{};
    f3 x = S.n_lights ? mix_sample(S, dummy, bn, bn, pos, us, u01(r.y), u01(r.z), u01(r.w)) : mk3(0, 0, 0);
    if (S.n_lights && !(us < (S.light_inline ? S.lights[S.n_lights - 1].cdf : S.lights_g[S.n_lights - 1].cdf))) x = mk3(0, 0, 0);
    w[3 * i] = x.x; w[3 * i + 1] = x.y; w[3 * i + 2] = x.z;
}

__global__ void k_philox_batch(const uint4* __restrict__ c, size_t n, PhiloxKeys keys, uint4* blocks, float4* uniforms) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint4 r = philox4x32(c[i].x, c[i].y, c[i].z, c[i].w, keys);
    if (blocks) blocks[i] = r;
    if (uniforms) uniforms[i] = make_float4(u01(r.x), u01(r.y), u01(r.z), u01(r.w));
}

// *out = max(*out, max of v[0..n)): the range check of device-resident material indices
__global__ void k_max_u32(const uint32_t* __restrict__ v, size_t n, uint32_t* out) {
    uint32_t m = 0;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) m = max(m, v[i]);
    for (int off = 16; off > 0; off >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, off));
    if ((threadIdx.x & 31) == 0) atomicMax(out, m);
}

// ---------------------------------------------------------------------------------------------------
// the scene's light tables (derive_lights, for ipt_scene_create and ipt_scene_update_lights) in the reference's operation
// order: every step is an explicit _rn intrinsic; oracle/ipt_oracle.c restates them (prepare_light, prepare_weights)
// ---------------------------------------------------------------------------------------------------
// One thread per light: the DevLight record (weight and cdf follow in k_light_weights / k_light_scan), the 64-byte record
// of DevScene::light_samp and, for a scene with a light LBVH, the tree's inputs: 9 floats and (kind, area, weight). The
// area-light arithmetic is that of k_lbvh_records (AreaLight::AreaLight, lighting.cpp:79-90). A kind that differs from
// the scene's light i is reported by the smallest such index in *mismatch; a new scene has no lights yet (`current` null).
__global__ void k_light_derive(const ipt_light* __restrict__ in, uint32_t n, const DevLight* __restrict__ current, DevLight* out, float4* samp,
                               float* ltris, float* extra, uint32_t* mismatch) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const ipt_light l = in[i];
    if (current && l.kind != current[i].kind) atomicMin(mismatch, i);
    DevLight o{};
    o.kind = l.kind;
    o.power = l.power;
    o.px = l.position[0]; o.py = l.position[1]; o.pz = l.position[2];
    o.radius = l.radius;
    o.xax = l.x_axis[0]; o.xay = l.x_axis[1]; o.xaz = l.x_axis[2];
    o.yax = l.y_axis[0]; o.yay = l.y_axis[1]; o.yaz = l.y_axis[2];
    if (l.kind == IPT_LIGHT_AREA_DIAMOND || l.kind == IPT_LIGHT_AREA_TRIANGLE) {
        const f3 e1 = mk3(o.xax, o.xay, o.xaz), e2 = mk3(o.yax, o.yay, o.yaz);
        const f3 cr = xcross3(e1, e2);
        const float full_area = xlength3(cr);
        o.area = l.kind == IPT_LIGHT_AREA_DIAMOND ? full_area : xdiv(full_area, 2.0f);
        // glm::inverse(mat3(e1, e2, cr)) rows 0 and 1, as k_lbvh_records
        float m00 = e1.x, m01 = e1.y, m02 = e1.z, m10 = e2.x, m11 = e2.y, m12 = e2.z, m20 = cr.x, m21 = cr.y, m22 = cr.z;
        float det = xadd(xsub(xmul(m00, xsub(xmul(m11, m22), xmul(m21, m12))), xmul(m10, xsub(xmul(m01, m22), xmul(m21, m02)))),
                         xmul(m20, xsub(xmul(m01, m12), xmul(m11, m02))));
        float ood = xdiv(1.0f, det);
        o.i0x = xmul(xsub(xmul(m11, m22), xmul(m21, m12)), ood);
        o.i0y = xmul(-xsub(xmul(m10, m22), xmul(m20, m12)), ood);
        o.i0z = xmul(xsub(xmul(m10, m21), xmul(m20, m11)), ood);
        o.i1x = xmul(-xsub(xmul(m01, m22), xmul(m21, m02)), ood);
        o.i1y = xmul(xsub(xmul(m00, m22), xmul(m20, m02)), ood);
        o.i1z = xmul(-xsub(xmul(m00, m21), xmul(m20, m01)), ood);
        const f3 nn = xnormalize3(cr);
        o.nx = nn.x; o.ny = nn.y; o.nz = nn.z;
        o.surface_power = xdiv(l.power, o.area);
    } else if (l.kind == IPT_LIGHT_SPHERE || l.kind == IPT_LIGHT_SPHERE_INVERTED) {
        const double r = (double)l.radius; // lighting.h:51, in double as the host evaluates 4.0 * M_PI * r * r
        o.area = __double2float_rn(__dmul_rn(__dmul_rn(4.0 * M_PI, r), r));
        o.surface_power = xdiv(l.power, o.area);
    } else if (l.kind == IPT_LIGHT_POINT) {
        o.area = 0.0f;
        o.surface_power = __uint_as_float(0x7FC00000u); // the host's NAN (lighting.cpp:204)
    }
    out[i] = o;
    samp[4 * (size_t)i] = make_float4(o.px, o.py, o.pz, __uint_as_float(o.kind));
    samp[4 * (size_t)i + 1] = make_float4(o.xax, o.xay, o.xaz, o.radius);
    samp[4 * (size_t)i + 2] = make_float4(o.yax, o.yay, o.yaz, 0.0f);
    samp[4 * (size_t)i + 3] = make_float4(o.nx, o.ny, o.nz, 0.0f);
    if (ltris) {
        float* t = ltris + 9 * (size_t)i;
        t[0] = o.px; t[1] = o.py; t[2] = o.pz;
        t[3] = o.xax; t[4] = o.xay; t[5] = o.xaz;
        t[6] = o.yax; t[7] = o.yay; t[8] = o.yaz;
        extra[3 * (size_t)i] = l.kind == IPT_LIGHT_AREA_TRIANGLE ? 1.0f : 0.0f;
        extra[3 * (size_t)i + 1] = o.area;
    }
}

// The mixture weights of CollectionLighting::distributionInPoint (src/CollectionLighting.cpp:12-21) through unite()'s
// union+simple branch (src/libddf/ddf.cpp:207-223): appending light j rescales every earlier weight by
// f_j = ka_j / (ka_j + p_j) and gives light j the weight r_j = p_j / (ka_j + p_j), where ka_j is the running float sum of
// the powers before j; main.cpp:143 then halves every weight. So w_i = r_i * f_{i+1} * ... * f_{n-1} * 0.5, multiplied
// left to right. Three stages keep every rounding: ka in order (one thread), f and r (one thread each), and each weight's
// chain of multiplies in order.
__global__ void k_light_power_prefix(const ipt_light* __restrict__ in, uint32_t n, float* ka) {
    if (blockIdx.x || threadIdx.x) return;
    float acc = 0.0f;
    for (uint32_t j = 0; j < n; ++j) {
        ka[j] = acc;
        acc = xadd(acc, in[j].power);
    }
}

__global__ void k_light_ratios(const ipt_light* __restrict__ in, const float* __restrict__ ka, uint32_t n, float* f, float* r) {
    uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const float a = ka[j], p = in[j].power, s = xadd(a, p);
    f[j] = xdiv(a, s);
    r[j] = xdiv(p, s);
}

// Four consecutive lights per thread: each f_j is loaded once for the four chains, which are independent multiplies.
// No reassociation: light i still multiplies r_i by f_{i+1}, f_{i+2}, ... in that order, then by 0.5 (main.cpp:143).
#define IPT_WEIGHTS_PER_THREAD 4
__global__ void k_light_weights(const float* __restrict__ f, const float* __restrict__ r, uint32_t n, float* w, DevLight* out, float* extra) {
    const uint32_t i0 = IPT_WEIGHTS_PER_THREAD * (blockIdx.x * blockDim.x + threadIdx.x);
    if (i0 >= n) return;
    float c[IPT_WEIGHTS_PER_THREAD];
#pragma unroll
    for (int k = 0; k < IPT_WEIGHTS_PER_THREAD; ++k) c[k] = i0 + k < n ? r[i0 + k] : 0.0f;
    const uint32_t common = min(i0 + IPT_WEIGHTS_PER_THREAD, n);
    for (uint32_t j = i0 + 1; j < common; ++j) {
        const float fj = f[j];
#pragma unroll
        for (int k = 0; k < IPT_WEIGHTS_PER_THREAD; ++k)
            if (i0 + k < j) c[k] = xmul(c[k], fj);
    }
#pragma unroll 4
    for (uint32_t j = common; j < n; ++j) {
        const float fj = f[j];
#pragma unroll
        for (int k = 0; k < IPT_WEIGHTS_PER_THREAD; ++k) c[k] = xmul(c[k], fj);
    }
#pragma unroll
    for (int k = 0; k < IPT_WEIGHTS_PER_THREAD; ++k) {
        const uint32_t i = i0 + k;
        if (i >= n) break;
        const float wi = xmul(c[k], 0.5f);
        w[i] = wi;
        out[i].weight = wi;
        if (extra) extra[3 * (size_t)i + 2] = wi;
    }
}

// The running float sum of the weights (DevLight::cdf, DevScene::light_cdf) and the guide table, in one thread: the sum
// keeps its order, and guide[b] is a monotone search, whose result on plateaus of the cdf (zero powers) is the contract.
// Without lights the guide is all zero.
__global__ void k_light_scan(const float* __restrict__ w, uint32_t n, float* cdf, DevLight* out, uint32_t* guide) {
    if (blockIdx.x || threadIdx.x) return;
    float acc = 0.0f;
    for (uint32_t i = 0; i < n; ++i) {
        acc = xadd(acc, w[i]);
        cdf[i] = acc;
        out[i].cdf = acc;
    }
    uint32_t i = 0;
    for (uint32_t b = 0; b <= IPT_LIGHT_GUIDE + 1; ++b) {
        const float edge = xdiv((float)b, (float)IPT_LIGHT_GUIDE);
        while (i < n && !(edge < cdf[i])) ++i;
        guide[b] = i;
    }
}

__global__ void k_plane_add_rays(RenderCtx C, size_t n, const float* __restrict__ x, const float* __restrict__ y, const float* __restrict__ v) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t cell = plane_cell(C, x[i], y[i], min((uint32_t)(x[i] * C.width), C.width - 1), min((uint32_t)(y[i] * C.height), C.height - 1));
    atomicAdd(&C.sum[cell], v[i]);
    atomicAdd(&C.sumsq[cell], v[i] * v[i]);
    atomicAdd(&C.count[cell], 1u);
}

__global__ void k_plane_merge(float* __restrict__ sum, float* __restrict__ sumsq, uint32_t* __restrict__ count, const float* __restrict__ s2,
                              const float* __restrict__ q2, const uint32_t* __restrict__ c2, size_t n) {
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        sum[i] += s2[i];
        sumsq[i] += q2[i];
        count[i] += c2[i];
    }
}

__global__ void k_plane_resolve(const float* __restrict__ sum, const uint32_t* __restrict__ count, size_t n, float* pixels) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) pixels[i] = count[i] ? sum[i] / (float)count[i] : 0.0f;
}

// ---------------------------------------------------------------------------------------------------
// scene flattening
// ---------------------------------------------------------------------------------------------------
static int flatten_prims(const ipt_scene_desc* d, std::vector<DevPrim>& out, bool& smallpt) {
    out.assign(d->n_prims, DevPrim{});
    smallpt = false;
    for (uint32_t i = 0; i < d->n_prims; ++i) {
        const ipt_prim& p = d->prims[i];
        DevPrim& o = out[i];
        o.px = p.p[0]; o.py = p.p[1]; o.pz = p.p[2];
        o.radius = p.radius;
        o.kind = p.kind;
        o.material = p.material;
        o.r2 = p.radius * p.radius;
        o.flags = p.flip_normal ? 8u : 0u;
        if (p.material >= d->n_materials) return fail(IPT_ERR_INVALID, "primitive material index out of range");
        if (p.kind == IPT_PRIM_BOX_PLANE) {
            int axis = -1, nz = 0;
            for (int a = 0; a < 3; ++a)
                if (p.p[a] != 0.0f) { axis = a; ++nz; }
            if (nz != 1 || std::fabs(p.p[axis]) != 1.0f)
                return fail(IPT_ERR_INVALID, "box planes must be +-unit axis vectors (geometric_utils.cpp:8)");
            o.flags |= (uint32_t)axis | (p.p[axis] < 0 ? 4u : 0u);
        } else if (p.kind == IPT_PRIM_SPHERE_SMALLPT) {
            smallpt = true;
        } else if (p.kind != IPT_PRIM_SPHERE) {
            return fail(IPT_ERR_INVALID, "unknown primitive kind");
        }
    }
    return IPT_OK;
}

static void set_camera(DevScene& dev, const ipt_camera& c) {
    std::memcpy(dev.cam.pos, c.position, 12);
    std::memcpy(dev.cam.dir, c.direction, 12);
    std::memcpy(dev.cam.right, c.right, 12);
    std::memcpy(dev.cam.up, c.up, 12);
}

// Philox key schedule of a seed (ipt_device.cuh: philox4x32)
static void philox_keys(uint64_t seed, PhiloxKeys& out) {
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    for (int r = 0; r < IPT_PHILOX_ROUNDS; ++r) {
        out.k[2 * r] = k0; out.k[2 * r + 1] = k1;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
}
// (mul, shift) of ipt_device.cuh's fastdiv: mul = floor(2^32 * (2^L - d) / d) + 1 with L = ceil(log2 d), shift = L - 1
static FastDiv make_fastdiv(uint32_t d) {
    FastDiv f{d, 0, 0};
    if (d <= 1) return f;
    uint32_t L = 0;
    while ((1ull << L) < d) ++L;
    f.mul = (uint32_t)((((1ull << L) - d) << 32) / d + 1);
    f.shift = L - 1;
    return f;
}

template <class K>
static int occupancy_grid(K kernel, int sm_count, size_t smem) {
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, IPT_BLOCK, smem) != cudaSuccess || per_sm < 1) per_sm = 1;
    return sm_count * per_sm;
}

// f(smallpt, mesh) with the scene's two flags as std::bool_constant, for the kernels compiled per <SMALLPT, MESH>
template <class F>
static void with_scene_kind(const ipt_scene* s, F&& f) {
    if (s->smallpt && s->mesh) f(std::true_type{}, std::true_type{});
    else if (s->smallpt) f(std::true_type{}, std::false_type{});
    else if (s->mesh) f(std::false_type{}, std::true_type{});
    else f(std::false_type{}, std::false_type{});
}

// the fused k_shade of a scene spec; SPEC_RUNTIME is the SmallPt kernel, which keeps the runtime light switch
template <int FUSE>
static RenderKernel::Fn fused_shade(SceneSpec spec) {
    switch (spec) {
        case SPEC_LIGHT_BVH: return k_shade<FUSE, false, SPEC_LIGHT_BVH>;
        case SPEC_LAMBERT_BOX: return k_shade<FUSE, false, SPEC_LAMBERT_BOX>;
        case SPEC_BOX_SCENE: return k_shade<FUSE, false, SPEC_BOX_SCENE>;
        case SPEC_ONE_AREA_LIGHT: return k_shade<FUSE, false, SPEC_ONE_AREA_LIGHT>;
        case SPEC_ONE_LIGHT: return k_shade<FUSE, false, SPEC_ONE_LIGHT>;
        case SPEC_FEW_LIGHTS: return k_shade<FUSE, false, SPEC_FEW_LIGHTS>;
        default: return k_shade<FUSE, true>;
    }
}

// the device scene's view of the mesh LBVH
static void bind_mesh(ipt_scene* s) {
    s->dev.tris = s->bvh.tri_records;
    s->dev.tri_id = s->bvh.sorted_ids;
    s->dev.nodes = s->bvh.nodes;
    s->dev.qnodes = s->bvh.qnodes;
    s->dev.grid = s->bvh.grid;
    s->dev.tri_mats = s->d_tri_mats;
}

// The input pointer of an entry that takes host or device memory (IPT_UPDATE_DEVICE_POINTER). A mislabelled pointer must be
// refused here: read from the other side it would fault. `align_what` names the required alignment in the message.
static int check_input_pointer(const ipt_scene* s, const void* p, bool device_input, size_t align, const char* entry, const char* arg,
                               const char* align_what) {
    cudaPointerAttributes pa{};
    if (cudaPointerGetAttributes(&pa, p) != cudaSuccess) {
        cudaGetLastError();
        pa.type = cudaMemoryTypeUnregistered;
    }
    const std::string who = std::string(entry) + ": `" + arg + "`";
    if (device_input && !((pa.type == cudaMemoryTypeDevice || pa.type == cudaMemoryTypeManaged) && pa.device == s->device))
        return fail(IPT_ERR_INVALID, std::string(entry) + ": IPT_UPDATE_DEVICE_POINTER given, but `" + arg +
                                         "` is not device or managed memory on the scene's device " + std::to_string(s->device));
    if (!device_input && pa.type == cudaMemoryTypeDevice) return fail(IPT_ERR_INVALID, who + " is device memory: pass IPT_UPDATE_DEVICE_POINTER");
    if (reinterpret_cast<uintptr_t>(p) % align) return fail(IPT_ERR_INVALID, who + " is not aligned to " + align_what);
    return IPT_OK;
}

// grouped box planes + inline spheres only (analytic_closest's first branch)
static bool geom_fast_scene(const ipt_scene* s) { return !s->smallpt && !s->mesh && s->dev.planes_grouped && s->dev.others_inline; }

// DevScene::lights_inside_box. Shadow rays of box scenes skip the wall planes: every non-plane primitive is a sphere inside
// the closed box [-1,1]^3 and every light is an area light whose corners keep a margin of 1e-3 to every wall, so origin (a
// point of a wall or of a sphere) and target lie in the convex box and no wall can come between them. `box_area_light`: a
// geom_fast scene whose lights are the inline ones, all of them area lights.
static uint32_t lights_inside_box(const DevScene& dv, bool box_area_light, const ipt_light* lights, uint32_t n_lights) {
    if (!box_area_light || dv.n_planes == 0) return 0;
    bool inside = true;
    for (uint32_t k = 0; k < dv.n_others; ++k) {
        const DevSphere& sp = dv.others[k];
        const float r = std::sqrt(sp.r2);
        for (float c : {sp.cx, sp.cy, sp.cz}) inside = inside && std::fabs(c) + r <= 1.0f;
    }
    for (uint32_t i = 0; i < n_lights; ++i) {
        const ipt_light& l = lights[i];
        for (int corner = 0; corner < 4; ++corner)
            for (int a = 0; a < 3; ++a) {
                const float q = l.position[a] + ((corner & 1) ? l.x_axis[a] : 0.0f) + ((corner & 2) ? l.y_axis[a] : 0.0f);
                inside = inside && std::fabs(q) <= 1.0f - 1e-3f;
            }
    }
    return inside ? 1u : 0u;
}

static size_t stack_smem(const ipt_scene* s) { return s->mesh ? (size_t)IPT_STACK_SHORT * IPT_BLOCK * sizeof(uint32_t) : 0; }

template <class T>
struct DevBuf {
    T* p = nullptr;
    ~DevBuf() { cudaFree(p); }
    cudaError_t alloc(size_t n) { return cudaMalloc((void**)&p, std::max<size_t>(n, 1) * sizeof(T)); }
};

// n elements of an entry's input on the device: `*d_p` is device memory as given, or host memory copied into `staged` on
// the scene stream
template <class T>
static cudaError_t stage_input(const ipt_scene* s, const T* p, size_t n, bool device_input, DevBuf<T>& staged, const T** d_p) {
    *d_p = p;
    if (device_input) return cudaSuccess;
    cudaError_t e = staged.alloc(n);
    if (e == cudaSuccess && n) e = cudaMemcpyAsync(staged.p, p, sizeof(T) * n, cudaMemcpyHostToDevice, s->stream);
    *d_p = staged.p;
    return e;
}

// The scene's light tables from n ipt_light records in device memory, for ipt_scene_create and ipt_scene_update_lights:
// the DevLight records, DevScene::light_cdf, light_guide and light_samp, the light LBVH of a scene that has one (built into
// a new tree when `rebuild`, else refitted), the inline records and lights_inside_box. The scene's shape (n_lights,
// light_inline, n_light_bvh) is decided already. Everything is derived into new buffers and checked before anything of the
// scene changes; the kinds are checked against the scene's current lights, which a new scene does not have yet (its
// d_lights is null). `who` starts the error messages.
static int derive_lights(ipt_scene* s, const ipt_light* d_in, uint32_t n, bool rebuild, const std::string& who) {
    DevScene& dv = s->dev;
    const bool tree = dv.n_light_bvh > 0;
    DevBuf<DevLight> d_lights;
    DevBuf<float> cdf, samp, scratch, ltris, extra;
    DevBuf<uint32_t> guide, word;
    CUDA_TRY(d_lights.alloc(n));
    CUDA_TRY(cdf.alloc(n));
    CUDA_TRY(samp.alloc(16 * (size_t)n));
    CUDA_TRY(scratch.alloc(4 * (size_t)n)); // ka, f, r, w
    CUDA_TRY(guide.alloc(IPT_LIGHT_GUIDE + 2));
    CUDA_TRY(word.alloc(1));
    if (tree) {
        CUDA_TRY(ltris.alloc(9 * (size_t)n));
        CUDA_TRY(extra.alloc(3 * (size_t)n));
    }
    float *ka = scratch.p, *f = ka + n, *r = f + n, *w = r + n;
    CUDA_TRY(cudaMemsetAsync(word.p, 0xFF, sizeof(uint32_t), s->stream));
    if (n) { // a grid of zero blocks is a launch error: without lights only k_light_scan runs
        const unsigned blocks = (n + 255) / 256;
        k_light_derive<<<blocks, 256, 0, s->stream>>>(d_in, n, s->d_lights, d_lights.p, reinterpret_cast<float4*>(samp.p), ltris.p, extra.p, word.p);
        k_light_power_prefix<<<1, 1, 0, s->stream>>>(d_in, n, ka);
        k_light_ratios<<<blocks, 256, 0, s->stream>>>(d_in, ka, n, f, r);
        const uint32_t weight_threads = (n + IPT_WEIGHTS_PER_THREAD - 1) / IPT_WEIGHTS_PER_THREAD;
        k_light_weights<<<(weight_threads + 127) / 128, 128, 0, s->stream>>>(f, r, n, w, d_lights.p, extra.p);
    }
    k_light_scan<<<1, 1, 0, s->stream>>>(w, n, cdf.p, d_lights.p, guide.p);
    CUDA_TRY(cudaGetLastError());
    // what the host needs back: the kind check and, for a scene that holds its light inline, the derived record and the
    // input record (DevScene::lights and lights_inside_box)
    uint32_t first_bad = 0;
    DevLight inline_derived[IPT_INLINE_LIGHTS];
    ipt_light inline_input[IPT_INLINE_LIGHTS];
    const uint32_t n_inline = dv.light_inline ? n : 0; // n <= IPT_INLINE_LIGHTS
    CUDA_TRY(cudaMemcpyAsync(&first_bad, word.p, sizeof first_bad, cudaMemcpyDeviceToHost, s->stream));
    if (n_inline) {
        CUDA_TRY(cudaMemcpyAsync(inline_derived, d_lights.p, sizeof(DevLight) * n_inline, cudaMemcpyDeviceToHost, s->stream));
        CUDA_TRY(cudaMemcpyAsync(inline_input, d_in, sizeof(ipt_light) * n_inline, cudaMemcpyDeviceToHost, s->stream));
    }
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    if (first_bad != 0xFFFFFFFFu)
        return fail(IPT_ERR_INVALID, who + "lights[" + std::to_string(first_bad) + "].kind differs from the kind of the scene's light " +
                                         std::to_string(first_bad) + " (a different kind needs a new scene)");
    // the light LBVH: a rebuild goes into a new tree, swapped in only if the build succeeds; a refit allocates all its scratch
    // before it writes the tree
    LbvhDevice fresh;
    if (tree) {
        std::string err;
        if (rebuild) {
            if (lbvh_build(ltris.p, n, s->stream, fresh, err, extra.p) != 0) return fail(IPT_ERR_CUDA, who + "light LBVH build failed: " + err);
        } else if (lbvh_refit(ltris.p, s->stream, s->light_bvh, err, extra.p) != 0) {
            return fail(IPT_ERR_CUDA, who + "light LBVH refit failed: " + err);
        }
    }
    // commit. The stream is idle (the read-back and the tree stages end with a synchronise): no enqueued render still reads
    // the buffers that are replaced, and the DevBufs free them on return.
    std::swap(s->d_lights, d_lights.p);
    std::swap(s->d_light_cdf, cdf.p);
    std::swap(s->d_light_guide, guide.p);
    std::swap(s->d_light_samp, samp.p);
    dv.lights_g = s->d_lights;
    dv.light_cdf = s->d_light_cdf;
    dv.light_guide = s->d_light_guide;
    dv.light_samp = reinterpret_cast<const float4*>(s->d_light_samp);
    if (tree && rebuild) {
        lbvh_free(s->light_bvh);
        s->light_bvh = fresh;
    }
    if (tree) {
        dv.light_nodes = s->light_bvh.nodes;
        dv.light_qnodes = s->light_bvh.qnodes;
        dv.light_grid = s->light_bvh.grid;
        dv.light_recs = s->light_bvh.tri_records;
    }
    bool inline_area_light = n_inline > 0;
    for (uint32_t i = 0; i < n_inline; ++i) {
        dv.lights[i] = inline_derived[i];
        if (inline_input[i].kind > IPT_LIGHT_AREA_TRIANGLE) inline_area_light = false;
    }
    dv.lights_inside_box = lights_inside_box(dv, geom_fast_scene(s) && inline_area_light, inline_input, n_inline);
    return IPT_OK;
}

extern "C" {

int ipt_abi_version(void) { return IPT_B200_ABI_VERSION; }
const char* ipt_last_error(void) { return g_last_error.c_str(); }
int ipt_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int ipt_light_derived(const ipt_light* light, float* area, float* surface_power, float normal[3]) {
    namespace H = ipt_host;
    if (!light) return fail(IPT_ERR_INVALID, "null light");
    const ipt_light& l = *light;
    float a = 0.0f, sp = NAN; // a point light (lighting.cpp:204)
    H::f3 nn{0.0f, 0.0f, 0.0f};
    if (l.kind == IPT_LIGHT_AREA_DIAMOND || l.kind == IPT_LIGHT_AREA_TRIANGLE) {
        // AreaLight::AreaLight (src/lighting/lighting.cpp:79-90)
        const H::f3 cr = H::cross(H::mk(l.x_axis), H::mk(l.y_axis));
        const float full_area = H::length(cr);
        a = l.kind == IPT_LIGHT_AREA_DIAMOND ? full_area : full_area / 2.0f;
        nn = H::normalize(cr);
        sp = l.power / a;
    } else if (l.kind == IPT_LIGHT_SPHERE || l.kind == IPT_LIGHT_SPHERE_INVERTED) {
        a = (float)(4.0 * M_PI * l.radius * l.radius); // lighting.h:51
        sp = l.power / a;
    } else if (l.kind != IPT_LIGHT_POINT) {
        return fail(IPT_ERR_INVALID, "unknown light kind");
    }
    if (area) *area = a;
    if (surface_power) *surface_power = sp;
    if (normal) { normal[0] = nn.x; normal[1] = nn.y; normal[2] = nn.z; }
    return IPT_OK;
}

int ipt_scene_create(const ipt_scene_desc* desc, int device, ipt_scene** out) {
    if (!desc || !out) return fail(IPT_ERR_INVALID, "null argument");
    if (!check_eps_constants()) return fail(IPT_ERR_INVALID, "float/double epsilon constants do not hold on this host");
    if (ipt_device_count() <= device || device < 0) return fail(IPT_ERR_NO_DEVICE, "no CUDA device (there is no CPU fallback)");
    if (desc->n_materials == 0) return fail(IPT_ERR_INVALID, "scene has no materials");
    if (desc->n_triangles && desc->triangle_material >= desc->n_materials) return fail(IPT_ERR_INVALID, "triangle material out of range");
    if (desc->n_triangles >= 0x7FFFFFFFull) return fail(IPT_ERR_INVALID, "too many triangles");
    for (uint32_t i = 0; i < desc->n_materials; ++i) {
        const ipt_material& m = desc->materials[i];
        if (m.ddf == IPT_DDF_GLOSSY && !(m.exponent >= 3.0f && m.exponent == std::floor(m.exponent) && m.kd + m.ks > 0.0f))
            return fail(IPT_ERR_INVALID, "glossy material needs an integer exponent >= 3 and kd+ks > 0");
        if (m.ddf > IPT_DDF_GLOSSY) return fail(IPT_ERR_INVALID, "unknown ddf kind");
    }
    std::vector<DevPrim> prims;
    bool smallpt = false;
    int rc = flatten_prims(desc, prims, smallpt);
    if (rc) return rc;
    for (uint32_t i = 0; i < desc->n_lights; ++i)
        if (desc->lights[i].kind > IPT_LIGHT_POINT) return fail(IPT_ERR_INVALID, "unknown light kind");
    std::vector<DevMaterial> mats(desc->n_materials);
    for (uint32_t i = 0; i < desc->n_materials; ++i) {
        const ipt_material& m = desc->materials[i];
        mats[i] = DevMaterial{};
        mats[i].ddf = m.ddf;
        mats[i].albedo = m.albedo;
        if (m.ddf == IPT_DDF_GLOSSY) {
            mats[i].wd = m.kd / (m.kd + m.ks);
            mats[i].ws = m.ks / (m.kd + m.ks);
        }
        mats[i].exponent = m.exponent;
        const float n_lobe = m.ddf == IPT_DDF_GLOSSY ? (float)(int)m.exponent : 1.0f;
        mats[i].inv_np1 = 1.0f / (n_lobe + 1.0f);
        mats[i].lobe_norm = (n_lobe + 1.0f) * (0.5f / IPT_PI_F);
    }

    CUDA_TRY(cudaSetDevice(device));
    // owned by `guard` until the very end: every early return below destroys what has been created so far
    struct SceneGuard {
        ipt_scene* s;
        ~SceneGuard() { if (s) ipt_scene_destroy(s); }
    } guard{new ipt_scene()};
    ipt_scene* s = guard.s;
    s->device = device;
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    s->sm_count = prop.multiProcessorCount;
    CUDA_TRY(cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking));
    CUDA_TRY(cudaEventCreate(&s->ev_begin));
    CUDA_TRY(cudaEventCreate(&s->ev_end));
    DevScene& dv = s->dev;
    std::memset(&dv, 0, sizeof dv);
    dv.n_prims = desc->n_prims;
    dv.n_lights = desc->n_lights;
    dv.n_materials = desc->n_materials;
    dv.has_smallpt = smallpt;
    dv.sdf_weight = desc->n_lights ? 0.5f : 1.0f; // main.cpp:143 unite(light_ddf, 1, sdf, 1); with no lights the sdf alone (ddf.cpp:209-210)
    dv.prim_inline = desc->n_prims <= IPT_INLINE_PRIMS;
    dv.light_inline = desc->n_lights <= IPT_INLINE_LIGHTS;
    bool inline_area_light = dv.light_inline && desc->n_lights > 0; // the lights are the inline ones, all of them area lights
    for (uint32_t i = 0; i < desc->n_lights && i < IPT_INLINE_LIGHTS; ++i)
        if (desc->lights[i].kind > IPT_LIGHT_AREA_TRIANGLE) inline_area_light = false;
    auto upload = [&](auto*& dptr, const auto& vec) -> cudaError_t {
        size_t bytes = std::max<size_t>(vec.size(), 1) * sizeof(vec[0]);
        cudaError_t e = cudaMalloc((void**)&dptr, bytes);
        if (e != cudaSuccess) return e;
        if (!vec.empty()) e = cudaMemcpy(dptr, vec.data(), vec.size() * sizeof(vec[0]), cudaMemcpyHostToDevice);
        return e;
    };
    CUDA_TRY(upload(s->d_prims, prims));
    CUDA_TRY(upload(s->d_mats, mats));
    dv.prims_g = s->d_prims;
    dv.mats_g = s->d_mats;
    for (uint32_t i = 0; i < desc->n_prims && i < IPT_INLINE_PRIMS; ++i) dv.prims[i] = prims[i];
    for (uint32_t i = 0; i < desc->n_materials && i < IPT_INLINE_MATS; ++i) dv.mats[i] = mats[i];
    // group the box planes by (axis, sign) for the branch-free plane test
    dv.planes_grouped = 1;
    dv.n_planes = 0;
    for (int k = 0; k < 6; ++k) dv.plane_of[k] = IPT_NO_HIT;
    for (uint32_t i = 0; i < desc->n_prims; ++i)
        if (prims[i].kind == IPT_PRIM_BOX_PLANE) {
            uint32_t slot = 2 * (prims[i].flags & 3u) + ((prims[i].flags & 4u) ? 1u : 0u);
            if (dv.plane_of[slot] != IPT_NO_HIT) dv.planes_grouped = 0; // duplicate plane: keep the generic ordered scan
            dv.plane_of[slot] = i;
            ++dv.n_planes;
        }
    dv.n_others = 0;
    dv.others_inline = 1;
    for (uint32_t i = 0; i < desc->n_prims; ++i) {
        if (prims[i].kind == IPT_PRIM_BOX_PLANE) continue;
        if (prims[i].kind != IPT_PRIM_SPHERE || dv.n_others == IPT_INLINE_OTHERS) { dv.others_inline = 0; break; }
        DevSphere& sp = dv.others[dv.n_others++];
        sp.cx = prims[i].px; sp.cy = prims[i].py; sp.cz = prims[i].pz; sp.r2 = prims[i].r2; sp.index = i;
    }
    set_camera(dv, desc->camera);
    s->smallpt = smallpt;
    s->mesh = desc->n_triangles > 0;
    // grouped box planes + inline spheres only (analytic_closest's first branch)
    const bool geom_fast = geom_fast_scene(s);
    bool all_lambert = true; // every material is the cosine DDF
    for (const DevMaterial& m : mats) if (m.ddf != IPT_DDF_COSINE) all_lambert = false;
    if (s->mesh) {
        DevBuf<float> staged;
        const float* d_tris;
        CUDA_TRY(stage_input(s, desc->triangles, 9 * (size_t)desc->n_triangles, false, staged, &d_tris));
        std::string err;
        if (lbvh_build(d_tris, (uint32_t)desc->n_triangles, s->stream, s->bvh, err) != 0) return fail(IPT_ERR_CUDA, "LBVH build failed: " + err);
        dv.n_tris = (uint32_t)desc->n_triangles;
        dv.tri_material = desc->triangle_material;
        bind_mesh(s);
    }
    // many area lights: LBVH over them (nearest-light and all-hits density queries instead of O(L) scans)
    bool all_area = desc->n_lights > 0;
    for (uint32_t i = 0; i < desc->n_lights; ++i) all_area = all_area && desc->lights[i].kind <= IPT_LIGHT_AREA_TRIANGLE;
    if (all_area && desc->n_lights > IPT_LIGHT_BVH_MIN) dv.n_light_bvh = desc->n_lights;
    {
        DevBuf<ipt_light> staged;
        const ipt_light* d_in;
        CUDA_TRY(stage_input(s, desc->lights, desc->n_lights, false, staged, &d_in));
        if (int rc = derive_lights(s, d_in, desc->n_lights, true, "")) return rc;
    }
    CUDA_TRY(cudaMalloc((void**)&s->d_cnt, sizeof(uint32_t) * IPT_CNT_WORDS));
    CUDA_TRY(cudaMalloc((void**)&s->d_stats, sizeof(unsigned long long) * ST_COUNT));

    // the kernels compiled for this kind of scene (SceneSpec in ipt_kernels.cuh)
    s->shade_spec = smallpt ? SPEC_RUNTIME
                    : dv.n_light_bvh ? SPEC_LIGHT_BVH
                    : (inline_area_light && geom_fast && all_lambert) ? SPEC_LAMBERT_BOX
                    : (inline_area_light && geom_fast) ? SPEC_BOX_SCENE
                    : inline_area_light ? SPEC_ONE_AREA_LIGHT
                    : dv.light_inline ? SPEC_ONE_LIGHT
                                      : SPEC_FEW_LIGHTS;
    const bool persistent_mesh = s->mesh && !smallpt;
    s->mesh_spec = persistent_mesh && inline_area_light && dv.planes_grouped && dv.others_inline ? SPEC_BOX_SCENE : SPEC_RUNTIME;
    auto entry = [&](RenderKernel::Fn k, size_t smem) { return RenderKernel{k, occupancy_grid(k, s->sm_count, smem), smem}; };
    s->grid_generate = occupancy_grid(k_generate, s->sm_count, 0);
    s->grid_accumulate = occupancy_grid(k_accumulate, s->sm_count, 0);
    s->shade = entry(smallpt ? k_shade<FUSE_NONE, true> : k_shade<FUSE_NONE, false>, 0);
    s->shade_next = entry(fused_shade<FUSE_NEXT>(s->shade_spec), 0);
    s->shade_last = entry(fused_shade<FUSE_LAST>(s->shade_spec), 0);
    if (persistent_mesh) {
        // persistent warps that refill idle lanes from the ray queue (ipt_trace.cuh), always in exact arithmetic
        const bool box = s->mesh_spec == SPEC_BOX_SCENE;
        s->extend[0][0] = s->extend[0][1] = entry(box ? k_extend_mesh<false, SPEC_BOX_SCENE> : k_extend_mesh<false>, IPT_MESH_SMEM_BYTES);
        s->extend[1][0] = s->extend[1][1] = entry(box ? k_extend_mesh<true, SPEC_BOX_SCENE> : k_extend_mesh<true>, IPT_MESH_SMEM_BYTES);
    } else {
        const size_t sm = stack_smem(s);
        with_scene_kind(s, [&](auto sp, auto ms) {
            s->extend[0][1] = entry(k_extend<sp, ms, false, true>, sm);
            s->extend[1][1] = entry(k_extend<sp, ms, true, true>, sm);
            // SmallPt scenes with a mesh trace every depth in exact arithmetic: k_extend has no contracted mesh form
            s->extend[0][0] = ms ? s->extend[0][1] : entry(k_extend<sp, false, false, false>, sm);
            s->extend[1][0] = ms ? s->extend[1][1] : entry(k_extend<sp, false, true, false>, sm);
        });
    }
    guard.s = nullptr;
    *out = s;
    return IPT_OK;
}

static void free_workspace(Workspace& w) {
    cudaFree(w.ray_o); cudaFree(w.ray_d); cudaFree(w.ray_x); cudaFree(w.hit_a); cudaFree(w.hit_b); cudaFree(w.hit_a2); cudaFree(w.hit_b2);
    cudaFree(w.pathval);
    w = Workspace();
}

int ipt_scene_destroy(ipt_scene* s) {
    if (!s) return fail(IPT_ERR_INVALID, "null scene");
    cudaSetDevice(s->device);
    if (s->stream) cudaStreamSynchronize(s->stream);
    if (s->host_plane) ipt_plane_destroy(s->host_plane);
    free_workspace(s->ws);
    lbvh_free(s->bvh);
    lbvh_free(s->light_bvh);
    cudaFree(s->d_tri_mats_orig); cudaFree(s->d_tri_mats);
    cudaFree(s->d_prims); cudaFree(s->d_lights); cudaFree(s->d_light_cdf); cudaFree(s->d_light_guide); cudaFree(s->d_light_samp); cudaFree(s->d_mats); cudaFree(s->d_cnt); cudaFree(s->d_stats);
    if (s->pinned) cudaFreeHost(s->pinned);
    for (cudaEvent_t e : s->events) cudaEventDestroy(e);
    if (s->ev_begin) cudaEventDestroy(s->ev_begin);
    if (s->ev_end) cudaEventDestroy(s->ev_end);
    if (s->stream) cudaStreamDestroy(s->stream);
    cudaGetLastError(); // a half-built scene may have tripped an error on the way: it has been reported already
    delete s;
    return IPT_OK;
}

int ipt_scene_set_camera(ipt_scene* s, const ipt_camera* camera) {
    if (!s || !camera) return fail(IPT_ERR_INVALID, "null argument");
    std::lock_guard<std::recursive_mutex> lock__(s->mu);
    set_camera(s->dev, *camera);
    return IPT_OK;
}

int ipt_scene_dispatch(ipt_scene* s, uint32_t out[IPT_DISPATCH_WORDS]) {
    if (!s || !out) return fail(IPT_ERR_INVALID, "null argument");
    std::lock_guard<std::recursive_mutex> lock__(s->mu);
    out[0] = (uint32_t)s->shade_spec;
    out[1] = s->smallpt;
    out[2] = s->mesh;
    out[3] = s->mesh_spec == SPEC_BOX_SCENE;
    out[4] = s->dev.lights_inside_box;
    out[5] = s->dev.light_inline;
    out[6] = s->dev.n_light_bvh;
    return IPT_OK;
}

int ipt_scene_update_triangles(ipt_scene* s, const float* triangles, uint64_t n_triangles, uint32_t flags) {
    if (!s || !triangles) return fail(IPT_ERR_INVALID, "ipt_scene_update_triangles: null argument");
    if (flags & ~(uint32_t)(IPT_UPDATE_DEVICE_POINTER | IPT_UPDATE_REBUILD))
        return fail(IPT_ERR_INVALID, "ipt_scene_update_triangles: unknown flag bits " + std::to_string(flags));
    std::lock_guard<std::recursive_mutex> lock__(s->mu);
    if (!s->mesh) return fail(IPT_ERR_INVALID, "ipt_scene_update_triangles: the scene has no triangle mesh");
    if (n_triangles != s->bvh.n)
        return fail(IPT_ERR_INVALID, "ipt_scene_update_triangles: " + std::to_string(n_triangles) + " triangles given, the scene has " +
                                         std::to_string(s->bvh.n) + " (a different count needs a new scene)");
    CUDA_TRY(cudaSetDevice(s->device));
    const bool device_input = flags & IPT_UPDATE_DEVICE_POINTER;
    if (int rc = check_input_pointer(s, triangles, device_input, alignof(float), "ipt_scene_update_triangles", "triangles", "a float")) return rc;
    const uint32_t n = s->bvh.n;
    DevBuf<float> staged;
    const float* d_tris;
    CUDA_TRY(stage_input(s, triangles, 9 * (size_t)n, device_input, staged, &d_tris));
    std::string err;
    if (flags & IPT_UPDATE_REBUILD) {
        // into a new tree: the scene keeps the old one unless the build succeeds. lbvh_build waits for the scene stream, so
        // no enqueued render still reads the old buffers when they are freed. Per-triangle materials follow the new sorted
        // order: their buffer is allocated before the build and filled from it before the swap.
        DevBuf<uint32_t> mats;
        if (s->d_tri_mats_orig) CUDA_TRY(mats.alloc(n));
        LbvhDevice fresh;
        if (lbvh_build(d_tris, n, s->stream, fresh, err) != 0) return fail(IPT_ERR_CUDA, "ipt_scene_update_triangles: LBVH build failed: " + err);
        if (mats.p) {
            k_lbvh_gather<<<(n + 255) / 256, 256, 0, s->stream>>>(s->d_tri_mats_orig, fresh.sorted_ids, n, mats.p);
            cudaError_t e = cudaGetLastError();
            if (e == cudaSuccess) e = cudaStreamSynchronize(s->stream);
            if (e != cudaSuccess) {
                lbvh_free(fresh);
                return fail(IPT_ERR_CUDA, std::string("ipt_scene_update_triangles: material gather failed: ") + cudaGetErrorString(e));
            }
            cudaFree(s->d_tri_mats);
            s->d_tri_mats = mats.p;
            mats.p = nullptr;
        }
        lbvh_free(s->bvh);
        s->bvh = fresh;
    } else if (lbvh_refit(d_tris, s->stream, s->bvh, err) != 0) {
        return fail(IPT_ERR_CUDA, "ipt_scene_update_triangles: LBVH refit failed: " + err);
    }
    bind_mesh(s);
    return IPT_OK;
}

int ipt_scene_set_triangle_materials(ipt_scene* s, const uint32_t* materials, uint64_t n_triangles, uint32_t flags) {
    static const char* entry = "ipt_scene_set_triangle_materials";
    if (!s || !materials) return fail(IPT_ERR_INVALID, std::string(entry) + ": null argument");
    if (flags & ~(uint32_t)IPT_UPDATE_DEVICE_POINTER) return fail(IPT_ERR_INVALID, std::string(entry) + ": unknown flag bits " + std::to_string(flags));
    std::lock_guard<std::recursive_mutex> lock__(s->mu);
    if (!s->mesh) return fail(IPT_ERR_INVALID, std::string(entry) + ": the scene has no triangle mesh");
    if (n_triangles != s->bvh.n)
        return fail(IPT_ERR_INVALID, std::string(entry) + ": " + std::to_string(n_triangles) + " materials given, the scene has " +
                                         std::to_string(s->bvh.n) + " triangles");
    CUDA_TRY(cudaSetDevice(s->device));
    const bool device_input = flags & IPT_UPDATE_DEVICE_POINTER;
    if (int rc = check_input_pointer(s, materials, device_input, alignof(uint32_t), entry, "materials", "4 bytes")) return rc;
    const uint32_t n = s->bvh.n, n_mats = s->dev.n_materials;
    if (!device_input)
        for (uint32_t k = 0; k < n; ++k)
            if (materials[k] >= n_mats)
                return fail(IPT_ERR_INVALID, std::string(entry) + ": materials[" + std::to_string(k) + "] = " + std::to_string(materials[k]) +
                                                 " is out of range: the scene has " + std::to_string(n_mats) + " materials");
    // new buffers, filled and checked before anything of the scene changes
    DevBuf<uint32_t> orig, sorted, max_word;
    CUDA_TRY(orig.alloc(n));
    CUDA_TRY(sorted.alloc(n));
    if (device_input) CUDA_TRY(max_word.alloc(1));
    CUDA_TRY(cudaMemcpyAsync(orig.p, materials, sizeof(uint32_t) * (size_t)n, device_input ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, s->stream));
    if (device_input) {
        uint32_t max_index = 0;
        CUDA_TRY(cudaMemsetAsync(max_word.p, 0, sizeof(uint32_t), s->stream));
        k_max_u32<<<std::min<uint32_t>((n + 255) / 256, 4 * (uint32_t)s->sm_count), 256, 0, s->stream>>>(orig.p, n, max_word.p);
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cudaMemcpyAsync(&max_index, max_word.p, sizeof(uint32_t), cudaMemcpyDeviceToHost, s->stream));
        CUDA_TRY(cudaStreamSynchronize(s->stream));
        if (max_index >= n_mats)
            return fail(IPT_ERR_INVALID, std::string(entry) + ": a material index is out of range (largest " + std::to_string(max_index) +
                                             "): the scene has " + std::to_string(n_mats) + " materials");
    }
    k_lbvh_gather<<<(n + 255) / 256, 256, 0, s->stream>>>(orig.p, s->bvh.sorted_ids, n, sorted.p);
    CUDA_TRY(cudaGetLastError());
    // the stream is idle after this: no enqueued render still reads the buffers replaced below
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    std::swap(s->d_tri_mats_orig, orig.p);
    std::swap(s->d_tri_mats, sorted.p);
    bind_mesh(s);
    return IPT_OK;
}

int ipt_scene_update_lights(ipt_scene* s, const ipt_light* lights, uint32_t n_lights, uint32_t flags) {
    static const char* entry = "ipt_scene_update_lights";
    if (!s || !lights) return fail(IPT_ERR_INVALID, std::string(entry) + ": null argument");
    if (flags & ~(uint32_t)(IPT_UPDATE_DEVICE_POINTER | IPT_UPDATE_REBUILD))
        return fail(IPT_ERR_INVALID, std::string(entry) + ": unknown flag bits " + std::to_string(flags));
    std::lock_guard<std::recursive_mutex> lock__(s->mu);
    DevScene& dv = s->dev;
    if (n_lights != dv.n_lights)
        return fail(IPT_ERR_INVALID, std::string(entry) + ": " + std::to_string(n_lights) + " lights given, the scene has " +
                                         std::to_string(dv.n_lights) + " (a different count needs a new scene)");
    CUDA_TRY(cudaSetDevice(s->device));
    const bool device_input = flags & IPT_UPDATE_DEVICE_POINTER;
    if (int rc = check_input_pointer(s, lights, device_input, alignof(uint32_t), entry, "lights", "4 bytes")) return rc;
    if (n_lights == 0) return IPT_OK;
    DevBuf<ipt_light> staged;
    const ipt_light* d_in;
    CUDA_TRY(stage_input(s, lights, n_lights, device_input, staged, &d_in));
    return derive_lights(s, d_in, n_lights, flags & IPT_UPDATE_REBUILD, std::string(entry) + ": ");
}

// ---- parity entries ----------------------------------------------------------------------------------
int ipt_trace_batch(ipt_scene* s, const float* origins, const float* directions, size_t n, uint32_t* prim_id, float* t,
                    uint32_t* light_id, float* light_pos, uint32_t* outcome) {
    if (!s || !origins || !directions) return fail(IPT_ERR_INVALID, "null argument");
    std::lock_guard<std::recursive_mutex> lock__(s->mu);
    if (n == 0) return IPT_OK;
    CUDA_TRY(cudaSetDevice(s->device));
    DevBuf<float> d_o, d_d, d_t, d_lp;
    DevBuf<uint32_t> d_prim, d_light, d_out;
    CUDA_TRY(d_o.alloc(3 * n)); CUDA_TRY(d_d.alloc(3 * n)); CUDA_TRY(d_t.alloc(n)); CUDA_TRY(d_lp.alloc(3 * n));
    CUDA_TRY(d_prim.alloc(n)); CUDA_TRY(d_light.alloc(n)); CUDA_TRY(d_out.alloc(n));
    CUDA_TRY(cudaMemcpyAsync(d_o.p, origins, 12 * n, cudaMemcpyHostToDevice, s->stream));
    CUDA_TRY(cudaMemcpyAsync(d_d.p, directions, 12 * n, cudaMemcpyHostToDevice, s->stream));
    unsigned blocks = (unsigned)((n + IPT_BLOCK - 1) / IPT_BLOCK);
    with_scene_kind(s, [&](auto sp, auto ms) {
        k_trace_batch<sp, ms><<<blocks, IPT_BLOCK, stack_smem(s), s->stream>>>(s->dev, d_o.p, d_d.p, n, d_prim.p, d_t.p, d_light.p, d_lp.p, d_out.p);
    });
    CUDA_TRY(cudaGetLastError());
    if (prim_id) CUDA_TRY(cudaMemcpyAsync(prim_id, d_prim.p, 4 * n, cudaMemcpyDeviceToHost, s->stream));
    if (t) CUDA_TRY(cudaMemcpyAsync(t, d_t.p, 4 * n, cudaMemcpyDeviceToHost, s->stream));
    if (light_id) CUDA_TRY(cudaMemcpyAsync(light_id, d_light.p, 4 * n, cudaMemcpyDeviceToHost, s->stream));
    if (light_pos) CUDA_TRY(cudaMemcpyAsync(light_pos, d_lp.p, 12 * n, cudaMemcpyDeviceToHost, s->stream));
    if (outcome) CUDA_TRY(cudaMemcpyAsync(outcome, d_out.p, 4 * n, cudaMemcpyDeviceToHost, s->stream));
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    return IPT_OK;
}

int ipt_preview_batch(ipt_scene* s, const float* origins, const float* directions, size_t n, float* value) {
    if (!s || !origins || !directions || !value) return fail(IPT_ERR_INVALID, "null argument");
    std::lock_guard<std::recursive_mutex> lock__(s->mu);
    if (n == 0) return IPT_OK;
    CUDA_TRY(cudaSetDevice(s->device));
    DevBuf<float> d_o, d_d, d_v;
    CUDA_TRY(d_o.alloc(3 * n)); CUDA_TRY(d_d.alloc(3 * n)); CUDA_TRY(d_v.alloc(n));
    CUDA_TRY(cudaMemcpyAsync(d_o.p, origins, 12 * n, cudaMemcpyHostToDevice, s->stream));
    CUDA_TRY(cudaMemcpyAsync(d_d.p, directions, 12 * n, cudaMemcpyHostToDevice, s->stream));
    unsigned blocks = (unsigned)((n + IPT_BLOCK - 1) / IPT_BLOCK);
    with_scene_kind(s, [&](auto sp, auto ms) {
        k_preview_batch<sp, ms><<<blocks, IPT_BLOCK, stack_smem(s), s->stream>>>(s->dev, d_o.p, d_d.p, n, d_v.p);
    });
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(value, d_v.p, 4 * n, cudaMemcpyDeviceToHost, s->stream));
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    return IPT_OK;
}

int ipt_camera_rays(ipt_scene* s, const float* xy, size_t n, float* origins, float* directions) {
    if (!s || !xy || !origins || !directions) return fail(IPT_ERR_INVALID, "null argument");
    std::lock_guard<std::recursive_mutex> lock__(s->mu);
    if (n == 0) return IPT_OK;
    CUDA_TRY(cudaSetDevice(s->device));
    DevBuf<float> d_xy, d_o, d_d;
    CUDA_TRY(d_xy.alloc(2 * n)); CUDA_TRY(d_o.alloc(3 * n)); CUDA_TRY(d_d.alloc(3 * n));
    CUDA_TRY(cudaMemcpyAsync(d_xy.p, xy, 8 * n, cudaMemcpyHostToDevice, s->stream));
    k_camera_rays<<<(unsigned)((n + 255) / 256), 256, 0, s->stream>>>(s->dev, d_xy.p, n, d_o.p, d_d.p);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(origins, d_o.p, 12 * n, cudaMemcpyDeviceToHost, s->stream));
    CUDA_TRY(cudaMemcpyAsync(directions, d_d.p, 12 * n, cudaMemcpyDeviceToHost, s->stream));
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    return IPT_OK;
}

int ipt_ddf_value(ipt_scene* s, int kind, const float* to, const float* dirs, size_t n, float* out) {
    if (!s || !dirs || !out || kind < 0) return fail(IPT_ERR_INVALID, "bad argument");
    std::lock_guard<std::recursive_mutex> lock__(s->mu);
    if (n == 0) return IPT_OK;
    CUDA_TRY(cudaSetDevice(s->device));
    DevBuf<float> d_w, d_out;
    CUDA_TRY(d_w.alloc(3 * n)); CUDA_TRY(d_out.alloc(n));
    CUDA_TRY(cudaMemcpyAsync(d_w.p, dirs, 12 * n, cudaMemcpyHostToDevice, s->stream));
    f3 tv = to ? f3{to[0], to[1], to[2]} : f3{0, 0, 1};
    k_ddf_value<<<(unsigned)((n + 255) / 256), 256, 0, s->stream>>>(kind, to != nullptr, tv, d_w.p, n, d_out.p);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(out, d_out.p, 4 * n, cudaMemcpyDeviceToHost, s->stream));
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    return IPT_OK;
}

int ipt_ddf_sample(ipt_scene* s, int kind, const float* to, uint64_t seed, size_t n, float* dirs) {
    if (!s || !dirs || kind < 0) return fail(IPT_ERR_INVALID, "bad argument");
    std::lock_guard<std::recursive_mutex> lock__(s->mu);
    if (n == 0) return IPT_OK;
    CUDA_TRY(cudaSetDevice(s->device));
    DevBuf<float> d_w;
    CUDA_TRY(d_w.alloc(3 * n));
    f3 tv = to ? f3{to[0], to[1], to[2]} : f3{0, 0, 1};
    k_ddf_sample<<<(unsigned)((n + 255) / 256), 256, 0, s->stream>>>(kind, to != nullptr, tv, (uint32_t)seed, (uint32_t)(seed >> 32), n, d_w.p);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(dirs, d_w.p, 12 * n, cudaMemcpyDeviceToHost, s->stream));
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    return IPT_OK;
}

int ipt_mix_sample(ipt_scene* s, const float origin[3], const float direction[3], uint64_t seed, size_t n, float* dirs,
                   float* mix_value_out, float* sdf_value_out) {
    if (!s || !origin || !direction || !dirs || !mix_value_out || !sdf_value_out) return fail(IPT_ERR_INVALID, "null argument");
    std::lock_guard<std::recursive_mutex> lock__(s->mu);
    if (n == 0) return IPT_OK;
    CUDA_TRY(cudaSetDevice(s->device));
    DevBuf<float> d_w, d_m, d_s;
    DevBuf<int> d_flag;
    CUDA_TRY(d_w.alloc(3 * n)); CUDA_TRY(d_m.alloc(n)); CUDA_TRY(d_s.alloc(n)); CUDA_TRY(d_flag.alloc(1));
    f3 o{origin[0], origin[1], origin[2]}, d{direction[0], direction[1], direction[2]};
    unsigned blocks = (unsigned)((n + IPT_BLOCK - 1) / IPT_BLOCK);
    with_scene_kind(s, [&](auto sp, auto ms) {
        k_mix_sample<sp, ms><<<blocks, IPT_BLOCK, stack_smem(s), s->stream>>>(s->dev, o, d, (uint32_t)seed, (uint32_t)(seed >> 32), n, d_w.p, d_m.p, d_s.p, d_flag.p);
    });
    CUDA_TRY(cudaGetLastError());
    int flag = 0;
    CUDA_TRY(cudaMemcpyAsync(&flag, d_flag.p, 4, cudaMemcpyDeviceToHost, s->stream));
    CUDA_TRY(cudaMemcpyAsync(dirs, d_w.p, 12 * n, cudaMemcpyDeviceToHost, s->stream));
    CUDA_TRY(cudaMemcpyAsync(mix_value_out, d_m.p, 4 * n, cudaMemcpyDeviceToHost, s->stream));
    CUDA_TRY(cudaMemcpyAsync(sdf_value_out, d_s.p, 4 * n, cudaMemcpyDeviceToHost, s->stream));
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    if (!flag) return fail(IPT_ERR_INVALID, "the ray does not hit the geometry");
    return IPT_OK;
}

int ipt_light_ddf_value(ipt_scene* s, const float pos[3], const float* dirs, size_t n, float* out) {
    if (!s || !pos || !dirs || !out) return fail(IPT_ERR_INVALID, "null argument");
    std::lock_guard<std::recursive_mutex> lock__(s->mu);
    if (n == 0) return IPT_OK;
    CUDA_TRY(cudaSetDevice(s->device));
    DevBuf<float> d_w, d_out;
    CUDA_TRY(d_w.alloc(3 * n)); CUDA_TRY(d_out.alloc(n));
    CUDA_TRY(cudaMemcpyAsync(d_w.p, dirs, 12 * n, cudaMemcpyHostToDevice, s->stream));
    k_light_ddf_value<<<(unsigned)((n + 255) / 256), 256, 0, s->stream>>>(s->dev, f3{pos[0], pos[1], pos[2]}, d_w.p, n, d_out.p);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(out, d_out.p, 4 * n, cudaMemcpyDeviceToHost, s->stream));
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    return IPT_OK;
}

int ipt_light_ddf_sample(ipt_scene* s, const float pos[3], uint64_t seed, size_t n, float* dirs) {
    if (!s || !pos || !dirs) return fail(IPT_ERR_INVALID, "null argument");
    std::lock_guard<std::recursive_mutex> lock__(s->mu);
    if (n == 0) return IPT_OK;
    CUDA_TRY(cudaSetDevice(s->device));
    DevBuf<float> d_w;
    CUDA_TRY(d_w.alloc(3 * n));
    k_light_ddf_sample<<<(unsigned)((n + 255) / 256), 256, 0, s->stream>>>(s->dev, f3{pos[0], pos[1], pos[2]}, (uint32_t)seed, (uint32_t)(seed >> 32), n, d_w.p);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(dirs, d_w.p, 12 * n, cudaMemcpyDeviceToHost, s->stream));
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    return IPT_OK;
}

int ipt_philox_batch(int device, const uint32_t* counters, size_t n, uint64_t seed, uint32_t* blocks, float* uniforms) {
    if (!counters) return fail(IPT_ERR_INVALID, "null argument");
    if (ipt_device_count() <= device || device < 0) return fail(IPT_ERR_NO_DEVICE, "no CUDA device (there is no CPU fallback)");
    if (n == 0) return IPT_OK;
    CUDA_TRY(cudaSetDevice(device));
    DevBuf<uint4> d_c, d_b;
    DevBuf<float4> d_u;
    CUDA_TRY(d_c.alloc(n)); CUDA_TRY(d_b.alloc(n)); CUDA_TRY(d_u.alloc(n));
    CUDA_TRY(cudaMemcpy(d_c.p, counters, 16 * n, cudaMemcpyHostToDevice));
    PhiloxKeys keys;
    philox_keys(seed, keys);
    k_philox_batch<<<(unsigned)((n + 255) / 256), 256>>>(d_c.p, n, keys, d_b.p, d_u.p);
    CUDA_TRY(cudaGetLastError());
    if (blocks) CUDA_TRY(cudaMemcpy(blocks, d_b.p, 16 * n, cudaMemcpyDeviceToHost));
    if (uniforms) CUDA_TRY(cudaMemcpy(uniforms, d_u.p, 16 * n, cudaMemcpyDeviceToHost));
    return IPT_OK;
}

int ipt_bvh_export(ipt_scene* s, ipt_bvh_node* nodes, uint32_t* sorted_prims, uint64_t* morton, uint64_t* n_nodes) {
    if (!s) return fail(IPT_ERR_INVALID, "null scene");
    std::lock_guard<std::recursive_mutex> lock__(s->mu);
    if (!s->mesh) return fail(IPT_ERR_INVALID, "scene has no triangle mesh");
    CUDA_TRY(cudaSetDevice(s->device));
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    uint32_t n = s->bvh.n;
    static_assert(sizeof(ipt_bvh_node) == sizeof(BvhNode), "ABI node layout");
    if (n_nodes) *n_nodes = n > 1 ? n - 1 : 0;
    if (nodes && n > 1) CUDA_TRY(cudaMemcpy(nodes, s->bvh.nodes, sizeof(BvhNode) * (n - 1), cudaMemcpyDeviceToHost));
    if (sorted_prims) CUDA_TRY(cudaMemcpy(sorted_prims, s->bvh.sorted_ids, 4 * (size_t)n, cudaMemcpyDeviceToHost));
    if (morton) CUDA_TRY(cudaMemcpy(morton, s->bvh.sorted_keys, 8 * (size_t)n, cudaMemcpyDeviceToHost));
    return IPT_OK;
}

int ipt_bvh_export_compact(ipt_scene* s, uint32_t* nodes32, float grid[6], uint64_t* n_nodes) {
    if (!s) return fail(IPT_ERR_INVALID, "null scene");
    std::lock_guard<std::recursive_mutex> lock__(s->mu);
    if (!s->mesh) return fail(IPT_ERR_INVALID, "scene has no triangle mesh");
    CUDA_TRY(cudaSetDevice(s->device));
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    uint32_t n = s->bvh.n;
    if (n_nodes) *n_nodes = n > 1 ? n - 1 : 0;
    if (nodes32 && n > 1) CUDA_TRY(cudaMemcpy(nodes32, s->bvh.qnodes, sizeof(BvhNodeQ) * (size_t)(n - 1), cudaMemcpyDeviceToHost));
    if (grid) for (int a = 0; a < 3; ++a) { grid[a] = s->bvh.grid.lo[a]; grid[3 + a] = s->bvh.grid.scale[a]; }
    return IPT_OK;
}

int ipt_light_tables_export(ipt_scene* s, float* area, float* surface_power, float* normal, float* weight, float* cdf,
                            uint32_t guide[IPT_LIGHT_GUIDE_WORDS]) {
    static_assert(IPT_LIGHT_GUIDE_WORDS == IPT_LIGHT_GUIDE + 2, "ABI guide size");
    if (!s) return fail(IPT_ERR_INVALID, "null scene");
    std::lock_guard<std::recursive_mutex> lock__(s->mu);
    CUDA_TRY(cudaSetDevice(s->device));
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    const uint32_t n = s->dev.n_lights;
    std::vector<DevLight> lights(n);
    if (n) CUDA_TRY(cudaMemcpy(lights.data(), s->d_lights, sizeof(DevLight) * n, cudaMemcpyDeviceToHost));
    for (uint32_t i = 0; i < n; ++i) {
        const DevLight& L = lights[i];
        if (area) area[i] = L.area;
        if (surface_power) surface_power[i] = L.surface_power;
        if (normal) { normal[3 * i] = L.nx; normal[3 * i + 1] = L.ny; normal[3 * i + 2] = L.nz; }
        if (weight) weight[i] = L.weight;
    }
    if (cdf && n) CUDA_TRY(cudaMemcpy(cdf, s->d_light_cdf, sizeof(float) * n, cudaMemcpyDeviceToHost));
    if (guide) CUDA_TRY(cudaMemcpy(guide, s->d_light_guide, sizeof(uint32_t) * IPT_LIGHT_GUIDE_WORDS, cudaMemcpyDeviceToHost));
    return IPT_OK;
}

// ---- render plane ---------------------------------------------------------------------------------------
int ipt_plane_create(ipt_scene* s, uint32_t width, uint32_t height, ipt_plane** out) {
    if (!s || !out || !width || !height) return fail(IPT_ERR_INVALID, "bad argument");
    CUDA_TRY(cudaSetDevice(s->device));
    // one packed block: sum | sumsq | count (12 B per cell), so that the all-reduce and the clear see contiguous memory
    size_t n = (size_t)width * height;
    float* block = nullptr;
    CUDA_TRY(cudaMalloc((void**)&block, 12 * n));
    ipt_plane* p = new ipt_plane();
    p->scene = s; p->width = width; p->height = height; p->owned = true;
    p->sum = block; p->sumsq = block + n; p->count = reinterpret_cast<uint32_t*>(block + 2 * n);
    int rc = ipt_plane_clear(p);
    if (rc) { ipt_plane_destroy(p); return rc; }
    *out = p;
    return IPT_OK;
}
int ipt_plane_wrap(ipt_scene* s, uint32_t width, uint32_t height, float* d_sum, float* d_sumsq, uint32_t* d_count, ipt_plane** out) {
    if (!s || !out || !width || !height || !d_sum || !d_sumsq || !d_count) return fail(IPT_ERR_INVALID, "bad argument");
    ipt_plane* p = new ipt_plane();
    p->scene = s; p->width = width; p->height = height; p->owned = false;
    p->sum = d_sum; p->sumsq = d_sumsq; p->count = d_count;
    *out = p;
    return IPT_OK;
}
int ipt_plane_clear(ipt_plane* p) {
    if (!p) return fail(IPT_ERR_INVALID, "null plane");
    std::lock_guard<std::recursive_mutex> lock__(p->scene->mu);
    CUDA_TRY(cudaSetDevice(p->scene->device));
    size_t n = (size_t)p->width * p->height;
    if (p->owned) CUDA_TRY(cudaMemsetAsync(p->sum, 0, 12 * n, p->scene->stream));
    else {
        CUDA_TRY(cudaMemsetAsync(p->sum, 0, 4 * n, p->scene->stream));
        CUDA_TRY(cudaMemsetAsync(p->sumsq, 0, 4 * n, p->scene->stream));
        CUDA_TRY(cudaMemsetAsync(p->count, 0, 4 * n, p->scene->stream));
    }
    CUDA_TRY(cudaStreamSynchronize(p->scene->stream));
    return IPT_OK;
}
int ipt_plane_add_rays(ipt_plane* p, uint32_t plane_mode, size_t n, const float* x, const float* y, const float* value) {
    if (!p || !x || !y || !value || plane_mode > IPT_PLANE_LINEAR) return fail(IPT_ERR_INVALID, "bad argument");
    std::lock_guard<std::recursive_mutex> lock__(p->scene->mu);
    if (n == 0) return IPT_OK;
    CUDA_TRY(cudaSetDevice(p->scene->device));
    cudaStream_t st = p->scene->stream;
    DevBuf<float> d_x, d_y, d_v;
    CUDA_TRY(d_x.alloc(n)); CUDA_TRY(d_y.alloc(n)); CUDA_TRY(d_v.alloc(n));
    CUDA_TRY(cudaMemcpyAsync(d_x.p, x, 4 * n, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(d_y.p, y, 4 * n, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(d_v.p, value, 4 * n, cudaMemcpyHostToDevice, st));
    RenderCtx C;
    std::memset(&C, 0, sizeof C);
    C.sum = p->sum; C.sumsq = p->sumsq; C.count = p->count;
    C.width = p->width; C.height = p->height; C.plane_mode = plane_mode;
    k_plane_add_rays<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(C, n, d_x.p, d_y.p, d_v.p);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaStreamSynchronize(st));
    return IPT_OK;
}
int ipt_plane_destroy(ipt_plane* p) {
    if (!p) return fail(IPT_ERR_INVALID, "null plane");
    if (p->owned) {
        cudaSetDevice(p->scene->device);
        cudaFree(p->sum); // the packed block
    }
    if (p->scene && p->scene->host_plane == p) p->scene->host_plane = nullptr;
    delete p;
    return IPT_OK;
}
int ipt_plane_download(ipt_plane* p, float* sum, float* sumsq, uint32_t* count) {
    if (!p) return fail(IPT_ERR_INVALID, "null plane");
    std::lock_guard<std::recursive_mutex> lock__(p->scene->mu);
    CUDA_TRY(cudaSetDevice(p->scene->device));
    size_t n = (size_t)p->width * p->height;
    cudaStream_t st = p->scene->stream;
    if (sum) CUDA_TRY(cudaMemcpyAsync(sum, p->sum, 4 * n, cudaMemcpyDeviceToHost, st));
    if (sumsq) CUDA_TRY(cudaMemcpyAsync(sumsq, p->sumsq, 4 * n, cudaMemcpyDeviceToHost, st));
    if (count) CUDA_TRY(cudaMemcpyAsync(count, p->count, 4 * n, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return IPT_OK;
}
int ipt_plane_upload(ipt_plane* p, const float* sum, const float* sumsq, const uint32_t* count) {
    if (!p || !sum || !sumsq || !count) return fail(IPT_ERR_INVALID, "null argument");
    std::lock_guard<std::recursive_mutex> lock__(p->scene->mu);
    CUDA_TRY(cudaSetDevice(p->scene->device));
    size_t n = (size_t)p->width * p->height;
    cudaStream_t st = p->scene->stream;
    CUDA_TRY(cudaMemcpyAsync(p->sum, sum, 4 * n, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(p->sumsq, sumsq, 4 * n, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(p->count, count, 4 * n, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return IPT_OK;
}
int ipt_plane_device_ptrs(ipt_plane* p, float** d_sum, float** d_sumsq, uint32_t** d_count) {
    if (!p) return fail(IPT_ERR_INVALID, "null plane");
    if (d_sum) *d_sum = p->sum;
    if (d_sumsq) *d_sumsq = p->sumsq;
    if (d_count) *d_count = p->count;
    return IPT_OK;
}
int ipt_plane_allreduce(ipt_plane* p, void* nccl_comm, float* ms) {
    if (!p || !nccl_comm) return fail(IPT_ERR_INVALID, "null argument");
    std::lock_guard<std::recursive_mutex> lock__(p->scene->mu);
    // ncclResult_t ncclAllReduce(const void* send, void* recv, size_t count, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t)
    typedef int (*allreduce_fn)(const void*, void*, size_t, int, int, void*, cudaStream_t);
    typedef int (*group_fn)(void);
    typedef const char* (*errstr_fn)(int);
    static allreduce_fn all_reduce = nullptr;
    static group_fn group_start = nullptr, group_end = nullptr;
    static errstr_fn err_string = nullptr;
    if (!all_reduce) {
        void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD); // the copy the host application already uses
        if (!h) h = dlopen("libnccl.so.2", RTLD_NOW);
        if (!h) h = dlopen("libnccl.so", RTLD_NOW);
        if (!h) return fail(IPT_ERR_UNSUPPORTED, "libnccl.so.2 is not loadable in this process");
        group_start = (group_fn)dlsym(h, "ncclGroupStart");
        group_end = (group_fn)dlsym(h, "ncclGroupEnd");
        err_string = (errstr_fn)dlsym(h, "ncclGetErrorString");
        all_reduce = (allreduce_fn)dlsym(h, "ncclAllReduce");
        if (!all_reduce || !group_start || !group_end) { all_reduce = nullptr; return fail(IPT_ERR_UNSUPPORTED, "ncclAllReduce / ncclGroupStart not found in libnccl"); }
    }
    CUDA_TRY(cudaSetDevice(p->scene->device));
    const size_t n = (size_t)p->width * p->height;
    cudaStream_t st = p->scene->stream;
    const int nccl_float32 = 7, nccl_uint32 = 3, nccl_sum = 0; // nccl.h: ncclFloat32, ncclUint32, ncclSum
    CUDA_TRY(cudaEventRecord(p->scene->ev_begin, st));
    // one grouped launch: the float accumulators (one call when they are contiguous, as in a library-owned plane) + the counters
    int rc = group_start();
    if (!rc) {
        if (p->sumsq == p->sum + n) rc = all_reduce(p->sum, p->sum, 2 * n, nccl_float32, nccl_sum, nccl_comm, st);
        else {
            rc = all_reduce(p->sum, p->sum, n, nccl_float32, nccl_sum, nccl_comm, st);
            if (!rc) rc = all_reduce(p->sumsq, p->sumsq, n, nccl_float32, nccl_sum, nccl_comm, st);
        }
        if (!rc) rc = all_reduce(p->count, p->count, n, nccl_uint32, nccl_sum, nccl_comm, st);
        int rc2 = group_end();
        if (!rc) rc = rc2;
    }
    if (rc) return fail(IPT_ERR_CUDA, std::string("ncclAllReduce: ") + (err_string ? err_string(rc) : "error"));
    CUDA_TRY(cudaEventRecord(p->scene->ev_end, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (ms) CUDA_TRY(cudaEventElapsedTime(ms, p->scene->ev_begin, p->scene->ev_end));
    return IPT_OK;
}
int ipt_plane_merge(ipt_plane* dst, ipt_plane* src) {
    if (!dst || !src) return fail(IPT_ERR_INVALID, "null plane");
    if (dst == src) return fail(IPT_ERR_INVALID, "a plane cannot be merged into itself");
    if (dst->width != src->width || dst->height != src->height) return fail(IPT_ERR_INVALID, "planes of different frame sizes");
    // both scenes are locked (in address order: two threads merging in opposite directions cannot deadlock)
    ipt_scene* a = dst->scene < src->scene ? dst->scene : src->scene;
    ipt_scene* b = dst->scene < src->scene ? src->scene : dst->scene;
    std::lock_guard<std::recursive_mutex> lock_a(a->mu);
    std::lock_guard<std::recursive_mutex> lock_b(b->mu);
    const size_t n = (size_t)dst->width * dst->height;
    const int ddev = dst->scene->device, sdev = src->scene->device;
    CUDA_TRY(cudaSetDevice(sdev));
    CUDA_TRY(cudaStreamSynchronize(src->scene->stream)); // src's last render / merge has landed
    CUDA_TRY(cudaSetDevice(ddev));
    cudaStream_t st = dst->scene->stream;
    const float *s2 = src->sum, *q2 = src->sumsq;
    const uint32_t* c2 = src->count;
    DevBuf<float> staged;
    if (ddev != sdev) {
        CUDA_TRY(staged.alloc(3 * n));
        CUDA_TRY(cudaMemcpyPeerAsync(staged.p, ddev, src->sum, sdev, 4 * n, st));
        CUDA_TRY(cudaMemcpyPeerAsync(staged.p + n, ddev, src->sumsq, sdev, 4 * n, st));
        CUDA_TRY(cudaMemcpyPeerAsync(staged.p + 2 * n, ddev, src->count, sdev, 4 * n, st));
        s2 = staged.p; q2 = staged.p + n; c2 = reinterpret_cast<const uint32_t*>(staged.p + 2 * n);
    }
    int blocks = (int)std::min<size_t>((n + 255) / 256, (size_t)dst->scene->sm_count * 8);
    k_plane_merge<<<blocks, 256, 0, st>>>(dst->sum, dst->sumsq, dst->count, s2, q2, c2, n);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaStreamSynchronize(st));
    return IPT_OK;
}
int ipt_plane_resolve(ipt_plane* p, float* pixels, uint64_t* pixel_counters, float* max_value) {
    if (!p || !pixels) return fail(IPT_ERR_INVALID, "null argument");
    std::lock_guard<std::recursive_mutex> lock__(p->scene->mu);
    CUDA_TRY(cudaSetDevice(p->scene->device));
    size_t n = (size_t)p->width * p->height;
    DevBuf<float> d_pix;
    CUDA_TRY(d_pix.alloc(n));
    k_plane_resolve<<<(unsigned)((n + 255) / 256), 256, 0, p->scene->stream>>>(p->sum, p->count, n, d_pix.p);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(pixels, d_pix.p, 4 * n, cudaMemcpyDeviceToHost, p->scene->stream));
    std::vector<uint32_t> cnt;
    if (pixel_counters) {
        cnt.resize(n);
        CUDA_TRY(cudaMemcpyAsync(cnt.data(), p->count, 4 * n, cudaMemcpyDeviceToHost, p->scene->stream));
    }
    CUDA_TRY(cudaStreamSynchronize(p->scene->stream));
    if (pixel_counters) for (size_t i = 0; i < n; ++i) pixel_counters[i] = cnt[i];
    if (max_value) {
        float m = 0.0f; // GridRenderPlane::max_value starts at 0 (GridRenderPlane.h:12)
        for (size_t i = 0; i < n; ++i) m = std::max(m, pixels[i]);
        *max_value = m;
    }
    return IPT_OK;
}

// ---- the hot path ------------------------------------------------------------------------------------------
void ipt_render_params_default(ipt_render_params* p) {
    if (!p) return;
    std::memset(p, 0, sizeof *p);
    p->width = 640; p->height = 640; // main.cpp:189-190
    p->depth_max = 4;                // main.cpp:95
    p->schedule[0] = 16; p->schedule[1] = 8; p->schedule[2] = 4; p->schedule[3] = 2; // main.cpp:94,177 (n_rays/2)
    p->seed = 0;
    p->pass_begin = 0; p->pass_count = 1;
    p->plane_mode = IPT_PLANE_GRID;
}

static size_t workspace_bytes(size_t ray_cap, size_t hit_cap, size_t path_cap, bool two_hit_sets) {
    return 36 * ray_cap + 32 * std::max<size_t>(hit_cap, 1) * (two_hit_sets ? 2 : 1) + 4 * path_cap;
}
// IPT_OK, IPT_ERR_OVERFLOW when the device cannot hold this workspace (the caller retries with a smaller batch), or an error
static int ensure_workspace(ipt_scene* s, size_t ray_cap, size_t hit_cap, size_t path_cap, bool two_hit_sets) {
    Workspace& w = s->ws;
    if (w.ray_cap >= ray_cap && w.hit_cap >= hit_cap && w.path_cap >= path_cap && (w.two_hit_sets || !two_hit_sets)) return IPT_OK;
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    free_workspace(w);
    void** slots[8] = {(void**)&w.ray_o, (void**)&w.ray_d, (void**)&w.ray_x, (void**)&w.hit_a, (void**)&w.hit_b, (void**)&w.pathval, (void**)&w.hit_a2, (void**)&w.hit_b2};
    const size_t bytes[8] = {16 * ray_cap, 16 * ray_cap, 4 * ray_cap, 16 * std::max<size_t>(hit_cap, 1), 16 * std::max<size_t>(hit_cap, 1), 4 * path_cap,
                             16 * std::max<size_t>(hit_cap, 1), 16 * std::max<size_t>(hit_cap, 1)};
    for (int k = 0; k < (two_hit_sets ? 8 : 6); ++k) {
        cudaError_t e = cudaMalloc(slots[k], bytes[k]);
        if (e == cudaErrorMemoryAllocation) {
            cudaGetLastError();
            free_workspace(w);
            return fail(IPT_ERR_OVERFLOW, "the device cannot hold the queue workspace of this batch size");
        }
        if (e != cudaSuccess) { free_workspace(w); return fail(IPT_ERR_CUDA, std::string("cudaMalloc (workspace): ") + cudaGetErrorString(e)); }
    }
    w.ray_cap = ray_cap; w.hit_cap = hit_cap; w.path_cap = path_cap; w.two_hit_sets = two_hit_sets;
    return IPT_OK;
}

// The paths per batch of a render (`requested`, or a default from the widest tree levels), and the scene's workspace
// grown to hold the queues of one batch
static int size_batch(ipt_scene* s, uint64_t requested, uint64_t total_paths, uint64_t tile_pixels, uint64_t max_ray_w,
                      uint64_t max_queued_w, uint64_t max_hit_w, uint32_t slot_bits, bool fuse_next, uint64_t& batch) {
    // default batch: as many paths as keep the widest tree level near 2^28 rays (2^19 paths at 16/8/4/2; up to 2^23
    // for narrow schedules such as depth 8 with one child per hit, whose deeper levels would otherwise be tiny launches)
    // (with the fused last level the widest level is not queued: 2^27 / widest queued level, i.e. 2^20 paths at 16/8/4/2)
    // (fused shade kernels: what is queued are the hits, 2^28 / widest hit level = 2^21 paths at 16/8/4/2, 17 GB of
    // hit records in the two sets; 2^20 paths is 1.5 % slower, 2^22 0.3 % faster)
    uint64_t batch_rays = (max_queued_w < max_ray_w && !fuse_next) ? (1ull << 27) : (1ull << 28);
    uint64_t batch_w = fuse_next ? max_hit_w : max_queued_w;
    // (narrow schedules such as depth 8 with one child per hit: up to 2^25 paths. Every launch of the persistent mesh kernel
    // ends with its longest ray — ~1000 dependent node visits walked by a single lane, ~0.9 ms whatever the launch holds —
    // so eight launches per batch want as many rays per launch as memory allows: 2^23 / 2^24 / 2^25 paths per batch give
    // C3 325 / 369 / 376 and C4 290 / 322 / 332 Mpaths/s; 2^25 paths are 2.4 GB of queues)
    batch = requested ? requested : std::min<uint64_t>(1ull << 25, std::max<uint64_t>(1ull << 16, batch_rays / batch_w));
    batch = std::min<uint64_t>(batch, slot_bits >= 32 ? 0xFFFFFFFFull : (1ull << slot_bits));
    // Queue memory is sized for the worst case of a batch (no overflow path). Budget: IPT_QUEUE_BUDGET_GB (default 24 GiB:
    // 2^21 paths at 16/8/4/2 need 2 x 8.6 GB of hit records; halving the batch costs ~1.5 %, profiles/tuning_r02.md), never
    // more than 80 % of what the device has free right now (plus what this scene's workspace already holds), and the
    // batch is halved again whenever the allocation itself fails.
    uint64_t budget = 24ull << 30;
    if (const char* e = std::getenv("IPT_QUEUE_BUDGET_GB")) { double gb = std::atof(e); if (gb > 0) budget = (uint64_t)(gb * (double)(1ull << 30)); }
    Workspace& ws = s->ws;
    const uint64_t choice_key[5] = {batch, max_queued_w, max_hit_w, budget, fuse_next ? 1ull : 0ull};
    if (ws.choice_batch && ws.path_cap && std::memcmp(choice_key, ws.choice_key, sizeof choice_key) == 0) {
        batch = ws.choice_batch; // same question as last time, and a workspace it led to is still allocated
    } else {
        size_t free_b = 0, total_b = 0;
        if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess) {
            uint64_t held = ws.path_cap ? workspace_bytes(ws.ray_cap, ws.hit_cap, ws.path_cap, ws.two_hit_sets) : 0;
            budget = std::min<uint64_t>(budget, (uint64_t)((double)(free_b + held) * 0.8));
        } else cudaGetLastError();
        while (batch > 1024 && workspace_bytes(batch * max_queued_w, batch * max_hit_w, batch, fuse_next) > budget) batch >>= 1;
    }
    const uint64_t batch_unclamped = batch;
    batch = std::max<uint64_t>(1, std::min<uint64_t>(batch, std::max<uint64_t>(total_paths, 1)));
    if (tile_pixels + batch > 0xFFFFFFFFull) return fail(IPT_ERR_UNSUPPORTED, "tile too large: tile pixels + batch must stay below 2^32");
    bool alloc_halved = false;
    for (;;) {
        int rc = ensure_workspace(s, batch * max_queued_w, batch * max_hit_w, batch, fuse_next);
        if (rc == IPT_OK) break;
        if (rc != IPT_ERR_OVERFLOW || batch <= 1024) return rc;
        batch >>= 1; // another tenant (torch, NCCL) took the memory between the query and the allocation
        alloc_halved = true;
    }
    if (!alloc_halved) {
        std::memcpy(ws.choice_key, choice_key, sizeof choice_key);
        ws.choice_batch = batch_unclamped;
    }
    return IPT_OK;
}

int ipt_render(ipt_scene* s, ipt_plane* plane, const ipt_render_params* p, ipt_render_stats* stats) {
    if (!s || !plane || !p) return fail(IPT_ERR_INVALID, "null argument");
    std::lock_guard<std::recursive_mutex> lock__(s->mu);
    if (plane->scene != s) return fail(IPT_ERR_INVALID, "plane belongs to another scene");
    if (!p->width || !p->height || plane->width != p->width || plane->height != p->height)
        return fail(IPT_ERR_INVALID, "plane size does not match render params");
    if (p->depth_max == 0 || p->depth_max > IPT_MAX_DEPTH) return fail(IPT_ERR_INVALID, "depth_max out of range");
    if ((uint64_t)p->width * p->height > 0xFFFFFFFFull) return fail(IPT_ERR_INVALID, "frame too large");
    uint32_t tx0 = p->tile_w ? p->tile_x0 : 0, ty0 = p->tile_w ? p->tile_y0 : 0;
    uint32_t tw = p->tile_w ? p->tile_w : p->width, th = p->tile_w ? p->tile_h : p->height;
    if (!tw || !th || tx0 + tw > p->width || ty0 + th > p->height) return fail(IPT_ERR_INVALID, "tile outside the frame");
    if (p->plane_mode > IPT_PLANE_LINEAR) return fail(IPT_ERR_INVALID, "unknown plane mode");
#ifndef IPT_DEBUG_PRINT
    if (p->flags & IPT_FLAG_DEBUG_PRINT) return fail(IPT_ERR_UNSUPPORTED, "IPT_FLAG_DEBUG_PRINT needs a library built with -DIPT_DEBUG_PRINT (the device printf is compiled out of the production kernels)");
#endif
    CUDA_TRY(cudaSetDevice(s->device));

    // analytic scenes: the shade kernels trace the children they spawn (FUSE_NEXT / FUSE_LAST in ipt_kernels.cuh)
    const bool fuse_last = !s->mesh && !(p->flags & (IPT_FLAG_DEBUG_PRINT | IPT_FLAG_RESOLVE_LAST_LEVEL | IPT_FLAG_NO_FUSED_LAST_LEVEL));
    const bool fuse_next = fuse_last && !(p->flags & IPT_FLAG_NO_FUSED_TRACE);
    // widest tree level among traced depths -> bits for the node index inside the ray tag
    uint64_t width_at[IPT_MAX_DEPTH];
    uint64_t w = 1, max_ray_w = 1, max_hit_w = 1, max_queued_w = 1;
    for (uint32_t d = 0; d < p->depth_max; ++d) {
        width_at[d] = w;
        max_ray_w = std::max(max_ray_w, w);
        // with the fused last level the rays of the last traced depth (> 0) are never queued
        bool is_last = d + 1 == p->depth_max || p->schedule[d] == 0;
        if (!(fuse_last && is_last && d > 0) && !(fuse_next && d > 0)) max_queued_w = std::max(max_queued_w, w);
        if (d + 1 < p->depth_max) max_hit_w = std::max(max_hit_w, w);
        w *= p->schedule[d];
        if (w > (1ull << 31)) return fail(IPT_ERR_UNSUPPORTED, "split schedule too wide (more than 2^31 nodes per tree level)");
        if (w == 0 && d + 1 < p->depth_max) { /* schedule[d]==0: deeper levels never exist */
            for (uint32_t e = d + 1; e < p->depth_max; ++e) width_at[e] = 0;
            break;
        }
    }
    uint32_t idx_bits = 0;
    while ((1ull << idx_bits) < max_ray_w) ++idx_bits;
    uint32_t slot_bits = 32 - idx_bits;
    uint64_t total_paths = (uint64_t)tw * th * p->pass_count;
    uint64_t batch = 0;
    int rc = size_batch(s, p->batch_paths, total_paths, (uint64_t)tw * th, max_ray_w, max_queued_w, max_hit_w, slot_bits, fuse_next, batch);
    if (rc) return rc;

    const Workspace& W = s->ws;
    RenderCtx C;
    std::memset(&C, 0, sizeof C);
    C.ray_o = W.ray_o; C.ray_d = W.ray_d; C.ray_x = W.ray_x; C.pathval = W.pathval;
    C.hit_a[0] = W.hit_a; C.hit_b[0] = W.hit_b;
    C.hit_a[1] = fuse_next ? W.hit_a2 : W.hit_a; C.hit_b[1] = fuse_next ? W.hit_b2 : W.hit_b;
    C.cnt = s->d_cnt; C.fetch = C.cnt + (2 * IPT_MAX_DEPTH + 2);
    C.stats = s->d_stats;
    C.sum = plane->sum; C.sumsq = plane->sumsq; C.count = plane->count;
    C.ray_cap = (uint32_t)std::min<size_t>(W.ray_cap, 0xFFFFFFFFull); C.hit_cap = (uint32_t)std::min<size_t>(W.hit_cap, 0xFFFFFFFFull);
    C.width = p->width; C.height = p->height;
    C.tile_x0 = tx0; C.tile_y0 = ty0; C.tile_w = tw; C.tile_h = th; C.tile_pixels = tw * th;
    C.pass_begin = p->pass_begin;
    C.slot_bits = slot_bits;
    C.slot_mask = slot_bits >= 32 ? 0xFFFFFFFFu : ((1u << slot_bits) - 1u);
    C.depth_max = p->depth_max;
    std::memcpy(C.schedule, p->schedule, sizeof C.schedule);
    philox_keys(p->seed, C.keys);
    C.div_tile_pixels = make_fastdiv(C.tile_pixels);
    C.div_tile_w = make_fastdiv(C.tile_w);
    C.plane_mode = p->plane_mode; C.flags = p->flags;

    const cudaStream_t st = s->stream;
    const bool timing = (p->flags & IPT_FLAG_TIME_KERNELS) != 0;
    bool timing_failed = false;
    std::vector<int> ev_kind; // 0 generate 1 extend 2 shade 3 accumulate, one entry per bracketed launch
    size_t ev_used = 0;
    auto ev_next = [&]() -> cudaEvent_t {
        if (ev_used == s->events.size()) {
            cudaEvent_t e = nullptr;
            if (cudaEventCreate(&e) != cudaSuccess) { timing_failed = true; return s->ev_begin; }
            s->events.push_back(e);
        }
        return s->events[ev_used++];
    };
    uint32_t launches = 0;
    auto timed = [&](int kind, auto&& launch) { // one launch, bracketed by events when the kernels are timed
        if (timing) cudaEventRecord(ev_next(), st);
        launch();
        ++launches;
        if (timing) { cudaEventRecord(ev_next(), st); ev_kind.push_back(kind); }
    };
    // a kernel of the scene's table at depth d, never with more blocks than the level has rays for
    auto run = [&](const RenderKernel& k, int kind, uint32_t d, int cap_blocks) {
        timed(kind, [&] { k.kernel<<<std::max(1, std::min(k.grid, cap_blocks)), IPT_BLOCK, k.smem, st>>>(s->dev, C, d); });
    };
    CUDA_TRY(cudaMemsetAsync(s->d_stats, 0, sizeof(unsigned long long) * ST_COUNT, st));
    CUDA_TRY(cudaEventRecord(s->ev_begin, st));
    uint32_t batches = 0;
    for (uint64_t g0 = 0; g0 < total_paths; g0 += batch, ++batches) {
        C.g0 = g0;
        C.pass0 = p->pass_begin + (uint32_t)(g0 / C.tile_pixels);
        C.rem0 = (uint32_t)(g0 % C.tile_pixels);
        C.batch = (uint32_t)std::min<uint64_t>(batch, total_paths - g0);
        CUDA_TRY(cudaMemsetAsync(C.cnt, 0, sizeof(uint32_t) * IPT_CNT_WORDS, st));
        int gg = std::min<int>(s->grid_generate, (int)((C.batch + IPT_BLOCK - 1) / IPT_BLOCK));
        timed(0, [&] { k_generate<<<gg, IPT_BLOCK, 0, st>>>(s->dev, C); });
        bool traced = false; // the shade kernel of the previous depth has already traced the rays of this depth
        for (uint32_t d = 0; d < p->depth_max; ++d) {
            if (width_at[d] == 0) break;
            bool last = (d + 1 == p->depth_max) || p->schedule[d] == 0;
            uint64_t max_rays = (uint64_t)C.batch * width_at[d];
            int cap_blocks = (int)std::min<uint64_t>((max_rays + IPT_BLOCK - 1) / IPT_BLOCK, 1u << 30);
            // camera rays are traced with the reference's exact arithmetic; rays downstream of a random number with the
            // contracted form the fused shade kernels use too (so fused and queued runs agree ray for ray)
            const bool exact_d = d == 0 || !IPT_FAST_SECONDARY;
            if (!traced) { // the rays of this depth wait in the ray queue (depth 0, or an unfused run)
                run(s->extend[last][exact_d], 1, d, cap_blocks);
                if (last) break;
            }
            traced = false;
            // the children of this level are the last traced depth: resolve them inside the shade kernel (no queue, no
            // k_extend<LAST> launch); analytic scenes only, and not when a flag asks for the unfused behaviour
            bool child_last = width_at[d + 1] != 0 && ((d + 2 == p->depth_max) || p->schedule[d + 1] == 0);
            if (child_last && fuse_last) {
                run(s->shade_last, 2, d, cap_blocks);
                break;
            }
            if (fuse_next && width_at[d + 1] != 0) {
                run(s->shade_next, 2, d, cap_blocks);
                traced = true; // the rays of depth d+1 are traced by this launch: no k_extend for them
                continue;
            }
            run(s->shade, 2, d, cap_blocks);
        }
        timed(3, [&] { k_accumulate<<<std::max(1, gg), IPT_BLOCK, 0, st>>>(C); });
        CUDA_TRY(cudaGetLastError());
    }
    CUDA_TRY(cudaEventRecord(s->ev_end, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaGetLastError());

#ifdef IPT_DEBUG_BOUNDS
    {
        unsigned long long over = 0;
        CUDA_TRY(cudaMemcpy(&over, s->d_stats + ST_OVERFLOW, sizeof over, cudaMemcpyDeviceToHost));
        if (over) return fail(IPT_ERR_OVERFLOW, std::to_string(over) + " queue append(s) beyond the allocated capacity (IPT_DEBUG_BOUNDS build)");
    }
#endif
    if (stats) {
        std::memset(stats, 0, sizeof *stats);
        unsigned long long h[ST_COUNT];
        CUDA_TRY(cudaMemcpy(h, s->d_stats, sizeof h, cudaMemcpyDeviceToHost));
        stats->paths = h[ST_PATHS];
        for (int d = 0; d < IPT_MAX_DEPTH; ++d) {
            stats->rays_at_depth[d] = h[ST_RAYS_AT_DEPTH + d];
            stats->rays += h[ST_RAYS_AT_DEPTH + d];
        }
        stats->surface_hits = h[ST_SURFACE];
        stats->light_hits = h[ST_LIGHT];
        stats->misses = h[ST_MISS];
        stats->failed_samples = h[ST_FAILED];
        stats->zero_weight_pruned = h[ST_PRUNED];
        stats->nonfinite_dropped = h[ST_DROPPED];
        stats->bvh_nodes_visited = h[ST_NODES];
        stats->triangles_tested = h[ST_TRIS];
        stats->lights_tested = h[ST_LIGHTS];
        stats->light_bvh_nodes_visited = h[ST_LIGHT_NODES];
        stats->batches = batches;
        stats->kernel_launches = launches;
        CUDA_TRY(cudaEventElapsedTime(&stats->ms_total, s->ev_begin, s->ev_end));
        if (timing && !timing_failed) {
            for (size_t k = 0; k < ev_kind.size(); ++k) {
                float ms = 0;
                cudaEventElapsedTime(&ms, s->events[2 * k], s->events[2 * k + 1]);
                switch (ev_kind[k]) {
                    case 0: stats->ms_generate += ms; break;
                    case 1: stats->ms_extend += ms; ++stats->n_extend; break;
                    case 2: stats->ms_shade += ms; ++stats->n_shade; break;
                    default: stats->ms_accumulate += ms; break;
                }
            }
        }
        // ray record written + read (2 x 36 B) per ray, hit record written + read per QUEUED surface hit, pathval RMW
        stats->queue_bytes = 72ull * stats->rays + 64ull * h[ST_QUEUED] + 8ull * stats->paths;
        stats->rays_resolved_in_shade = h[ST_FUSED];
    }
    return IPT_OK;
}

int ipt_render_host(ipt_scene* s, const ipt_render_params* p, float* sum, float* sumsq, uint32_t* count, ipt_render_stats* stats) {
    if (!s || !p || !sum) return fail(IPT_ERR_INVALID, "null argument");
    std::lock_guard<std::recursive_mutex> lock__(s->mu);
    if (s->host_plane && (s->host_plane->width != p->width || s->host_plane->height != p->height)) {
        ipt_plane_destroy(s->host_plane);
        s->host_plane = nullptr;
    }
    if (!s->host_plane) {
        int rc = ipt_plane_create(s, p->width, p->height, &s->host_plane);
        if (rc) return rc;
    } else {
        int rc = ipt_plane_clear(s->host_plane);
        if (rc) return rc;
    }
    int rc = ipt_render(s, s->host_plane, p, stats);
    if (rc) return rc;
    return ipt_plane_download(s->host_plane, sum, sumsq, count);
}

} // extern "C"

#include "ipt_output.cuh"
