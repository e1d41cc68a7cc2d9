// ipt_lbvh.cuh — GPU-built linear BVH over the triangle mesh (BASELINE.json north_star item 1):
// Morton codes + hand-written LSD radix sort + Karras 2012 hierarchy + bottom-up refit. Integer work is
// bit-exact by construction; the few float steps (bounds, centroid quantisation, padding) use explicit
// round-to-nearest intrinsics in a fixed order so that oracle/ipt_oracle_mesh.inc reproduces every byte.
// The reference has no acceleration structure (it scans linearly: FractalSpheres.cpp:75-84,
// GeometrySmallPt.cpp:39-47); parity for this file is against our own CPU restatement (SURVEY.md §8c).
#pragma once
#include "ipt_device.cuh"

#include <cmath>
#include <string>

namespace iptd {

struct LbvhDevice {
    uint32_t n = 0;
    float4* tri_records = nullptr;       // 4 float4 (64 B) per sorted triangle (see DevScene::tris)
    uint32_t* sorted_ids = nullptr;      // sorted position -> original index
    unsigned long long* sorted_keys = nullptr; // 63-bit Morton keys, ascending
    BvhNode* nodes = nullptr;            // n-1 internal nodes, root = 0
    BvhNodeQ* qnodes = nullptr;          // the same nodes in the 32-byte traversal form
    GridMap grid{};                      // world -> grid space of qnodes
};

// order-preserving float <-> uint map for atomicMin/atomicMax
__device__ __forceinline__ uint32_t f2ord(float f) { uint32_t b = __float_as_uint(f); return (b & 0x80000000u) ? ~b : (b | 0x80000000u); }
__device__ __forceinline__ float ord2f(uint32_t u) { return __uint_as_float((u & 0x80000000u) ? (u & 0x7FFFFFFFu) : ~u); }

// per triangle: tight box of (v0, v0+e1, v0+e2); scene bounds of the box centres
__global__ void k_lbvh_bounds(const float* __restrict__ tris, uint32_t n, float4* lo, float4* hi, uint32_t* cbounds /*[6] ord: min xyz, max xyz*/,
                              const float* __restrict__ extra /* per primitive (kind, area, weight) or null; kind 0 = parallelogram */) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t mn[3] = {0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu}, mx[3] = {0, 0, 0};
    if (i < n) {
        const float* t = tris + 9 * (size_t)i;
        float l[3], h[3];
        for (int a = 0; a < 3; ++a) {
            float v0 = t[a], v1 = xadd(t[a], t[3 + a]), v2 = xadd(t[a], t[6 + a]);
            l[a] = fminf(v0, fminf(v1, v2));
            h[a] = fmaxf(v0, fmaxf(v1, v2));
            if (extra && extra[3 * (size_t)i] == 0.0f) { // parallelogram ("diamond" area light): the fourth corner
                float v3 = xadd(v1, t[6 + a]);
                l[a] = fminf(l[a], v3);
                h[a] = fmaxf(h[a], v3);
            }
            float c = xmul(xadd(l[a], h[a]), 0.5f);
            mn[a] = mx[a] = f2ord(c);
        }
        lo[i] = make_float4(l[0], l[1], l[2], 0.0f);
        hi[i] = make_float4(h[0], h[1], h[2], 0.0f);
    }
    for (int a = 0; a < 3; ++a) {
        uint32_t vmin = mn[a], vmax = mx[a];
        for (int off = 16; off > 0; off >>= 1) {
            vmin = min(vmin, __shfl_xor_sync(0xffffffffu, vmin, off));
            vmax = max(vmax, __shfl_xor_sync(0xffffffffu, vmax, off));
        }
        if ((threadIdx.x & 31) == 0) {
            atomicMin(&cbounds[a], vmin);
            atomicMax(&cbounds[3 + a], vmax);
        }
    }
}

__device__ __forceinline__ unsigned long long expand21(uint32_t v) { // spread 21 bits to every third bit
    unsigned long long x = v & 0x1FFFFFull;
    x = (x | x << 32) & 0x1F00000000FFFFull;
    x = (x | x << 16) & 0x1F0000FF0000FFull;
    x = (x | x << 8) & 0x100F00F00F00F00Full;
    x = (x | x << 4) & 0x10C30C30C30C30C3ull;
    x = (x | x << 2) & 0x1249249249249249ull;
    return x;
}

__global__ void k_lbvh_morton(const float4* __restrict__ lo, const float4* __restrict__ hi, uint32_t n, const uint32_t* __restrict__ cbounds,
                              unsigned long long* keys, uint32_t* ids) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float4 l = lo[i], h = hi[i];
    float c[3] = {xmul(xadd(l.x, h.x), 0.5f), xmul(xadd(l.y, h.y), 0.5f), xmul(xadd(l.z, h.z), 0.5f)};
    uint32_t q[3];
    for (int a = 0; a < 3; ++a) {
        float cmin = ord2f(cbounds[a]), cmax = ord2f(cbounds[3 + a]);
        float ext = xsub(cmax, cmin);
        float f = ext > 0.0f ? xdiv(xsub(c[a], cmin), ext) : 0.0f;
        float v = xmul(f, 2097152.0f);
        v = fminf(fmaxf(v, 0.0f), 2097151.0f);
        q[a] = (uint32_t)v; // truncation
    }
    keys[i] = (expand21(q[0]) << 2) | (expand21(q[1]) << 1) | expand21(q[2]);
    ids[i] = i;
}

// ---- LSD radix sort, 8-bit digits, stable; one tile of RS_TILE consecutive elements per block ---------
#define RS_THREADS 256
#define RS_ITEMS 8
#define RS_TILE (RS_THREADS * RS_ITEMS)

__global__ void __launch_bounds__(RS_THREADS) k_rs_hist(const unsigned long long* __restrict__ keys, uint32_t n, int shift, uint32_t nb,
                                                       uint32_t* counters) {
    __shared__ uint32_t hist[256];
    hist[threadIdx.x] = 0;
    __syncthreads();
    uint32_t base = blockIdx.x * RS_TILE;
    for (int k = 0; k < RS_ITEMS; ++k) {
        uint32_t i = base + k * RS_THREADS + threadIdx.x;
        if (i < n) atomicAdd(&hist[(uint32_t)(keys[i] >> shift) & 255u], 1u);
    }
    __syncthreads();
    counters[threadIdx.x * nb + blockIdx.x] = hist[threadIdx.x]; // digit-major
}

// exclusive scan of m counters by ONE block (m = 256 * tiles, a few million at most)
__global__ void __launch_bounds__(1024) k_rs_scan(uint32_t* counters, uint32_t m) {
    __shared__ uint32_t part[1024];
    uint32_t per = (m + 1023u) / 1024u;
    uint32_t lo = min(threadIdx.x * per, m), hi = min(lo + per, m);
    uint32_t s = 0;
    for (uint32_t i = lo; i < hi; ++i) s += counters[i];
    part[threadIdx.x] = s;
    __syncthreads();
    for (uint32_t off = 1; off < 1024; off <<= 1) { // Hillis-Steele inclusive
        uint32_t v = threadIdx.x >= off ? part[threadIdx.x - off] : 0;
        __syncthreads();
        part[threadIdx.x] += v;
        __syncthreads();
    }
    uint32_t run = threadIdx.x ? part[threadIdx.x - 1] : 0;
    for (uint32_t i = lo; i < hi; ++i) {
        uint32_t c = counters[i];
        counters[i] = run;
        run += c;
    }
}

__global__ void __launch_bounds__(RS_THREADS) k_rs_scatter(const unsigned long long* __restrict__ keys_in, const uint32_t* __restrict__ vals_in,
                                                          unsigned long long* keys_out, uint32_t* vals_out, uint32_t n, int shift, uint32_t nb,
                                                          const uint32_t* __restrict__ offsets) {
    __shared__ uint32_t whist[RS_THREADS / 32][256];
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (uint32_t k = threadIdx.x; k < (RS_THREADS / 32) * 256; k += RS_THREADS) (&whist[0][0])[k] = 0;
    __syncthreads();
    const uint32_t per_warp = RS_TILE / (RS_THREADS / 32); // consecutive elements owned by one warp
    const uint32_t wbase = blockIdx.x * RS_TILE + warp * per_warp;
    // A: per-warp digit histograms (one leader per distinct digit and step: no atomics)
    for (uint32_t st = 0; st < per_warp / 32; ++st) {
        uint32_t i = wbase + st * 32 + lane;
        uint32_t digit = i < n ? ((uint32_t)(keys_in[i] >> shift) & 255u) : 0xFFFFu;
        uint32_t peers = __match_any_sync(0xffffffffu, digit);
        if (digit != 0xFFFFu && lane == (uint32_t)(__ffs(peers) - 1)) whist[warp][digit] += __popc(peers);
        __syncwarp();
    }
    __syncthreads();
    // B: turn counts into output bases: global (digit, tile) offset, then warps of the tile in order
    {
        uint32_t d = threadIdx.x;
        uint32_t run = offsets[d * nb + blockIdx.x];
        for (uint32_t w = 0; w < RS_THREADS / 32; ++w) {
            uint32_t c = whist[w][d];
            whist[w][d] = run;
            run += c;
        }
    }
    __syncthreads();
    // C: replay in the same order; rank inside a step = number of lower lanes with the same digit
    for (uint32_t st = 0; st < per_warp / 32; ++st) {
        uint32_t i = wbase + st * 32 + lane;
        unsigned long long key = i < n ? keys_in[i] : 0ull;
        uint32_t digit = i < n ? ((uint32_t)(key >> shift) & 255u) : 0xFFFFu;
        uint32_t peers = __match_any_sync(0xffffffffu, digit);
        uint32_t rank = __popc(peers & ((1u << lane) - 1u));
        if (digit != 0xFFFFu) {
            uint32_t pos = whist[warp][digit] + rank;
            keys_out[pos] = key;
            vals_out[pos] = vals_in[i];
        }
        __syncwarp();
        if (digit != 0xFFFFu && lane == (uint32_t)(__ffs(peers) - 1)) whist[warp][digit] += __popc(peers);
        __syncwarp();
    }
}

// ---- Karras 2012: one thread per internal node ----------------------------------------------------------
__device__ __forceinline__ int lbvh_delta(const unsigned long long* __restrict__ keys, uint32_t n, long long i, long long j) {
    if (j < 0 || j >= (long long)n) return -1;
    unsigned long long a = keys[i], b = keys[j];
    if (a == b) return 64 + __clz((uint32_t)i ^ (uint32_t)j); // duplicate keys: fall back to the sorted position
    return __clzll((long long)(a ^ b));
}

__global__ void k_lbvh_hierarchy(const unsigned long long* __restrict__ keys, uint32_t n, BvhNode* nodes, uint32_t* leaf_parent) {
    uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n - 1) return;
    long long i = idx;
    int d = (lbvh_delta(keys, n, i, i + 1) - lbvh_delta(keys, n, i, i - 1)) > 0 ? 1 : -1;
    int dmin = lbvh_delta(keys, n, i, i - d);
    long long lmax = 2;
    while (lbvh_delta(keys, n, i, i + lmax * d) > dmin) lmax *= 2;
    long long l = 0;
    for (long long t = lmax / 2; t >= 1; t /= 2)
        if (lbvh_delta(keys, n, i, i + (l + t) * d) > dmin) l += t;
    long long j = i + l * d;
    int dnode = lbvh_delta(keys, n, i, j);
    long long s = 0, t = l;
    do {
        t = (t + 1) / 2;
        if (lbvh_delta(keys, n, i, i + (s + t) * d) > dnode) s += t;
    } while (t > 1);
    long long gamma = i + s * d + (d < 0 ? d : 0);
    long long lo = i < j ? i : j, hi = i < j ? j : i;
    uint32_t left = (lo == gamma) ? (0x80000000u | (uint32_t)gamma) : (uint32_t)gamma;
    uint32_t right = (hi == gamma + 1) ? (0x80000000u | (uint32_t)(gamma + 1)) : (uint32_t)(gamma + 1);
    nodes[idx].left = left;
    nodes[idx].right = right;
    nodes[idx].pad = 0;
    if (idx == 0) nodes[0].parent = IPT_NO_HIT;
    if (left & 0x80000000u) leaf_parent[gamma] = idx; else nodes[gamma].parent = idx;
    if (right & 0x80000000u) leaf_parent[gamma + 1] = idx; else nodes[gamma + 1].parent = idx;
}

// leaf box = triangle box padded by 2^-17 * (1 + max |coordinate|): conservative against the rounding of the
// exact intersection routine, so that traversal can never cull a triangle the linear scan would hit
__device__ __forceinline__ void padded_box(float4 l, float4 h, float* lo, float* hi) {
    float m = fmaxf(fmaxf(fmaxf(fabsf(l.x), fabsf(l.y)), fmaxf(fabsf(l.z), fabsf(h.x))), fmaxf(fabsf(h.y), fabsf(h.z)));
    float pad = xmul(xadd(m, 1.0f), 7.62939453125e-06f);
    lo[0] = xsub(l.x, pad); lo[1] = xsub(l.y, pad); lo[2] = xsub(l.z, pad);
    hi[0] = xadd(h.x, pad); hi[1] = xadd(h.y, pad); hi[2] = xadd(h.z, pad);
}

__global__ void k_lbvh_refit(const float4* __restrict__ tlo, const float4* __restrict__ thi, const uint32_t* __restrict__ ids, uint32_t n,
                             BvhNode* nodes, const uint32_t* __restrict__ leaf_parent, uint32_t* flags) {
    uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    float lo[3], hi[3];
    uint32_t id = ids[k];
    padded_box(tlo[id], thi[id], lo, hi);
    uint32_t child = 0x80000000u | k;
    uint32_t cur = leaf_parent[k];
    while (cur != IPT_NO_HIT) {
        volatile BvhNode* nd = nodes + cur;
        bool is_left = nd->left == child;
        if (is_left) { nd->lo0x = lo[0]; nd->lo0y = lo[1]; nd->lo0z = lo[2]; nd->hi0x = hi[0]; nd->hi0y = hi[1]; nd->hi0z = hi[2]; }
        else { nd->lo1x = lo[0]; nd->lo1y = lo[1]; nd->lo1z = lo[2]; nd->hi1x = hi[0]; nd->hi1y = hi[1]; nd->hi1z = hi[2]; }
        __threadfence();
        if (atomicAdd(&flags[cur], 1u) == 0u) return; // the sibling subtree is not finished: its thread continues
        __threadfence();
        lo[0] = fminf(nd->lo0x, nd->lo1x); lo[1] = fminf(nd->lo0y, nd->lo1y); lo[2] = fminf(nd->lo0z, nd->lo1z);
        hi[0] = fmaxf(nd->hi0x, nd->hi1x); hi[1] = fmaxf(nd->hi0y, nd->hi1y); hi[2] = fmaxf(nd->hi0z, nd->hi1z);
        child = cur;
        cur = nd->parent;
    }
}

// per sorted position: the constants AreaLight's constructor derives (lighting.cpp:79-90) for the triangle
__global__ void k_lbvh_records(const float* __restrict__ tris, const uint32_t* __restrict__ ids, uint32_t n, float4* rec, const float* __restrict__ extra) {
    uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const float* t = tris + 9 * (size_t)ids[k];
    f3 v0 = mk3(t[0], t[1], t[2]), e1 = mk3(t[3], t[4], t[5]), e2 = mk3(t[6], t[7], t[8]);
    f3 cr = xcross3(e1, e2);
    f3 nn = xnormalize3(cr);
    // glm::inverse(mat3(e1, e2, cr)) rows 0 and 1 (include/glm/detail/func_matrix.inl:269-291); m[i][j]: column i, row j
    float m00 = e1.x, m01 = e1.y, m02 = e1.z, m10 = e2.x, m11 = e2.y, m12 = e2.z, m20 = cr.x, m21 = cr.y, m22 = cr.z;
    float det = xadd(xsub(xmul(m00, xsub(xmul(m11, m22), xmul(m21, m12))), xmul(m10, xsub(xmul(m01, m22), xmul(m21, m02)))),
                     xmul(m20, xsub(xmul(m01, m12), xmul(m11, m02))));
    float ood = xdiv(1.0f, det);
    float i00 = xmul(xsub(xmul(m11, m22), xmul(m21, m12)), ood);
    float i10 = xmul(-xsub(xmul(m10, m22), xmul(m20, m12)), ood);
    float i20 = xmul(xsub(xmul(m10, m21), xmul(m20, m11)), ood);
    float i01 = xmul(-xsub(xmul(m01, m22), xmul(m21, m02)), ood);
    float i11 = xmul(xsub(xmul(m00, m22), xmul(m20, m02)), ood);
    float i21 = xmul(-xsub(xmul(m00, m21), xmul(m20, m01)), ood);
    // coord.x = i00*r.x + i10*r.y + i20*r.z ; coord.y = i01*r.x + i11*r.y + i21*r.z
    rec[4 * (size_t)k] = make_float4(v0.x, v0.y, v0.z, nn.x);
    rec[4 * (size_t)k + 1] = make_float4(nn.y, nn.z, i00, i10);
    rec[4 * (size_t)k + 2] = make_float4(i20, i01, i11, i21);
    // the original index rides in the 64-byte record; light sets add (kind, area, mixture weight)
    const float* ex = extra ? extra + 3 * (size_t)ids[k] : nullptr;
    rec[4 * (size_t)k + 3] = make_float4(__uint_as_float(ids[k]), ex ? ex[0] : 1.0f, ex ? ex[1] : 0.0f, ex ? ex[2] : 0.0f);
}

// 64-byte node -> 32-byte node (see BvhNodeQ): one thread per node. Low bounds round down, high bounds up, then one more
// cell outwards. Float steps: (x - lo) with __fsub_rn, then one __fmaf_rn — oracle/ipt_oracle_mesh.inc restates them.
__device__ __forceinline__ uint32_t grid_quant(float x, float lo, float scale, bool upper) {
    float g = __fmaf_rn(__fsub_rn(x, lo), scale, IPT_GRID_BASE);
    g = fminf(fmaxf(g, 1.0f), 1.99993896484375f);
    uint32_t m = __float_as_uint(g) & 0x007FFFFFu; // 23-bit mantissa of a float in [1, 2)
    int q = upper ? (int)((m + 127u) >> 7) + 1 : (int)(m >> 7) - 1;
    return (uint32_t)min(max(q, 0), 65535);
}
__global__ void k_lbvh_compact(const BvhNode* __restrict__ nodes, uint32_t n_nodes, GridMap G, BvhNodeQ* out) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_nodes) return;
    BvhNode nd = nodes[i];
    uint32_t l0x = grid_quant(nd.lo0x, G.lo[0], G.scale[0], false), l0y = grid_quant(nd.lo0y, G.lo[1], G.scale[1], false), l0z = grid_quant(nd.lo0z, G.lo[2], G.scale[2], false);
    uint32_t h0x = grid_quant(nd.hi0x, G.lo[0], G.scale[0], true), h0y = grid_quant(nd.hi0y, G.lo[1], G.scale[1], true), h0z = grid_quant(nd.hi0z, G.lo[2], G.scale[2], true);
    uint32_t l1x = grid_quant(nd.lo1x, G.lo[0], G.scale[0], false), l1y = grid_quant(nd.lo1y, G.lo[1], G.scale[1], false), l1z = grid_quant(nd.lo1z, G.lo[2], G.scale[2], false);
    uint32_t h1x = grid_quant(nd.hi1x, G.lo[0], G.scale[0], true), h1y = grid_quant(nd.hi1y, G.lo[1], G.scale[1], true), h1z = grid_quant(nd.hi1z, G.lo[2], G.scale[2], true);
    BvhNodeQ q;
    q.w[0] = l0x | (l0y << 16); q.w[1] = l0z | (h0x << 16); q.w[2] = h0y | (h0z << 16);
    q.w[3] = l1x | (l1y << 16); q.w[4] = l1z | (h1x << 16); q.w[5] = h1y | (h1z << 16);
    q.w[6] = nd.left; q.w[7] = nd.right;
    out[i] = q;
}

// leaf -> parent links of an existing tree, for a refit: each internal node writes the entry of its leaf children (the
// parent links of internal nodes are kept in BvhNode::parent)
__global__ void k_lbvh_leaf_parents(const BvhNode* __restrict__ nodes, uint32_t n_nodes, uint32_t* leaf_parent) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_nodes) return;
    uint32_t l = nodes[i].left, r = nodes[i].right;
    if (l & 0x80000000u) leaf_parent[l & 0x7FFFFFFFu] = i;
    if (r & 0x80000000u) leaf_parent[r & 0x7FFFFFFFu] = i;
}

static inline void lbvh_free(LbvhDevice& b) {
    cudaFree(b.tri_records); cudaFree(b.sorted_ids); cudaFree(b.sorted_keys); cudaFree(b.nodes); cudaFree(b.qnodes);
    b = LbvhDevice();
}

#define LB_TRY(expr)                                                     \
    do {                                                                 \
        cudaError_t e__ = (expr);                                        \
        if (e__ != cudaSuccess) { err = std::string(#expr) + ": " + cudaGetErrorString(e__); goto fail; } \
    } while (0)

// Shared by build and refit, over the kept sorted order and topology: the internal boxes bottom-up from the leaf boxes
// (lo, hi: tight boxes per original triangle; flags: n words of scratch) and the 64-byte records of the sorted triangles.
static inline cudaError_t lbvh_fit(const float* tris, const float* extra, const float4* lo, const float4* hi, const uint32_t* leaf_parent,
                                   uint32_t* flags, LbvhDevice& b, cudaStream_t st) {
    const uint32_t n = b.n;
    const unsigned blocks = (n + 255) / 256;
    k_lbvh_records<<<blocks, 256, 0, st>>>(tris, b.sorted_ids, n, b.tri_records, extra);
    if (n > 1) {
        cudaError_t e = cudaMemsetAsync(flags, 0, 4 * (size_t)n, st);
        if (e != cudaSuccess) return e;
        k_lbvh_refit<<<blocks, 256, 0, st>>>(lo, hi, b.sorted_ids, n, b.nodes, leaf_parent, flags);
    }
    return cudaGetLastError();
}

// Shared by build and refit: the grid of the 32-byte nodes spans the root box (the union of the root's two child boxes);
// quantises b.nodes into b.qnodes under it. Waits for the stream.
static inline int lbvh_grid_compact(LbvhDevice& b, cudaStream_t st, std::string& err) {
    if (b.n < 2) return 0;
    BvhNode root;
    LB_TRY(cudaMemcpyAsync(&root, b.nodes, sizeof root, cudaMemcpyDeviceToHost, st));
    LB_TRY(cudaStreamSynchronize(st));
    {
        const float rlo[3] = {std::fmin(root.lo0x, root.lo1x), std::fmin(root.lo0y, root.lo1y), std::fmin(root.lo0z, root.lo1z)};
        const float rhi[3] = {std::fmax(root.hi0x, root.hi1x), std::fmax(root.hi0y, root.hi1y), std::fmax(root.hi0z, root.hi1z)};
        for (int a = 0; a < 3; ++a) {
            float ext = rhi[a] - rlo[a];
            b.grid.lo[a] = rlo[a];
            b.grid.scale[a] = ext > 0.0f ? IPT_GRID_FILL / ext : 1.0f; // a flat scene: every coordinate maps to 1
        }
    }
    k_lbvh_compact<<<(b.n - 1 + 255) / 256, 256, 0, st>>>(b.nodes, b.n - 1, b.grid, b.qnodes);
    LB_TRY(cudaGetLastError());
    LB_TRY(cudaStreamSynchronize(st));
    return 0;
fail:
    return 1;
}

// Builds the LBVH for n triangles (9 floats each) and their optional per-primitive extras, both in DEVICE memory on the
// stream's device. Returns 0 on success; on failure `out` holds nothing.
static inline int lbvh_build(const float* d_tris, uint32_t n, cudaStream_t st, LbvhDevice& out, std::string& err, const float* d_extra = nullptr) {
    float4 *d_lo = nullptr, *d_hi = nullptr;
    uint32_t *d_cb = nullptr, *d_ids2 = nullptr, *d_counters = nullptr, *d_leaf_parent = nullptr, *d_flags = nullptr;
    unsigned long long* d_keys2 = nullptr;
    const uint32_t nb = (n + RS_TILE - 1) / RS_TILE;
    const unsigned blocks = (n + 255) / 256;
    out = LbvhDevice();
    out.n = n;
    {
        LB_TRY(cudaMalloc((void**)&d_lo, 16 * (size_t)n));
        LB_TRY(cudaMalloc((void**)&d_hi, 16 * (size_t)n));
        LB_TRY(cudaMalloc((void**)&d_cb, 24));
        const uint32_t cb_init[6] = {0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0, 0, 0};
        LB_TRY(cudaMemcpyAsync(d_cb, cb_init, 24, cudaMemcpyHostToDevice, st));
        LB_TRY(cudaMalloc((void**)&out.sorted_keys, 8 * (size_t)n));
        LB_TRY(cudaMalloc((void**)&out.sorted_ids, 4 * (size_t)n));
        LB_TRY(cudaMalloc((void**)&d_keys2, 8 * (size_t)n));
        LB_TRY(cudaMalloc((void**)&d_ids2, 4 * (size_t)n));
        LB_TRY(cudaMalloc((void**)&d_counters, 4 * (size_t)256 * nb));
        k_lbvh_bounds<<<blocks, 256, 0, st>>>(d_tris, n, d_lo, d_hi, d_cb, d_extra);
        k_lbvh_morton<<<blocks, 256, 0, st>>>(d_lo, d_hi, n, d_cb, out.sorted_keys, out.sorted_ids);
        unsigned long long *ka = out.sorted_keys, *kb = d_keys2;
        uint32_t *va = out.sorted_ids, *vb = d_ids2;
        for (int pass = 0; pass < 8; ++pass) { // 8 passes: the result lands back in (ka, va) == out.*
            int shift = 8 * pass;
            k_rs_hist<<<nb, RS_THREADS, 0, st>>>(ka, n, shift, nb, d_counters);
            k_rs_scan<<<1, 1024, 0, st>>>(d_counters, 256 * nb);
            k_rs_scatter<<<nb, RS_THREADS, 0, st>>>(ka, va, kb, vb, n, shift, nb, d_counters);
            std::swap(ka, kb);
            std::swap(va, vb);
        }
        LB_TRY(cudaGetLastError());
        LB_TRY(cudaMalloc((void**)&out.tri_records, 64 * (size_t)n));
        if (n > 1) {
            LB_TRY(cudaMalloc((void**)&out.nodes, sizeof(BvhNode) * (size_t)(n - 1)));
            LB_TRY(cudaMemsetAsync(out.nodes, 0, sizeof(BvhNode) * (size_t)(n - 1), st));
            LB_TRY(cudaMalloc((void**)&out.qnodes, sizeof(BvhNodeQ) * (size_t)(n - 1)));
            LB_TRY(cudaMalloc((void**)&d_leaf_parent, 4 * (size_t)n));
            LB_TRY(cudaMalloc((void**)&d_flags, 4 * (size_t)n));
            k_lbvh_hierarchy<<<blocks, 256, 0, st>>>(out.sorted_keys, n, out.nodes, d_leaf_parent);
        }
        LB_TRY(lbvh_fit(d_tris, d_extra, d_lo, d_hi, d_leaf_parent, d_flags, out, st));
        if (lbvh_grid_compact(out, st, err)) goto fail;
        LB_TRY(cudaStreamSynchronize(st));
    }
    cudaFree(d_lo); cudaFree(d_hi); cudaFree(d_cb); cudaFree(d_keys2); cudaFree(d_ids2);
    cudaFree(d_counters); cudaFree(d_leaf_parent); cudaFree(d_flags);
    return 0;
fail:
    cudaFree(d_lo); cudaFree(d_hi); cudaFree(d_cb); cudaFree(d_keys2); cudaFree(d_ids2);
    cudaFree(d_counters); cudaFree(d_leaf_parent); cudaFree(d_flags);
    lbvh_free(out);
    return 1;
}

// The same from HOST memory: the triangles (and extras) are staged on the stream, then built.
static inline int lbvh_build_host(const float* host_tris, uint32_t n, cudaStream_t st, LbvhDevice& out, std::string& err,
                                  const float* host_extra = nullptr) {
    float* d_tris = nullptr;
    float* d_extra = nullptr;
    int rc = 1;
    out = LbvhDevice();
    LB_TRY(cudaMalloc((void**)&d_tris, sizeof(float) * 9 * (size_t)n));
    LB_TRY(cudaMemcpyAsync(d_tris, host_tris, sizeof(float) * 9 * (size_t)n, cudaMemcpyHostToDevice, st));
    if (host_extra) {
        LB_TRY(cudaMalloc((void**)&d_extra, sizeof(float) * 3 * (size_t)n));
        LB_TRY(cudaMemcpyAsync(d_extra, host_extra, sizeof(float) * 3 * (size_t)n, cudaMemcpyHostToDevice, st));
    }
    rc = lbvh_build(d_tris, n, st, out, err, d_extra);
fail:
    cudaFree(d_extra); cudaFree(d_tris);
    return rc;
}

// Refit: new vertices (DEVICE memory, the triangle count of the tree) under the tree's kept topology and sorted order.
// Recomputes the leaf boxes, the internal boxes, the records, the grid and the 32-byte nodes in place; the Morton keys and
// sorted order stay those of the build. All scratch is allocated before anything of `b` is written: on an allocation
// failure `b` is unchanged. Returns 0 on success.
static inline int lbvh_refit(const float* d_tris, cudaStream_t st, LbvhDevice& b, std::string& err) {
    const uint32_t n = b.n;
    float4 *d_lo = nullptr, *d_hi = nullptr;
    uint32_t *d_cb = nullptr, *d_leaf_parent = nullptr, *d_flags = nullptr;
    int rc = 1;
    LB_TRY(cudaMalloc((void**)&d_lo, 16 * (size_t)n));
    LB_TRY(cudaMalloc((void**)&d_hi, 16 * (size_t)n));
    LB_TRY(cudaMalloc((void**)&d_cb, 24)); // the centre bounds k_lbvh_bounds also gathers: unused here
    if (n > 1) {
        LB_TRY(cudaMalloc((void**)&d_leaf_parent, 4 * (size_t)n));
        LB_TRY(cudaMalloc((void**)&d_flags, 4 * (size_t)n));
        k_lbvh_leaf_parents<<<(n - 1 + 255) / 256, 256, 0, st>>>(b.nodes, n - 1, d_leaf_parent);
    }
    k_lbvh_bounds<<<(n + 255) / 256, 256, 0, st>>>(d_tris, n, d_lo, d_hi, d_cb, nullptr);
    LB_TRY(lbvh_fit(d_tris, nullptr, d_lo, d_hi, d_leaf_parent, d_flags, b, st));
    if (lbvh_grid_compact(b, st, err)) goto fail;
    LB_TRY(cudaStreamSynchronize(st));
    rc = 0;
fail:
    cudaFree(d_lo); cudaFree(d_hi); cudaFree(d_cb); cudaFree(d_leaf_parent); cudaFree(d_flags);
    return rc;
}
#undef LB_TRY

} // namespace iptd
