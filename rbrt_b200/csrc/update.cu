// update.cu — refit of one mesh's LBVH to new vertices, in place (rbrt_gpu_scene_update_mesh, RBRT_UPDATE_REFIT).
//
// Built into its own shared object (librbrt_gpu_update.so), which librbrt_gpu.so loads at run time: the device code of
// librbrt_gpu.so stays exactly the build the GPU tests verified.  The refit keeps the tree's topology — the child refs of every
// 4-wide node, the Morton order of the triangle records, the node count — and recomputes everything derived from the vertices:
//   1. the exact mesh AABB over ALL real triangles (aabbox.rs:62-88, mesh.rs:61), NaN coordinates ignored;
//   2. MeshDev.lo/hi/qorg/qstep and the leaf padding (k_mesh_setup's formula);
//   3. each triangle record {v0 | orig, e1, e2} in place (orig kept) and the unit normal of `orig` (original order);
//   4. the child boxes of every 4-wide node, bottom up: a leaf child's float box is the min / max of its triangles' padded boxes,
//      an internal child's the union of its own children's float boxes (kept in scratch, never read back from the quantised
//      bytes), each quantised outward onto the new grid.  Unused slots keep their inverted box.
// min / max are exact whatever the order, so a refit with the vertices the mesh was built from reproduces the build's bytes.
// Formulas restated from bvh_build.cu cite the line they copy; the two must stay in step.
#include "update.cuh"

namespace rbrt {
namespace {

struct RefitParams { float pad; float org[3], step[3]; };

// ------------------------------------------------------------------ 1. exact AABB (= k_aabb_init / k_aabb, bvh_build.cu:314-337)
__device__ __forceinline__ int f2ord(float f) { int i = __float_as_int(f); return i >= 0 ? i : i ^ 0x7FFFFFFF; }
__device__ __forceinline__ float ord2f(int i) { int b = i >= 0 ? i : i ^ 0x7FFFFFFF; return __int_as_float(b); }

__global__ void k_upd_aabb_init(int* mm) { if (threadIdx.x < 3) mm[threadIdx.x] = 0x7F7FFFFF; else if (threadIdx.x < 6) mm[threadIdx.x] = (int)0xFF7FFFFF ^ 0x7FFFFFFF; }

__global__ void k_upd_aabb(const float* __restrict__ raw, uint64_t n_vertices, int* __restrict__ mm) {
    float lo[3] = {3.40282347e+38f, 3.40282347e+38f, 3.40282347e+38f}, hi[3] = {-3.40282347e+38f, -3.40282347e+38f, -3.40282347e+38f};
    for (uint64_t v = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; v < n_vertices; v += (uint64_t)gridDim.x * blockDim.x) {
#pragma unroll
        for (int k = 0; k < 3; ++k) { float x = raw[3 * v + k]; lo[k] = fminf(lo[k], x); hi[k] = fmaxf(hi[k], x); }
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        for (int off = 16; off; off >>= 1) { lo[k] = fminf(lo[k], __shfl_down_sync(0xFFFFFFFFu, lo[k], off)); hi[k] = fmaxf(hi[k], __shfl_down_sync(0xFFFFFFFFu, hi[k], off)); }
        if ((threadIdx.x & 31) == 0) { atomicMin(&mm[k], f2ord(lo[k])); atomicMax(&mm[3 + k], f2ord(hi[k])); }
    }
}

// ------------------------------------------------------------------ 2. MeshDev box + grid (= k_mesh_setup, bvh_build.cu:341-369)
// Only lo/hi/qorg/qstep change; tri_base, n_tris, node_base, root_ref, nrm_base and elem are the device record's own.
__global__ void k_upd_setup(const int* __restrict__ mm, uint32_t n_eff, float pad_rel, MeshDev* __restrict__ md_io, RefitParams* __restrict__ rp) {
    if (threadIdx.x || blockIdx.x) return;
    MeshDev md = *md_io;
    float lo[3], hi[3], mx = 0.0f;
    for (int k = 0; k < 3; ++k) {
        lo[k] = ord2f(mm[k]); hi[k] = ord2f(mm[3 + k]);
        md.lo[k] = lo[k]; md.hi[k] = hi[k];
        mx = fmaxf(mx, fmaxf(fabsf(lo[k]), fabsf(hi[k]))); mx = fmaxf(mx, hi[k] - lo[k]);
    }
    // the relative padding with its floor of 2^-21 * (mx + 1000) (bvh_build.cu:357; profiles/r2_device_code.md)
    const float pad = pad_rel > 0.0f ? fmaxf(pad_rel * mx, 4.7683716e-7f * (mx + 1000.0f)) : 0.0f;
    rp->pad = pad;
    for (int k = 0; k < 3; ++k) {                                          // bvh_build.cu:359-367
        float ext = (hi[k] + pad) - (lo[k] - pad);
        float step = ext / 65500.0f;
        if (!(step > 1e-30f)) step = 1e-30f;
        const float org = (lo[k] - pad) - 8.0f * step;
        rp->step[k] = step; rp->org[k] = org;
        md.qstep[k] = n_eff ? (step <= RBRT_QSTEP_MAX ? step : __int_as_float(0x7FFFFFFF)) : 0.0f; md.qorg[k] = n_eff ? org : 0.0f;   // bvh_build.cu:365
    }
    *md_io = md;
}

// ------------------------------------------------------------------ 3. triangle records, normals, padded leaf boxes
// record p keeps bits(orig) in .w; v0, e1, e2 as k_emit_tris (bvh_build.cu:58-72), the normal as k_prepare (bvh_build.cu:40-43)
__global__ void k_upd_tris(const float* __restrict__ raw, uint32_t n, const RefitParams* __restrict__ rp, float4* __restrict__ tris,
                           float4* __restrict__ normals, float4* __restrict__ leaf_lo, float4* __restrict__ leaf_hi) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const float pad = rp->pad;
    const float w = tris[3 * (size_t)p].w;
    const uint32_t orig = __float_as_uint(w);
    const float* t = raw + 9 * (size_t)orig;
    f3 a = mk3(t[0], t[1], t[2]), b = mk3(t[3], t[4], t[5]), c = mk3(t[6], t[7], t[8]);
    f3 e1 = b - a, e2 = c - a;                                            // mesh.rs:57-60
    tris[3 * (size_t)p] = make_float4(a.x, a.y, a.z, w);
    tris[3 * (size_t)p + 1] = make_float4(e1.x, e1.y, e1.z, 0.0f);
    tris[3 * (size_t)p + 2] = make_float4(e2.x, e2.y, e2.z, 0.0f);
    f3 nn = norm3(cross3(e1, e2));                                        // triangle.rs:30-34
    normals[orig] = make_float4(nn.x, nn.y, nn.z, 0.0f);
    leaf_lo[p] = make_float4(fminf(a.x, fminf(b.x, c.x)) - pad, fminf(a.y, fminf(b.y, c.y)) - pad, fminf(a.z, fminf(b.z, c.z)) - pad, 0.0f);
    leaf_hi[p] = make_float4(fmaxf(a.x, fmaxf(b.x, c.x)) + pad, fmaxf(a.y, fmaxf(b.y, c.y)) + pad, fmaxf(a.z, fmaxf(b.z, c.z)) + pad, 0.0f);
}

// ------------------------------------------------------------------ 4. bottom-up refit of the 4-wide nodes
// Outward quantisation onto the 16-bit grid (= quant_lo / quant_hi, bvh_build.cu:191-200)
__device__ __forceinline__ uint32_t quant_lo(float v, float org, float step) {
    float q = floorf((v - org) / step) - 1.0f;
    while (q > 0.0f && __fmaf_rn(q, step, org) > v) q -= 1.0f;             // never above the true bound
    return (uint32_t)fminf(fmaxf(q, 0.0f), 65535.0f);
}
__device__ __forceinline__ uint32_t quant_hi(float v, float org, float step) {
    float q = ceilf((v - org) / step) + 1.0f;
    while (q < 65535.0f && __fmaf_rn(q, step, org) < v) q += 1.0f;         // never below the true bound
    return (uint32_t)fminf(fmaxf(q, 0.0f), 65535.0f);
}

// A node is 12 box words (word 3k + axis = child k's lo | hi << 16 on that axis) and 4 child refs (collapse_node, bvh_build.cu:253-256).
struct Node { uint32_t w[12]; int32_t ref[4]; };
__device__ __forceinline__ Node load_node(const uint4* __restrict__ nodes, uint32_t j) {
    Node n;
    const uint4 a = nodes[4 * (size_t)j], b = nodes[4 * (size_t)j + 1], c = nodes[4 * (size_t)j + 2], d = nodes[4 * (size_t)j + 3];
    n.w[0] = a.x; n.w[1] = a.y; n.w[2] = a.z; n.w[3] = a.w; n.w[4] = b.x; n.w[5] = b.y; n.w[6] = b.z; n.w[7] = b.w;
    n.w[8] = c.x; n.w[9] = c.y; n.w[10] = c.z; n.w[11] = c.w;
    n.ref[0] = (int32_t)d.x; n.ref[1] = (int32_t)d.y; n.ref[2] = (int32_t)d.z; n.ref[3] = (int32_t)d.w;
    return n;
}
// unused slot: inverted box on every axis (lo 65535, hi 0) and the dummy leaf ref (bvh_build.cu:248-250); a real child's box has lo <= hi
__device__ __forceinline__ bool slot_used(const Node& n, int k) {
    return !(n.w[3 * k] == 0x0000FFFFu && n.w[3 * k + 1] == 0x0000FFFFu && n.w[3 * k + 2] == 0x0000FFFFu && n.ref[k] == make_leaf_ref(0, 1));
}

// parent[c] = 4 * j + slot of every internal child c of node j; need[j] = how many internal children j has
__global__ void k_upd_links(const uint4* __restrict__ nodes, const BuildResult* __restrict__ res, uint32_t* __restrict__ parent,
                            uint32_t* __restrict__ need, uint32_t* __restrict__ arrive) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= res->live_nodes) return;
    const Node n = load_node(nodes, j);
    uint32_t cnt = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if (slot_used(n, k) && n.ref[k] >= 0) { parent[n.ref[k]] = 4 * j + (uint32_t)k; ++cnt; }
    need[j] = cnt; arrive[j] = 0;
}

// One thread starts at every node without internal children; the last child to arrive at a node carries on with it (Karras 2012 §4
// on the 4-wide tree).  cbox[8 j + 2 k], [8 j + 2 k + 1]: float box of internal child k of node j, written by that child's thread.
__global__ void k_upd_nodes(uint4* __restrict__ nodes, const BuildResult* __restrict__ res, const RefitParams* __restrict__ rp,
                            const float4* __restrict__ leaf_lo, const float4* __restrict__ leaf_hi, const uint32_t* __restrict__ parent,
                            const uint32_t* __restrict__ need, uint32_t* __restrict__ arrive, float4* cbox) {
    uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= res->live_nodes || need[j]) return;
    const float org[3] = {rp->org[0], rp->org[1], rp->org[2]}, step[3] = {rp->step[0], rp->step[1], rp->step[2]};
    for (;;) {
        Node n = load_node(nodes, j);
        float4 ulo = make_float4(0.0f, 0.0f, 0.0f, 0.0f), uhi = ulo;
        bool first = true;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (!slot_used(n, k)) continue;
            float4 lo, hi;
            if (n.ref[k] < 0) {                                           // leaf: its triangles' padded boxes (a contiguous run of records)
                const uint32_t code = (uint32_t)~n.ref[k], f = code >> 3, cnt = (code & 7u) + 1u;
                lo = leaf_lo[f]; hi = leaf_hi[f];
                for (uint32_t i = 1; i < cnt; ++i) {
                    const float4 a = leaf_lo[f + i], b = leaf_hi[f + i];
                    lo.x = fminf(lo.x, a.x); lo.y = fminf(lo.y, a.y); lo.z = fminf(lo.z, a.z);
                    hi.x = fmaxf(hi.x, b.x); hi.y = fmaxf(hi.y, b.y); hi.z = fmaxf(hi.z, b.z);
                }
            } else {                                                      // internal: the union its own thread left in scratch
                lo = __ldcg(&cbox[8 * (size_t)j + 2 * k]); hi = __ldcg(&cbox[8 * (size_t)j + 2 * k + 1]);
            }
            n.w[3 * k] = quant_lo(lo.x, org[0], step[0]) | (quant_hi(hi.x, org[0], step[0]) << 16);
            n.w[3 * k + 1] = quant_lo(lo.y, org[1], step[1]) | (quant_hi(hi.y, org[1], step[1]) << 16);
            n.w[3 * k + 2] = quant_lo(lo.z, org[2], step[2]) | (quant_hi(hi.z, org[2], step[2]) << 16);
            if (first) { ulo = lo; uhi = hi; first = false; }             // (a copy, not a min with a neutral value: an all-NaN union stays NaN, as in the build)
            else {
                ulo.x = fminf(ulo.x, lo.x); ulo.y = fminf(ulo.y, lo.y); ulo.z = fminf(ulo.z, lo.z);
                uhi.x = fmaxf(uhi.x, hi.x); uhi.y = fmaxf(uhi.y, hi.y); uhi.z = fmaxf(uhi.z, hi.z);
            }
        }
        nodes[4 * (size_t)j] = make_uint4(n.w[0], n.w[1], n.w[2], n.w[3]);
        nodes[4 * (size_t)j + 1] = make_uint4(n.w[4], n.w[5], n.w[6], n.w[7]);
        nodes[4 * (size_t)j + 2] = make_uint4(n.w[8], n.w[9], n.w[10], n.w[11]);
        if (j == 0) return;                                               // the root: its box is the mesh AABB's business
        const uint32_t p = parent[j], pj = p >> 2, slot = p & 3u;
        __stcg(&cbox[8 * (size_t)pj + 2 * slot], ulo);
        __stcg(&cbox[8 * (size_t)pj + 2 * slot + 1], uhi);
        __threadfence();
        if (atomicAdd(&arrive[pj], 1u) + 1u != need[pj]) return;         // a sibling subtree is still on its way up
        __threadfence();
        j = pj;
    }
}

inline size_t al256(size_t b) { return (b + 255) & ~(size_t)255; }

struct Carve { size_t params, leaf_lo, leaf_hi, parent, need, arrive, cbox, total; };
Carve carve(uint64_t n_eff) {
    const uint64_t n = n_eff ? n_eff : 1, ni = n_eff > 1 ? n_eff - 1 : 1;
    Carve c; size_t off = 0;
    c.params = off; off += 256;                                           // AABB cell (6 ints) + RefitParams
    c.leaf_lo = off; off += al256(16 * n);
    c.leaf_hi = off; off += al256(16 * n);
    c.parent = off; off += al256(4 * ni);
    c.need = off; off += al256(4 * ni);
    c.arrive = off; off += al256(4 * ni);
    c.cbox = off; off += al256(128 * ni);
    c.total = off;
    return c;
}

}  // namespace
}  // namespace rbrt

using namespace rbrt;

extern "C" {

size_t rbrt_update_scratch_bytes(uint64_t n_eff) { return carve(n_eff).total; }

int rbrt_update_refit(const RefitArgs* a, void* scratch, cudaStream_t st) {
    const Carve c = carve(a->n_eff);
    char* base = (char*)scratch;
    int* mm = (int*)(base + c.params);
    RefitParams* rp = (RefitParams*)(base + c.params + 64);
    float4* leaf_lo = (float4*)(base + c.leaf_lo); float4* leaf_hi = (float4*)(base + c.leaf_hi);
    uint32_t* parent = (uint32_t*)(base + c.parent); uint32_t* need = (uint32_t*)(base + c.need); uint32_t* arrive = (uint32_t*)(base + c.arrive);
    float4* cbox = (float4*)(base + c.cbox);
    const int Bk = 256;
    k_upd_aabb_init<<<1, 32, 0, st>>>(mm);
    if (a->n_all) k_upd_aabb<<<148 * 4, 256, 0, st>>>(a->raw, a->n_all * 3, mm);    // the build's grid (bvh_build.cu:496)
    k_upd_setup<<<1, 32, 0, st>>>(mm, a->n_eff, a->pad_rel, a->mesh, rp);
    if (a->n_eff) k_upd_tris<<<(a->n_eff + Bk - 1) / Bk, Bk, 0, st>>>(a->raw, a->n_eff, rp, a->tris, a->normals, leaf_lo, leaf_hi);
    if (a->n_eff > 1) {                                                   // live_nodes (0 for a one-leaf mesh) is read on the device
        const uint32_t g = (uint32_t)((a->n_eff - 1 + Bk - 1) / Bk);
        k_upd_links<<<g, Bk, 0, st>>>(a->nodes, a->res, parent, need, arrive);
        k_upd_nodes<<<g, Bk, 0, st>>>(a->nodes, a->res, rp, leaf_lo, leaf_hi, parent, need, arrive, cbox);
    }
    return (int)cudaGetLastError();
}

}  // extern "C"
