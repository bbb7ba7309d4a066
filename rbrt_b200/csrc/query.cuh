// query.cuh — ray queries on device memory (rbrt_gpu_query_closest_device / rbrt_gpu_query_occluded_device, DESIGN.md section 12).
// The launch interface of the query module (query.cu, built into librbrt_gpu_query.so, which librbrt_gpu.so loads at run time) and the
// per-ray steps of the occlusion query.  The kernels run these steps warp-voted for 32 rays at a time; occluded_ray() below runs them for
// one ray, and the host build of the device headers (tests/host_device) checks it against Scene::hit composed with the max_dist compare.
#pragma once
#include "../../include/rbrt_gpu.h"
#include "intersect.cuh"

namespace rbrt {

enum { QRY_ST_HEAD = 0, QRY_ST_NAN = 1, QRY_ST_NODES = 2, QRY_ST_TRIS = 3, QRY_ST_COUNT = 4 };

struct QueryArgs {
    SceneDev S;                  // replica 0 of the scene
    const rbrt_ray* rays;        // n rays, device memory
    uint64_t n;                  // < 2^32
    rbrt_query_out out;          // closest query: device planes, a NULL member is not written
    const float* max_dist;       // occlusion query: n bounds, or NULL = +inf
    uint8_t* occluded;           // occlusion query: n results; NULL for a closest query
    unsigned long long* ctr;     // QRY_ST_COUNT counters, zeroed before the launch: [QRY_ST_HEAD] is the ray cursor
    int count;                   // also fill QRY_ST_NAN / NODES / TRIS
    uint32_t blocks;             // persistent grid
};

// The t bound of a mesh traversal for a hit that must have dist < c: scene_hit's conversion (intersect.cuh), op for op.  dist is
// monotone in t and ~ t*|d|; the margin keeps the bound from cutting a triangle whose dist is below c.
__device__ __forceinline__ float query_t_limit(f3 o, f3 d, float c) {
    float t_limit = RBRT_T_CAP;
    if (c < 3.0e38f) {
        float dl = len3(d);
        float omax = fmaxf(fmaxf(fabsf(o.x), fabsf(o.y)), fabsf(o.z));
        float lim = (c * 1.001f + 1e-5f * (omax + c) + 1e-6f) / dl;
        if (lim == lim) t_limit = fminf(t_limit, lim);
    }
    return t_limit;
}

// ------------------------------------------------------------------ occlusion: is Scene::hit(ray) a hit with dist < max_dist?
// 0 no, 1 yes, 2 a NaN ray (Scene::hit reports a NaN sphere discriminant, sphere.rs:33, wherever that sphere is in the element list).

// The elements, all of them: a NaN discriminant on ANY sphere makes the ray a NaN ray, even after an earlier hit, so nothing is
// concluded before the last element.  An element hit counts when its dist < max_dist (a NaN dist, possible for a BasicTriangle, is
// never recorded by Scene::hit and fails the compare too).
__device__ __forceinline__ int occluded_elements(const SceneDev& S, f3 o, f3 d, float max_dist) {
    int res = 0;
    for (uint32_t i = 0; i < S.n_spheres; ++i) {
        float t, dist;
        const int r = element_intersect(S, i, o, d, t, dist);
        if (r < 0) return 2;
        if (r && dist < max_dist) res = 1;
    }
    return res;
}

// A mesh hit at parameter t occludes: the window of mesh.rs:249 and the strict compare with max_dist.
__device__ __forceinline__ bool mesh_hit_occludes(f3 o, f3 d, float t, float max_dist) {
    const f3 p = o + t * d;
    const float dist = len3(o - p);
    return dist > RBRT_MIN_DIST && dist < RBRT_MAX_DIST && dist < max_dist;
}

// Whether the first accepted triangle with a small enough dist may end the traversal (DESIGN.md section 12).  A mesh hit is decided by its
// minimum-t triangle alone, and its dist must exceed 0.001.  For a finite ray, dist(t) = len3(o - (o + t*d)) is non-decreasing in t under
// this f32 op sequence, and a triangle is only accepted at t > 0.001, i.e. t >= nextafterf(0.001f, inf).  If dist there already exceeds
// 0.001, every accepted triangle lies above the lower window, the minimum-t triangle has the smallest dist of all, and ANY accepted
// triangle with dist < min(max_dist, 2000) proves occlusion.  Otherwise (short directions: t > 0.001 but t*|d| <= 0.001), or for a ray
// with an inf or NaN component, the mesh needs the exact closest search.
__device__ __forceinline__ bool occluded_early_exit_ok(f3 o, f3 d) {
    const float big = 3.40282347e+38f;
    if (!(fabsf(o.x) <= big && fabsf(o.y) <= big && fabsf(o.z) <= big && fabsf(d.x) <= big && fabsf(d.y) <= big && fabsf(d.z) <= big)) return false;
    const float t0 = __uint_as_float(0x3A831270u);                        // nextafterf(0.001f, inf); 0.001f = 0x3A83126F
    const f3 p = o + t0 * d;
    return len3(o - p) > RBRT_MIN_DIST;
}

// ONE triangle of the current leaf, as leaf_step_one (intersect.cuh), and with `early` the exit: an accepted triangle that occludes ends
// the lane's traversal (occ = 1, cur = sentinel).
template <class STK>
__device__ __forceinline__ void occluded_leaf_step_one(const float4* __restrict__ tris, uint32_t tri_base, int32_t& cur, f3 o, f3 d, float t_limit,
                                                       float max_dist, bool early, float& best_t, uint32_t& best_idx, float& t_prune, int& occ,
                                                       const STK& stack, int& sp) {
    const uint32_t code = (uint32_t)(~cur);
    f3 v0, e1, e2; uint32_t orig; float t;
    load_tri(tris, tri_base + (code >> 3), v0, e1, e2, orig);
    if (tri_intersect_masks(v0, e1, e2, o, d, t)) {
        keep_min(t, orig, best_t, best_idx);
        t_prune = fminf(t_limit, __fmaf_rn(best_t, 1.0001f, 1e-4f));
        if (early && mesh_hit_occludes(o, d, t, max_dist)) { occ = 1; cur = RBRT_SENTINEL; return; }
    }
    cur = (code & 7u) ? (int32_t)~(code + 7u) : stack.get(--sp);
}

// traverse_voted (intersect.cuh) with the occlusion leaf step: one node visit or one triangle test per step, whichever more lanes wait for.
template <bool COUNT, class STK>
__device__ __forceinline__ void traverse_voted_occluded(const uint4* __restrict__ nodes, const float4* __restrict__ tris, uint32_t tri_base,
                                                        const RaySlabs& R, f3 o, f3 d, float t_limit, float max_dist, bool early, const STK& stack,
                                                        int& sp, int32_t& cur, float& best_t, uint32_t& best_idx, float& t_prune, int& occ,
                                                        int threshold, uint32_t& n_nodes, uint32_t& n_tris) {
    asm volatile("" : "+r"(threshold));
    for (;;) {
        const bool at_node = (uint32_t)cur < (uint32_t)RBRT_SENTINEL, at_leaf = cur < 0;
        const int nn = __popc(__ballot_sync(0xFFFFFFFFu, at_node)), nl = __popc(__ballot_sync(0xFFFFFFFFu, at_leaf));
        if (nn + nl < threshold) break;
        if (nn * RBRT_VOTE_N >= nl * RBRT_VOTE_L) {
            if (at_node) { cur = bvh4_step<false>(nodes + 4 * (size_t)cur, nodes, tris + 3 * (size_t)tri_base, R, t_prune, stack, sp); if (COUNT) ++n_nodes; }
        } else if (at_leaf) {
            occluded_leaf_step_one(tris, tri_base, cur, o, d, t_limit, max_dist, early, best_t, best_idx, t_prune, occ, stack, sp);
            if (COUNT) ++n_tris;
        }
    }
}

// The whole occlusion rule for one ray, one lane (the kernel interleaves the same steps over a warp).  The traversal's t bound comes from
// max_dist: by the time a mesh is traversed no earlier element or mesh had a dist below max_dist (that would have ended the query), so
// max_dist is the smaller of max_dist and Scene::hit's running `closest`.
template <class STK>
__device__ __forceinline__ int occluded_ray(const SceneDev& S, f3 o, f3 d, float max_dist, const STK& stack, TraceCounters* cnt) {
    int occ = occluded_elements(S, o, d, max_dist);
    if (occ || !(max_dist > RBRT_MIN_DIST)) return occ;                   // a NaN ray, an element below max_dist, or nothing can be below it
    const bool early = occluded_early_exit_ok(o, d);
    uint32_t n_nodes = 0, n_tris = 0;
    for (uint32_t mi = 0; mi < S.n_meshes && !occ; ++mi) {
        const MeshDev& M = S.meshes[mi];
        if (M.n_tris == 0 || !mesh_bbox_hit(M, o, d)) continue;
        const float t_limit = query_t_limit(o, d, max_dist);
        float t_prune = t_limit, best_t = 1000000.0f; uint32_t best_idx = 0xFFFFFFFFu;
        const uint4* nodes = reinterpret_cast<const uint4*>(S.nodes) + 4 * (size_t)M.node_base;
        const RaySlabs R = ray_slabs(M, o, d);
        int sp = 0; stack.put(sp++, RBRT_SENTINEL);
        int32_t cur = M.root_ref;
        traverse_voted_occluded<true>(nodes, S.tris, M.tri_base, R, o, d, t_limit, max_dist, early, stack, sp, cur, best_t, best_idx, t_prune, occ,
                                      1, n_nodes, n_tris);
        if (!early && best_idx != 0xFFFFFFFFu && mesh_hit_occludes(o, d, best_t, max_dist)) occ = 1;
    }
    if (cnt) { cnt->nodes += n_nodes; cnt->tris += n_tris; }
    return occ;
}

}  // namespace rbrt

#ifdef __CUDACC__                                                         // (not in the host build of the tests)
extern "C" {
// Enqueues the query kernel on `stream` (a closest query when args->occluded is NULL); returns a cudaError_t.
typedef int (*rbrt_query_launch_fn)(const rbrt::QueryArgs* args, cudaStream_t stream);
}
#endif
