// motion.cu — per-object motion vectors (rbrt_gpu_scene_snapshot, rbrt_gpu_render_motion*; DESIGN.md section 16).
//   k_snapshot: the scene's geometry as the previous frame — mesh triangle records scattered by original triangle index, element and
//               BasicTriangle records as stored.
//   k_motion:   per pixel the centre ray of the current camera (tp_pixel_dir), its closest hit = Scene::hit as rbrt_gpu_trace_rays
//               (RBRT_TRACE_BVH) reports it, bit for bit, then motion.cuh's mv_pixel with the hit element's current and snapshot records.
//
// Built into its own shared object (librbrt_gpu_motion.so), which librbrt_gpu.so loads at run time: the device code of librbrt_gpu.so
// stays exactly the build the GPU tests verified.  One warp is one 8x4-pixel tile (neighbouring lanes trace neighbouring rays), one lane
// one pixel.  The lanes run the elements on their own, then mesh by mesh the box pre-test and the warp-voted BVH traversal of the query
// module (section 12), whose leaf step here also keeps the slot of the winning triangle: the mesh hit reports the ORIGINAL index (the
// snapshot's key), the slot gives the current record.  A lane's own sequence of visits and tests is the one-lane loop's, so the hit is
// the same bits (DESIGN.md section 2).
#include "motion.cuh"
#include "intersect.cuh"
#include "query.cuh"

namespace rbrt {
namespace {

#define MV_THREADS 128
#define MV_SMEM_STACK 16        // traversal-stack entries per lane in shared memory (8 KB per block); deeper entries go to local memory
#define MV_SNAP_THREADS 256

__global__ void __launch_bounds__(MV_SNAP_THREADS) k_snapshot(SnapshotArgs A) {
    const SceneDev& S = A.S;
    const uint32_t stride = A.blocks * MV_SNAP_THREADS;
    const uint32_t g = blockIdx.x * MV_SNAP_THREADS + threadIdx.x;
    for (uint32_t mi = 0; mi < S.n_meshes; ++mi) {
        const MeshDev& M = S.meshes[mi];
        for (uint32_t i = g; i < M.n_tris; i += stride) {
            const float4* r = S.tris + 3 * ((size_t)M.tri_base + i);
            const float4 a = r[0], b = r[1], c = r[2];
            float4* w = A.snap.tris + 3 * ((size_t)M.tri_base + __float_as_uint(a.w));
            w[0] = a; w[1] = b; w[2] = c;
        }
    }
    for (uint32_t i = g; i < S.n_spheres; i += stride) A.snap.elems[i] = S.spheres[i];
    for (uint32_t i = g; i < S.n_etris; i += stride)
        for (int k = 0; k < 3; ++k) A.snap.etris[3 * (size_t)i + k] = S.etris[4 * (size_t)i + k];
}

// traverse_voted (intersect.cuh) with leaf_step_one's test and tie rule, keeping the slot of the running minimum in best_slot.
template <bool COUNT, class STK>
__device__ __forceinline__ void mv_traverse(const uint4* __restrict__ nodes, const float4* __restrict__ tris, uint32_t tri_base, const RaySlabs& R,
                                            f3 o, f3 d, float t_limit, const STK& stack, int& sp, int32_t& cur, float& best_t,
                                            uint32_t& best_idx, uint32_t& best_slot, float& t_prune, uint32_t& n_nodes, uint32_t& n_tris) {
    for (;;) {
        const bool at_node = (uint32_t)cur < (uint32_t)RBRT_SENTINEL, at_leaf = cur < 0;
        const int nn = __popc(__ballot_sync(0xFFFFFFFFu, at_node)), nl = __popc(__ballot_sync(0xFFFFFFFFu, at_leaf));
        if (nn + nl == 0) break;
        if (nn * RBRT_VOTE_N >= nl * RBRT_VOTE_L) {
            if (at_node) { cur = bvh4_step<false>(nodes + 4 * (size_t)cur, nodes, tris + 3 * (size_t)tri_base, R, t_prune, stack, sp); if (COUNT) ++n_nodes; }
        } else if (at_leaf) {
            const uint32_t code = (uint32_t)(~cur), slot = tri_base + (code >> 3);
            f3 v0, e1, e2; uint32_t orig; float t;
            load_tri(tris, slot, v0, e1, e2, orig);
            if (tri_intersect_masks(v0, e1, e2, o, d, t)) {
                if (t < best_t || (t == best_t && orig < best_idx)) { best_t = t; best_idx = orig; best_slot = slot; }   // keep_min
                t_prune = fminf(t_limit, __fmaf_rn(best_t, 1.0001f, 1e-4f));
            }
            cur = (code & 7u) ? (int32_t)~(code + 7u) : stack.get(--sp);
            if (COUNT) ++n_tris;
        }
    }
}

template <bool STATS>
__global__ void __launch_bounds__(MV_THREADS) k_motion(MotionArgs A) {
    const SceneDev& S = A.S;
    __shared__ int32_t s_stack[MV_SMEM_STACK][MV_THREADS];
    int32_t lstack[RBRT_STACK];
    const StackS<MV_SMEM_STACK, MV_THREADS> stack = {&s_stack[0][threadIdx.x], lstack};
    const uint32_t gt = blockIdx.x * MV_THREADS + threadIdx.x;
    const uint32_t T = gt >> 5, lane = gt & 31;
    const uint32_t ty = T / A.tiles_x, tx = T - ty * A.tiles_x;
    const uint32_t col = tx * 8 + (lane & 7), row = ty * 4 + (lane >> 3);
    const bool mine = T < A.tiles_total && col < A.cam.width && row < A.cam.height;
    const f3 o = mk3(A.cam.pos[0], A.cam.pos[1], A.cam.pos[2]);
    const f3 d = mine ? tp_pixel_dir(A.cam, col, row) : mk3(0.0f, 0.0f, 0.0f);
    uint32_t n_nodes = 0, n_tris = 0;

    // Scene::hit (intersect.cuh scene_hit): the elements in order, then the meshes in order
    Hit best; best.kind = -1; best.elem = 0; best.tri = 0; best.t = 0.0f; best.dist = 0.0f;
    uint32_t best_slot = 0;
    float closest = 3.40282347e+38f;                                      // f32::MAX (scene.rs:21)
    for (uint32_t i = 0; mine && i < S.n_spheres; ++i) {
        float t, dist;
        const int r = element_intersect(S, i, o, d, t, dist);
        if (r < 0) { best.kind = -2; break; }
        if (r && dist < closest) { closest = dist; best.kind = 0; best.elem = i; best.t = t; best.dist = dist; }
    }
    for (uint32_t mi = 0; mi < S.n_meshes; ++mi) {                        // every lane takes part in every mesh's vote
        const MeshDev& M = S.meshes[mi];
        RaySlabs R = {0, 0, 0, 0, 0, 0, RBRT_SEL_LO, RBRT_SEL_LO, RBRT_SEL_LO, RBRT_SEL_HI, RBRT_SEL_HI, RBRT_SEL_HI};
        int32_t cur = RBRT_SENTINEL; int sp = 0;
        float best_t = 1000000.0f, t_limit = 0.0f, t_prune = 0.0f;        // min_param init (triangle.rs:398)
        uint32_t best_idx = 0xFFFFFFFFu, slot = 0;
        if (mine && best.kind != -2 && M.n_tris != 0 && mesh_bbox_hit(M, o, d)) {
            t_limit = query_t_limit(o, d, closest); t_prune = t_limit;
            R = ray_slabs(M, o, d);
            stack.put(sp++, RBRT_SENTINEL); cur = M.root_ref;
        }
        mv_traverse<STATS>(reinterpret_cast<const uint4*>(S.nodes) + 4 * (size_t)M.node_base, S.tris, M.tri_base, R, o, d, t_limit, stack, sp,
                           cur, best_t, best_idx, slot, t_prune, n_nodes, n_tris);
        if (best_idx != 0xFFFFFFFFu) {
            const f3 p = o + best_t * d;                                  // ray.point_at (mesh.rs:247)
            const float dist = len3(o - p);                               // mesh.rs:248
            if (dist > RBRT_MIN_DIST && dist < RBRT_MAX_DIST && dist < closest) {   // mesh.rs:249 + scene.rs:36
                closest = dist; best.kind = 1; best.elem = mi; best.tri = best_idx; best.t = best_t; best.dist = dist; best_slot = slot;
            }
        }
    }

    uint32_t n_nan = 0;
    if (mine) {
        float mx = __uint_as_float(0x7FC00000u), my = mx, pd = __uint_as_float(0x7F800000u);   // a miss or a NaN ray: NaN, +inf
        if (best.kind == -2) ++n_nan;
        else if (best.kind >= 0) {
            float4 cur[3], old[3];
            bool tri = true;
            if (best.kind == 1) {
                const float4* c = S.tris + 3 * (size_t)best_slot;
                const float4* w = A.snap.tris + 3 * ((size_t)S.meshes[best.elem].tri_base + best.tri);
                for (int k = 0; k < 3; ++k) { cur[k] = __ldg(c + k); old[k] = w[k]; }
            } else {
                const float4 e = __ldg(S.spheres + best.elem);
                if (S.n_etris && __ldg(S.elem_kind + best.elem)) {
                    const size_t ti = __float_as_uint(e.x);
                    for (int k = 0; k < 3; ++k) { cur[k] = __ldg(S.etris + 4 * ti + k); old[k] = A.snap.etris[3 * ti + k]; }
                } else {
                    cur[0] = e; old[0] = A.snap.elems[best.elem]; tri = false;
                }
            }
            mv_pixel(A.cam, A.prev, tri, o, d, best.t, cur, old, &mx, &my, &pd);
        }
        const size_t px = (size_t)row * A.cam.width + col;
        if (A.out.motion) { A.out.motion[2 * px] = mx; A.out.motion[2 * px + 1] = my; }
        if (A.out.prev_dist) A.out.prev_dist[px] = pd;
    }
    if (STATS) {
        unsigned long long nan = n_nan, nd = n_nodes, tr = n_tris;
        for (int off = 16; off; off >>= 1) {
            nan += __shfl_down_sync(0xFFFFFFFFu, nan, off);
            nd += __shfl_down_sync(0xFFFFFFFFu, nd, off);
            tr += __shfl_down_sync(0xFFFFFFFFu, tr, off);
        }
        if (lane == 0) {
            if (nan) atomicAdd(&A.stats[MV_ST_NAN], nan);
            if (nd) atomicAdd(&A.stats[MV_ST_NODES], nd);
            if (tr) atomicAdd(&A.stats[MV_ST_TRIS], tr);
        }
    }
}

}  // namespace
}  // namespace rbrt

extern "C" int rbrt_snapshot_launch(const rbrt::SnapshotArgs* a, cudaStream_t stream) {
    if (!a->blocks) return (int)cudaSuccess;
    rbrt::k_snapshot<<<a->blocks, MV_SNAP_THREADS, 0, stream>>>(*a);
    return (int)cudaGetLastError();
}

extern "C" int rbrt_motion_launch(const rbrt::MotionArgs* a, cudaStream_t stream) {
    const uint64_t threads = 32ull * a->tiles_total;
    if (!threads) return (int)cudaSuccess;
    const unsigned grid = (unsigned)((threads + MV_THREADS - 1) / MV_THREADS);
    if (a->stats) rbrt::k_motion<true><<<grid, MV_THREADS, 0, stream>>>(*a);
    else rbrt::k_motion<false><<<grid, MV_THREADS, 0, stream>>>(*a);
    return (int)cudaGetLastError();
}
