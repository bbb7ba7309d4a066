// query.cu — ray queries on device memory (rbrt_gpu_query_closest_device / rbrt_gpu_query_occluded_device, DESIGN.md section 12).
//
// Built into its own shared object (librbrt_gpu_query.so), which librbrt_gpu.so loads at run time: the device code of librbrt_gpu.so stays
// exactly the build the GPU tests verified.  Both queries are defined by Scene::hit as rbrt_gpu_trace_rays(RBRT_TRACE_BVH) reports it:
//   closest  = that hit, field for field (k_trace_rays' record, split into planes);
//   occluded = 1 when it is a hit with dist < max_dist, 2 for a NaN ray, 0 otherwise.
// Persistent warps take rays from a global cursor, 32 lanes at a time.  A lane runs its ray's element loop on its own, then mesh by mesh the
// box pre-test and the warp-voted BVH traversal of the renderer's k_trace (one node visit or one triangle test per step, whichever more
// lanes wait for), with the first stack entries in shared memory.  Lanes may be in different meshes at the same step.  When fewer than
// QRY_FETCH_THRESHOLD lanes still traverse, the warp closes finished meshes and re-fills idle lanes from the cursor.  The result does not
// depend on the tree or the order of visits (DESIGN.md section 2), only on every prune bound being conservative.
#include "query.cuh"

namespace rbrt {
namespace {

#define QRY_THREADS 128
#define QRY_BLOCKS 8            // resident blocks per SM: 8 x 128 threads = 64 registers per thread, as k_trace
#define QRY_SMEM_STACK 16       // traversal-stack entries per lane in shared memory (8 KB per block); deeper entries go to local memory
#define QRY_FETCH_THRESHOLD 8   // re-fill the warp when fewer lanes than this still traverse (k_trace's FETCH_THRESHOLD)
#define QRY_FULL 0xFFFFFFFFu

template <bool OCC, bool COUNT>
__global__ void __launch_bounds__(QRY_THREADS, QRY_BLOCKS) k_query(QueryArgs A) {
    const SceneDev& S = A.S;
    __shared__ int32_t s_stack[QRY_SMEM_STACK][QRY_THREADS];
    int32_t lstack[RBRT_STACK];
    const StackS<QRY_SMEM_STACK, QRY_THREADS> stack = {&s_stack[0][threadIdx.x], lstack};
    const uint32_t lane = threadIdx.x & 31, lt = (1u << lane) - 1;
    // ---- ray state
    bool has_ray = false, exhausted = false;
    uint32_t ri = 0, mi = 0;
    f3 o = mk3(0, 0, 0), d = mk3(0, 0, 0);
    float max_dist = 0.0f;                                                // OCC
    int occ = 0;                                                          // OCC: 0 / 1 / 2
    bool early = false;                                                   // OCC: the first occluding triangle ends a mesh
    Hit best; best.kind = -1; best.elem = 0; best.tri = 0; best.t = 0.0f; best.dist = 0.0f;   // closest: over elements + finished meshes
    float closest = 0.0f;
    // ---- traversal state of the current mesh
    RaySlabs R = {0, 0, 0, 0, 0, 0, RBRT_SEL_LO, RBRT_SEL_LO, RBRT_SEL_LO, RBRT_SEL_HI, RBRT_SEL_HI, RBRT_SEL_HI};
    int32_t cur = RBRT_SENTINEL; int sp = 0;
    float best_t = 0.0f, t_prune = 0.0f, t_limit = 0.0f; uint32_t best_idx = 0xFFFFFFFFu;
    const uint4* __restrict__ nodes = reinterpret_cast<const uint4*>(S.nodes); uint32_t tri_base = 0;
    uint32_t n_nodes = 0, n_tris = 0, n_nan = 0;

    auto finish_ray = [&]() {
        if (OCC) {
            A.occluded[ri] = (uint8_t)occ;
            if (occ == 2) ++n_nan;
            return;
        }
        int32_t kind = RBRT_HIT_NONE;                                     // a miss: zeros, as k_trace_rays writes it
        uint32_t e = 0, tri = 0; float t = 0.0f, dist = 0.0f;
        f3 p = mk3(0, 0, 0), nrm = mk3(0, 0, 0);
        if (best.kind >= 0) {
            p = o + best.t * d;
            if (best.kind == 0) {
                nrm = element_normal(S, best.elem, p);                    // sphere: p - c, un-normalised
                kind = (S.n_etris && __ldg(S.elem_kind + best.elem)) ? RBRT_HIT_TRIANGLE : RBRT_HIT_SPHERE;
            } else {
                const float4 nn = __ldg(S.normals + S.meshes[best.elem].nrm_base + best.tri);
                nrm = mk3(nn.x, nn.y, nn.z); kind = RBRT_HIT_MESH;
            }
            e = best.elem; tri = best.tri; t = best.t; dist = best.dist;
        } else if (best.kind == -2) ++n_nan;
        const rbrt_query_out& q = A.out;
        if (q.t) q.t[ri] = t;
        if (q.dist) q.dist[ri] = dist;
        if (q.kind) q.kind[ri] = kind;
        if (q.elem_idx) q.elem_idx[ri] = e;
        if (q.tri_idx) q.tri_idx[ri] = tri;
        if (q.point) { float* w = q.point + 3 * (size_t)ri; w[0] = p.x; w[1] = p.y; w[2] = p.z; }
        if (q.normal) { float* w = q.normal + 3 * (size_t)ri; w[0] = nrm.x; w[1] = nrm.y; w[2] = nrm.z; }
    };
    // A lane whose traversal ended: close the mesh, start the next one whose box the ray enters, or write the result.
    auto advance = [&]() {
        if (!has_ray || cur != RBRT_SENTINEL) return;
        if (best_idx != 0xFFFFFFFFu) {
            if (OCC) { if (!early && mesh_hit_occludes(o, d, best_t, max_dist)) occ = 1; }
            else {
                const f3 p = o + best_t * d;                              // ray.point_at (mesh.rs:247)
                const float dist = len3(o - p);                           // mesh.rs:248
                if (dist > RBRT_MIN_DIST && dist < RBRT_MAX_DIST && dist < closest) {   // mesh.rs:249 + scene.rs:36
                    closest = dist; best.kind = 1; best.elem = mi; best.tri = best_idx; best.t = best_t; best.dist = dist;
                }
            }
            best_idx = 0xFFFFFFFFu;
        }
        if (OCC ? occ == 0 && max_dist > RBRT_MIN_DIST : best.kind != -2) {   // (max_dist <= 0.001 or NaN: no mesh hit can be below it)
            while (++mi < S.n_meshes) {                                   // later meshes, in order (scene.rs:33-41)
                const MeshDev& M = S.meshes[mi];
                if (M.n_tris == 0 || !mesh_bbox_hit(M, o, d)) continue;
                t_limit = query_t_limit(o, d, OCC ? max_dist : closest);
                t_prune = t_limit; best_t = 1000000.0f; best_idx = 0xFFFFFFFFu;   // min_param init (triangle.rs:398)
                nodes = reinterpret_cast<const uint4*>(S.nodes) + 4 * (size_t)M.node_base; tri_base = M.tri_base;
                R = ray_slabs(M, o, d);
                sp = 0; stack.put(sp++, RBRT_SENTINEL); cur = M.root_ref;
                return;
            }
        }
        finish_ray();
        has_ray = false;
    };

    for (;;) {
        advance();
        // ---- idle lanes take the next rays (one atomic per warp)
        if (!exhausted) {
            const uint32_t m = __ballot_sync(QRY_FULL, !has_ray);
            if (m) {
                const uint32_t leader = __ffs(m) - 1;
                unsigned long long base = 0;
                if (lane == leader) base = atomicAdd(&A.ctr[QRY_ST_HEAD], (unsigned long long)__popc(m));
                base = __shfl_sync(QRY_FULL, base, leader);
                if (!has_ray) {
                    const unsigned long long qi = base + __popc(m & lt);
                    if (qi < A.n) {
                        ri = (uint32_t)qi;
                        const float* r = reinterpret_cast<const float*>(A.rays + ri);
                        o = mk3(r[0], r[1], r[2]); d = mk3(r[3], r[4], r[5]);
                        if (OCC) {                                        // elements first, every one of them (query.cuh)
                            max_dist = A.max_dist ? A.max_dist[ri] : __int_as_float(0x7F800000);
                            occ = occluded_elements(S, o, d, max_dist);
                            early = occluded_early_exit_ok(o, d);
                        } else {
                            best.kind = -1; best.elem = 0; best.tri = 0; best.t = 0.0f; best.dist = 0.0f;
                            closest = 3.40282347e+38f;                    // f32::MAX (scene.rs:21)
                            for (uint32_t i = 0; i < S.n_spheres; ++i) {  // spheres first, in order (scene.rs:23-31)
                                float t, dist;
                                const int rr = element_intersect(S, i, o, d, t, dist);
                                if (rr < 0) { best.kind = -2; break; }
                                if (rr && dist < closest) { closest = dist; best.kind = 0; best.elem = i; best.t = t; best.dist = dist; }
                            }
                        }
                        mi = 0xFFFFFFFFu; best_idx = 0xFFFFFFFFu; cur = RBRT_SENTINEL;
                        has_ray = true;
                        advance();
                    }
                }
                if (base + __popc(m) >= A.n) exhausted = true;
            }
        }
        const uint32_t active = __ballot_sync(QRY_FULL, cur != RBRT_SENTINEL);
        if (active == 0) { if (exhausted) break; continue; }
        const int threshold = exhausted ? 1 : QRY_FETCH_THRESHOLD;
        if (OCC) traverse_voted_occluded<COUNT>(nodes, S.tris, tri_base, R, o, d, t_limit, max_dist, early, stack, sp, cur, best_t, best_idx, t_prune,
                                                occ, threshold, n_nodes, n_tris);
        else traverse_voted<COUNT, false>(nodes, S.tris, tri_base, R, o, d, t_limit, stack, sp, cur, best_t, best_idx, t_prune, threshold, n_nodes, n_tris);
    }
    if (COUNT) {
        unsigned long long nan = n_nan, nd = n_nodes, tr = n_tris;
        for (int off = 16; off; off >>= 1) {
            nan += __shfl_down_sync(QRY_FULL, nan, off);
            nd += __shfl_down_sync(QRY_FULL, nd, off);
            tr += __shfl_down_sync(QRY_FULL, tr, off);
        }
        if (lane == 0) {
            if (nan) atomicAdd(&A.ctr[QRY_ST_NAN], nan);
            if (nd) atomicAdd(&A.ctr[QRY_ST_NODES], nd);
            if (tr) atomicAdd(&A.ctr[QRY_ST_TRIS], tr);
        }
    }
}

}  // namespace
}  // namespace rbrt

extern "C" int rbrt_query_launch(const rbrt::QueryArgs* a, cudaStream_t stream) {
    if (!a->n || !a->blocks) return (int)cudaSuccess;
    if (a->occluded) {
        if (a->count) rbrt::k_query<true, true><<<a->blocks, QRY_THREADS, 0, stream>>>(*a);
        else rbrt::k_query<true, false><<<a->blocks, QRY_THREADS, 0, stream>>>(*a);
    } else {
        if (a->count) rbrt::k_query<false, true><<<a->blocks, QRY_THREADS, 0, stream>>>(*a);
        else rbrt::k_query<false, false><<<a->blocks, QRY_THREADS, 0, stream>>>(*a);
    }
    return (int)cudaGetLastError();
}
