// wind.cu — generalized winding numbers on device memory (rbrt_gpu_query_winding_device, DESIGN.md section 18).
//
// Built into its own shared object (librbrt_gpu_wind.so), which librbrt_gpu.so loads at run time: the device code of librbrt_gpu.so stays
// exactly the build the GPU tests verified.  Two parts:
//  - k_wind_links / k_wind_nodes: the moments of every child slot of one mesh's 4-wide tree and of its root, bottom up on the refit's
//    scheme (update.cu): parent links from the child refs, an arrival counter per node, and the last child to arrive carries on.
//  - k_winding: the query, shaped like k_nearest (point.cu): persistent warps take points from a global cursor, one lane per point; a
//    lane sums its elements on its own, then mesh by mesh a warp-voted traversal of one node step or one leaf-triangle term per step.  A
//    node step reads the node's child refs and the four moment records; a far child adds its expansion, any other is entered or pushed.
//    Nothing is pruned, so the stack holds refs only.  Terms are f32, the sum is f64 (winding.cuh).
#include "winding.cuh"
#include "intersect.cuh"

namespace rbrt {
namespace {

#define WD_THREADS 128
#define WD_BLOCKS 8             // resident blocks per SM: 8 x 128 threads = 64 registers per thread, as k_nearest
#define WD_SMEM_STACK 32        // traversal-stack entries per lane in shared memory (16 KB per block); deeper ones in local memory
#define WD_FETCH_THRESHOLD 8    // re-fill the warp when fewer lanes than this still traverse (k_nearest's PT_FETCH_THRESHOLD)
#define WD_FULL 0xFFFFFFFFu

// ------------------------------------------------------------------ moments
// unused slot: inverted box on every axis (lo 65535, hi 0) and the dummy leaf ref (bvh_build.cu:248-250), the test of update.cu's
// slot_used on the raw words: the boxes are never decoded, so a qstep = NaN axis does not matter
__device__ __forceinline__ bool wd_slot_used(const uint4& a, const uint4& b, const uint4& c, int32_t ref, int k) {
    const uint32_t w[12] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, c.x, c.y, c.z, c.w};
    return !(w[3 * k] == 0x0000FFFFu && w[3 * k + 1] == 0x0000FFFFu && w[3 * k + 2] == 0x0000FFFFu && ref == make_leaf_ref(0, 1));
}

// parent[c] = 4 * j + slot of every internal child c of node j; need[j] = how many internal children j has.  A mesh whose root is a
// leaf gets its root record here.
__global__ void k_wind_links(WindMomentArgs A) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j == 0 && A.mesh->root_ref < 0) {
        const uint32_t code = (uint32_t)~A.mesh->root_ref;
        WindMom m;
        wind_leaf(A.tris + 3 * (size_t)(code >> 3), (code & 7u) + 1u, m);
        float4 r[4];
        wind_store(m, r);
        for (int i = 0; i < 4; ++i) A.root[i] = r[i];
    }
    if (j >= *A.live_nodes) return;
    const uint4* nd = A.nodes + 4 * (size_t)j;
    const uint4 a = nd[0], b = nd[1], c = nd[2], d = nd[3];
    const int32_t ref[4] = {(int32_t)d.x, (int32_t)d.y, (int32_t)d.z, (int32_t)d.w};
    uint32_t cnt = 0;
    for (int k = 0; k < 4; ++k)
        if (wd_slot_used(a, b, c, ref[k], k) && ref[k] >= 0) { A.parent[ref[k]] = 4 * j + (uint32_t)k; ++cnt; }
    A.need[j] = cnt; A.arrive[j] = 0;
}

// One thread starts at every node without internal children.  At node j it forms the records of j's leaf children from their triangles,
// reads those of its internal children (written by their threads), stores all four, and merges them into j's own record: the root
// record for node 0, else the record of j's slot in its parent.  The last child to arrive at the parent carries on with it.
__global__ void k_wind_nodes(WindMomentArgs A) {
    uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= *A.live_nodes || A.need[j]) return;
    for (;;) {
        const uint4* nd = A.nodes + 4 * (size_t)j;
        const uint4 a = nd[0], b = nd[1], c = nd[2], d = nd[3];
        const int32_t ref[4] = {(int32_t)d.x, (int32_t)d.y, (int32_t)d.z, (int32_t)d.w};
        float4 rec[4][4];
        double area[4];
        for (int k = 0; k < 4; ++k) {
            float4* dst = A.mom + 4 * (4 * (size_t)j + k);
            if (!wd_slot_used(a, b, c, ref[k], k)) {
                wind_unused(rec[k]); area[k] = 0.0;
                for (int i = 0; i < 4; ++i) dst[i] = rec[k][i];
            } else if (ref[k] < 0) {
                const uint32_t code = (uint32_t)~ref[k];
                WindMom m;
                wind_leaf(A.tris + 3 * (size_t)(code >> 3), (code & 7u) + 1u, m);
                wind_store(m, rec[k]); area[k] = m.area;
                for (int i = 0; i < 4; ++i) dst[i] = rec[k][i];
            } else {                                                      // written by the child's thread before it arrived here
                for (int i = 0; i < 4; ++i) rec[k][i] = __ldcg(dst + i);
                area[k] = __ldcg(A.area + 4 * (size_t)j + k);
            }
        }
        WindMom m;
        if (!wind_merge(rec, area, m)) { m = WindMom(); m.R = -1.0f; }
        float4 out[4];
        wind_store(m, out);
        if (j == 0) { for (int i = 0; i < 4; ++i) A.root[i] = out[i]; return; }
        const uint32_t p = A.parent[j], pj = p >> 2;
        for (int i = 0; i < 4; ++i) __stcg(A.mom + 4 * (size_t)p + i, out[i]);
        __stcg(A.area + p, m.area);
        __threadfence();
        if (atomicAdd(&A.arrive[pj], 1u) + 1u != A.need[pj]) return;    // a sibling subtree is still on its way up
        __threadfence();
        j = pj;
    }
}

// ------------------------------------------------------------------ the query
// The traversal stack of refs: entry i of all lanes shares a row in shared memory ([entry][thread], conflict-free), entries from
// WD_SMEM_STACK on live in the lane's local array.
struct WdStack {
    int32_t* sr;                 // &s_ref[0][threadIdx.x]
    int32_t* lr;
    __device__ __forceinline__ void put(int i, int32_t r) const { if (i < WD_SMEM_STACK) sr[i * WD_THREADS] = r; else lr[i - WD_SMEM_STACK] = r; }
    __device__ __forceinline__ int32_t get(int i) const { return i < WD_SMEM_STACK ? sr[i * WD_THREADS] : lr[i - WD_SMEM_STACK]; }
};

// One node step: the four children's records; a far child adds its expansion to acc, a near one is pushed (an unused slot, R < 0, is
// skipped).  Returns the next ref: the top of the stack.
__device__ __forceinline__ int32_t wd_node_step(const uint4* __restrict__ nd, const float4* __restrict__ mom, f3 p, float beta, double& acc,
                                                const WdStack& stack, int& sp) {
    const uint4 refs = __ldg(nd + 3);
    const int32_t ref[4] = {(int32_t)refs.x, (int32_t)refs.y, (int32_t)refs.z, (int32_t)refs.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float4 m0 = __ldg(mom + 4 * k);
        if (!(m0.w >= 0.0f)) continue;
        f3 u; float inv;
        if (wind_far(p, m0, beta, u, inv)) acc += (double)wind_expand(u, inv, __ldg(mom + 4 * k + 1), __ldg(mom + 4 * k + 2), __ldg(mom + 4 * k + 3));
        else stack.put(sp++, ref[k]);
    }
    return stack.get(--sp);
}

template <bool COUNT>
__global__ void __launch_bounds__(WD_THREADS, WD_BLOCKS) k_winding(WindQueryArgs A) {
    const SceneDev& S = A.S;
    __shared__ int32_t s_ref[WD_SMEM_STACK][WD_THREADS];
    int32_t lref[RBRT_STACK - WD_SMEM_STACK];
    const WdStack stack = {&s_ref[0][threadIdx.x], lref};
    const uint32_t lane = threadIdx.x & 31, lt = (1u << lane) - 1;
    // ---- point state
    bool has_pt = false, exhausted = false, nan = false;
    uint32_t pi = 0, mi = 0;
    f3 p = mk3(0, 0, 0);
    double acc = 0.0;
    // ---- traversal state of the current mesh
    int32_t cur = RBRT_SENTINEL; int sp = 0;
    const uint4* __restrict__ nodes = reinterpret_cast<const uint4*>(S.nodes);
    const float4* __restrict__ mom = A.mom;
    uint32_t tri_base = 0;
    uint32_t n_nodes = 0, n_tris = 0, n_nan = 0;

    auto finish_point = [&]() {
        const float w = nan ? __uint_as_float(0x7FC00000u) : (float)(acc / WD_FOUR_PI);
        if (A.out.winding) A.out.winding[pi] = w;
        if (A.out.inside) A.out.inside[pi] = fabsf(w) > 0.5f ? 1 : 0;
    };
    // A lane whose traversal ended: the next mesh (a far root adds its expansion), or the result.
    auto advance = [&]() {
        if (!has_pt || cur != RBRT_SENTINEL) return;
        while (++mi < S.n_meshes) {
            const MeshDev& M = S.meshes[mi];
            if (M.n_tris == 0) continue;
            const float4* rr = A.root + 4 * (size_t)mi;
            const float4 m0 = __ldg(rr);
            f3 u; float inv;
            if (wind_far(p, m0, A.beta, u, inv)) { acc += (double)wind_expand(u, inv, __ldg(rr + 1), __ldg(rr + 2), __ldg(rr + 3)); continue; }
            nodes = reinterpret_cast<const uint4*>(S.nodes) + 4 * (size_t)M.node_base;
            mom = A.mom + 16 * (size_t)M.node_base;
            tri_base = M.tri_base;
            sp = 0; stack.put(sp++, RBRT_SENTINEL); cur = M.root_ref;
            return;
        }
        finish_point();
        has_pt = false;
    };

    for (;;) {
        advance();
        // ---- idle lanes take the next points (one atomic per warp)
        if (!exhausted) {
            const uint32_t m = __ballot_sync(WD_FULL, !has_pt);
            if (m) {
                const uint32_t leader = __ffs(m) - 1;
                unsigned long long base = 0;
                if (lane == leader) base = atomicAdd(&A.ctr[WD_ST_HEAD], (unsigned long long)__popc(m));
                base = __shfl_sync(WD_FULL, base, leader);
                if (!has_pt) {
                    const unsigned long long qi = base + __popc(m & lt);
                    if (qi < A.n) {
                        pi = (uint32_t)qi;
                        const float* r = A.points + 3 * (size_t)pi;
                        p = mk3(r[0], r[1], r[2]);
                        acc = 0.0; mi = 0xFFFFFFFFu; cur = RBRT_SENTINEL;
                        nan = p.x != p.x || p.y != p.y || p.z != p.z;
                        if (nan) { ++n_nan; mi = S.n_meshes; }
                        else {
                            for (uint32_t i = 0; i < S.n_spheres; ++i) {      // the elements
                                const float4 el = __ldg(S.spheres + i);
                                if (S.n_etris && __ldg(S.elem_kind + i)) {
                                    const float4* rec = S.etris + 4 * (size_t)__float_as_uint(el.x);
                                    const float4 a = __ldg(rec), b = __ldg(rec + 1), c = __ldg(rec + 2);
                                    acc += (double)wind_tri(p, mk3(a.x, a.y, a.z), mk3(b.x, b.y, b.z), mk3(c.x, c.y, c.z));
                                } else acc += WD_TWO_PI * wind_sphere(p, el);
                            }
                        }
                        has_pt = true;
                        advance();
                    }
                }
                if (base + __popc(m) >= A.n) exhausted = true;
            }
        }
        const uint32_t active = __ballot_sync(WD_FULL, cur != RBRT_SENTINEL);
        if (active == 0) { if (exhausted) break; continue; }
        const int threshold = exhausted ? 1 : WD_FETCH_THRESHOLD;
        // ---- warp-voted traversal: one node step or one triangle term per step, whichever more lanes wait for
        for (;;) {
            const bool at_node = (uint32_t)cur < (uint32_t)RBRT_SENTINEL, at_leaf = cur < 0;
            const int nn = __popc(__ballot_sync(WD_FULL, at_node)), nl = __popc(__ballot_sync(WD_FULL, at_leaf));
            if (nn + nl < threshold) break;
            if (nn >= nl) {
                if (at_node) {
                    cur = wd_node_step(nodes + 4 * (size_t)cur, mom + 16 * (size_t)cur, p, A.beta, acc, stack, sp);
                    if (COUNT) ++n_nodes;
                }
            } else if (at_leaf) {
                const uint32_t code = (uint32_t)(~cur);
                f3 v0, e1, e2; uint32_t orig;
                load_tri(S.tris, tri_base + (code >> 3), v0, e1, e2, orig);
                acc += (double)wind_tri(p, v0, e1, e2);
                cur = (code & 7u) ? (int32_t)~(code + 7u) : stack.get(--sp);   // {first + 1, count - 1}, or the stack
                if (COUNT) ++n_tris;
            }
        }
    }
    if (COUNT) {
        unsigned long long nn = n_nan, nd = n_nodes, tr = n_tris;
        for (int off = 16; off; off >>= 1) {
            nn += __shfl_down_sync(WD_FULL, nn, off);
            nd += __shfl_down_sync(WD_FULL, nd, off);
            tr += __shfl_down_sync(WD_FULL, tr, off);
        }
        if (lane == 0) {
            if (nn) atomicAdd(&A.ctr[WD_ST_NAN], nn);
            if (nd) atomicAdd(&A.ctr[WD_ST_NODES], nd);
            if (tr) atomicAdd(&A.ctr[WD_ST_TRIS], tr);
        }
    }
}

}  // namespace
}  // namespace rbrt

extern "C" int rbrt_wind_query_launch(const rbrt::WindQueryArgs* a, cudaStream_t stream) {
    if (!a->n || !a->blocks) return (int)cudaSuccess;
    if (a->count) rbrt::k_winding<true><<<a->blocks, WD_THREADS, 0, stream>>>(*a);
    else rbrt::k_winding<false><<<a->blocks, WD_THREADS, 0, stream>>>(*a);
    return (int)cudaGetLastError();
}

extern "C" int rbrt_wind_moments_launch(const rbrt::WindMomentArgs* a, cudaStream_t stream) {
    if (!a->n_tris) return (int)cudaSuccess;
    const uint32_t B = 128, g = (a->n_tris + B - 1) / B;                  // live nodes <= n_tris - 1; thread 0 also covers a leaf root
    rbrt::k_wind_links<<<g, B, 0, stream>>>(*a);
    rbrt::k_wind_nodes<<<g, B, 0, stream>>>(*a);
    return (int)cudaGetLastError();
}
