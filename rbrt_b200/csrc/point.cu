// point.cu — nearest-surface queries on device memory (rbrt_gpu_query_nearest_device, DESIGN.md section 17).
//
// Built into its own shared object (librbrt_gpu_point.so), which librbrt_gpu.so loads at run time: the device code of librbrt_gpu.so stays
// exactly the build the GPU tests verified.  The shape is the query module's k_query (section 12): persistent warps take points from a
// global cursor, one lane per point.  A lane runs every element on its own, then mesh by mesh the box pre-test and a warp-voted traversal of
// the mesh's 4-wide tree (one node visit or one triangle test per step, whichever more lanes wait for), with the first stack entries in
// shared memory.  When fewer than PT_FETCH_THRESHOLD lanes still traverse, the warp closes finished meshes and re-fills idle lanes.
// What differs from the ray traversal is the prune: a child box is entered, and a stacked entry is kept, while the lower bound of its squared
// distance to the point does not exceed pt_prune_d2 (point.cuh, with the proof that it never drops a triangle that could be recorded).
// The winner is the lexicographic minimum of (d2, scene order), so the answer does not depend on the tree or on the order of visits.
#include "point.cuh"
#include "intersect.cuh"

namespace rbrt {
namespace {

#define PT_THREADS 128
#define PT_BLOCKS 8             // resident blocks per SM: 8 x 128 threads = 64 registers per thread, as k_query
#define PT_SMEM_STACK 16        // traversal-stack entries per lane in shared memory (16 KB per block: ref and bound); deeper ones in local memory
#define PT_FETCH_THRESHOLD 8    // re-fill the warp when fewer lanes than this still traverse (k_query's QRY_FETCH_THRESHOLD)
#define PT_FULL 0xFFFFFFFFu

// The traversal stack of (ref, lower bound) pairs: entry i of all lanes shares a row in shared memory ([entry][thread], conflict-free),
// entries from PT_SMEM_STACK on live in the lane's local arrays.
struct PtStack {
    int32_t* sr; float* sb;      // &s_ref[0][threadIdx.x], &s_lb[0][threadIdx.x]
    int32_t* lr; float* lb;
    __device__ __forceinline__ void put(int i, int32_t r, float b) const {
        if (i < PT_SMEM_STACK) { sr[i * PT_THREADS] = r; sb[i * PT_THREADS] = b; } else { lr[i - PT_SMEM_STACK] = r; lb[i - PT_SMEM_STACK] = b; }
    }
    __device__ __forceinline__ int32_t get(int i, float& b) const {
        if (i < PT_SMEM_STACK) { b = sb[i * PT_THREADS]; return sr[i * PT_THREADS]; }
        b = lb[i - PT_SMEM_STACK]; return lr[i - PT_SMEM_STACK];
    }
};

// The next entry of the stack whose bound does not exceed prune_d2 (the sentinel's bound is 0: it always stops the loop).
__device__ __forceinline__ int32_t pt_pop(const PtStack& stack, int& sp, float prune_d2) {
    for (;;) {
        float b;
        const int32_t r = stack.get(--sp, b);
        if (!(b > prune_d2)) return r;
    }
}

// One node visit: each child's box decoded from its 16-bit words with the builder's own fmaf(q, qstep, qorg) (quant_lo / quant_hi check
// exactly that value against the box they cover), its lower bound, and the accepted children: the nearest is returned, the others pushed
// with their bounds.  An unused slot holds an inverted box (lo 65535, hi 0 on every axis) and is skipped.
__device__ __forceinline__ int32_t pt_node_step(const uint4* __restrict__ nd, f3 p, const float (&org)[3], const float (&step)[3], float prune_d2,
                                                const PtStack& stack, int& sp) {
    uint4 w0, w1, w2, w3;
    ldg256(nd, w0, w1); ldg256(nd + 2, w2, w3);
    float b[4]; int32_t r[4];
#define PT_DEC(W, SEL, K) __fmaf_rn(q16(W, SEL) - 8388608.0f, step[K], org[K])
#define PT_CHILD(k, X, Y, Z, REF) { \
        const float lb_ = pt_box_d2(p, PT_DEC(X, RBRT_SEL_LO, 0), PT_DEC(Y, RBRT_SEL_LO, 1), PT_DEC(Z, RBRT_SEL_LO, 2), \
                                    PT_DEC(X, RBRT_SEL_HI, 0), PT_DEC(Y, RBRT_SEL_HI, 1), PT_DEC(Z, RBRT_SEL_HI, 2)); \
        const bool in_ = ((X) & 0xFFFFu) <= ((X) >> 16) && !(lb_ > prune_d2); \
        b[k] = in_ ? lb_ : __int_as_float(0x7F800000); r[k] = in_ ? (int32_t)(REF) : RBRT_SENTINEL; }
    PT_CHILD(0, w0.x, w0.y, w0.z, w3.x) PT_CHILD(1, w0.w, w1.x, w1.y, w3.y) PT_CHILD(2, w1.z, w1.w, w2.x, w3.z) PT_CHILD(3, w2.y, w2.z, w2.w, w3.w)
#undef PT_CHILD
#undef PT_DEC
    // bring the nearest child to slot 0 (three exchanges, as bvh4_step); the other accepted children are pushed in slot order
#define PT_CSWAP(a, c) { const bool sw = b[c] < b[a]; const float bl = sw ? b[c] : b[a], bh = sw ? b[a] : b[c]; \
        const int32_t ra = sw ? r[c] : r[a], rc = sw ? r[a] : r[c]; b[a] = bl; b[c] = bh; r[a] = ra; r[c] = rc; }
    PT_CSWAP(0, 1) PT_CSWAP(2, 3) PT_CSWAP(0, 2)
#undef PT_CSWAP
    if (r[3] != RBRT_SENTINEL) stack.put(sp++, r[3], b[3]);
    if (r[2] != RBRT_SENTINEL) stack.put(sp++, r[2], b[2]);
    if (r[1] != RBRT_SENTINEL) stack.put(sp++, r[1], b[1]);
    return r[0] != RBRT_SENTINEL ? r[0] : pt_pop(stack, sp, prune_d2);
}

// The running winner of one point: kind -1 none, 0 an element, 1 a mesh triangle (elem = mesh index, tri = original index, slot = record).
struct PtBest { float d2; int kind; uint32_t elem, tri, slot; };

template <bool COUNT>
__global__ void __launch_bounds__(PT_THREADS, PT_BLOCKS) k_nearest(PointArgs A) {
    const SceneDev& S = A.S;
    __shared__ int32_t s_ref[PT_SMEM_STACK][PT_THREADS];
    __shared__ float s_lb[PT_SMEM_STACK][PT_THREADS];
    int32_t lref[RBRT_STACK - PT_SMEM_STACK];
    float llb[RBRT_STACK - PT_SMEM_STACK];
    const PtStack stack = {&s_ref[0][threadIdx.x], &s_lb[0][threadIdx.x], lref, llb};
    const uint32_t lane = threadIdx.x & 31, lt = (1u << lane) - 1;
    // ---- point state
    bool has_pt = false, exhausted = false;
    uint32_t pi = 0, mi = 0;
    f3 p = mk3(0, 0, 0);
    float md = 0.0f;                                                      // max_dist
    PtBest best; best.d2 = 0.0f; best.kind = -1; best.elem = 0; best.tri = 0; best.slot = 0;
    // ---- traversal state of the current mesh
    float org[3] = {0, 0, 0}, step[3] = {0, 0, 0}, s = 0.0f, prune_d2 = 0.0f;
    int32_t cur = RBRT_SENTINEL; int sp = 0;
    const uint4* __restrict__ nodes = reinterpret_cast<const uint4*>(S.nodes); uint32_t tri_base = 0;
    uint32_t n_nodes = 0, n_tris = 0, n_nan = 0;

    auto finish_point = [&]() {
        int32_t kind = RBRT_HIT_NONE;                                     // no candidate: dist +inf, zeros elsewhere
        uint32_t e = 0, tri = 0;
        float dist = __int_as_float(0x7F800000), u = 0.0f, v = 0.0f;
        f3 q = mk3(0, 0, 0), nrm = mk3(0, 0, 0);
        if (best.kind >= 0) {                                             // the winner's routine again: the same bits as when it was recorded
            dist = XSQRT(best.d2); e = best.elem;
            if (best.kind == 0) {
                const float4 el = __ldg(S.spheres + e);
                if (S.n_etris && __ldg(S.elem_kind + e)) {
                    const float4* rec = S.etris + 4 * (size_t)__float_as_uint(el.x);
                    const float4 a = __ldg(rec), b = __ldg(rec + 1), c = __ldg(rec + 2);
                    closest_on_triangle(p, mk3(a.x, a.y, a.z), mk3(b.x, b.y, b.z), mk3(c.x, c.y, c.z), q, u, v);
                    kind = RBRT_HIT_TRIANGLE;
                } else {
                    closest_on_sphere(p, el, q);
                    kind = RBRT_HIT_SPHERE;
                }
                nrm = element_normal(S, e, q);
            } else {
                f3 v0, e1, e2; uint32_t orig;
                load_tri(S.tris, best.slot, v0, e1, e2, orig);
                closest_on_triangle(p, v0, e1, e2, q, u, v);
                const float4 nn = __ldg(S.normals + S.meshes[e].nrm_base + best.tri);
                nrm = mk3(nn.x, nn.y, nn.z); kind = RBRT_HIT_MESH; tri = best.tri;
            }
        }
        const rbrt_nearest_out& o = A.out;
        if (o.dist) o.dist[pi] = dist;
        if (o.kind) o.kind[pi] = kind;
        if (o.elem_idx) o.elem_idx[pi] = e;
        if (o.tri_idx) o.tri_idx[pi] = tri;
        if (o.point) { float* w = o.point + 3 * (size_t)pi; w[0] = q.x; w[1] = q.y; w[2] = q.z; }
        if (o.normal) { float* w = o.normal + 3 * (size_t)pi; w[0] = nrm.x; w[1] = nrm.y; w[2] = nrm.z; }
        if (o.uv) { float* w = o.uv + 2 * (size_t)pi; w[0] = u; w[1] = v; }
    };
    // A lane whose traversal ended: start the next mesh whose box passes the bound, or write the result.
    auto advance = [&]() {
        if (!has_pt || cur != RBRT_SENTINEL) return;
        while (++mi < S.n_meshes) {                                       // later meshes, in order
            const MeshDev& M = S.meshes[mi];
            if (M.n_tris == 0) continue;
            s = pt_scale(p, M);
            prune_d2 = pt_prune_d2(md, best.d2, s);
            if (pt_box_d2(p, M.lo[0], M.lo[1], M.lo[2], M.hi[0], M.hi[1], M.hi[2]) > prune_d2) continue;
            for (int k = 0; k < 3; ++k) { org[k] = M.qorg[k]; step[k] = M.qstep[k]; }
            nodes = reinterpret_cast<const uint4*>(S.nodes) + 4 * (size_t)M.node_base; tri_base = M.tri_base;
            sp = 0; stack.put(sp++, RBRT_SENTINEL, 0.0f); cur = M.root_ref;
            return;
        }
        finish_point();
        has_pt = false;
    };

    for (;;) {
        advance();
        // ---- idle lanes take the next points (one atomic per warp)
        if (!exhausted) {
            const uint32_t m = __ballot_sync(PT_FULL, !has_pt);
            if (m) {
                const uint32_t leader = __ffs(m) - 1;
                unsigned long long base = 0;
                if (lane == leader) base = atomicAdd(&A.ctr[PT_ST_HEAD], (unsigned long long)__popc(m));
                base = __shfl_sync(PT_FULL, base, leader);
                if (!has_pt) {
                    const unsigned long long qi = base + __popc(m & lt);
                    if (qi < A.n) {
                        pi = (uint32_t)qi;
                        const float* r = A.points + 3 * (size_t)pi;
                        p = mk3(r[0], r[1], r[2]);
                        md = A.max_dist ? A.max_dist[pi] : __int_as_float(0x7F800000);
                        best.d2 = __int_as_float(0x7F800000); best.kind = -1; best.elem = 0; best.tri = 0; best.slot = 0;
                        mi = 0xFFFFFFFFu; cur = RBRT_SENTINEL;
                        const bool nan = p.x != p.x || p.y != p.y || p.z != p.z;
                        if (nan) ++n_nan;
                        // A point with a NaN or inf coordinate has a non-finite d2 for every candidate, and a bound that is NaN, 0 or negative
                        // accepts nothing: such a point is a miss without a look at the scene.
                        if (nan || !(fabsf(p.x) <= 3.40282347e+38f && fabsf(p.y) <= 3.40282347e+38f && fabsf(p.z) <= 3.40282347e+38f) || !(md > 0.0f)) {
                            mi = S.n_meshes;
                        } else {
                            for (uint32_t i = 0; i < S.n_spheres; ++i) {      // the elements, in order (a strict < keeps the first minimum)
                                const float4 el = __ldg(S.spheres + i);
                                f3 q; float u, v, d2;
                                if (S.n_etris && __ldg(S.elem_kind + i)) {
                                    const float4* rec = S.etris + 4 * (size_t)__float_as_uint(el.x);
                                    const float4 a = __ldg(rec), b = __ldg(rec + 1), c = __ldg(rec + 2);
                                    d2 = closest_on_triangle(p, mk3(a.x, a.y, a.z), mk3(b.x, b.y, b.z), mk3(c.x, c.y, c.z), q, u, v);
                                } else d2 = closest_on_sphere(p, el, q);
                                if (d2 < best.d2 && pt_accept(d2, md)) { best.d2 = d2; best.kind = 0; best.elem = i; }
                            }
                        }
                        has_pt = true;
                        advance();
                    }
                }
                if (base + __popc(m) >= A.n) exhausted = true;
            }
        }
        const uint32_t active = __ballot_sync(PT_FULL, cur != RBRT_SENTINEL);
        if (active == 0) { if (exhausted) break; continue; }
        const int threshold = exhausted ? 1 : PT_FETCH_THRESHOLD;
        // ---- warp-voted traversal: one node visit or one triangle test per step, whichever more lanes wait for
        for (;;) {
            const bool at_node = (uint32_t)cur < (uint32_t)RBRT_SENTINEL, at_leaf = cur < 0;
            const int nn = __popc(__ballot_sync(PT_FULL, at_node)), nl = __popc(__ballot_sync(PT_FULL, at_leaf));
            if (nn + nl < threshold) break;
            if (nn >= nl) {
                if (at_node) { cur = pt_node_step(nodes + 4 * (size_t)cur, p, org, step, prune_d2, stack, sp); if (COUNT) ++n_nodes; }
            } else if (at_leaf) {
                const uint32_t code = (uint32_t)(~cur), slot = tri_base + (code >> 3);
                f3 v0, e1, e2, q; uint32_t orig; float u, v;
                load_tri(S.tris, slot, v0, e1, e2, orig);
                const float d2 = closest_on_triangle(p, v0, e1, e2, q, u, v);
                // lexicographic (d2, scene order): within this mesh the lower original index wins a tie; an earlier element or mesh keeps it
                if ((d2 < best.d2 || (d2 == best.d2 && best.kind == 1 && best.elem == mi && orig < best.tri)) && pt_accept(d2, md)) {
                    best.d2 = d2; best.kind = 1; best.elem = mi; best.tri = orig; best.slot = slot;
                    prune_d2 = pt_prune_d2(md, best.d2, s);
                }
                cur = (code & 7u) ? (int32_t)~(code + 7u) : pt_pop(stack, sp, prune_d2);   // {first + 1, count - 1}, or the stack
                if (COUNT) ++n_tris;
            }
        }
    }
    if (COUNT) {
        unsigned long long nan = n_nan, nd = n_nodes, tr = n_tris;
        for (int off = 16; off; off >>= 1) {
            nan += __shfl_down_sync(PT_FULL, nan, off);
            nd += __shfl_down_sync(PT_FULL, nd, off);
            tr += __shfl_down_sync(PT_FULL, tr, off);
        }
        if (lane == 0) {
            if (nan) atomicAdd(&A.ctr[PT_ST_NAN], nan);
            if (nd) atomicAdd(&A.ctr[PT_ST_NODES], nd);
            if (tr) atomicAdd(&A.ctr[PT_ST_TRIS], tr);
        }
    }
}

}  // namespace
}  // namespace rbrt

extern "C" int rbrt_point_launch(const rbrt::PointArgs* a, cudaStream_t stream) {
    if (!a->n || !a->blocks) return (int)cudaSuccess;
    if (a->count) rbrt::k_nearest<true><<<a->blocks, PT_THREADS, 0, stream>>>(*a);
    else rbrt::k_nearest<false><<<a->blocks, PT_THREADS, 0, stream>>>(*a);
    return (int)cudaGetLastError();
}
