// bvh_build.cu — scene upload kernels + GPU LBVH build (north_star (1),(2)).
//
// Replaces the reference's per-mesh SoA conversion (mesh.rs:41-74,123-181): per triangle
// e1 = v1-v0, e2 = v2-v0 (mesh.rs:57-60) and the unit geometric normal normalize(cross(e1,e2))
// (triangle.rs:30-34) are computed with the same individually rounded f32 ops, then the
// triangles are put in Morton order and a binary LBVH is built over them:
//   63-bit Morton code of the triangle-box centre -> radix sort (CUB) -> Karras 2012 topology
//   -> bottom-up AABB refit with atomic arrival flags -> top-down collapse into 4-wide nodes of 64 bytes (child
//   boxes on a 16-bit grid over the mesh box), subtrees of <= leaf_size triangles collapsed into leaves.
#include "bvh_build.cuh"
#include <cub/device/device_radix_sort.cuh>
#include <cstring>
#include <cstdlib>

namespace rbrt {

// ------------------------------------------------------------------ per-triangle preparation
__device__ __forceinline__ uint64_t expand21(uint32_t v) {   // spread the low 21 bits, 2 zero bits between
    uint64_t x = v & 0x1FFFFFu;
    x = (x | x << 32) & 0x1F00000000FFFFull;
    x = (x | x << 16) & 0x1F0000FF0000FFull;
    x = (x | x << 8) & 0x100F00F00F00F00Full;
    x = (x | x << 4) & 0x10C30C30C30C30C3ull;
    x = (x | x << 2) & 0x1249249249249249ull;
    return x;
}

// traversal node emission: child boxes quantised OUTWARD (plus one step of margin, see intersect.cuh) onto the mesh's
// 16-bit grid  bound = qorg + q * qstep
struct QGrid { float org[3], step[3]; };
// Per-mesh build parameters, produced ON THE DEVICE by k_mesh_setup from the exact AABB (no host round trip)
struct BuildParams { float lo[3], inv_ext[3]; float pad; QGrid grid; };

__global__ void k_prepare(const float* __restrict__ raw, uint32_t n, const BuildParams* __restrict__ bp,
                          float4* __restrict__ normals, uint64_t* __restrict__ keys, uint32_t* __restrict__ vals) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float3 lo = make_float3(bp->lo[0], bp->lo[1], bp->lo[2]), inv_ext = make_float3(bp->inv_ext[0], bp->inv_ext[1], bp->inv_ext[2]);
    const float* t = raw + 9 * (size_t)i;
    f3 a = mk3(t[0], t[1], t[2]), b = mk3(t[3], t[4], t[5]), c = mk3(t[6], t[7], t[8]);
    f3 e1 = b - a, e2 = c - a;
    f3 nn = norm3(cross3(e1, e2));                                        // triangle.rs:30-34
    normals[i] = make_float4(nn.x, nn.y, nn.z, 0.0f);
    float cx = 0.5f * (fminf(a.x, fminf(b.x, c.x)) + fmaxf(a.x, fmaxf(b.x, c.x)));
    float cy = 0.5f * (fminf(a.y, fminf(b.y, c.y)) + fmaxf(a.y, fmaxf(b.y, c.y)));
    float cz = 0.5f * (fminf(a.z, fminf(b.z, c.z)) + fmaxf(a.z, fmaxf(b.z, c.z)));
    float fx = fminf(fmaxf((cx - lo.x) * inv_ext.x, 0.0f), 1.0f);
    float fy = fminf(fmaxf((cy - lo.y) * inv_ext.y, 0.0f), 1.0f);
    float fz = fminf(fmaxf((cz - lo.z) * inv_ext.z, 0.0f), 1.0f);
    uint32_t qx = min((uint32_t)(fx * 2097152.0f), 2097151u);
    uint32_t qy = min((uint32_t)(fy * 2097152.0f), 2097151u);
    uint32_t qz = min((uint32_t)(fz * 2097152.0f), 2097151u);
    keys[i] = (expand21(qx) << 2) | (expand21(qy) << 1) | expand21(qz);
    vals[i] = i;
}

// sorted position p -> triangle record {v0|orig, e1, e2} and padded leaf box
__global__ void k_emit_tris(const float* __restrict__ raw, const uint32_t* __restrict__ order, uint32_t n, const BuildParams* __restrict__ bp,
                            float4* __restrict__ tris, float4* __restrict__ leaf_lo, float4* __restrict__ leaf_hi) {
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const float pad = bp->pad;
    uint32_t orig = order[p];
    const float* t = raw + 9 * (size_t)orig;
    f3 a = mk3(t[0], t[1], t[2]), b = mk3(t[3], t[4], t[5]), c = mk3(t[6], t[7], t[8]);
    f3 e1 = b - a, e2 = c - a;                                            // mesh.rs:57-60
    tris[3 * (size_t)p] = make_float4(a.x, a.y, a.z, __uint_as_float(orig));
    tris[3 * (size_t)p + 1] = make_float4(e1.x, e1.y, e1.z, 0.0f);
    tris[3 * (size_t)p + 2] = make_float4(e2.x, e2.y, e2.z, 0.0f);
    leaf_lo[p] = make_float4(fminf(a.x, fminf(b.x, c.x)) - pad, fminf(a.y, fminf(b.y, c.y)) - pad, fminf(a.z, fminf(b.z, c.z)) - pad, 0.0f);
    leaf_hi[p] = make_float4(fmaxf(a.x, fmaxf(b.x, c.x)) + pad, fmaxf(a.y, fmaxf(b.y, c.y)) + pad, fmaxf(a.z, fmaxf(b.z, c.z)) + pad, 0.0f);
}

// ------------------------------------------------------------------ Karras 2012
__device__ __forceinline__ int delta(const uint64_t* __restrict__ keys, int n, int i, int j) {
    if (j < 0 || j >= n) return -1;
    uint64_t a = keys[i], b = keys[j];
    if (a == b) return 64 + __clz(i ^ j);                                 // tie-break on position
    return __clzll((long long)(a ^ b));
}

// child reference inside the build: >= 0 internal node, < 0 -> ~leaf position
__global__ void k_karras(const uint64_t* __restrict__ keys, int n, int2* __restrict__ children, int2* __restrict__ range,
                         int* __restrict__ parent_int, int* __restrict__ parent_leaf) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n - 1) return;
    int d = (delta(keys, n, i, i + 1) - delta(keys, n, i, i - 1)) >= 0 ? 1 : -1;
    int dmin = delta(keys, n, i, i - d);
    int lmax = 2;
    while (delta(keys, n, i, i + lmax * d) > dmin) lmax <<= 1;
    int l = 0;
    for (int t = lmax >> 1; t >= 1; t >>= 1)
        if (delta(keys, n, i, i + (l + t) * d) > dmin) l += t;
    int j = i + l * d;
    int dnode = delta(keys, n, i, j);
    int s = 0, t = l;
    do {
        t = (t + 1) >> 1;
        if (delta(keys, n, i, i + (s + t) * d) > dnode) s += t;
    } while (t > 1);
    int gamma = i + s * d + min(d, 0);
    int first = min(i, j), last = max(i, j);
    int left = (first == gamma) ? ~gamma : gamma;
    int right = (last == gamma + 1) ? ~(gamma + 1) : gamma + 1;
    children[i] = make_int2(left, right);
    range[i] = make_int2(first, last);
    if (left >= 0) parent_int[left] = i; else parent_leaf[~left] = i;
    if (right >= 0) parent_int[right] = i; else parent_leaf[~right] = i;
    if (i == 0) parent_int[0] = -1;
}

// bottom-up refit: the second thread to arrive at a node merges its children (Karras 2012 §4).
// ROT: on the way up every node also tries the four TREE ROTATIONS that exchange one of its children with a grandchild
// on the other side (Kensler 2008) and keeps the one that shrinks the surface area of the child being rebuilt most —
// the SAH term that changes.  The Morton-order tree splits space at fixed planes; a rotation lets a subtree pair up with
// the neighbour it overlaps least.  Safe without locks: a node is handled by exactly one thread, after both of its
// subtrees are complete, and only that thread ever touches those subtrees again (on its way up).
struct BoxH { float lx, ly, lz, hx, hy, hz; int h; };
__device__ __forceinline__ BoxH load_box(int c, const float4* __restrict__ leaf_lo, const float4* __restrict__ leaf_hi,
                                         volatile const float4* nl, volatile const float4* nh, volatile const int* height) {
    BoxH b;
    if (c >= 0) { b.lx = nl[c].x; b.ly = nl[c].y; b.lz = nl[c].z; b.hx = nh[c].x; b.hy = nh[c].y; b.hz = nh[c].z; b.h = height[c]; }
    else { const float4 a = leaf_lo[~c], d = leaf_hi[~c]; b.lx = a.x; b.ly = a.y; b.lz = a.z; b.hx = d.x; b.hy = d.y; b.hz = d.z; b.h = 0; }
    return b;
}
__device__ __forceinline__ BoxH merge_box(const BoxH& a, const BoxH& b) {
    BoxH m; m.lx = fminf(a.lx, b.lx); m.ly = fminf(a.ly, b.ly); m.lz = fminf(a.lz, b.lz);
    m.hx = fmaxf(a.hx, b.hx); m.hy = fmaxf(a.hy, b.hy); m.hz = fmaxf(a.hz, b.hz); m.h = max(a.h, b.h) + 1;
    return m;
}
__device__ __forceinline__ float box_area(const BoxH& b) {
    const float dx = b.hx - b.lx, dy = b.hy - b.ly, dz = b.hz - b.lz;
    return dx * dy + dy * dz + dz * dx;
}

template <bool ROT>
__global__ void k_refit(int n, int rot_min_leaves, const int2* __restrict__ range, int2* children, int* parent_int,
                        int* parent_leaf, const float4* __restrict__ leaf_lo, const float4* __restrict__ leaf_hi,
                        float4* node_lo, float4* node_hi, int* __restrict__ flags, int* height) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    int cur = parent_leaf[p];
    volatile const float4* nl = node_lo; volatile const float4* nh = node_hi; volatile const int* vh = height;
    volatile int* vch = reinterpret_cast<volatile int*>(children);
    while (cur >= 0) {
        __threadfence();
        if (atomicAdd(&flags[cur], 1) == 0) return;
        __threadfence();
        int c0 = vch[2 * cur], c1 = vch[2 * cur + 1];
        BoxH b0 = load_box(c0, leaf_lo, leaf_hi, nl, nh, vh), b1 = load_box(c1, leaf_lo, leaf_hi, nl, nh, vh);
        // (only where the node covers at least rot_min_leaves triangles — a node's own leaf set is invariant under rotations below it:
        //  the bottom levels hold most of the nodes, i.e. most of the pass's cost, but few of the levels a ray descends through)
        if (ROT && range[cur].y - range[cur].x + 1 >= rot_min_leaves) {
            float best = 0.0f; int bside = -1, bwhich = 0; BoxH bnew = b0;
#pragma unroll
            for (int side = 0; side < 2; ++side) {                         // X = the child that is rebuilt, Y = the other child, moved down
                const int X = side ? c1 : c0;
                if (X < 0) continue;
                const BoxH& bx = side ? b1 : b0; const BoxH& by = side ? b0 : b1;
                const int g0 = vch[2 * X], g1 = vch[2 * X + 1];
                const BoxH bg0 = load_box(g0, leaf_lo, leaf_hi, nl, nh, vh), bg1 = load_box(g1, leaf_lo, leaf_hi, nl, nh, vh);
                const float ax = box_area(bx);
                const BoxH m0 = merge_box(by, bg1), m1 = merge_box(bg0, by);   // Y replaces g0 / Y replaces g1
                const float d0 = box_area(m0) - ax, d1 = box_area(m1) - ax;
                if (d0 < best) { best = d0; bside = side; bwhich = 0; bnew = m0; }
                if (d1 < best) { best = d1; bside = side; bwhich = 1; bnew = m1; }
            }
            if (bside >= 0) {
                const int X = bside ? c1 : c0, Y = bside ? c0 : c1;
                const int g0 = vch[2 * X], g1 = vch[2 * X + 1];
                const int up = bwhich ? g1 : g0;                              // the grandchild that moves up, Y takes its place
                if (bwhich) vch[2 * X + 1] = Y; else vch[2 * X] = Y;
                node_lo[X] = make_float4(bnew.lx, bnew.ly, bnew.lz, 0.0f); node_hi[X] = make_float4(bnew.hx, bnew.hy, bnew.hz, 0.0f);
                height[X] = bnew.h;
                const BoxH bup = load_box(up, leaf_lo, leaf_hi, nl, nh, vh);
                if (bside) { c0 = up; b0 = bup; b1 = bnew; } else { c1 = up; b1 = bup; b0 = bnew; }
                vch[2 * cur] = c0; vch[2 * cur + 1] = c1;
                // parents of the two moved subtrees (both complete: nobody reads these again in this pass; the next pass walks them)
                if (Y >= 0) parent_int[Y] = X; else parent_leaf[~Y] = X;
                if (up >= 0) parent_int[up] = cur; else parent_leaf[~up] = cur;
            }
        }
        const BoxH m = merge_box(b0, b1);
        node_lo[cur] = make_float4(m.lx, m.ly, m.lz, 0.0f);
        node_hi[cur] = make_float4(m.hx, m.hy, m.hz, 0.0f);
        height[cur] = m.h;
        cur = parent_int[cur];
    }
}

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

// ------------------------------------------------------------------ binary LBVH -> 4-wide nodes (64 bytes)
// Level-synchronous top-down collapse.  `queue[j]` = the binary node that becomes wide node j (its position in the
// queue IS its output slot); every launch handles one BFS level [begin, end) and appends the internal children it
// keeps to the tail.  A binary node's two children are expanded greedily — largest surface area first — until there
// are four (subtrees of <= leaf_size triangles count as leaves and are never expanded).
struct CollapseState { uint32_t begin[2], end[2], tail, done, depth, base_level; };

__device__ __forceinline__ float half_area(float4 lo, float4 hi) {
    float dx = hi.x - lo.x, dy = hi.y - lo.y, dz = hi.z - lo.z;
    return dx * dy + dy * dz + dz * dx;
}

__device__ __forceinline__ void collapse_node(uint32_t j, uint32_t leaf_size, const QGrid& g, const int2* __restrict__ children, const int2* __restrict__ range,
                                              const float4* __restrict__ leaf_lo, const float4* __restrict__ leaf_hi,
                                              const float4* __restrict__ node_lo, const float4* __restrict__ node_hi,
                                              uint32_t* queue, CollapseState* st, uint4* __restrict__ out) {
    const int i = (int)queue[j];
    int src[4]; int32_t ref[4]; int nc = 2;
    auto effective = [&](int c, int k) {                                   // binary child -> (source of its box, traversal ref)
        src[k] = c;
        if (c < 0) { ref[k] = make_leaf_ref((uint32_t)(~c), 1); return; }
        int2 r = range[c];
        uint32_t cnt = (uint32_t)(r.y - r.x + 1);
        ref[k] = cnt <= leaf_size ? make_leaf_ref((uint32_t)r.x, cnt) : c;
    };
    int2 ch = children[i];
    effective(ch.x, 0); effective(ch.y, 1);
    for (int round = 0; round < 2; ++round) {
        int best = -1; float best_a = -1.0f;
        for (int k = 0; k < nc; ++k)
            if (ref[k] >= 0) { float a = half_area(node_lo[src[k]], node_hi[src[k]]); if (a > best_a) { best_a = a; best = k; } }
        if (best < 0) break;
        int2 c2 = children[src[best]];
        effective(c2.x, best); effective(c2.y, nc); ++nc;
    }
    uint32_t q[4][3]; int32_t refs[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        if (k < nc) {
            float4 lo, hi;
            if (src[k] < 0) { lo = leaf_lo[~src[k]]; hi = leaf_hi[~src[k]]; } else { lo = node_lo[src[k]]; hi = node_hi[src[k]]; }
            q[k][0] = quant_lo(lo.x, g.org[0], g.step[0]) | (quant_hi(hi.x, g.org[0], g.step[0]) << 16);
            q[k][1] = quant_lo(lo.y, g.org[1], g.step[1]) | (quant_hi(hi.y, g.org[1], g.step[1]) << 16);
            q[k][2] = quant_lo(lo.z, g.org[2], g.step[2]) | (quant_hi(hi.z, g.org[2], g.step[2]) << 16);
            if (ref[k] >= 0) { uint32_t pos = atomicAdd(&st->tail, 1u); queue[pos] = (uint32_t)src[k]; refs[k] = (int32_t)pos; }
            else refs[k] = ref[k];
        } else {                                                           // unused slot: inverted box (lo 65535, hi 0), never hit
            q[k][0] = q[k][1] = q[k][2] = 0x0000FFFFu;
            refs[k] = make_leaf_ref(0, 1);
        }
    }
    out[4 * (size_t)j] = make_uint4(q[0][0], q[0][1], q[0][2], q[1][0]);
    out[4 * (size_t)j + 1] = make_uint4(q[1][1], q[1][2], q[2][0], q[2][1]);
    out[4 * (size_t)j + 2] = make_uint4(q[2][2], q[3][0], q[3][1], q[3][2]);
    out[4 * (size_t)j + 3] = make_uint4((uint32_t)refs[0], (uint32_t)refs[1], (uint32_t)refs[2], (uint32_t)refs[3]);
}

// One BFS level per launch, all blocks of the GPU; level index = st->base_level (how many levels the single-block kernel below has
// already done: constant while these launches run) + launch index.
__global__ void k_collapse4(uint32_t launch_idx, uint32_t leaf_size, const BuildParams* __restrict__ bp, const int2* __restrict__ children, const int2* __restrict__ range,
                            const float4* __restrict__ leaf_lo, const float4* __restrict__ leaf_hi,
                            const float4* __restrict__ node_lo, const float4* __restrict__ node_hi,
                            uint32_t* queue, CollapseState* st, uint4* __restrict__ out) {
    const uint32_t level = st->base_level + launch_idx;
    const uint32_t begin = st->begin[level & 1], end = st->end[level & 1];
    if (begin == end) {                                                    // the tree is complete: the remaining launches of the fixed sequence only
        if (blockIdx.x == 0 && threadIdx.x == 0) { st->begin[(level + 1) & 1] = end; st->end[(level + 1) & 1] = end; }   // pass the empty level on
        return;
    }
    const QGrid g = bp->grid;
    for (uint32_t j = begin + blockIdx.x * blockDim.x + threadIdx.x; j < end; j += gridDim.x * blockDim.x)
        collapse_node(j, leaf_size, g, children, range, leaf_lo, leaf_hi, node_lo, node_hi, queue, st, out);
    // the last block to finish publishes the next level (in the other parity slot: blocks of THIS launch that become
    // resident late still read the current one)
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(&st->done, 1u) == gridDim.x - 1) {
            st->begin[(level + 1) & 1] = end; st->end[(level + 1) & 1] = st->tail; st->done = 0;
            if (end > begin) st->depth = level + 1;
        }
    }
}

// Levels handled by ONE block, from level st->base_level + skip on: the small top levels of the tree (while a level has at most
// max_nodes nodes; a launch per level would cost more than the level), and — after the fixed number of whole-GPU launches —
// whatever is left of a very deep tree (max_nodes = all).  Leaves st->base_level = the next level to do.
__global__ void __launch_bounds__(1024) k_collapse_block(uint32_t skip, uint32_t max_nodes, uint32_t leaf_size, const BuildParams* __restrict__ bp,
                                                         const int2* __restrict__ children, const int2* __restrict__ range,
                                                         const float4* __restrict__ leaf_lo, const float4* __restrict__ leaf_hi,
                                                         const float4* __restrict__ node_lo, const float4* __restrict__ node_hi,
                                                         uint32_t* queue, CollapseState* st, uint4* __restrict__ out) {
    const QGrid g = bp->grid;
    uint32_t level = st->base_level + skip;
    __syncthreads();                                                       // everybody has read base_level before thread 0 rewrites it
    for (;; ++level) {
        const uint32_t begin = st->begin[level & 1], end = st->end[level & 1];
        if (begin == end || end - begin > max_nodes) break;
        for (uint32_t j = begin + threadIdx.x; j < end; j += blockDim.x)
            collapse_node(j, leaf_size, g, children, range, leaf_lo, leaf_hi, node_lo, node_hi, queue, st, out);
        __threadfence();
        __syncthreads();
        if (threadIdx.x == 0) { st->begin[(level + 1) & 1] = end; st->end[(level + 1) & 1] = st->tail; st->depth = level + 1; }
        __threadfence();
        __syncthreads();
    }
    if (threadIdx.x == 0) st->base_level = level;
}

// ------------------------------------------------------------------ exact mesh AABB (aabbox.rs:62-88) on the device
// min / max are exact whatever the order, so a parallel reduction gives the reference's bounds bit for bit
// (NaN coordinates are ignored like the reference's `<` / `>` comparisons ignore them).
__device__ __forceinline__ int f2ord(float f) { int i = __float_as_int(f); return i >= 0 ? i : i ^ 0x7FFFFFFF; }
__host__ __device__ __forceinline__ float ord2f(int i) {
    int b = i >= 0 ? i : i ^ 0x7FFFFFFF;
#ifdef __CUDA_ARCH__
    return __int_as_float(b);
#else
    float f; memcpy(&f, &b, 4); return f;
#endif
}

__global__ void k_aabb_init(int* mm) { if (threadIdx.x < 3) mm[threadIdx.x] = 0x7F7FFFFF; else if (threadIdx.x < 6) mm[threadIdx.x] = (int)0xFF7FFFFF ^ 0x7FFFFFFF; }

__global__ void k_aabb(const float* __restrict__ raw, uint64_t n_vertices, int* __restrict__ mm) {
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

// ------------------------------------------------------------------ device-side set-up / wrap-up of one mesh
// MeshDev record + build parameters from the exact AABB (mm: ordered-int min/max cell filled by k_aabb)
__global__ void k_mesh_setup(const int* __restrict__ mm, MeshDev proto, float pad_rel, MeshDev* __restrict__ out, BuildParams* __restrict__ bp) {
    if (threadIdx.x || blockIdx.x) return;
    MeshDev md = proto;
    float lo[3], hi[3], mx = 0.0f;
    for (int k = 0; k < 3; ++k) {
        lo[k] = ord2f(mm[k]); hi[k] = ord2f(mm[3 + k]);
        md.lo[k] = lo[k]; md.hi[k] = hi[k];
        mx = fmaxf(mx, fmaxf(fabsf(lo[k]), fabsf(hi[k]))); mx = fmaxf(mx, hi[k] - lo[k]);
    }
    // Padding of the leaf boxes.  Relative to the mesh's coordinates it covers the rounding of the reference's own arithmetic for rays that start
    // near the mesh; a ray may start up to t < 1000 away (triangle.rs:146), and then `o - v0` and the direction carry ~ulp(|o|): for a SMALL mesh
    // NEAR THE WORLD ORIGIN the exact test shifts by more than 2e-5 * mx and accepts rays that miss the padded box (found with the host build of
    // the traversal, tests/test_device_source_on_host.py: 0.5 % of edge-aimed rays from 990 units away on a mesh of size 0.2; a padding of 6e-5
    // made them vanish).  Hence a floor of 2^-21 * (mx + 1000) = 4.8e-4 and up: it also covers the slab test's own reciprocal (MUFU.RCP, ~1 ulp:
    // 1.2e-4 at t = 1000; the host build emulates 2 ulp of it and stays clean) and exceeds the relative pad only for mx < 24.4.
    // pad_rel = 0 (box_pad_rel < 0: "none") stays none.
    const float pad = pad_rel > 0.0f ? fmaxf(pad_rel * mx, 4.7683716e-7f * (mx + 1000.0f)) : 0.0f;
    bp->pad = pad;
    for (int k = 0; k < 3; ++k) {                                          // 16-bit grid over the padded mesh box, 8 steps of slack per side
        float ext = (hi[k] + pad) - (lo[k] - pad);
        float step = ext / 65500.0f;
        if (!(step > 1e-30f)) step = 1e-30f;
        bp->grid.step[k] = step; bp->grid.org[k] = (lo[k] - pad) - 8.0f * step;
        // a step the slab test cannot take without overflow (huge extents, inf coordinates): NaN, the axis is not culled (common.cuh)
        md.qstep[k] = md.n_tris ? (step <= RBRT_QSTEP_MAX ? step : __int_as_float(0x7FFFFFFF)) : 0.0f; md.qorg[k] = md.n_tris ? bp->grid.org[k] : 0.0f;
        bp->lo[k] = lo[k]; bp->inv_ext[k] = hi[k] > lo[k] ? 1.0f / (hi[k] - lo[k]) : 0.0f;
    }
    *out = md;
}

__global__ void k_collapse_init(CollapseState* st, uint32_t* queue) {
    if (threadIdx.x || blockIdx.x) return;
    CollapseState init; init.begin[0] = 0; init.begin[1] = 0; init.end[0] = 1; init.end[1] = 0; init.tail = 1; init.done = 0; init.depth = 0; init.base_level = 0;
    *st = init; queue[0] = 0u;
}

// The tree is in place: publish its root, or — if it is deeper than the traversal stack allows (pathological input) — take the
// mesh out of the scene (n_tris = 0: never traversed) and raise the error the host reports at its next synchronising call.
__global__ void k_build_finish(const CollapseState* __restrict__ st, MeshDev* __restrict__ md, BuildResult* __restrict__ res) {
    if (threadIdx.x || blockIdx.x) return;
    BuildResult r; r.pad = 0;
    if (!st) { r.live_nodes = 0; r.depth = 0; r.error = 0; *res = r; return; }   // the whole mesh is one leaf (root_ref came with the proto)
    const bool unfinished = st->begin[st->base_level & 1] != st->end[st->base_level & 1];
    const bool bad = unfinished || 3 * st->depth + 2 > RBRT_STACK;
    r.live_nodes = bad ? 0u : st->tail; r.depth = st->depth; r.error = bad ? 1u : 0u;
    if (bad) md->n_tris = 0; else md->root_ref = 0;
    *res = r;
}

// ------------------------------------------------------------------ scratch + streams, per device
// Two grow-only scratch slots per device: a scene's create uploads into one while the previous scene's build may still be
// reading the other.  A slot's `busy` event marks the last build kernel that reads it.
struct ScratchSlot { void* p = nullptr; size_t bytes = 0; cudaEvent_t busy = nullptr, up = nullptr; };
struct DeviceBuild { ScratchSlot slot[2]; int next = 0; cudaStream_t copy = nullptr, build = nullptr; };
static DeviceBuild g_build[64];

void release_build_scratch() {
    int cur = 0; cudaGetDevice(&cur);
    for (int d = 0; d < 64; ++d) {
        DeviceBuild& B = g_build[d];
        if (!B.copy && !B.slot[0].p && !B.slot[1].p) continue;
        cudaSetDevice(d);
        if (B.build) cudaStreamSynchronize(B.build);
        if (B.copy) cudaStreamSynchronize(B.copy);
        for (auto& s : B.slot) { cudaFree(s.p); if (s.busy) cudaEventDestroy(s.busy); if (s.up) cudaEventDestroy(s.up); s = ScratchSlot(); }
        if (B.copy) cudaStreamDestroy(B.copy);
        if (B.build) cudaStreamDestroy(B.build);
        B = DeviceBuild();
    }
    cudaSetDevice(cur);
}

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) return e_; } while (0)

cudaError_t build_begin(int device, BuildCtx* ctx) {
    DeviceBuild& B = g_build[device & 63];
    if (!B.copy) {
        CK(cudaStreamCreateWithFlags(&B.copy, cudaStreamNonBlocking));
        // The build's ~80 small dependent kernels run in the gaps the render kernels of earlier frames leave; with the highest stream
        // priority a freed SM goes to them first (RBRT_BUILD_PRIORITY=0: default priority, for A/B measurements).
        int pr_least = 0, pr_greatest = 0;
        CK(cudaDeviceGetStreamPriorityRange(&pr_least, &pr_greatest));
        static const bool prio = !(getenv("RBRT_BUILD_PRIORITY") && atoi(getenv("RBRT_BUILD_PRIORITY")) == 0);
        CK(cudaStreamCreateWithPriority(&B.build, cudaStreamNonBlocking, prio ? pr_greatest : 0));
        for (auto& s : B.slot) { CK(cudaEventCreateWithFlags(&s.busy, cudaEventDisableTiming)); CK(cudaEventCreateWithFlags(&s.up, cudaEventDisableTiming)); }
    }
    ctx->device = device; ctx->slot = B.next; B.next ^= 1;
    ctx->copy = B.copy; ctx->build = B.build;
    return cudaSuccess;
}

cudaError_t build_uploads_done(BuildCtx& ctx, cudaEvent_t ev) { return cudaEventRecord(ev, ctx.copy); }


static cudaError_t slot_reserve(ScratchSlot& S, cudaStream_t cs, size_t bytes) {
    if (S.bytes < bytes) {                                                 // grow (rare): nothing may still be using the slot
        CK(cudaEventSynchronize(S.busy));
        CK(cudaStreamSynchronize(cs));
        cudaFree(S.p); S.p = nullptr; S.bytes = 0;
        const size_t want = bytes + bytes / 8 + (1u << 20);
        CK(cudaMalloc(&S.p, want)); S.bytes = want;
    }
    return cudaSuccess;
}

cudaError_t build_slot_acquire(BuildCtx& ctx, size_t bytes, char** base) {
    ScratchSlot& S = g_build[ctx.device & 63].slot[ctx.slot];
    CK(slot_reserve(S, ctx.copy, bytes));
    CK(cudaStreamWaitEvent(ctx.copy, S.busy, 0));
    *base = (char*)S.p;
    return cudaSuccess;
}

cudaError_t build_slot_uploaded(BuildCtx& ctx, cudaEvent_t* uploaded) {
    ScratchSlot& S = g_build[ctx.device & 63].slot[ctx.slot];
    CK(cudaEventRecord(S.up, ctx.copy));
    CK(cudaStreamWaitEvent(ctx.build, S.up, 0));
    *uploaded = S.up;
    return cudaSuccess;
}

cudaError_t build_slot_release(BuildCtx& ctx) { return cudaEventRecord(g_build[ctx.device & 63].slot[ctx.slot].busy, ctx.build); }

cudaError_t build_mesh(BuildCtx& ctx, const float* h_tris, uint64_t n_all, uint32_t n, float pad_rel, uint32_t leaf_size, bool sah,
                       const MeshDev& proto, MeshDev* d_mesh, float4* d_tris, float4* d_normals, float4* d_nodes, BuildResult* d_res,
                       cudaEvent_t src_ready) {
    DeviceBuild& B = g_build[ctx.device & 63];
    ScratchSlot& S = B.slot[ctx.slot];
    cudaStream_t cs = ctx.copy, st = ctx.build;
    const int Bk = 256;
    const uint32_t g = (n + Bk - 1) / Bk, ni = n > 1 ? n - 1 : 1;
    size_t tmp_bytes = 0;
    if (n) CK(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, (uint64_t*)nullptr, (uint64_t*)nullptr, (uint32_t*)nullptr, (uint32_t*)nullptr, (int)n, 0, 63, st));
    // carve the slot: raw triangle soup | AABB cell + build parameters | build arrays | sort temp
    const size_t raw_bytes = (36ull * n_all + 255) & ~255ull;
    size_t off = raw_bytes + 512;
    auto take_off = [&](size_t bytes) { size_t o = off; off += (bytes + 255) & ~255ull; return o; };
    const size_t o_keys = take_off(8ull * n), o_keys_s = take_off(8ull * n), o_vals = take_off(4ull * n), o_vals_s = take_off(4ull * n);
    const size_t o_leaf_lo = take_off(16ull * n), o_leaf_hi = take_off(16ull * n), o_node_lo = take_off(16ull * ni), o_node_hi = take_off(16ull * ni);
    const size_t o_children = take_off(8ull * ni), o_range = take_off(8ull * ni), o_parent_int = take_off(4ull * ni), o_parent_leaf = take_off(4ull * n);
    const size_t o_flags = take_off(4ull * ni), o_height = take_off(4ull * ni), o_queue = take_off(4ull * ni), o_cstate = take_off(sizeof(CollapseState));
    const size_t o_tmp = take_off(tmp_bytes ? tmp_bytes : 16);
    CK(slot_reserve(S, cs, off));
    char* base = (char*)S.p;
    // ---- upload (copy stream): after the previous build that read this slot (and, for device vertices, after their producer)
    CK(cudaStreamWaitEvent(cs, S.busy, 0));
    if (src_ready) CK(cudaStreamWaitEvent(cs, src_ready, 0));
    if (n_all) CK(cudaMemcpyAsync(base, h_tris, 36ull * n_all, cudaMemcpyDefault, cs));
    CK(cudaEventRecord(S.up, cs));
    // ---- build (build stream)
    CK(cudaStreamWaitEvent(st, S.up, 0));
    const float* d_raw = (const float*)base;
    int* mm = (int*)(base + raw_bytes);
    BuildParams* bp = (BuildParams*)(base + raw_bytes + 64);
    k_aabb_init<<<1, 32, 0, st>>>(mm);
    if (n_all) k_aabb<<<148 * 4, 256, 0, st>>>(d_raw, n_all * 3, mm);    // exact AABB over ALL real triangles, also those the SIMD tail rule drops (aabbox.rs:62-88, mesh.rs:61)
    MeshDev pr = proto;
    const bool one_leaf = n && (n <= leaf_size || n == 1);
    if (one_leaf) pr.root_ref = make_leaf_ref(0, n);
    k_mesh_setup<<<1, 32, 0, st>>>(mm, pr, pad_rel, d_mesh, bp);
    CK(cudaGetLastError());
    if (n) {
        uint64_t* keys = (uint64_t*)(base + o_keys); uint64_t* keys_s = (uint64_t*)(base + o_keys_s);
        uint32_t* vals = (uint32_t*)(base + o_vals); uint32_t* vals_s = (uint32_t*)(base + o_vals_s);
        float4* leaf_lo = (float4*)(base + o_leaf_lo); float4* leaf_hi = (float4*)(base + o_leaf_hi);
        float4* node_lo = (float4*)(base + o_node_lo); float4* node_hi = (float4*)(base + o_node_hi);
        int2* children = (int2*)(base + o_children); int2* range = (int2*)(base + o_range);
        int* parent_int = (int*)(base + o_parent_int); int* parent_leaf = (int*)(base + o_parent_leaf);
        int* flags = (int*)(base + o_flags); int* height = (int*)(base + o_height);
        uint32_t* queue = (uint32_t*)(base + o_queue); CollapseState* cstate = (CollapseState*)(base + o_cstate);
        void* tmp = base + o_tmp;
        k_prepare<<<g, Bk, 0, st>>>(d_raw, n, bp, d_normals, keys, vals);
        CK(cudaGetLastError());
        CK(cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, keys, keys_s, vals, vals_s, (int)n, 0, 63, st));
        k_emit_tris<<<g, Bk, 0, st>>>(d_raw, vals_s, n, bp, d_tris, leaf_lo, leaf_hi);
        CK(cudaGetLastError());
        if (!one_leaf) {
            CK(cudaMemsetAsync(flags, 0, 4ull * ni, st));
            k_karras<<<(ni + Bk - 1) / Bk, Bk, 0, st>>>(keys_s, (int)n, children, range, parent_int, parent_leaf);
            CK(cudaGetLastError());
            // SAH pass: tree rotations during the refit; only with one-triangle leaves (a rotated subtree no longer covers a
            // contiguous run of the Morton order, which multi-triangle leaves rely on).  RBRT_SAH_PASSES: tuning knob.
            static const int sah_passes_env = getenv("RBRT_SAH_PASSES") ? atoi(getenv("RBRT_SAH_PASSES")) : 1;
            const int passes = (sah && leaf_size == 1) ? sah_passes_env : 0;
            static const int rot_min_env = getenv("RBRT_SAH_MIN_LEAVES") ? atoi(getenv("RBRT_SAH_MIN_LEAVES")) : 16;
            if (passes <= 0) k_refit<false><<<g, Bk, 0, st>>>((int)n, 0, range, children, parent_int, parent_leaf, leaf_lo, leaf_hi, node_lo, node_hi, flags, height);
            for (int pass = 0; pass < passes; ++pass) {
                if (pass) CK(cudaMemsetAsync(flags, 0, 4ull * ni, st));
                k_refit<true><<<g, Bk, 0, st>>>((int)n, rot_min_env, range, children, parent_int, parent_leaf, leaf_lo, leaf_hi, node_lo, node_hi, flags, height);
            }
            CK(cudaGetLastError());
            k_collapse_init<<<1, 32, 0, st>>>(cstate, queue);
            uint32_t gcol = (ni + Bk - 1) / Bk; if (gcol > 148u * 8u) gcol = 148u * 8u;
            // Top-down collapse into 4-wide nodes, level-synchronous.  The depth is only known on the device, so the launch sequence
            // is fixed: ONE block does the small top levels (up to 2048 nodes each: ~7 levels that would each cost a launch), then
            // ceil(log2 n) + 2 whole-GPU launches, one level each (a level of a finished tree returns at once), then one block again
            // for whatever a pathologically deep tree has left.  C3: 24 launches; the 64 of the first asynchronous version cost 0.45 ms.
            k_collapse_block<<<1, 1024, 0, st>>>(0u, 2048u, leaf_size, bp, children, range, leaf_lo, leaf_hi, node_lo, node_hi, queue, cstate, reinterpret_cast<uint4*>(d_nodes));
            uint32_t n_multi = 2; while ((1ull << (n_multi - 2)) < n) ++n_multi;
            for (uint32_t k = 0; k < n_multi; ++k)
                k_collapse4<<<gcol, Bk, 0, st>>>(k, leaf_size, bp, children, range, leaf_lo, leaf_hi, node_lo, node_hi, queue, cstate,
                                                reinterpret_cast<uint4*>(d_nodes));
            k_collapse_block<<<1, 1024, 0, st>>>(n_multi, 0xFFFFFFFFu, leaf_size, bp, children, range, leaf_lo, leaf_hi, node_lo, node_hi, queue, cstate, reinterpret_cast<uint4*>(d_nodes));
            CK(cudaGetLastError());
            k_build_finish<<<1, 32, 0, st>>>(cstate, d_mesh, d_res);
        } else k_build_finish<<<1, 32, 0, st>>>(nullptr, d_mesh, d_res);
    } else k_build_finish<<<1, 32, 0, st>>>(nullptr, d_mesh, d_res);
    CK(cudaGetLastError());
    CK(cudaEventRecord(S.busy, st));
    return cudaSuccess;
}

}  // namespace rbrt
