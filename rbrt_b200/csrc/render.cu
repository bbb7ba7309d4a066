// render.cu — the wavefront path tracer: render_scene + colorize (rbrt_lib/src/lib.rs:43-124).
//
// One batch = every pixel of this rank's shard x a run of consecutive samples.  Path id
// pid = s_local * P + j (j = pixel enumeration of the shard, 8x4 tiles, one warp = one tile); every
// per-path record (ray, hit, radiance, scatter history) lives at index pid, queues hold pids.
//
// A ray's closest-hit query (Scene::hit, scene.rs:19-43) is split in two stages:
//   stage A  (coherent, runs in the kernel that PRODUCES the ray: k_generate / k_shade): the sphere
//            tests and the whole-mesh AABB pre-tests.  Rays that touch no mesh box are resolved on the
//            spot — sphere hit -> material queue, miss -> sky + attenuation unwinding -> out[pid];
//            only rays that enter a mesh box are queued for traversal.
//   stage B  (k_trace): persistent warps traverse the LBVH for queued rays only and re-fill lanes
//            whose ray has finished from the queue INSIDE the traversal loop (dynamic fetch), so lanes
//            do not idle behind the longest traversal of their warp.
// Per bounce iteration `it` (= depth 50-it of the reference's recursion): k_trace(it) -> k_shade(it).
// k_shade pulls 32 hits of ONE material, runs its scatter() and stage A of the continuation ray.
// After the last iteration k_accumulate adds the batch's per-path radiances to the per-pixel sums in
// sample order — the reference's `color += colorize(..)` (lib.rs:96-100) — with no float atomics,
// so an image is bit-reproducible and independent of scheduling.
#include <cstdio>
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include "engine.cuh"
#include "intersect.cuh"
#include "cull.cuh"
#include "shade.cuh"

namespace rbrt {

#define FULL_MASK 0xFFFFFFFFu
#define CLS_CAND 3            // queue classes of a produced ray: 0..2 material queues, 3 traversal queue
#define CLS_NONE 7            // resolved on the spot (or no ray)
#define ROUNDS 4              // 32-ray rounds a producer warp handles per queue reservation

// ------------------------------------------------------------------ warp helpers
// Every lane of a converged warp calls this; lanes with pred get consecutive slots.
__device__ __forceinline__ uint32_t warp_append(uint32_t* counter, bool pred) {
    uint32_t mask = __ballot_sync(FULL_MASK, pred);
    if (mask == 0) return 0;
    uint32_t lane = threadIdx.x & 31;
    uint32_t leader = __ffs(mask) - 1;
    uint32_t base = 0;
    if (lane == leader) base = atomicAdd(counter, __popc(mask));
    base = __shfl_sync(FULL_MASK, base, leader);
    return base + __popc(mask & ((1u << lane) - 1));
}

__device__ __forceinline__ uint32_t warp_grab(uint32_t* head, uint32_t count) {
    uint32_t base = 0;
    if ((threadIdx.x & 31) == 0) base = atomicAdd(head, count);
    return __shfl_sync(FULL_MASK, base, 0);
}

// Deferred queue appends of a producer warp: each lane remembers the class and pid of the ray it
// produced in each of ROUNDS rounds; flush() reserves space with ONE atomic per non-empty class for
// all rounds together (same-address atomics are the scarce resource: ~1 per ns per address).
struct Deferred {
    uint32_t cls;            // 3 bits per round
    uint32_t pid[ROUNDS];
    __device__ __forceinline__ void clear() { cls = 0; for (int r = 0; r < ROUNDS; ++r) { cls |= (uint32_t)CLS_NONE << (3 * r); pid[r] = 0; } }
    __device__ __forceinline__ void set(int r, uint32_t c, uint32_t p) { cls = (cls & ~(7u << (3 * r))) | (c << (3 * r)); pid[r] = p; }
};

__device__ __forceinline__ void flush(const WaveParams& P, uint32_t it, const Deferred& df) {
    IterCtr* c = P.ctr + it;
    const uint32_t lane = threadIdx.x & 31, lt = (1u << lane) - 1;
#pragma unroll
    for (uint32_t k = 0; k < 4; ++k) {
        uint32_t m[ROUNDS], total = 0;
#pragma unroll
        for (int r = 0; r < ROUNDS; ++r) { m[r] = __ballot_sync(FULL_MASK, ((df.cls >> (3 * r)) & 7u) == k); total += __popc(m[r]); }
        if (total == 0) continue;
        uint32_t base = 0;
        if (lane == 0) base = atomicAdd(k == CLS_CAND ? &c->cand_count : &c->mat_count[k], total);
        base = __shfl_sync(FULL_MASK, base, 0);
        uint32_t* q = k == CLS_CAND ? P.candq : P.matq[it & 1][k];
#pragma unroll
        for (int r = 0; r < ROUNDS; ++r) {
            if (m[r] & (1u << lane)) q[base + __popc(m[r] & lt)] = df.pid[r];
            base += __popc(m[r]);
        }
    }
}

// ------------------------------------------------------------------ path record
// Everything a path's queued work item needs sits in ONE 32-byte, 32-byte-aligned record = ONE DRAM sector, always read with one
// 256-bit load and always written WHOLE with one 256-bit store (a partly written sector costs a read: L2 completes it from DRAM
// before it can write it back).  Two formats, told apart by the queue the path sits in:
//   traversal candidate (candq)   {bits(t_sphere), sphere | first_mesh << 16, origin.xyz, direction.xyz}
//       stage A's sphere pre-result (sphere = 0xFFFF: none) and the first mesh whose box the ray entered; `closest`, the distance the
//       mesh must beat (scene.rs:36), is re-derived from t_sphere with the expression the sphere test itself uses (sphere.rs:49-50)
//   pending hit (matq[kind])      {hit_point.xyz, direction.xyz, element | is_mesh << 16, triangle}
//       what scatter() takes: the hit point (= ray.point_at(t), computed where t is known), the incoming direction, and where the
//       normal comes from.  Neither the ray's origin nor t is needed after the hit.
// The scatter history (element ids, for the attenuation product when the path ends) lives in per-iteration rows, WaveParams::hist:
// a 2-byte entry inside the record would be a partial write to it at every bounce.
// History of this layout (C3 frame, one frame at a time): five separate arrays 37.6 ms -> one 64-byte record {hit, ray, 12 history
// entries} 36.5 -> camera rays in one sector (34.65 -> 33.80, profiles/r2_exp_camera_records.jsonl) -> this one-sector record.
#define NO_SPHERE 0xFFFFu
__device__ __forceinline__ uint4* rec_ptr(const WaveParams& P, uint32_t pid) { return P.rec + 2 * (size_t)pid; }
__device__ __forceinline__ void store_rec(const WaveParams& P, uint32_t pid, uint32_t w0, uint32_t w1, uint32_t w2, uint32_t w3,
                                          uint32_t w4, uint32_t w5, uint32_t w6, uint32_t w7) {
    asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" :: "l"(rec_ptr(P, pid)), "r"(w0), "r"(w1), "r"(w2), "r"(w3),
                 "r"(w4), "r"(w5), "r"(w6), "r"(w7) : "memory");
}
__device__ __forceinline__ void load_rec(const WaveParams& P, uint32_t pid, uint4& a, uint4& b) {
    asm volatile("ld.global.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(a.x), "=r"(a.y), "=r"(a.z), "=r"(a.w), "=r"(b.x), "=r"(b.y), "=r"(b.z), "=r"(b.w) : "l"(rec_ptr(P, pid)) : "memory");
}
#define FB(x) __float_as_uint(x)
#define BF(x) __uint_as_float(x)
__device__ __forceinline__ void store_candidate(const WaveParams& P, uint32_t pid, float t_s, uint32_t sphere, uint32_t mi, f3 o, f3 d) {
    store_rec(P, pid, FB(t_s), sphere | (mi << 16), FB(o.x), FB(o.y), FB(o.z), FB(d.x), FB(d.y), FB(d.z));
}
// closest = dist_from_ray_orig of the sphere pre-result: `p = o + t*d; dist = length(o - p)` (sphere.rs:49-50, triangle.rs:425-426)
__device__ __forceinline__ void load_candidate_rec(const WaveParams& P, uint32_t pid, float& t_s, uint32_t& sphere, uint32_t& mi, float& closest, f3& o, f3& d) {
    uint4 a, b; load_rec(P, pid, a, b);
    t_s = BF(a.x); sphere = a.y & 0xFFFFu; mi = a.y >> 16;
    o = mk3(BF(a.z), BF(a.w), BF(b.x)); d = mk3(BF(b.y), BF(b.z), BF(b.w));
    closest = 3.40282347e+38f;                                            // f32::MAX (scene.rs:21)
    if (sphere != NO_SPHERE) { const f3 p = o + t_s * d; closest = len3(o - p); }
}
__device__ __forceinline__ void store_pending(const WaveParams& P, uint32_t pid, f3 point, f3 d, uint32_t elem, bool is_mesh, uint32_t tri) {
    store_rec(P, pid, FB(point.x), FB(point.y), FB(point.z), FB(d.x), FB(d.y), FB(d.z), elem | (is_mesh ? 0x10000u : 0u), tri);
}
__device__ __forceinline__ void load_pending(const WaveParams& P, uint32_t pid, f3& point, f3& d, uint32_t& elem, bool& is_mesh, uint32_t& tri) {
    uint4 a, b; load_rec(P, pid, a, b);
    point = mk3(BF(a.x), BF(a.y), BF(a.z)); d = mk3(BF(a.w), BF(b.x), BF(b.y));
    elem = b.z & 0xFFFFu; is_mesh = (b.z >> 16) != 0u; tri = b.w;
}
__device__ __forceinline__ uint32_t load_hist(const WaveParams& P, uint32_t pid, uint32_t k) { return P.hist[(size_t)k * P.cap + pid]; }
__device__ __forceinline__ void store_hist(const WaveParams& P, uint32_t pid, uint32_t k, uint32_t elem) { P.hist[(size_t)k * P.cap + pid] = (uint16_t)elem; }

// Path id -> (frame of the batch, sample of the batch, pixel enumeration index): pid = ((f * s_count) + s_local) * paths_px + j
__device__ __forceinline__ void path_coords(const WaveParams& P, uint32_t pid, uint32_t& f, uint32_t& s_local, uint32_t& j) {
    const uint32_t v = fast_div(pid, P.fd_paths_px);
    j = pid - v * P.paths_px;
    f = P.n_frames > 1u ? fast_div(v, P.fd_s_count) : 0u;
    s_local = v - f * P.s_count;
}

// att_1 * (att_2 * (... * leaf)): the recursion of lib.rs:62 unwinds innermost first
__device__ __forceinline__ f3 unwind(const WaveParams& P, f3 col, uint32_t n_scatters, uint32_t pid) {
    for (int k = (int)n_scatters - 1; k >= 0; --k) {
        uint32_t e = load_hist(P, pid, (uint32_t)k);
        float4 m = __ldg(P.S.mat + e);
        f3 att = __ldg(P.S.mat_kind + e) == 2u ? mk3(1.0f, 1.0f, 1.0f) : mk3(m.x, m.y, m.z);
        col = att * col;
    }
    return col;
}

__device__ __forceinline__ void end_path(const WaveParams& P, uint32_t pid, f3 col) { P.out[pid] = make_float4(col.x, col.y, col.z, 0.0f); }

// ------------------------------------------------------------------ stage A of Scene::hit (scene.rs:19-31 + mesh.rs:233)
// `it` = bounce iteration of the ray (number of scatters before it).  Returns the queue class of the ray.
// Camera rays share ONE origin, so whether a sphere (or a mesh box) can be hit at all depends on the direction alone: it
// must lie inside the cone the sphere subtends from the camera.  k_generate builds, per frame and element, the cone's axis and
// cos^2 of its half-angle (minus a margin) in shared memory; stage A then SKIPS the exact test of an element whose cone the
// ray misses — a test the reference would run and that would return "no hit" (discriminant < 0, or both roots behind the
// origin; slab test t_min > t_max).  Only provable misses are skipped (margin 1e-4 on cos^2 against ~1e-6 of f32 rounding in the
// reference's discriminant; origin inside or within 1 % of the sphere, BasicTriangle elements and NaN directions: never
// skipped), so every result bit is unchanged.  C3: 4 spheres + 1 box, 2.9 -> see profiles/ for the measured k_generate time.
#define CULL_MAX 256
// cone_of_sphere, outside_cone, outside_double_cone: cull.cuh
template <bool ET, bool PRIMARY = false>   // ET: Scene.elements holds BasicTriangles besides spheres (separate kernel instantiations, so the usual
                    // sphere-only kernels carry no trace of the triangle path); PRIMARY: camera ray, `cull` = this frame's cone table
__device__ __forceinline__ uint32_t stage_a(const WaveParams& P, uint32_t it, uint32_t pid, f3 o, f3 d, uint32_t& nan_count, const float4* cull = nullptr) {
    float closest = 3.40282347e+38f;                                     // f32::MAX (scene.rs:21)
    int kind = -1; uint32_t elem = 0; float t_s = 0.0f;
    for (uint32_t i = 0; i < P.S.n_spheres; ++i) {                       // elements first, in order (scene.rs:23-31)
        if (PRIMARY && cull && outside_double_cone(cull[i], d)) continue;
        float t, dist;
        int r = ET ? element_intersect(P.S, i, o, d, t, dist) : sphere_intersect(__ldg(P.S.spheres + i), o, d, t, dist);
        if (r < 0) { ++nan_count; end_path(P, pid, mk3(0, 0, 0)); return CLS_NONE; }   // reference panics (sphere.rs:33)
        if (r && dist < closest) { closest = dist; kind = 0; elem = i; t_s = t; }
    }
    for (uint32_t mi = 0; mi < P.S.n_meshes; ++mi) {                     // whole-mesh AABB pre-test (mesh.rs:233)
        const MeshDev& M = P.S.meshes[mi];
        if (PRIMARY && cull && outside_cone(cull[P.S.n_spheres + mi], d)) continue;
        if (M.n_tris == 0 || !mesh_bbox_hit(M, o, d)) continue;
        store_candidate(P, pid, t_s, kind == 0 ? elem : NO_SPHERE, mi, o, d);
        return CLS_CAND;
    }
    if (kind == 0) {
        if (it < P.max_depth) {                                           // depth > 0: scatter() will run (lib.rs:54)
            store_pending(P, pid, o + t_s * d, d, elem, false, 0u);       // ray.point_at(t) (sphere.rs:49)
            if (P.keep_t) reinterpret_cast<float*>(P.out + pid)[0] = t_s;
            return __ldg(P.S.mat_kind + elem);
        }
        end_path(P, pid, mk3(0, 0, 0));                                   // depth exhausted -> black (lib.rs:63-66)
        return CLS_NONE;
    }
    end_path(P, pid, unwind(P, sky(d), it, pid));                         // miss: sky (lib.rs:68-71)
    return CLS_NONE;
}

// ------------------------------------------------------------------ generate (cam.rs:64-82) + stage A
template <bool ET>
__global__ void __launch_bounds__(256) k_generate(WaveParams P) {
    const uint32_t n_paths = P.n_frames * P.s_count * P.paths_px;         // multiple of 32
    const uint32_t n_groups = n_paths >> 5, lane = threadIdx.x & 31;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    uint32_t nan_count = 0, rays = 0;
    // cone table of this launch's frames: [frame][element | mesh] (see cone_of_sphere)
    __shared__ float4 s_cull[CULL_MAX];
    const uint32_t n_tab = P.S.n_spheres + P.S.n_meshes;
    const bool use_cull = P.use_cull && n_tab * P.n_frames <= CULL_MAX;
    if (use_cull) {
        for (uint32_t i = threadIdx.x; i < n_tab * P.n_frames; i += blockDim.x) {
            const uint32_t f = i / n_tab, e = i - f * n_tab;
            const f3 o = mk3(P.cam[f].pos[0], P.cam[f].pos[1], P.cam[f].pos[2]);
            float4 q = make_float4(0.0f, 0.0f, 0.0f, -2.0f);
            if (e < P.S.n_spheres) {
                if (!(ET && __ldg(P.S.elem_kind + e))) { const float4 sp = __ldg(P.S.spheres + e); q = cone_of_sphere(o, sp.x, sp.y, sp.z, fabsf(sp.w)); }
            } else {                                                       // the mesh AABB's bounding sphere, 0.1 % larger
                const MeshDev& M = P.S.meshes[e - P.S.n_spheres];
                const float hx = 0.5f * (M.hi[0] - M.lo[0]), hy = 0.5f * (M.hi[1] - M.lo[1]), hz = 0.5f * (M.hi[2] - M.lo[2]);
                q = cone_of_sphere(o, M.lo[0] + hx, M.lo[1] + hy, M.lo[2] + hz, 1.001f * sqrtf(hx * hx + hy * hy + hz * hz) + 1e-6f);
            }
            s_cull[i] = q;
        }
        __syncthreads();
    }
    for (uint32_t g0 = warp * ROUNDS; g0 < n_groups; g0 += n_warps * ROUNDS) {
        Deferred df; df.clear();
#pragma unroll 1                                                          // keep the body once: unrolled x4 the kernel outgrows the instruction cache
        for (int r = 0; r < ROUNDS; ++r) {
            uint32_t g = g0 + r;
            if (g >= n_groups) break;
            uint32_t pid = (g << 5) + lane;
            uint32_t f, s_local, j;
            path_coords(P, pid, f, s_local, j);
            uint32_t row, col;
            if (shard_pixel(P.sh, P.cam[0], j, row, col)) {
                f3 o, d;
                RngKey key; key.k0 = P.key0[f]; key.k1 = P.key1[f];
                camera_ray(P.cam[f], row, col, key, row * P.cam[0].width + col, P.s_base + s_local, o, d);
                ++rays;
                df.set(r, stage_a<ET, true>(P, 0, pid, o, d, nan_count, use_cull ? s_cull + f * n_tab : nullptr), pid);
            }
        }
        flush(P, 0, df);
    }
    for (int off = 16; off; off >>= 1) { rays += __shfl_down_sync(FULL_MASK, rays, off); nan_count += __shfl_down_sync(FULL_MASK, nan_count, off); }
    if (lane == 0) {
        if (rays) atomicAdd(&P.ctr[0].ray_count, rays);
        if (nan_count) atomicAdd(&P.stats[ST_NAN], (unsigned long long)nan_count);
    }
}

// ------------------------------------------------------------------ stage B: BVH traversal with dynamic fetch
// Resolution of a queued ray once all its meshes are done: the rest of Scene::hit + the miss arm of colorize.
__device__ __forceinline__ int resolve(const WaveParams& P, uint32_t it, uint32_t pid, f3 o, f3 d, int kind, uint32_t elem, uint32_t tri, float t) {
    if (kind >= 0) {
        if (it < P.max_depth) {
            uint32_t e = kind == 0 ? elem : P.S.n_spheres + elem;
            store_pending(P, pid, o + t * d, d, e, kind == 1, tri);       // ray.point_at(t) (sphere.rs:49, mesh.rs:247)
            if (P.keep_t) reinterpret_cast<float*>(P.out + pid)[0] = t;   // rbrt_gpu_trace_rays reports t (k_rays_collect)
            return (int)__ldg(P.S.mat_kind + e);
        }
        end_path(P, pid, mk3(0, 0, 0));
        return -1;
    }
    end_path(P, pid, unwind(P, sky(d), it, pid));
    return -1;
}

#define TRACE_THREADS 128
#define FETCH_THRESHOLD 8      // re-fill the warp when fewer lanes than this are still traversing (WaveParams::fetch_thr; swept 1..24 on C3,
                               // profiles/r1_summary.md: a re-fill stalls the whole warp on an atomic -> queue -> ray chain, so fewer is better)

#ifndef TRACE_SMEM_STACK
#define TRACE_SMEM_STACK 0     // traversal-stack entries per lane kept in shared memory (intersect.cuh StackS); 0 = all in local memory
#endif
#ifndef TRACE_BLOCKS
#define TRACE_BLOCKS 8         // resident blocks per SM: 8 x 128 threads = 64 registers per thread
#endif
template <bool COUNT>
__global__ void __launch_bounds__(TRACE_THREADS, TRACE_BLOCKS) k_trace(WaveParams P, uint32_t it) {
    IterCtr* c = P.ctr + it;
    const uint32_t n = c->cand_count;
    if (n == 0 || P.ctr[0].pad) return;
    if (COUNT && blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&P.stats[ST_CAND], (unsigned long long)n);
    const uint32_t lane = threadIdx.x & 31, lt = (1u << lane) - 1;
    const int32_t SENTINEL = 0x7FFFFFFF;
    int32_t lstack[RBRT_STACK];
#if TRACE_SMEM_STACK > 0
    __shared__ int32_t s_stack[TRACE_SMEM_STACK][TRACE_THREADS];
    const StackS<TRACE_SMEM_STACK, TRACE_THREADS> stack = {&s_stack[0][threadIdx.x], lstack};
#else
    const StackL stack = {lstack};
#endif
    // ---- ray state
    bool has_ray = false;
    uint32_t pid = 0, mi = 0;
    f3 o = mk3(0, 0, 0), d = mk3(0, 0, 0);
    RaySlabs R = {0, 0, 0, 0, 0, 0, RBRT_SEL_LO, RBRT_SEL_LO, RBRT_SEL_LO, RBRT_SEL_HI, RBRT_SEL_HI, RBRT_SEL_HI};
    float closest = 0.0f, bt = 0.0f; int bkind = -1; uint32_t belem = 0, btri = 0;   // best over spheres + finished meshes
    // ---- traversal state of the current mesh
    int32_t cur = SENTINEL; int sp = 0;
    float best_t = 0.0f, t_prune = 0.0f, t_limit = 0.0f; uint32_t best_idx = 0xFFFFFFFFu;
    const uint4* __restrict__ nodes = reinterpret_cast<const uint4*>(P.S.nodes); uint32_t tri_base = 0;
    bool exhausted = false;                                               // warp-uniform: the queue has no more rays
    uint32_t n_nodes = 0, n_tris = 0;
    // With few rays (tail iterations) a warp must not take 32 of them while others idle: every ray is a
    // latency-bound chain, so spread them over all resident warps.
    const uint32_t n_warps = (gridDim.x * blockDim.x) >> 5;
    const uint32_t quota = min(32u, max(1u, (n + n_warps - 1) / n_warps));

    auto start_mesh = [&](const MeshDev& M) {
        // A mesh hit only matters if its dist beats `closest` (strict <).  dist is monotone in t and ~ t*|d|;
        // convert with a generous margin so the bound never cuts a winning hit.
        t_limit = RBRT_T_CAP;
        if (closest < 3.0e38f) {
            float dl = len3(d);
            float omax = fmaxf(fmaxf(fabsf(o.x), fabsf(o.y)), fabsf(o.z));
            float lim = (closest * 1.001f + 1e-5f * (omax + closest) + 1e-6f) / dl;
            if (lim == lim) t_limit = fminf(t_limit, lim);
        }
        t_prune = t_limit; best_t = 1000000.0f; best_idx = 0xFFFFFFFFu;     // min_param init (triangle.rs:398)
        nodes = reinterpret_cast<const uint4*>(P.S.nodes) + 4 * (size_t)M.node_base; tri_base = M.tri_base;
        R = ray_slabs(M, o, d);
        sp = 0; stack.put(sp++, SENTINEL); cur = M.root_ref;
    };

    for (;;) {
        // ---- lanes whose traversal ended: close the mesh, move to the next one or resolve the ray
        bool want_fetch = (cur == SENTINEL);
        int done_kind = -1;
        if (want_fetch && has_ray) {
            if (best_idx != 0xFFFFFFFFu) {
                f3 p = o + best_t * d;                                    // ray.point_at (mesh.rs:247)
                float dist = len3(o - p);                                 // mesh.rs:248
                if (dist > RBRT_MIN_DIST && dist < RBRT_MAX_DIST && dist < closest) {   // mesh.rs:249 + scene.rs:36
                    closest = dist; bkind = 1; belem = mi; btri = best_idx; bt = best_t;
                }
            }
            while (++mi < P.S.n_meshes) {                                 // later meshes, in order (scene.rs:33-41)
                const MeshDev& M = P.S.meshes[mi];
                if (M.n_tris == 0 || !mesh_bbox_hit(M, o, d)) continue;
                start_mesh(M); want_fetch = false; break;
            }
            if (want_fetch) { done_kind = resolve(P, it, pid, o, d, bkind, belem, btri, bt); has_ray = false; }
        }
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            uint32_t slot = warp_append(&c->mat_count[k], done_kind == k);
            if (done_kind == k) P.matq[it & 1][k][slot] = pid;
        }
        // ---- dynamic fetch: idle lanes take the next rays of the queue (one atomic per warp)
        if (!exhausted) {
            uint32_t m = __ballot_sync(FULL_MASK, want_fetch);
            if (quota < 32u) {                                            // keep at most `quota` lanes of this warp busy
                uint32_t busy = 32u - __popc(m);
                uint32_t allow = busy < quota ? quota - busy : 0u;
                if (allow == 0u) m = 0u;
                else if (allow < (uint32_t)__popc(m)) m &= (1u << __fns(m, 0, allow + 1)) - 1u;
                want_fetch = want_fetch && ((m >> lane) & 1u);
            }
            if (m) {
                uint32_t base = warp_grab(&c->cand_head, __popc(m));
                if (want_fetch) {
                    uint32_t qi = base + __popc(m & lt);
                    if (qi < n) {
                        pid = P.candq[qi];
                        load_candidate_rec(P, pid, bt, belem, mi, closest, o, d);
                        bkind = belem != NO_SPHERE ? 0 : -1; btri = 0;
                        has_ray = true;
                        start_mesh(P.S.meshes[mi]);                       // stage A found this mesh's box hit
                    }
                }
                if (base + __popc(m) >= n) exhausted = true;
            }
        }
        uint32_t active = __ballot_sync(FULL_MASK, cur != SENTINEL);
        if (active == 0) { if (exhausted) break; continue; }
        const int threshold = exhausted ? 1 : min((int)P.fetch_thr, (int)quota);
        // ---- warp-voted traversal: one node visit or one triangle test per step, whichever more lanes wait for (intersect.cuh)
        traverse_voted<COUNT, false>(nodes, P.S.tris, tri_base, R, o, d, t_limit, stack, sp, cur, best_t, best_idx, t_prune, threshold, n_nodes, n_tris);
    }
    if (COUNT) {
        for (int off = 16; off; off >>= 1) { n_nodes += __shfl_down_sync(FULL_MASK, n_nodes, off); n_tris += __shfl_down_sync(FULL_MASK, n_tris, off); }
        if (lane == 0) { atomicAdd(&P.stats[ST_NODES], (unsigned long long)n_nodes); atomicAdd(&P.stats[ST_TRIS], (unsigned long long)n_tris); }
    }
}

// One queued ray, start to finish, by one lane (no dynamic fetch): the rest of Scene::hit for the meshes from the
// first one whose box it entered.  Used by the brute-force integrator and by the tail kernel.  Returns the
// material kind to shade, or -1 when the path ended.
template <bool BRUTE>
__device__ __forceinline__ int process_candidate(const WaveParams& P, uint32_t it, uint32_t pid, TraceCounters* cnt) {
    f3 o, d; float bt, closest; uint32_t belem, mi0, btri = 0;
    load_candidate_rec(P, pid, bt, belem, mi0, closest, o, d);
    int bkind = belem != NO_SPHERE ? 0 : -1;
    for (uint32_t mi = mi0; mi < P.S.n_meshes; ++mi) {
        const MeshDev& M = P.S.meshes[mi];
        if (M.n_tris == 0 || !mesh_bbox_hit(M, o, d)) continue;
        float t; uint32_t ti; bool ok;
        if (BRUTE) ok = mesh_closest_brute(P.S, M, o, d, t, ti, cnt);
        else {
            float t_limit = RBRT_T_CAP;
            if (closest < 3.0e38f) {
                float dl = len3(d);
                float omax = fmaxf(fmaxf(fabsf(o.x), fabsf(o.y)), fabsf(o.z));
                float lim = (closest * 1.001f + 1e-5f * (omax + closest) + 1e-6f) / dl;
                if (lim == lim) t_limit = fminf(t_limit, lim);
            }
            ok = mesh_closest_bvh(P.S, M, o, d, t_limit, t, ti, cnt);
        }
        if (!ok) continue;
        f3 p = o + t * d;
        float dist = len3(o - p);
        if (dist > RBRT_MIN_DIST && dist < RBRT_MAX_DIST && dist < closest) { closest = dist; bkind = 1; belem = mi; btri = ti; bt = t; }
    }
    return resolve(P, it, pid, o, d, bkind, belem, btri, bt);
}

// Brute-force stage B (RBRT_TRACE_BRUTE): the reference's own every-triangle loop, no dynamic fetch.
template <bool COUNT>
__global__ void __launch_bounds__(256) k_trace_brute(WaveParams P, uint32_t it) {
    IterCtr* c = P.ctr + it;
    const uint32_t n = c->cand_count;
    if (n == 0 || P.ctr[0].pad) return;
    if (COUNT && blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&P.stats[ST_CAND], (unsigned long long)n);
    TraceCounters cnt; cnt.nodes = 0; cnt.tris = 0;
    for (;;) {
        uint32_t base = warp_grab(&c->cand_head, 32u);
        if (base >= n) break;
        uint32_t qi = base + (threadIdx.x & 31);
        int done_kind = -1; uint32_t pid = 0;
        if (qi < n) { pid = P.candq[qi]; done_kind = process_candidate<true>(P, it, pid, COUNT ? &cnt : nullptr); }
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            uint32_t slot = warp_append(&c->mat_count[k], done_kind == k);
            if (done_kind == k) P.matq[it & 1][k][slot] = pid;
        }
    }
    if (COUNT) { atomicAdd(&P.stats[ST_NODES], (unsigned long long)cnt.nodes); atomicAdd(&P.stats[ST_TRIS], (unsigned long long)cnt.tris); }
}

// ------------------------------------------------------------------ shade (lib.rs:54-62 + the scatter impls) + stage A
// One hit of material `kind` at iteration `it`: scatter, then stage A of the continuation ray.  Returns its queue class.
template <bool ET>
__device__ __forceinline__ uint32_t shade_item(const WaveParams& P, uint32_t it, uint32_t kind, uint32_t pid,
                                               uint32_t& rays, uint32_t& nan_count) {
    f3 point, d; uint32_t elem, tri; bool is_mesh;
    load_pending(P, pid, point, d, elem, is_mesh, tri);
    f3 normal;
    if (!is_mesh) {                                                       // sphere: p - c, un-normalised (sphere.rs:56); BasicTriangle: stored normal
        if (ET) normal = element_normal(P.S, elem, point);
        else { float4 s4 = __ldg(P.S.spheres + elem); normal = point - mk3(s4.x, s4.y, s4.z); }
    }
    else {                                                              // mesh: stored unit normal (mesh.rs:253-257)
        const MeshDev& M = P.S.meshes[elem - P.S.n_spheres];
        float4 nn = __ldg(P.S.normals + M.nrm_base + tri);
        normal = mk3(nn.x, nn.y, nn.z);
    }
    uint32_t f, s_local, jp;
    path_coords(P, pid, f, s_local, jp);
    uint32_t row, col;
    shard_pixel(P.sh, P.cam[0], jp, row, col);
    RngKey key; key.k0 = P.key0[f]; key.k1 = P.key1[f];
    f3 out_d;
    bool cont = scatter(kind, __ldg(P.S.mat + elem), d, point, normal, key, row * P.cam[0].width + col,
                        P.s_base + s_local, it + 1, out_d);
    if (!cont) { end_path(P, pid, mk3(0, 0, 0)); return CLS_NONE; }       // absorbed (metal.rs:24) -> black
    store_hist(P, pid, it, elem);
    ++rays;
    return stage_a<ET>(P, it + 1, pid, point, out_d, nan_count);
}

#ifndef SHADE_BLOCKS
#define SHADE_BLOCKS 4
#endif
template <bool ET>
__global__ void __launch_bounds__(256, SHADE_BLOCKS) k_shade(WaveParams P, uint32_t it) {
    IterCtr* c = P.ctr + it;
    const uint32_t n0 = c->mat_count[0], n1 = c->mat_count[1], n2 = c->mat_count[2];
    // virtual index space: each material's run is padded to a multiple of 32 so a warp round never mixes kinds
    const uint32_t a0 = (n0 + 31u) & ~31u, a1 = a0 + ((n1 + 31u) & ~31u), total = a1 + ((n2 + 31u) & ~31u);
    if (total == 0 || P.ctr[0].pad) return;
    const uint32_t lane = threadIdx.x & 31;
    uint32_t nan_count = 0, rays = 0;
    const uint32_t n_warps = (gridDim.x * blockDim.x) >> 5;
    const uint32_t rounds = min((uint32_t)ROUNDS, max(1u, (total / 32u + n_warps - 1) / n_warps));   // tail iterations: spread the work
    for (;;) {
        uint32_t base = warp_grab(&c->shade_head, 32u * rounds);
        if (base >= total) break;
        Deferred df; df.clear();
        // The queue entries of all rounds first (independent, coalesced loads).  Prefetching the records they point to
        // (prefetch.global.L1 / .L2) was measured and made every iteration slower (it 1: 1.51 -> 1.78 ms): dropped.
        uint32_t kinds = 0;
#pragma unroll
        for (int r = 0; r < ROUNDS; ++r) {
            const uint32_t w = base + 32u * r + lane;
            uint32_t kind = 3u, j = 0, nk = 0;
            if ((uint32_t)r < rounds && w < total) {
                if (w < a0) { kind = 0; j = w; nk = n0; }
                else if (w < a1) { kind = 1; j = w - a0; nk = n1; }
                else { kind = 2; j = w - a1; nk = n2; }
                if (j >= nk) kind = 3u;
            }
            if (kind < 3u) df.pid[r] = P.matq[it & 1][kind][j];
            kinds |= kind << (2 * r);
        }
#pragma unroll 1                                                          // (measured: stall_no_instruction 5.7 per issue with the x4 unrolled body)
        for (int r = 0; r < ROUNDS; ++r) {
            const uint32_t kind = (kinds >> (2 * r)) & 3u;
            if (kind == 3u) continue;
            const uint32_t pid = df.pid[r];
            df.set(r, shade_item<ET>(P, it, kind, pid, rays, nan_count), pid);
        }
        flush(P, it + 1, df);
    }
    for (int off = 16; off; off >>= 1) { rays += __shfl_down_sync(FULL_MASK, rays, off); nan_count += __shfl_down_sync(FULL_MASK, nan_count, off); }
    if (lane == 0) {
        if (rays) atomicAdd(&P.ctr[it + 1].ray_count, rays);
        if (nan_count) atomicAdd(&P.stats[ST_NAN], (unsigned long long)nan_count);
    }
}

// ------------------------------------------------------------------ tail: finish every surviving path in ONE launch
// Each bounce iteration costs a trace and a shade launch whose durations are bounded below by their slowest ray
// (~0.2 ms together), however few rays are left, and paths trapped between surfaces use all 50 bounces.  Once the
// rays of iteration `it` fit the lanes of one resident grid, this kernel takes every queued item (traversal
// candidates and pending hits of iteration `it`) and runs each path to its end inside one lane — colorize's own
// loop (lib.rs:43-73) — with the same device functions as the wavefront kernels, so results are bit-identical.
// It raises ctr[0].pad; the remaining trace / shade / finish launches of the batch return at once.
template <bool BRUTE, bool COUNT, bool ET>
__global__ void __launch_bounds__(256) k_finish(WaveParams P, uint32_t it0, uint32_t max_rays) {
    if (P.ctr[0].pad) return;
    const IterCtr c = P.ctr[it0];
    if (c.ray_count > max_rays) return;
    const uint32_t nc = c.cand_count, n0 = c.mat_count[0], n1 = c.mat_count[1], n2 = c.mat_count[2];
    const uint32_t total = nc + n0 + n1 + n2;
    const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x, stride = gridDim.x * blockDim.x;
    uint32_t nan_count = 0, rays = 0;
    TraceCounters cnt; cnt.nodes = 0; cnt.tris = 0;
    uint32_t n_cand = 0;
    for (uint32_t w = tid; w < total; w += stride) {
        uint32_t it = it0, pid; int kind;                                 // kind: 0..2 pending hit of that material, CLS_CAND queued ray
        if (w < nc) { pid = P.candq[w]; kind = CLS_CAND; }
        else if (w < nc + n0) { pid = P.matq[it0 & 1][0][w - nc]; kind = 0; }
        else if (w < nc + n0 + n1) { pid = P.matq[it0 & 1][1][w - nc - n0]; kind = 1; }
        else { pid = P.matq[it0 & 1][2][w - nc - n0 - n1]; kind = 2; }
        for (;;) {
            if (kind == CLS_CAND) { ++n_cand; kind = process_candidate<BRUTE>(P, it, pid, COUNT ? &cnt : nullptr); }
            if (kind < 0) break;                                          // path ended (miss / depth exhausted)
            uint32_t cls = shade_item<ET>(P, it, (uint32_t)kind, pid, rays, nan_count);
            if (cls == CLS_NONE) break;                                   // absorbed / resolved on the spot
            kind = (int)cls; ++it;
        }
    }
    for (int off = 16; off; off >>= 1) { rays += __shfl_down_sync(FULL_MASK, rays, off); nan_count += __shfl_down_sync(FULL_MASK, nan_count, off); }
    if ((threadIdx.x & 31) == 0) {
        if (rays) atomicAdd(&P.ctr[P.max_depth + 1].ray_count, rays);     // statistics slot past the last iteration
        if (nan_count) atomicAdd(&P.stats[ST_NAN], (unsigned long long)nan_count);
    }
    if (COUNT) {
        atomicAdd(&P.stats[ST_TAIL_NODES], (unsigned long long)cnt.nodes); atomicAdd(&P.stats[ST_TAIL_TRIS], (unsigned long long)cnt.tris);
        atomicAdd(&P.stats[ST_TAIL_CAND], (unsigned long long)n_cand);
    }
    // Raise the flag only when EVERY block of this launch has finished (blocks that become resident late must still
    // pass the entry check above): the last block to leave sets it; later launches see it (stream order).
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(&P.ctr[1].pad, 1u) == gridDim.x - 1) P.ctr[0].pad = 1u + it0;
    }
}

// statistics: rays = sum over iterations of ray_count (one tiny launch per batch)
__global__ void k_sum_rays(WaveParams P) {
    unsigned long long r = 0;
    for (uint32_t it = threadIdx.x; it <= P.max_depth + 1; it += blockDim.x) r += P.ctr[it].ray_count;
    for (int off = 16; off; off >>= 1) r += __shfl_down_sync(FULL_MASK, r, off);
    if ((threadIdx.x & 31) == 0 && r) atomicAdd(&P.stats[ST_RAYS], r);
}

// ------------------------------------------------------------------ tail, asynchronous form (BVH mode)
// Same hand-over as k_finish, but built like k_trace: persistent warps, every lane owns a PATH (not a ray), lanes whose
// path has ended take the next queued item inside the loop, and traversal is the shared warp-voted loop with dynamic
// fetch.  There is no barrier between bounces of different paths, so the hand-over can happen while millions of rays are
// still alive: the sparsely populated iterations (each bounded by its slowest ray) disappear instead of being paid one
// after another.  A lane's step: [traversal of the meshes its ray entered] -> resolve -> scatter + stage A (possibly
// several times in a row for sphere-only bounces) -> next traversal, or end of path -> next item.
#define TAIL_THREADS 128
#define TAIL_FETCH_THRESHOLD 8  // WaveParams::tail_thr
#define TAIL_FORCE_IT 12        // from this bounce iteration on, the tail kernel takes whatever is left

template <bool COUNT, bool ET>
__global__ void __launch_bounds__(TAIL_THREADS, 4) k_tail(WaveParams P, uint32_t it0, uint32_t max_rays) {
    if (P.ctr[0].pad) return;
    const IterCtr c = P.ctr[it0];
    if (c.ray_count > max_rays) return;
    const uint32_t nc = c.cand_count, n0 = c.mat_count[0], n1 = c.mat_count[1], n2 = c.mat_count[2];
    const uint32_t total = nc + n0 + n1 + n2;
    uint32_t* head = &P.ctr[it0].shade_head;                              // unused by k_shade(it0) from now on: queue cursor of this kernel
    const uint32_t lane = threadIdx.x & 31, lt = (1u << lane) - 1;
    const int32_t SENTINEL = 0x7FFFFFFF;
    int32_t lstack[RBRT_STACK];
    const StackL stack = {lstack};
    // ---- path state
    uint32_t pid = 0, it = it0;
    int pending = -1;                                                     // material kind of a hit waiting to be shaded, -1 none
    // ---- ray state (as k_trace)
    bool has_ray = false;
    uint32_t mi = 0;
    f3 o = mk3(0, 0, 0), d = mk3(0, 0, 0);
    RaySlabs R = {0, 0, 0, 0, 0, 0, RBRT_SEL_LO, RBRT_SEL_LO, RBRT_SEL_LO, RBRT_SEL_HI, RBRT_SEL_HI, RBRT_SEL_HI};
    float closest = 0.0f, bt = 0.0f; int bkind = -1; uint32_t belem = 0, btri = 0;
    int32_t cur = SENTINEL; int sp = 0;
    float best_t = 0.0f, t_prune = 0.0f, t_limit = 0.0f; uint32_t best_idx = 0xFFFFFFFFu;
    const uint4* __restrict__ nodes = reinterpret_cast<const uint4*>(P.S.nodes); uint32_t tri_base = 0;
    bool exhausted = total == 0;
    uint32_t n_nodes = 0, n_tris = 0, n_cand = 0, rays = 0, nan_count = 0;
    const uint32_t n_warps = (gridDim.x * blockDim.x) >> 5;
    const uint32_t quota = min(32u, max(1u, (total + n_warps - 1) / n_warps));

    auto start_mesh = [&](const MeshDev& M) {
        t_limit = RBRT_T_CAP;
        if (closest < 3.0e38f) {
            float dl = len3(d);
            float omax = fmaxf(fmaxf(fabsf(o.x), fabsf(o.y)), fabsf(o.z));
            float lim = (closest * 1.001f + 1e-5f * (omax + closest) + 1e-6f) / dl;
            if (lim == lim) t_limit = fminf(t_limit, lim);
        }
        t_prune = t_limit; best_t = 1000000.0f; best_idx = 0xFFFFFFFFu;
        nodes = reinterpret_cast<const uint4*>(P.S.nodes) + 4 * (size_t)M.node_base; tri_base = M.tri_base;
        R = ray_slabs(M, o, d);
        sp = 0; stack.put(sp++, SENTINEL); cur = M.root_ref;
    };
    auto load_candidate = [&]() {                                         // the ray stage A queued for this path
        load_candidate_rec(P, pid, bt, belem, mi, closest, o, d);
        bkind = belem != NO_SPHERE ? 0 : -1; btri = 0;
        has_ray = true;
        if (COUNT) ++n_cand;
        start_mesh(P.S.meshes[mi]);
    };

    for (;;) {
        // ---- (1) lanes whose traversal ended: close the mesh, move to the next one or resolve the ray
        bool idle = (cur == SENTINEL);
        if (idle && has_ray) {
            if (best_idx != 0xFFFFFFFFu) {
                f3 p = o + best_t * d;
                float dist = len3(o - p);
                if (dist > RBRT_MIN_DIST && dist < RBRT_MAX_DIST && dist < closest) { closest = dist; bkind = 1; belem = mi; btri = best_idx; bt = best_t; }
            }
            bool more = false;
            while (++mi < P.S.n_meshes) {
                const MeshDev& M = P.S.meshes[mi];
                if (M.n_tris == 0 || !mesh_bbox_hit(M, o, d)) continue;
                start_mesh(M); more = true; break;
            }
            if (!more) { pending = resolve(P, it, pid, o, d, bkind, belem, btri, bt); has_ray = false; }   // -1: the path ended
            else idle = false;
        }
        // ---- (2) lanes without a path take the next queued item (one atomic per warp)
        bool want_fetch = idle && !has_ray && pending < 0;
        if (!exhausted) {
            uint32_t m = __ballot_sync(FULL_MASK, want_fetch);
            if (quota < 32u) {
                uint32_t busy = 32u - __popc(m);
                uint32_t allow = busy < quota ? quota - busy : 0u;
                if (allow == 0u) m = 0u;
                else if (allow < (uint32_t)__popc(m)) m &= (1u << __fns(m, 0, allow + 1)) - 1u;
                want_fetch = want_fetch && ((m >> lane) & 1u);
            }
            if (m) {
                uint32_t base = warp_grab(head, __popc(m));
                if (want_fetch) {
                    uint32_t w = base + __popc(m & lt);
                    if (w < total) {
                        it = it0;
                        if (w < nc) { pid = P.candq[w]; load_candidate(); }
                        else if (w < nc + n0) { pid = P.matq[it0 & 1][0][w - nc]; pending = 0; }
                        else if (w < nc + n0 + n1) { pid = P.matq[it0 & 1][1][w - nc - n0]; pending = 1; }
                        else { pid = P.matq[it0 & 1][2][w - nc - n0 - n1]; pending = 2; }
                    }
                }
                if (base + __popc(m) >= total) exhausted = true;
            }
        }
        // ---- (3) pending hits: scatter + stage A, repeated while the continuation ray is resolved by a sphere alone
        while (pending >= 0) {
            uint32_t cls = shade_item<ET>(P, it, (uint32_t)pending, pid, rays, nan_count);
            ++it;
            if (cls == CLS_CAND) { pending = -1; load_candidate(); }
            else if (cls == CLS_NONE) pending = -1;                       // absorbed, missed, depth exhausted: path over
            else pending = (int)cls;
        }
        uint32_t active = __ballot_sync(FULL_MASK, cur != SENTINEL);
        if (active == 0) { if (exhausted) break; continue; }
        const int threshold = exhausted ? 1 : min((int)P.tail_thr, (int)quota);
        // ---- (4) traversal, as k_trace
#ifndef RBRT_TAIL_PREFETCH      // measured (profiles/r2_summary.md): prefetching the four children of every visited node into L1 makes the tail kernel SLOWER
                                // (1/8 shard of C3: 1.3 -> 2.3 ms, full frame 2.9 -> 4.0 ms): it is not a pure latency chain, the extra L1TEX requests cost more
        traverse_voted<COUNT, false>(nodes, P.S.tris, tri_base, R, o, d, t_limit, stack, sp, cur, best_t, best_idx, t_prune, threshold, n_nodes, n_tris);
#else
        traverse_voted<COUNT, true>(nodes, P.S.tris, tri_base, R, o, d, t_limit, stack, sp, cur, best_t, best_idx, t_prune, threshold, n_nodes, n_tris);
#endif
    }
    for (int off = 16; off; off >>= 1) { rays += __shfl_down_sync(FULL_MASK, rays, off); nan_count += __shfl_down_sync(FULL_MASK, nan_count, off); }
    if (lane == 0) {
        if (rays) atomicAdd(&P.ctr[P.max_depth + 1].ray_count, rays);
        if (nan_count) atomicAdd(&P.stats[ST_NAN], (unsigned long long)nan_count);
    }
    if (COUNT) {
        for (int off = 16; off; off >>= 1) { n_nodes += __shfl_down_sync(FULL_MASK, n_nodes, off); n_tris += __shfl_down_sync(FULL_MASK, n_tris, off); n_cand += __shfl_down_sync(FULL_MASK, n_cand, off); }
        if (lane == 0) { atomicAdd(&P.stats[ST_TAIL_NODES], (unsigned long long)n_nodes); atomicAdd(&P.stats[ST_TAIL_TRIS], (unsigned long long)n_tris); atomicAdd(&P.stats[ST_TAIL_CAND], (unsigned long long)n_cand); }
    }
    __syncthreads();
    if (threadIdx.x == 0) {                                               // last block out raises the flag (see k_finish)
        __threadfence();
        if (atomicAdd(&P.ctr[1].pad, 1u) == gridDim.x - 1) P.ctr[0].pad = 1u + it0;
    }
}

// ------------------------------------------------------------------ accumulate (lib.rs:95-100)
struct AccumPtrs { float4* p[RBRT_MAX_FRAMES]; };
__global__ void __launch_bounds__(256) k_accumulate(WaveParams P, AccumPtrs A) {
    uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t f = blockIdx.y;                                        // frame of the batch
    if (j >= P.paths_px) return;
    uint32_t row, col;
    if (!shard_pixel(P.sh, P.cam[0], j, row, col)) return;
    size_t px = (size_t)row * P.cam[0].width + col;
    float4* __restrict__ accum = A.p[f];
    float4 acc = accum[px];
    for (uint32_t s = 0; s < P.s_count; ++s) {
        float4 c = P.out[((size_t)f * P.s_count + s) * P.paths_px + j];
        acc.x = XADD(acc.x, c.x); acc.y = XADD(acc.y, c.y); acc.z = XADD(acc.z, c.z);
    }
    accum[px] = acc;
}

// ------------------------------------------------------------------ finalize (lib.rs:101,116-122)
__global__ void __launch_bounds__(256) k_finalize(const float4* __restrict__ accum, size_t n_px, float inv_spp,
                                                  uint8_t* __restrict__ rgb, float* __restrict__ hdr) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_px) return;
    float4 a = accum[i];
    f3 c = mk3(a.x, a.y, a.z) * inv_spp;
    if (hdr) { hdr[3 * i] = c.x; hdr[3 * i + 1] = c.y; hdr[3 * i + 2] = c.z; }
    if (rgb) {
        rgb[3 * i] = as_u8(XMUL(XSQRT(c.x), 256.0f));
        rgb[3 * i + 1] = as_u8(XMUL(XSQRT(c.y), 256.0f));
        rgb[3 * i + 2] = as_u8(XMUL(XSQRT(c.z), 256.0f));
    }
}

// ------------------------------------------------------------------ parity hooks
template <bool BRUTE>
__global__ void __launch_bounds__(256) k_trace_rays(SceneDev S, const rbrt_ray* __restrict__ rays, uint64_t n,
                                                    rbrt_hit* __restrict__ hits, unsigned long long* stats) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    TraceCounters cnt; cnt.nodes = 0; cnt.tris = 0;
    if (i < n) {
        rbrt_ray r = rays[i];
        f3 o = mk3(r.origin.x, r.origin.y, r.origin.z), d = mk3(r.direction.x, r.direction.y, r.direction.z);
        Hit h = scene_hit<BRUTE>(S, o, d, stats ? &cnt : nullptr);
        rbrt_hit out;
        out.kind = h.kind >= 0 ? h.kind : RBRT_HIT_NONE;
        out.elem_idx = 0; out.tri_idx = 0; out.t = 0.0f; out.dist = 0.0f;
        out.point.x = out.point.y = out.point.z = 0.0f;
        out.normal.x = out.normal.y = out.normal.z = 0.0f;
        if (h.kind >= 0) {
            f3 p = o + h.t * d;
            f3 nrm;
            if (h.kind == 0) { nrm = element_normal(S, h.elem, p); if (S.n_etris && __ldg(S.elem_kind + h.elem)) out.kind = RBRT_HIT_TRIANGLE; }
            else { float4 nn = __ldg(S.normals + S.meshes[h.elem].nrm_base + h.tri); nrm = mk3(nn.x, nn.y, nn.z); }
            out.elem_idx = h.elem; out.tri_idx = h.tri; out.t = h.t; out.dist = h.dist;
            out.point.x = p.x; out.point.y = p.y; out.point.z = p.z;
            out.normal.x = nrm.x; out.normal.y = nrm.y; out.normal.z = nrm.z;
        } else if (h.kind == -2 && stats) atomicAdd(&stats[ST_NAN], 1ull);
        hits[i] = out;
    }
    if (stats) {
        if (cnt.nodes) atomicAdd(&stats[ST_NODES], (unsigned long long)cnt.nodes);
        if (cnt.tris) atomicAdd(&stats[ST_TRIS], (unsigned long long)cnt.tris);
    }
}

__global__ void __launch_bounds__(256) k_primary_rays(CamDev cam, uint32_t key0, uint32_t key1, uint32_t sample, rbrt_ray* __restrict__ rays) {
    uint32_t px = blockIdx.x * blockDim.x + threadIdx.x;
    if (px >= cam.width * cam.height) return;
    uint32_t row = px / cam.width, col = px - row * cam.width;
    RngKey key; key.k0 = key0; key.k1 = key1;
    f3 o, d;
    camera_ray(cam, row, col, key, px, sample, o, d);
    rbrt_ray r; r.origin.x = o.x; r.origin.y = o.y; r.origin.z = o.z; r.direction.x = d.x; r.direction.y = d.y; r.direction.z = d.z;
    rays[px] = r;
}

// scatter() in isolation (materials.rs:4-12): the same device function the shade kernels call, one item per thread
__global__ void __launch_bounds__(256) k_scatter_kat(const rbrt_scatter_in* __restrict__ in, uint64_t n, uint32_t key0, uint32_t key1,
                                                     rbrt_scatter_out* __restrict__ out) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const rbrt_scatter_in q = in[i];
    RngKey key; key.k0 = key0; key.k1 = key1;
    const f3 point = mk3(q.hit_point.x, q.hit_point.y, q.hit_point.z), normal = mk3(q.hit_normal.x, q.hit_normal.y, q.hit_normal.z);
    f3 out_d = mk3(0, 0, 0);
    const bool ok = scatter(q.material.kind, make_float4(q.material.albedo.x, q.material.albedo.y, q.material.albedo.z, q.material.param),
                            mk3(q.in_ray.direction.x, q.in_ray.direction.y, q.in_ray.direction.z), point, normal, key, q.pixel, q.sample, q.bounce, out_d);
    rbrt_scatter_out r;
    r.scattered = ok ? 1 : 0;
    const bool glass = q.material.kind == 2u;                             // attenuation: albedo, or (1,1,1) for dielectrics (dielectric.rs:19)
    r.attenuation.x = glass ? 1.0f : q.material.albedo.x; r.attenuation.y = glass ? 1.0f : q.material.albedo.y; r.attenuation.z = glass ? 1.0f : q.material.albedo.z;
    r.out_ray.origin = q.hit_point;
    r.out_ray.direction.x = out_d.x; r.out_ray.direction.y = out_d.y; r.out_ray.direction.z = out_d.z;
    out[i] = r;
}

// ------------------------------------------------------------------ parity hook through the renderer's own kernels
// Caller-supplied rays become "paths" pid = ray index at bounce iteration 0: stage A exactly as k_generate runs it, then
// k_trace itself (persistent warps, quota, dynamic fetch, warp-voted traversal), then the records are read back.
// out[pid].w is pre-set to a NaN pattern; a path that ended (miss -> sky, NaN -> black) has it overwritten with 0.
template <bool ET>
__global__ void __launch_bounds__(256) k_rays_stage_a(WaveParams P, const rbrt_ray* __restrict__ rays, uint32_t n) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    const uint32_t n_groups = (n + 31) >> 5;
    uint32_t nan_count = 0;
    for (uint32_t g0 = warp * ROUNDS; g0 < n_groups; g0 += n_warps * ROUNDS) {
        Deferred df; df.clear();
#pragma unroll 1
        for (int r = 0; r < ROUNDS; ++r) {
            const uint32_t pid = ((g0 + r) << 5) + lane;
            if (g0 + r >= n_groups || pid >= n) continue;
            const rbrt_ray q = rays[pid];
            df.set(r, stage_a<ET>(P, 0, pid, mk3(q.origin.x, q.origin.y, q.origin.z), mk3(q.direction.x, q.direction.y, q.direction.z), nan_count), pid);
        }
        flush(P, 0, df);
    }
    for (int off = 16; off; off >>= 1) nan_count += __shfl_down_sync(FULL_MASK, nan_count, off);
    if (lane == 0 && nan_count) atomicAdd(&P.stats[ST_NAN], (unsigned long long)nan_count);
}

__global__ void __launch_bounds__(256) k_rays_collect(WaveParams P, const rbrt_ray* __restrict__ rays, uint32_t n, rbrt_hit* __restrict__ hits) {
    const uint32_t pid = blockIdx.x * blockDim.x + threadIdx.x;
    if (pid >= n) return;
    rbrt_hit out;
    out.kind = RBRT_HIT_NONE; out.elem_idx = 0; out.tri_idx = 0; out.t = 0.0f; out.dist = 0.0f;
    out.point.x = out.point.y = out.point.z = 0.0f; out.normal.x = out.normal.y = out.normal.z = 0.0f;
    if (__float_as_uint(P.out[pid].w) == 0xFFFFFFFFu) {                   // the path did not end: a hit is waiting to be shaded
        f3 p, d_rec; uint32_t elem, tri; bool is_mesh;
        load_pending(P, pid, p, d_rec, elem, is_mesh, tri);
        const rbrt_ray q = rays[pid];
        const f3 o = mk3(q.origin.x, q.origin.y, q.origin.z);
        const float t = P.out[pid].x;                                     // WaveParams::keep_t
        f3 nrm;
        if (!is_mesh) {
            nrm = element_normal(P.S, elem, p);
            out.kind = (P.S.n_etris && __ldg(P.S.elem_kind + elem)) ? RBRT_HIT_TRIANGLE : RBRT_HIT_SPHERE;
            out.elem_idx = elem;
        } else {
            const uint32_t mi = elem - P.S.n_spheres;
            const float4 nn = __ldg(P.S.normals + P.S.meshes[mi].nrm_base + tri); nrm = mk3(nn.x, nn.y, nn.z);
            out.kind = RBRT_HIT_MESH; out.elem_idx = mi; out.tri_idx = tri;
        }
        out.t = t; out.dist = len3(o - p);                                // sphere.rs:50, mesh.rs:248
        out.point.x = p.x; out.point.y = p.y; out.point.z = p.z;
        out.normal.x = nrm.x; out.normal.y = nrm.y; out.normal.z = nrm.z;
    }
    hits[pid] = out;
}

// ====================================================================== host side
CamDev make_cam(const rbrt_camera& c) {
    CamDev d;
    d.pos[0] = c.position.x; d.pos[1] = c.position.y; d.pos[2] = c.position.z;
    d.right[0] = c.right.x; d.right[1] = c.right.y; d.right[2] = c.right.z;
    d.up[0] = c.up.x; d.up[1] = c.up.y; d.up[2] = c.up.z;
    d.center[0] = c.img_center_point.x; d.center[1] = c.img_center_point.y; d.center[2] = c.img_center_point.z;
    d.mm_per_pix_hor = c.mm_per_pix_hor; d.mm_per_pix_vert = c.mm_per_pix_vert;
    d.width = c.img_width_pix; d.height = c.img_height_pix;
    return d;
}

static WaveBuffers g_wave[8][64];                                       // [pool][device]; pools 1..3 = RBRT_OPT_POOL_* (more frames in flight);
                                                                        // 4..7 = the second lane of pools 0..3 (RBRT_OPT_SPLIT_BATCHES)
WaveBuffers& device_wave_buffers(int device, int pool) { return g_wave[pool & 7][(device >= 0 && device < 64) ? device : 0]; }
// Second lane of a pool: its own stream and the events that order the two lanes of one frame
struct SplitLane { cudaStream_t aux = nullptr; cudaEvent_t fork = nullptr, acc[2] = {nullptr, nullptr}, join = nullptr; };
static SplitLane g_lane[4][64];
static int ensure_lane(SplitLane& L) {
    if (L.aux) return RBRT_OK;
    cudaError_t e = cudaStreamCreateWithFlags(&L.aux, cudaStreamNonBlocking);
    for (cudaEvent_t* ev : {&L.fork, &L.acc[0], &L.acc[1], &L.join}) if (e == cudaSuccess) e = cudaEventCreateWithFlags(ev, cudaEventDisableTiming);
    if (e != cudaSuccess) return cuda_fail(e, "split lane");
    return RBRT_OK;
}
void release_device_wave_buffers() {
    int cur = 0; cudaGetDevice(&cur);
    for (int p = 0; p < 8; ++p)
        for (int d = 0; d < 64; ++d) if (g_wave[p][d].cap || g_wave[p][d].accum || g_wave[p][d].rgb) { cudaSetDevice(d); free_wave_buffers(g_wave[p][d]); }
    for (int p = 0; p < 4; ++p)
        for (int d = 0; d < 64; ++d) {
            SplitLane& L = g_lane[p][d];
            if (!L.aux) continue;
            cudaSetDevice(d); cudaStreamSynchronize(L.aux); cudaStreamDestroy(L.aux);
            for (cudaEvent_t ev : {L.fork, L.acc[0], L.acc[1], L.join}) if (ev) cudaEventDestroy(ev);
            L = SplitLane();
        }
    cudaSetDevice(cur);
}

void free_wave_buffers(WaveBuffers& wb) {
    cudaFree(wb.rec); cudaFree(wb.candq);
    for (int i = 0; i < 6; ++i) cudaFree(wb.matq[i / 3][i % 3]);
    cudaFree(wb.out); cudaFree(wb.hist); cudaFree(wb.ctr); cudaFree(wb.stats); cudaFree(wb.accum);
    cudaFree(wb.rgb); cudaFree(wb.hdr);
    for (cudaEvent_t e : wb.ev) cudaEventDestroy(e);
    wb = WaveBuffers();
}

#define CKR(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) return cuda_fail(e_, #x); } while (0)

static int ensure_wave_buffers(WaveBuffers& wb, uint32_t cap, uint32_t depth) {
    if (wb.cap >= cap && wb.depth_cap >= depth && wb.stats) return RBRT_OK;
    float4* accum = wb.accum; size_t accum_px = wb.accum_px; uint8_t* rgb = wb.rgb; float* hdr = wb.hdr; size_t out_px = wb.out_px;
    std::vector<cudaEvent_t> ev; ev.swap(wb.ev);
    wb.accum = nullptr; wb.rgb = nullptr; wb.hdr = nullptr;
    free_wave_buffers(wb);
    wb.accum = accum; wb.accum_px = accum_px; wb.rgb = rgb; wb.hdr = hdr; wb.out_px = out_px; wb.ev.swap(ev);
    size_t b = 0;
    CKR(cudaMalloc(&wb.rec, 32ull * cap)); b += 32ull * cap;
    CKR(cudaMalloc(&wb.candq, 4ull * cap)); b += 4ull * cap;
    for (int i = 0; i < 6; ++i) { CKR(cudaMalloc(&wb.matq[i / 3][i % 3], 4ull * cap)); b += 4ull * cap; }
    CKR(cudaMalloc(&wb.out, 16ull * cap)); b += 16ull * cap;
    { const uint64_t rows = std::max<uint64_t>(depth, 1); CKR(cudaMalloc(&wb.hist, 2ull * cap * rows)); b += 2ull * cap * rows; }
    CKR(cudaMalloc(&wb.ctr, sizeof(IterCtr) * (depth + 2)));
    CKR(cudaMalloc(&wb.stats, 8 * ST_COUNT));
    wb.cap = cap; wb.depth_cap = depth; wb.bytes = b;
    return RBRT_OK;
}

// Renders n_frames (1..RBRT_MAX_FRAMES) frames of ONE scene — a camera and a Philox key each, same image size and
// sample count — in the same wavefront batches: a rank's share of a frame can be small (1/8 of C3: launches of
// 0.3-1 M rays that run at a third of the dense rate and each end in a drain as long as their slowest ray), and two
// or four frames per batch give the kernels the size they have on fewer GPUs.  Every path keeps its own (pixel,
// sample, frame) identity, so each image is bit-identical to a lone render of that frame.
void note_scene_use(const Scene& sc, int device, cudaStream_t st) {
    static std::mutex mu;                                                 // the per-GPU enqueue threads of one collective render share the scene
    std::lock_guard<std::mutex> g(mu);
    for (SceneUse& u : sc.uses)
        if (u.device == device && u.stream == st) { cudaEventRecord(u.ev, st); return; }
    SceneUse u{device, st, nullptr};
    if (cudaEventCreateWithFlags(&u.ev, cudaEventDisableTiming) != cudaSuccess) { cudaGetLastError(); return; }
    cudaEventRecord(u.ev, st);
    sc.uses.push_back(u);
}

// Pixel / sample shard of one rank (common.cuh ShardDev) from the render options
int make_shard(const rbrt_render_opts& o, uint32_t W, uint32_t H, uint32_t spp, ShardDev* out) {
    ShardDev sh;
    sh.rank = 0; sh.count = 1; sh.s0 = 0; sh.s1 = spp;
    sh.tiles_x = (W + 7) / 8;
    sh.fd_tiles_x = make_fastdiv(sh.tiles_x);
    sh.tiles_total = sh.tiles_x * ((H + 3) / 4);
    if (o.shard_count > 1) {
        if (o.shard_rank >= o.shard_count) { set_error("shard_rank >= shard_count"); return RBRT_E_INVALID; }
        if (o.shard_mode == RBRT_SHARD_TILES) { sh.rank = o.shard_rank; sh.count = o.shard_count; }
        else if (o.shard_mode == RBRT_SHARD_SAMPLES) {
            sh.s0 = (uint32_t)((uint64_t)spp * o.shard_rank / o.shard_count);
            sh.s1 = (uint32_t)((uint64_t)spp * (o.shard_rank + 1) / o.shard_count);
        } else { set_error("shard_count > 1 needs shard_mode TILES or SAMPLES"); return RBRT_E_INVALID; }
    }
    sh.tiles_mine = sh.tiles_total > sh.rank ? (sh.tiles_total - sh.rank + sh.count - 1) / sh.count : 0;
    *out = sh;
    return RBRT_OK;
}

int render_accum(const Scene& sc, int li, const rbrt_camera* cams, const uint64_t* seeds, uint32_t n_frames, uint32_t spp,
                 const rbrt_render_opts* opts, float4* const* d_accum, cudaStream_t st, rbrt_stats* stats, RenderJob* job_out,
                 int pool_arg) {
    const Replica& rp = sc.rep[li];
    RenderJob local_job;
    RenderJob& job = job_out ? *job_out : local_job;
    if (!n_frames || n_frames > RBRT_MAX_FRAMES) { set_error("n_frames must be 1..%d", RBRT_MAX_FRAMES); return RBRT_E_INVALID; }
    const rbrt_camera& cam = cams[0];
    const uint32_t W = cam.img_width_pix, H = cam.img_height_pix;
    for (uint32_t f = 1; f < n_frames; ++f)
        if (cams[f].img_width_pix != W || cams[f].img_height_pix != H) { set_error("frames of one batch must have the same image size"); return RBRT_E_INVALID; }
    if (!W || !H || !spp) { set_error("empty image or zero samples"); return RBRT_E_INVALID; }
    if ((uint64_t)W * H > 0x7FFFFFFFull) { set_error("image too large"); return RBRT_E_INVALID; }
    rbrt_render_opts o{}; if (opts) o = *opts;
    const uint32_t max_depth = o.max_depth ? o.max_depth : 50;
    if (max_depth > 1024) { set_error("max_depth > 1024"); return RBRT_E_INVALID; }
    if (o.integrator != 0) { set_error("unknown integrator %u", o.integrator); return RBRT_E_INVALID; }
    ShardDev sh;
    { int rc_sh = make_shard(o, W, H, spp, &sh); if (rc_sh) return rc_sh; }
    const uint32_t P = sh.tiles_mine * 32;
    CKR(cudaEventCreate(&job.ev0)); CKR(cudaEventCreate(&job.ev1));
    const cudaEvent_t ev0 = job.ev0, ev1 = job.ev1;
    wait_scene_ready(sc, li, st);                                         // the scene's build / replication is asynchronous
    for (uint32_t f = 0; f < n_frames; ++f) CKR(cudaMemsetAsync(d_accum[f], 0, 16ull * W * H, st));
    uint32_t launches = 0, iterations = 0, batch_iters = 0;
    const int pool = pool_arg >= 0 ? pool_arg & 7 : (int)((o.flags & RBRT_OPT_POOL_MASK) >> RBRT_OPT_POOL_SHIFT);
    // TWO LANES (RBRT_OPT_SPLIT_BATCHES).  A batch ends sparsely: its last bounce iterations and the tail kernel are latency chains
    // that leave most SMs idle (1/8 shard of C3: ~2.3 of 6.3 ms), and for a LONE frame no other frame is there to fill them.  So the
    // frame's samples are cut into at least two batches that alternate between two lanes — the caller's stream with pool p, an
    // internal stream with pool 4 + p — and the dense start of one batch runs under the sparse end of the previous one.  The
    // per-pixel sums keep their sample order: a batch's k_accumulate waits (event) for the previous batch's.
    const bool split = (o.flags & RBRT_OPT_SPLIT_BATCHES) && !(o.flags & RBRT_OPT_TIME_KERNELS) && sh.s1 - sh.s0 >= 2 && pool < 4;
    WaveBuffers* wbs[2] = {&device_wave_buffers(rp.device, pool), split ? &device_wave_buffers(rp.device, 4 + pool) : nullptr};
    WaveBuffers& wb = *wbs[0];
    SplitLane& SL = g_lane[pool & 3][rp.device & 63];
    if (split) { int rc_l = ensure_lane(SL); if (rc_l) return rc_l; }
    cudaStream_t lane_st[2] = {st, split ? SL.aux : st};
    uint32_t lane_iters[2] = {0, 0};
    CKR(cudaEventRecord(ev0, st));
    if (P && sh.s1 > sh.s0) {
        // Paths in flight per batch.  Every bounce iteration is one trace + one shade launch whose duration is
        // bounded below by its slowest ray, so the ~45 sparsely populated tail iterations cost the same for a
        // small batch as for a large one: the default is therefore "as many paths as fit" — up to 2^27 paths
        // (108 + 2*(max_depth - 12) bytes of wavefront state each: 24.7 GB at depth 50) and at most half of the free HBM.
        uint32_t target = o.batch_paths;
        const uint64_t PF = (uint64_t)P * n_frames;                                           // paths of one sample of every frame of the batch
        if (PF > 0x7FFFFFFFull) { set_error("batch too large"); return RBRT_E_INVALID; }
        const uint64_t per_path = 76ull + 2ull * std::max<uint64_t>(max_depth, 1);            // record 32 + queues 28 + radiance 16 + history rows
        const uint64_t limit_paths = pool_limit_bytes() ? std::max<uint64_t>(pool_limit_bytes() / per_path, 1) : ~0ull;   // rbrt_gpu_set_pool_limit
        const uint32_t S_all = sh.s1 - sh.s0, S_half = (S_all + 1) / 2;
        if (!target) {
            const uint64_t want = std::min<uint64_t>(std::min<uint64_t>((uint64_t)(split ? S_half : S_all) * PF, 1ull << 27), limit_paths);
            const uint64_t want_sb = std::max<uint64_t>(want / PF, 1);                      // whole samples per batch
            bool have = true;
            for (int l = 0; l < (split ? 2 : 1); ++l) have = have && wbs[l]->cap >= want_sb * PF && wbs[l]->depth_cap >= max_depth;
            if (have) target = (uint32_t)want;                            // the pools already hold it: no driver query (cudaMemGetInfo takes tens of ms at times)
            else {
                size_t free_b = 0, total_b = 0;
                CKR(cudaMemGetInfo(&free_b, &total_b));
                free_b += wb.bytes + (split ? wbs[1]->bytes : 0);         // what a re-allocation would release first
                uint64_t fit = (free_b / 2) / per_path / (split ? 2 : 1);
                target = (uint32_t)(fit < (1ull << 21) ? (1ull << 21) : (fit > (1ull << 27) ? (1ull << 27) : fit));
            }
        }
        if ((uint64_t)target > limit_paths) target = (uint32_t)limit_paths;
        uint64_t S_b64 = (uint64_t)target / PF; if (S_b64 < 1) S_b64 = 1; if (S_b64 > S_all) S_b64 = S_all;
        if (split && S_b64 > S_half) S_b64 = S_half;                      // at least two batches, one per lane
        if (S_b64 * PF > 0x7FFFFFFFull) { set_error("batch too large"); return RBRT_E_INVALID; }
        const uint32_t S_b = (uint32_t)S_b64;
        const uint32_t cap = (uint32_t)(S_b64 * PF);
        WaveParams wps[2];
        for (int l = 0; l < (split ? 2 : 1); ++l) {
            WaveBuffers& w = *wbs[l];
            int rc = ensure_wave_buffers(w, cap, max_depth);
            if (rc) return rc;
            WaveParams& wp = wps[l];
            wp.S = rp.dev; wp.sh = sh; wp.n_frames = n_frames;
            for (uint32_t f = 0; f < RBRT_MAX_FRAMES; ++f) {
                const uint32_t g = f < n_frames ? f : 0;
                const uint64_t seed = seeds ? seeds[g] : o.seed;
                wp.cam[f] = make_cam(cams[g]); wp.key0[f] = (uint32_t)seed; wp.key1[f] = (uint32_t)(seed >> 32);
            }
            wp.cap = w.cap; wp.paths_px = P; wp.fd_paths_px = make_fastdiv(P); wp.max_depth = max_depth;
            static const bool no_cull_env = getenv("RBRT_NO_PRIMARY_CULL") != nullptr;      // tuning / A-B knob
            wp.use_cull = no_cull_env ? 0u : 1u;
            wp.keep_t = 0u;
            const char* thr_env = getenv("RBRT_FETCH_THRESHOLD");             // tuning knob
            wp.fetch_thr = thr_env ? (uint32_t)std::min(32, std::max(1, atoi(thr_env))) : FETCH_THRESHOLD;
            const char* tthr_env = getenv("RBRT_TAIL_FETCH_THRESHOLD");
            wp.tail_thr = tthr_env ? (uint32_t)std::min(32, std::max(1, atoi(tthr_env))) : TAIL_FETCH_THRESHOLD;
            wp.rec = w.rec; wp.candq = w.candq;
            for (int i = 0; i < 6; ++i) wp.matq[i / 3][i % 3] = w.matq[i / 3][i % 3];
            wp.out = w.out; wp.hist = w.hist; wp.ctr = w.ctr; wp.stats = w.stats;
        }
        AccumPtrs ap; for (uint32_t f = 0; f < RBRT_MAX_FRAMES; ++f) ap.p[f] = d_accum[f < n_frames ? f : 0];
        if (split) {                                                      // fork: the second lane starts behind the caller's stream (scene ready, accumulators cleared)
            CKR(cudaEventRecord(SL.fork, st));
            CKR(cudaStreamWaitEvent(SL.aux, SL.fork, 0));
        }
        for (int l = 0; l < (split ? 2 : 1); ++l) CKR(cudaMemsetAsync(wbs[l]->stats, 0, 8 * ST_COUNT, lane_st[l]));
        const int sm_count = rp.sm_count;
        const int grid = sm_count * 8;                                     // producers / brute: 256-thread blocks
        int per_sm = 0;                                                   // k_trace: persistent blocks, exactly one resident wave
        static int per_sm_cached = 0, fin_per_sm_cached = 0;             // occupancy queries are pure functions of the kernels
        if (!per_sm_cached) CKR(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_cached, k_trace<false>, TRACE_THREADS, 0));
        per_sm = per_sm_cached;
        const int grid_trace = sm_count * (per_sm > 0 ? per_sm : 4);
        if (!fin_per_sm_cached) CKR(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&fin_per_sm_cached, k_finish<false, false, false>, 256, 0));
        const int fin_per_sm = fin_per_sm_cached;                         // k_finish: one resident wave of 256-thread blocks
        const int grid_fin = sm_count * (fin_per_sm > 0 ? fin_per_sm : 2);
        static int tail_per_sm_cached = 0;
        if (!tail_per_sm_cached) CKR(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&tail_per_sm_cached, k_tail<false, true>, TAIL_THREADS, 0));
        const int grid_tail = sm_count * (tail_per_sm_cached > 0 ? tail_per_sm_cached : 2);
        const char* tail_env = getenv("RBRT_TAIL_RAYS");                  // tuning knob
        // hand-over threshold: brute mode one ray per resident lane of k_finish; BVH mode (asynchronous k_tail) 2^18 rays (swept on C2, C3, C4 at 1 and 8 ranks: scripts/tail_sweep.py)
        const uint32_t tail_rays = (o.flags & RBRT_OPT_NO_TAIL_KERNEL) ? 0u : (tail_env ? (uint32_t)atoi(tail_env) : (o.trace_mode == RBRT_TRACE_BRUTE ? (uint32_t)grid_fin * 256u : (1u << 18)));
        const bool brute = o.trace_mode == RBRT_TRACE_BRUTE;
        const bool et = rp.dev.n_etris > 0;                               // BasicTriangle elements present: the ET kernel instantiations
        const bool count = (o.flags & RBRT_OPT_COUNT_VISITS) != 0;
        const bool time_kernels = (o.flags & RBRT_OPT_TIME_KERNELS) != 0;      // bracket every trace launch with events -> stats.ms_trace
        // The launch sequence of a batch is fixed on the host, but how fast its rays die out is only known on the device: the hand-over
        // to the tail kernel becomes unconditional at iteration `force_it`, where the sequence ends.  Rays roughly halve per bounce, so
        // the threshold (2^18 rays) is expected near log2(paths / 2^18); two iterations of slack, at most TAIL_FORCE_IT.  (A 1/8 shard
        // of C3 hands over at iteration 6; with the fixed 12 it then ran 18 launches that found the "tail done" flag and returned.)
        uint32_t force_it = TAIL_FORCE_IT;
        {
            const char* fenv = getenv("RBRT_TAIL_FORCE_IT");               // tuning knob
            uint32_t lg = 0; while (lg < 31 && ((uint64_t)cap >> lg) > (1ull << 18)) ++lg;
            const uint32_t guess = lg + 2 < 2 ? 2 : lg + 2;
            force_it = fenv ? (uint32_t)std::max(1, atoi(fenv)) : std::min<uint32_t>(TAIL_FORCE_IT, guess);
            if (brute) force_it = TAIL_FORCE_IT;
        }
        size_t ev_used = 0;
        auto next_event = [&]() -> cudaEvent_t {
            if (ev_used == wb.ev.size()) { cudaEvent_t e = nullptr; cudaEventCreate(&e); wb.ev.push_back(e); }
            return wb.ev[ev_used++];
        };
        uint32_t batch_no = 0;
        for (uint32_t s_base = sh.s0; s_base < sh.s1; s_base += S_b, ++batch_no) {
            const int l = split ? (int)(batch_no & 1u) : 0;
            WaveParams& wp = wps[l];
            cudaStream_t bs = lane_st[l];
            wp.s_base = s_base; wp.s_count = (sh.s1 - s_base < S_b) ? sh.s1 - s_base : S_b;
            wp.fd_s_count = make_fastdiv(wp.s_count);
            CKR(cudaMemsetAsync(wbs[l]->ctr, 0, sizeof(IterCtr) * (max_depth + 2), bs));
            if (et) k_generate<true><<<grid, 256, 0, bs>>>(wp); else k_generate<false><<<grid, 256, 0, bs>>>(wp);
            ++launches;
            batch_iters = 0;
            // A scene without mesh triangles (C1) has nothing to traverse: every closest-hit query is resolved by stage A inside the
            // kernel that produced the ray, so the whole path runs in ONE lane of the tail kernel right after k_generate
            // (5 launches per frame instead of 40; C1 is launch-bound).
            const bool no_mesh = sc.info.num_triangles_tested == 0;
            for (uint32_t it = 0; it <= max_depth; ++it) {
                if ((it >= 1 || no_mesh) && tail_rays) {                   // see k_finish / k_tail
                    const bool force = it >= force_it || no_mesh;
                    const uint32_t lim = force ? 0xFFFFFFFFu : tail_rays;
                    if (brute) {
                        if (et) { if (count) k_finish<true, true, true><<<grid_fin, 256, 0, bs>>>(wp, it, lim); else k_finish<true, false, true><<<grid_fin, 256, 0, bs>>>(wp, it, lim); }
                        else { if (count) k_finish<true, true, false><<<grid_fin, 256, 0, bs>>>(wp, it, lim); else k_finish<true, false, false><<<grid_fin, 256, 0, bs>>>(wp, it, lim); }
                    } else if (et) { if (count) k_tail<true, true><<<grid_tail, TAIL_THREADS, 0, bs>>>(wp, it, lim); else k_tail<false, true><<<grid_tail, TAIL_THREADS, 0, bs>>>(wp, it, lim); }
                    else { if (count) k_tail<true, false><<<grid_tail, TAIL_THREADS, 0, bs>>>(wp, it, lim); else k_tail<false, false><<<grid_tail, TAIL_THREADS, 0, bs>>>(wp, it, lim); }
                    ++launches;
                    if (force) break;
                }
                if (time_kernels) CKR(cudaEventRecord(next_event(), bs));
                if (brute) { if (count) k_trace_brute<true><<<grid, 256, 0, bs>>>(wp, it); else k_trace_brute<false><<<grid, 256, 0, bs>>>(wp, it); }
                else if (count) k_trace<true><<<grid_trace, TRACE_THREADS, 0, bs>>>(wp, it);
                else k_trace<false><<<grid_trace, TRACE_THREADS, 0, bs>>>(wp, it);
                ++launches; ++iterations; ++batch_iters; ++lane_iters[l];
                if (time_kernels) CKR(cudaEventRecord(next_event(), bs));
                if (it < max_depth) { if (et) k_shade<true><<<grid, 256, 0, bs>>>(wp, it); else k_shade<false><<<grid, 256, 0, bs>>>(wp, it); ++launches; }
            }
            if (split && batch_no > 0) CKR(cudaStreamWaitEvent(bs, SL.acc[l ^ 1], 0));   // sample order: after the previous batch's accumulate (other lane)
            k_accumulate<<<dim3((P + 255) / 256, n_frames), 256, 0, bs>>>(wp, ap); ++launches;
            if (split) CKR(cudaEventRecord(SL.acc[l], bs));
            k_sum_rays<<<1, 64, 0, bs>>>(wp); ++launches;
            CKR(cudaGetLastError());
        }
        if (split) {                                                      // join: the caller's stream continues behind the second lane
            CKR(cudaEventRecord(SL.join, SL.aux));
            CKR(cudaStreamWaitEvent(st, SL.join, 0));
        }
    }
    CKR(cudaEventRecord(ev1, st));
    note_scene_use(sc, rp.device, st);
    job.wb = &wb; job.wb2 = split ? wbs[1] : nullptr; job.sh = sh; job.P = P; job.n_frames = n_frames; job.W = W; job.H = H; job.launches = launches; job.iterations = iterations;
    job.batch_iters = batch_iters; job.flags = o.flags; job.max_depth = max_depth; job.rendered = P && sh.s1 > sh.s0;
    if (stats && !job_out) return collect_stats(job, stats);
    return RBRT_OK;
}

int collect_stats(RenderJob& job, rbrt_stats* stats) {
    WaveBuffers& wb = *job.wb;
    const ShardDev& sh = job.sh;
    const uint32_t W = job.W, H = job.H, iterations = job.iterations, max_depth = job.max_depth;
    const cudaEvent_t ev0 = job.ev0, ev1 = job.ev1;
    {
        CKR(cudaEventSynchronize(ev1));
        float ms = 0; CKR(cudaEventElapsedTime(&ms, ev0, ev1));
        unsigned long long h[ST_COUNT] = {0, 0, 0, 0, 0, 0, 0, 0};
        if (wb.stats && job.rendered) CKR(cudaMemcpy(h, wb.stats, sizeof(h), cudaMemcpyDeviceToHost));
        if (job.wb2 && job.wb2->stats && job.rendered) {                  // second lane (RBRT_OPT_SPLIT_BATCHES)
            unsigned long long h2[ST_COUNT];
            CKR(cudaMemcpy(h2, job.wb2->stats, sizeof(h2), cudaMemcpyDeviceToHost));
            for (int k = 0; k < ST_COUNT; ++k) h[k] += h2[k];
        }
        stats->rays = h[ST_RAYS]; stats->nan_rays = h[ST_NAN]; stats->node_visits = h[ST_NODES]; stats->tri_tests = h[ST_TRIS] + h[ST_TAIL_TRIS]; stats->traversed_rays = h[ST_CAND] + h[ST_TAIL_CAND];
        stats->node_visits += h[ST_TAIL_NODES];
        stats->tail_node_visits = h[ST_TAIL_NODES]; stats->tail_tri_tests = h[ST_TAIL_TRIS]; stats->tail_traversed_rays = h[ST_TAIL_CAND];
        uint64_t valid_px = 0;
        for (uint32_t tj = 0; tj < sh.tiles_mine; ++tj) {
            uint32_t T = tj * sh.count + sh.rank, ty = T / sh.tiles_x, tx = T - ty * sh.tiles_x;
            uint32_t w = W - tx * 8 < 8 ? W - tx * 8 : 8, hh = H - ty * 4 < 4 ? H - ty * 4 : 4;
            valid_px += (uint64_t)w * hh;
        }
        stats->paths = valid_px * (sh.s1 - sh.s0) * job.n_frames;
        stats->ms_device = ms; stats->launches = job.launches; stats->iterations = iterations;
        if (job.rendered && (job.flags & RBRT_OPT_TIME_KERNELS)) {
            double tr = 0;
            for (size_t i = 0; i + 1 < wb.ev.size() && i + 1 < 2ull * iterations; i += 2) {
                float t = 0; CKR(cudaEventElapsedTime(&t, wb.ev[i], wb.ev[i + 1])); tr += t;
            }
            stats->ms_trace = tr;
            if (getenv("RBRT_DEBUG_ITERS")) {                              // per-iteration trace time + queue sizes of the LAST batch
                std::vector<IterCtr> hc(max_depth + 2);
                CKR(cudaMemcpy(hc.data(), wb.ctr, sizeof(IterCtr) * (max_depth + 2), cudaMemcpyDeviceToHost));
                size_t per_batch = job.batch_iters, first = 2 * (iterations - per_batch);
                float t_first = 0; cudaEventElapsedTime(&t_first, ev0, wb.ev[first]);
                fprintf(stderr, "setup + generate (ev0 -> first trace): %.3f ms; tail kernel ran at it %d\n", t_first, (int)hc[0].pad - 1);
                for (uint32_t it = 0; it < per_batch; ++it) {
                    float t = 0, g = 0; cudaEventElapsedTime(&t, wb.ev[first + 2 * it], wb.ev[first + 2 * it + 1]);
                    if (it + 1 < per_batch) cudaEventElapsedTime(&g, wb.ev[first + 2 * it + 1], wb.ev[first + 2 * it + 2]);
                    else cudaEventElapsedTime(&g, wb.ev[first + 2 * it + 1], ev1);
                    fprintf(stderr, "it %2u rays %9u traversed %9u  lambert %9u metal %9u glass %9u  trace %8.3f ms  then shade+finish %8.3f ms\n", it, hc[it].ray_count,
                            hc[it].cand_count, hc[it].mat_count[0], hc[it].mat_count[1], hc[it].mat_count[2], t, g);
                }
            }
        }
    }
    return RBRT_OK;
}

int finalize(const float4* d_accum, uint32_t W, uint32_t H, uint32_t spp, uint8_t* d_rgb, float* d_hdr, cudaStream_t st) {
    size_t n = (size_t)W * H;
    if (!n || !spp) { set_error("empty image or zero samples"); return RBRT_E_INVALID; }
    float inv = 1.0f / (float)spp;                                        // lib.rs:101
    k_finalize<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_accum, n, inv, d_rgb, d_hdr);
    CKR(cudaGetLastError());
    return RBRT_OK;
}

int trace_rays_device(const Scene& sc, const rbrt_ray* d_rays, uint64_t n, uint32_t mode, rbrt_hit* d_hits,
                      unsigned long long* d_stats, cudaStream_t st) {
    if (!n) return RBRT_OK;
    wait_scene_ready(sc, 0, st);
    unsigned g = (unsigned)((n + 255) / 256);
    if (mode == RBRT_TRACE_BRUTE) k_trace_rays<true><<<g, 256, 0, st>>>(sc.dev, d_rays, n, d_hits, d_stats);
    else k_trace_rays<false><<<g, 256, 0, st>>>(sc.dev, d_rays, n, d_hits, d_stats);
    CKR(cudaGetLastError());
    return RBRT_OK;
}

int scatter_device(const rbrt_scatter_in* d_in, uint64_t n, uint64_t seed, rbrt_scatter_out* d_out, cudaStream_t st) {
    if (!n) return RBRT_OK;
    k_scatter_kat<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_in, n, (uint32_t)seed, (uint32_t)(seed >> 32), d_out);
    CKR(cudaGetLastError());
    return RBRT_OK;
}

// RBRT_TRACE_WAVEFRONT: the caller's rays through stage A + k_trace (see k_rays_stage_a).  Uses wavefront pool 0 of the device.
int trace_rays_wavefront(const Scene& sc, const rbrt_ray* d_rays, uint64_t n, rbrt_hit* d_hits, unsigned long long* d_stats, cudaStream_t st) {
    const Replica& rp = sc.rep[0];
    WaveBuffers& wb = device_wave_buffers(rp.device, 0);
    wait_scene_ready(sc, 0, st);
    const uint64_t chunk = 1ull << 24;
    static int per_sm_cached = 0;
    if (!per_sm_cached) CKR(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_cached, k_trace<false>, TRACE_THREADS, 0));
    const bool et = rp.dev.n_etris > 0;
    for (uint64_t base = 0; base < n; base += chunk) {
        const uint32_t m = (uint32_t)std::min<uint64_t>(chunk, n - base);
        const uint32_t cap = (m + 31u) & ~31u;
        int rc = ensure_wave_buffers(wb, std::max<uint32_t>(cap, 1u << 16), 50);
        if (rc) return rc;
        WaveParams wp;
        memset(&wp, 0, sizeof(wp));
        wp.S = rp.dev; wp.n_frames = 1; wp.cap = wb.cap; wp.paths_px = cap; wp.fd_paths_px = make_fastdiv(cap); wp.fd_s_count = make_fastdiv(1);
        wp.s_count = 1; wp.max_depth = 50; wp.fetch_thr = FETCH_THRESHOLD; wp.tail_thr = TAIL_FETCH_THRESHOLD; wp.keep_t = 1u;
        wp.rec = wb.rec; wp.candq = wb.candq;
        for (int i = 0; i < 6; ++i) wp.matq[i / 3][i % 3] = wb.matq[i / 3][i % 3];
        wp.out = wb.out; wp.hist = wb.hist; wp.ctr = wb.ctr; wp.stats = wb.stats;
        CKR(cudaMemsetAsync(wb.ctr, 0, sizeof(IterCtr) * 52, st));
        CKR(cudaMemsetAsync(wb.stats, 0, 8 * ST_COUNT, st));
        CKR(cudaMemsetAsync(wb.out, 0xFF, 16ull * cap, st));
        const int grid = rp.sm_count * 8;
        if (et) k_rays_stage_a<true><<<grid, 256, 0, st>>>(wp, d_rays + base, m); else k_rays_stage_a<false><<<grid, 256, 0, st>>>(wp, d_rays + base, m);
        if (d_stats) k_trace<true><<<rp.sm_count * std::max(per_sm_cached, 1), TRACE_THREADS, 0, st>>>(wp, 0);
        else k_trace<false><<<rp.sm_count * std::max(per_sm_cached, 1), TRACE_THREADS, 0, st>>>(wp, 0);
        k_rays_collect<<<(m + 255) / 256, 256, 0, st>>>(wp, d_rays + base, m, d_hits + base);
        CKR(cudaGetLastError());
        if (d_stats) {                                                    // accumulate this chunk's counters into the caller's block
            CKR(cudaStreamSynchronize(st));
            unsigned long long h[ST_COUNT], acc[ST_COUNT];
            CKR(cudaMemcpy(h, wb.stats, sizeof(h), cudaMemcpyDeviceToHost));
            CKR(cudaMemcpy(acc, d_stats, sizeof(acc), cudaMemcpyDeviceToHost));
            for (int k = 0; k < ST_COUNT; ++k) acc[k] += h[k];
            CKR(cudaMemcpy(d_stats, acc, sizeof(acc), cudaMemcpyHostToDevice));
        }
    }
    note_scene_use(sc, rp.device, st);
    return RBRT_OK;
}

int primary_rays_device(const rbrt_camera& cam, uint64_t seed, uint32_t sample, rbrt_ray* d_rays, cudaStream_t st) {
    size_t n = (size_t)cam.img_width_pix * cam.img_height_pix;
    if (!n) return RBRT_OK;
    k_primary_rays<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(make_cam(cam), (uint32_t)seed, (uint32_t)(seed >> 32), sample, d_rays);
    CKR(cudaGetLastError());
    return RBRT_OK;
}

}  // namespace rbrt
