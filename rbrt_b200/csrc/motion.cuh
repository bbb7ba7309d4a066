// motion.cuh — per-object motion vectors (rbrt_gpu_scene_snapshot, rbrt_gpu_render_motion*; include/rbrt_gpu.h, DESIGN.md section 16):
// steps 3-5 of the motion pass as __host__ __device__ code, and the launch interface of the module that runs it (motion.cu, built into
// librbrt_gpu_motion.so).
//
// mv_pixel below IS the definition of what a hit pixel reports: the kernel calls it with the hit element's current and snapshot records,
// tests/host_device/motion_harness.cpp compiles it with g++ for the host, and tests/motion_ref.py restates it in numpy.  The camera
// arithmetic is temporal.cuh's (tp_pixel_dir, tp_project), so the motion pass lines up with step 3 of the temporal accumulation.
// Every operation is one IEEE f32 operation, correctly rounded, or a compare of bit patterns.
#pragma once
#include "../../include/rbrt_gpu.h"
#include <string.h>
#include "temporal.cuh"

namespace rbrt {

enum { MV_ST_NAN = 0, MV_ST_NODES = 1, MV_ST_TRIS = 2, MV_ST_COUNT = 3 };

// A scene's snapshot (rbrt_gpu_scene_snapshot): one device block owned by the scene.
struct SnapshotDev {
    float4* tris;                // 3 per tested mesh triangle at index tri_base + ORIGINAL triangle index: the record {v0|orig, e1, e2}
                                 // of SceneDev::tris (whose slots follow the BVH order, which RBRT_UPDATE_REBUILD permutes)
    float4* elems;               // per element: SceneDev::spheres' record (sphere {c, r}; BasicTriangle {bits(index into etris)})
    float4* etris;               // 3 per BasicTriangle: v0, e1, e2 of SceneDev::etris (the values its intersection test reads)
};

struct SnapshotArgs {
    SceneDev S;                  // replica 0 of the scene
    SnapshotDev snap;
    uint32_t blocks;             // grid-stride launch
};

struct MotionArgs {
    SceneDev S;                  // replica 0 of the scene
    SnapshotDev snap;            // the latest snapshot (read only)
    CamDev cam;                  // the current frame's camera
    CamDev prev;                 // the history's camera
    uint32_t tiles_x, tiles_total;   // 8x4-pixel tiles of the image: one warp per tile, one lane per pixel
    rbrt_motion_out out;         // device planes; a NULL member is not written
    unsigned long long* stats;   // MV_ST_COUNT counters, or NULL (no counting)
};

// Bit patterns of f32 values (the device intrinsics are device-only).
__host__ __device__ __forceinline__ uint32_t mv_bits(float f) {
#ifdef __CUDA_ARCH__
    return __float_as_uint(f);
#else
    uint32_t u; memcpy(&u, &f, 4); return u;
#endif
}
__host__ __device__ __forceinline__ float mv_nan() {
#ifdef __CUDA_ARCH__
    return __uint_as_float(0x7FC00000u);
#else
    const uint32_t u = 0x7FC00000u; float f; memcpy(&f, &u, 4); return f;
#endif
}
__host__ __device__ __forceinline__ bool mv_same(float4 a, float4 b, bool w) {
    return mv_bits(a.x) == mv_bits(b.x) && mv_bits(a.y) == mv_bits(b.y) && mv_bits(a.z) == mv_bits(b.z) && (!w || mv_bits(a.w) == mv_bits(b.w));
}
__host__ __device__ __forceinline__ f3 mv_xyz(float4 a) { return mk3(a.x, a.y, a.z); }

// Steps 3-5 for a hit at parameter t of the ray (o, d) of the current camera.  tri: the hit element is a mesh triangle or a BasicTriangle,
// cur / old its current and snapshot records v0, e1, e2 (xyz); otherwise a sphere, cur[0] / old[0] = {c, r}.
//  3. P = o + t * d per component.
//  4. P' = P when the element is unchanged: v0, e1, e2 (sphere: c and r) bit for bit equal to the snapshot's.  Otherwise, for a triangle,
//     u and v as the Moller-Trumbore test computes them for the current record (h = d x e2, a = e1 . h, f = 1 / a, s = o - v0,
//     u = f * (s . h), q = s x e1, v = f * (d . q)) and P' = (v0' + u * e1') + v * e2'; for a sphere P' = c' + (P - c) * (r' / r).
//  5. q = tp_project(cam, P - pos), q' = tp_project(prev, P' - pos'); motion = q' - q per component, (NaN, NaN) when either projection
//     fails or a coordinate is not finite; prev_dist = sqrt(D' . D'), D' = P' - pos'.
__host__ __device__ __forceinline__ void mv_pixel(const CamDev& cam, const CamDev& prev, bool tri, f3 o, f3 d, float t, const float4* cur,
                                                  const float4* old, float* mx, float* my, float* prev_dist) {
    const f3 P = mk3(XADD(o.x, XMUL(t, d.x)), XADD(o.y, XMUL(t, d.y)), XADD(o.z, XMUL(t, d.z)));
    f3 Pp = P;
    if (tri) {
        if (!(mv_same(cur[0], old[0], false) && mv_same(cur[1], old[1], false) && mv_same(cur[2], old[2], false))) {
            const f3 v0 = mv_xyz(cur[0]), e1 = mv_xyz(cur[1]), e2 = mv_xyz(cur[2]);
            const f3 h = tp_cross(d, e2);
            const float f = XDIV(1.0f, tp_dot(e1, h));
            const f3 s = tp_sub(o, v0);
            const float u = XMUL(f, tp_dot(s, h));
            const float v = XMUL(f, tp_dot(d, tp_cross(s, e1)));
            const f3 w0 = mv_xyz(old[0]), w1 = mv_xyz(old[1]), w2 = mv_xyz(old[2]);
            Pp = mk3(XADD(XADD(w0.x, XMUL(u, w1.x)), XMUL(v, w2.x)), XADD(XADD(w0.y, XMUL(u, w1.y)), XMUL(v, w2.y)),
                     XADD(XADD(w0.z, XMUL(u, w1.z)), XMUL(v, w2.z)));
        }
    } else if (!mv_same(cur[0], old[0], true)) {
        const float k = XDIV(old[0].w, cur[0].w);
        Pp = mk3(XADD(old[0].x, XMUL(XSUB(P.x, cur[0].x), k)), XADD(old[0].y, XMUL(XSUB(P.y, cur[0].y), k)),
                 XADD(old[0].z, XMUL(XSUB(P.z, cur[0].z), k)));
    }
    const f3 Dp = tp_sub(Pp, tp_v(prev.pos));
    float qx, qy, px, py;
    const bool ok_q = tp_project(cam, tp_sub(P, tp_v(cam.pos)), &qx, &qy);
    const bool ok_p = tp_project(prev, Dp, &px, &py);
    if (ok_q && ok_p && dn_finite(qx) && dn_finite(qy) && dn_finite(px) && dn_finite(py)) {
        *mx = XSUB(px, qx); *my = XSUB(py, qy);
    } else {
        *mx = mv_nan(); *my = mv_nan();
    }
    *prev_dist = XSQRT(tp_dot(Dp, Dp));
}

}  // namespace rbrt

#ifdef __CUDACC__                                                         // (not in the host build of the tests)
extern "C" {
// Enqueues the snapshot of args->S into args->snap on `stream`; returns a cudaError_t.
typedef int (*rbrt_snapshot_launch_fn)(const rbrt::SnapshotArgs* args, cudaStream_t stream);
// Enqueues the motion pass on `stream`; returns a cudaError_t.
typedef int (*rbrt_motion_launch_fn)(const rbrt::MotionArgs* args, cudaStream_t stream);
}
#endif
