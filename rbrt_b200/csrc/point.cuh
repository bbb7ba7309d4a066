// point.cuh — nearest-surface queries on device memory (rbrt_gpu_query_nearest_device, DESIGN.md section 17).
// The per-candidate routines (the closest point of one triangle record or one sphere), the point-to-box lower bound and the prune bound of
// the traversal, and the launch interface of the point module (point.cu, built into librbrt_gpu_point.so, which librbrt_gpu.so loads at
// run time).  Every f32 operation of the routines is written out with XMUL / XADD / XSUB / XDIV / XSQRT, so the host build of this header
// (tests/host_device/point_harness.cpp) and the device build agree bit for bit, and tests/point_ref.py restates them op for op.
#pragma once
#include "../../include/rbrt_gpu.h"
#include "common.cuh"

namespace rbrt {

enum { PT_ST_HEAD = 0, PT_ST_NAN = 1, PT_ST_NODES = 2, PT_ST_TRIS = 3, PT_ST_COUNT = 4 };

struct PointArgs {
    SceneDev S;                  // replica 0 of the scene
    const float* points;         // n points, xyz, device memory
    uint64_t n;                  // < 2^32
    const float* max_dist;       // n bounds, or NULL = +inf
    rbrt_nearest_out out;        // device planes, a NULL member is not written
    unsigned long long* ctr;     // PT_ST_COUNT counters, zeroed before the launch: [PT_ST_HEAD] is the point cursor
    int count;                   // also fill PT_ST_NAN / NODES / TRIS
    uint32_t blocks;             // persistent grid
};

// ------------------------------------------------------------------ one candidate
// The closest point q of the real triangle v0 + u*e1 + v*e2 (u, v >= 0, u + v <= 1) to p, its (u, v), and d2 = dot3(p - q, p - q).
// Ericson's ClosestPtPointTriangle (Real-Time Collision Detection, 5.1.5) on the record: the vertex regions of a, b, c, the edge regions of
// ab, ac, bc, then the face.  b - p and c - p are formed from ap = p - v0 as ap - e1 and ap - e2, so the routine reads nothing but the record.
//   a:  q = v0                (0, 0)         ab: q = v0 + u*e1   (u, 0)         bc and face: q = (v0 + u*e1) + v*e2
//   b:  q = v0 + e1           (1, 0)         ac: q = v0 + v*e2   (0, v)
//   c:  q = v0 + e2           (0, 1)
// Degenerate records: when cross3(e1, e2) is exactly zero (collinear vertices, a zero-length edge, three equal vertices) the triangle is the
// segment or point it collapses to, and q is the closest of the three segments ab, ac, bc (pt_segments, first minimum in that order).  The
// edge parameters divide by a sum of two terms of the same sign that is 0 only when both are (then the parameter is 0); the face divides
// by va + vb + vc only when all three are >= 0 and the sum > 0, else (rounding on a sliver, an overflowed product) the segments decide.
// So no input made of finite values gives a NaN; NaN or inf in p or the record gives a non-finite d2, which is never recorded.
__device__ __forceinline__ float pt_seg(f3 ap, f3 e, float& t) {   // parameter of the closest point of the segment 0 + t*e to ap
    const float ee = dot3(e, e);
    const float x = ee > 0.0f ? XDIV(dot3(ap, e), ee) : 0.0f;
    t = x > 0.0f ? (x < 1.0f ? x : 1.0f) : 0.0f;                          // (a NaN quotient and -0 give +0)
    return ee;
}
__device__ __forceinline__ f3 pt_q(f3 v0, f3 e1, f3 e2, float u, float v) {   // (v0 + u*e1) + v*e2
    return mk3(XADD(XADD(v0.x, XMUL(u, e1.x)), XMUL(v, e2.x)), XADD(XADD(v0.y, XMUL(u, e1.y)), XMUL(v, e2.y)),
               XADD(XADD(v0.z, XMUL(u, e1.z)), XMUL(v, e2.z)));
}
__device__ __forceinline__ float pt_d2(f3 p, f3 q) {
    const f3 w = mk3(XSUB(p.x, q.x), XSUB(p.y, q.y), XSUB(p.z, q.z));
    return dot3(w, w);
}
// The segments of a degenerate record: ab (u, 0), ac (0, v), bc (1 - w, w); the first of equal d2 wins.
__device__ __forceinline__ float pt_segments(f3 p, f3 v0, f3 e1, f3 e2, f3 ap, f3& q, float& u, float& v) {
    float t;
    pt_seg(ap, e1, t);
    f3 qa = mk3(XADD(v0.x, XMUL(t, e1.x)), XADD(v0.y, XMUL(t, e1.y)), XADD(v0.z, XMUL(t, e1.z)));
    float best = pt_d2(p, qa), bu = t, bv = 0.0f;
    q = qa;
    pt_seg(ap, e2, t);
    qa = mk3(XADD(v0.x, XMUL(t, e2.x)), XADD(v0.y, XMUL(t, e2.y)), XADD(v0.z, XMUL(t, e2.z)));
    float d = pt_d2(p, qa);
    if (d < best) { best = d; bu = 0.0f; bv = t; q = qa; }
    const f3 bc = mk3(XSUB(e2.x, e1.x), XSUB(e2.y, e1.y), XSUB(e2.z, e1.z));
    const f3 bp = mk3(XSUB(ap.x, e1.x), XSUB(ap.y, e1.y), XSUB(ap.z, e1.z));
    pt_seg(bp, bc, t);
    const float w1 = XSUB(1.0f, t);
    qa = pt_q(v0, e1, e2, w1, t);
    d = pt_d2(p, qa);
    if (d < best) { best = d; bu = w1; bv = t; q = qa; }
    u = bu; v = bv;
    return best;
}
__device__ __forceinline__ float closest_on_triangle(f3 p, f3 v0, f3 e1, f3 e2, f3& q, float& u, float& v) {
    const f3 ap = mk3(XSUB(p.x, v0.x), XSUB(p.y, v0.y), XSUB(p.z, v0.z));
    const f3 n = cross3(e1, e2);
    if (n.x == 0.0f && n.y == 0.0f && n.z == 0.0f) return pt_segments(p, v0, e1, e2, ap, q, u, v);
    const float d1 = dot3(e1, ap), d2 = dot3(e2, ap);
    if (d1 <= 0.0f && d2 <= 0.0f) { q = v0; u = 0.0f; v = 0.0f; return pt_d2(p, q); }
    const f3 bp = mk3(XSUB(ap.x, e1.x), XSUB(ap.y, e1.y), XSUB(ap.z, e1.z));
    const float d3 = dot3(e1, bp), d4 = dot3(e2, bp);
    if (d3 >= 0.0f && d4 <= d3) { q = mk3(XADD(v0.x, e1.x), XADD(v0.y, e1.y), XADD(v0.z, e1.z)); u = 1.0f; v = 0.0f; return pt_d2(p, q); }
    const float vc = XSUB(XMUL(d1, d4), XMUL(d3, d2));
    if (vc <= 0.0f && d1 >= 0.0f && d3 <= 0.0f) {
        const float s = XSUB(d1, d3);
        u = s > 0.0f ? XDIV(d1, s) : 0.0f; v = 0.0f;
        q = mk3(XADD(v0.x, XMUL(u, e1.x)), XADD(v0.y, XMUL(u, e1.y)), XADD(v0.z, XMUL(u, e1.z)));
        return pt_d2(p, q);
    }
    const f3 cp = mk3(XSUB(ap.x, e2.x), XSUB(ap.y, e2.y), XSUB(ap.z, e2.z));
    const float d5 = dot3(e1, cp), d6 = dot3(e2, cp);
    if (d6 >= 0.0f && d5 <= d6) { q = mk3(XADD(v0.x, e2.x), XADD(v0.y, e2.y), XADD(v0.z, e2.z)); u = 0.0f; v = 1.0f; return pt_d2(p, q); }
    const float vb = XSUB(XMUL(d5, d2), XMUL(d1, d6));
    if (vb <= 0.0f && d2 >= 0.0f && d6 <= 0.0f) {
        const float s = XSUB(d2, d6);
        u = 0.0f; v = s > 0.0f ? XDIV(d2, s) : 0.0f;
        q = mk3(XADD(v0.x, XMUL(v, e2.x)), XADD(v0.y, XMUL(v, e2.y)), XADD(v0.z, XMUL(v, e2.z)));
        return pt_d2(p, q);
    }
    const float va = XSUB(XMUL(d3, d6), XMUL(d5, d4));
    const float x = XSUB(d4, d3), y = XSUB(d5, d6);
    if (va <= 0.0f && x >= 0.0f && y >= 0.0f) {
        const float s = XADD(x, y);
        const float w = s > 0.0f ? XDIV(x, s) : 0.0f;
        u = XSUB(1.0f, w); v = w;
        q = pt_q(v0, e1, e2, u, v);
        return pt_d2(p, q);
    }
    const float s = XADD(XADD(va, vb), vc);
    if (va >= 0.0f && vb >= 0.0f && vc >= 0.0f && s > 0.0f) {            // the face: u, v in [0, 1] (each term <= s)
        u = XDIV(vb, s); v = XDIV(vc, s);
        q = pt_q(v0, e1, e2, u, v);
        return pt_d2(p, q);
    }
    return pt_segments(p, v0, e1, e2, ap, q, u, v);
}

// The closest point of the sphere |x - c| = |r| (a negative radius is the same surface, r = 0 the point c):
// q = c + (p - c) * (|r| / |p - c|) per component, and q = c + (|r|, 0, 0) when p = c.
__device__ __forceinline__ float closest_on_sphere(f3 p, float4 s, f3& q) {
    const float r = fabsf(s.w);
    const f3 w = mk3(XSUB(p.x, s.x), XSUB(p.y, s.y), XSUB(p.z, s.z));
    const float l = len3(w);
    if (l == 0.0f) q = mk3(XADD(s.x, r), XADD(s.y, 0.0f), XADD(s.z, 0.0f));
    else {
        const float k = XDIV(r, l);
        q = mk3(XADD(s.x, XMUL(w.x, k)), XADD(s.y, XMUL(w.y, k)), XADD(s.z, XMUL(w.z, k)));
    }
    return pt_d2(p, q);
}

// d2 is a candidate: finite, and its distance sqrt_rn(d2) below max_dist (strict; a NaN max_dist accepts nothing).
__device__ __forceinline__ bool pt_accept(float d2, float max_dist) {
    return d2 <= 3.40282347e+38f && XSQRT(d2) < max_dist;
}

// ------------------------------------------------------------------ pruning (DESIGN.md section 17)
// Lower bound of the squared distance from p to the box [lo, hi]: per axis the gap max(lo - p, p - hi, 0), then (gx*gx + gy*gy) + gz*gz.
// fmaxf ignores NaN, so an axis whose bounds are NaN (qstep = NaN, common.cuh) contributes 0: never NaN, never a rejection.
__device__ __forceinline__ float pt_gap(float lo, float hi, float p) { return fmaxf(fmaxf(XSUB(lo, p), XSUB(p, hi)), 0.0f); }
__device__ __forceinline__ float pt_box_d2(f3 p, float lx, float ly, float lz, float hx, float hy, float hz) {
    const float gx = pt_gap(lx, hx, p.x), gy = pt_gap(ly, hy, p.y), gz = pt_gap(lz, hz, p.z);
    return XADD(XADD(XMUL(gx, gx), XMUL(gy, gy)), XMUL(gz, gz));
}

// The prune bound: a box whose lower bound exceeds it holds no triangle that can be recorded.  b = min(max_dist, sqrt(best d2)) bounds the
// distance of anything that can still be recorded; s = max(|p|, the mesh's largest |coordinate|) (per axis, max over lo and hi of the exact
// mesh box), u = 2^-23 * s.
//   prune_d2 = ((b * 1.0001 + 64 u) + 1e-18)^2
// PROOF that it is conservative (eps = 2^-24, every f32 operation rounds to nearest, and rounding is monotone).  Let T be the real triangle
// {v0 + u e1 + v e2} of a tested record in the box B, D = dist(p, T), and d2 the routine's result for it.
//  (1) T lies within u of the mesh box on every axis: v0 is a vertex, v0 + e1 differs from the vertex b by |a + fl(b - a) - b| <= eps |b - a|
//      <= 2 eps s = u, likewise c.  The node boxes contain the exact box of each vertex triple (the leaf box min - pad / max + pad, and
//      quant_lo / quant_hi check fmaf(q, qstep, qorg) against it: the decode below is that fmaf).  So D >= dist(p, B) - sqrt(3) u, for the
//      node boxes and for the exact mesh box of the pre-test alike.
//  (2) The routine's q is within 11 u per axis of a point of T: its u, v lie in [0, 1] with u + v <= 1 + 5 eps (each edge and face
//      parameter is a quotient of a non-negative term by a sum that contains it, or a clamped segment parameter), and forming
//      (v0 + u e1) + v e2 from |v0| <= s, |e| <= 2 s (1 + eps) rounds by at most 12 eps s = 6 u; being off T by the excess of u + v adds
//      at most 5 u.  So |p - q| >= D - 20 u.
//  (3) d2 >= |p - q|^2 (1 - eps)^5 (a rounded difference, three squares, two sums), and the box bound is at most dist(p, B)^2 (1 + eps)^5.
// A recorded candidate needs sqrt(d2) <= sqrt(best d2) or sqrt_rn(d2) < max_dist, so sqrt(d2) <= b (1 + eps).  Chaining (1)-(3):
// sqrt(box bound) <= (sqrt(d2) (1 - eps)^-2.5 + 22 u) (1 + eps)^2.5 <= b (1 + 7 eps) + 23 u, which is below sqrt(prune_d2) even after the
// four roundings of prune_d2 (b * 1.0001 leaves 1e-4 b of room, 64 u leaves 41 u).  Equal d2 are covered (<=), so ties are never pruned.
// Underflow: the term 1e-18 keeps prune_d2 >= 1e-36, a normal number, so the absolute errors of subnormal squares (2^-149 each) are far
// below the room left; u itself may underflow to 0.  An infinite or NaN s (a mesh with inf coordinates) makes prune_d2 inf or NaN, and
// nothing is pruned.
__device__ __forceinline__ float pt_prune_d2(float max_dist, float best_d2, float s) {
    const float b = fminf(max_dist, XSQRT(best_d2));
    const float pd = XADD(XADD(XMUL(b, 1.0001f), XMUL(s, 7.62939453125e-06f)), 1e-18f);   // 64 * 2^-23 = 7.62939453125e-06
    return XMUL(pd, pd);
}
// s of p and a mesh: max(|p.x|, |p.y|, |p.z|, |lo|, |hi|) over the mesh's exact box.
__device__ __forceinline__ float pt_scale(f3 p, const MeshDev& M) {
    float s = fmaxf(fmaxf(fabsf(p.x), fabsf(p.y)), fabsf(p.z));
    for (int k = 0; k < 3; ++k) s = fmaxf(s, fmaxf(fabsf(M.lo[k]), fabsf(M.hi[k])));
    return s;
}

}  // namespace rbrt

#ifdef __CUDACC__                                                         // (not in the host build of the tests)
extern "C" {
// Enqueues the nearest-surface kernel on `stream`; returns a cudaError_t.
typedef int (*rbrt_point_launch_fn)(const rbrt::PointArgs* args, cudaStream_t stream);
}
#endif
