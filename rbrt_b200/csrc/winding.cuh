// winding.cuh — inside tests on device memory: generalized winding numbers (rbrt_gpu_query_winding_device, DESIGN.md section 18).
// The per-candidate terms (the solid angle of one triangle record, the sphere rule), the moments of a subtree's triangles with their merge
// and their far-field expansion, and the launch interfaces of the winding module (wind.cu, built into librbrt_gpu_wind.so, which
// librbrt_gpu.so loads at run time).  Everything here also builds on the host (tests/host_device/winding_harness.cpp), so
// tests/test_winding_host.py checks the same source against float64.
#pragma once
#include "../../include/rbrt_gpu.h"
#include "common.cuh"

namespace rbrt {

enum { WD_ST_HEAD = 0, WD_ST_NAN = 1, WD_ST_NODES = 2, WD_ST_TRIS = 3, WD_ST_COUNT = 4 };

// One moment record, 64 bytes: m[0] = {c, R}, m[1] = {N, T00}, m[2] = {T01, T02, T10, T11}, m[3] = {T12, T20, T21, T22}.
//   c  the area-weighted centroid of the subtree's triangles (the plain mean of their centroids when the area is 0);
//   R  a bound on the distance from c to every vertex of the subtree, rounded up; +inf when a moment is not finite (the subtree is then
//      always descended), -1 for an unused child slot;
//   N  sum of 1/2 (e1 x e2);  T  sum of N_t (x) (c_t - c), T_ij = sum N_t,i (c_t - c)_j (Barill et al. 2018, section 3).
struct WindQueryArgs {
    SceneDev S;                  // replica 0 of the scene
    const float4* mom;           // 4 records per node slot: node j of a mesh, child k at 4 * (4 * (node_base + j) + k)
    const float4* root;          // one record per mesh (4 float4 each)
    const float* points;         // n points, xyz, device memory
    uint64_t n;                  // < 2^32
    float beta;                  // > 1, or +inf
    rbrt_winding_out out;        // device planes, a NULL member is not written
    unsigned long long* ctr;     // WD_ST_COUNT counters, zeroed before the launch: [WD_ST_HEAD] is the point cursor
    int count;                   // also fill WD_ST_NAN / NODES / TRIS
    uint32_t blocks;             // persistent grid
};

// The moments of one mesh (k_wind_moments): its nodes, records and BuildResult in replica 0's block, and scratch for n_eff - 1 nodes.
struct WindMomentArgs {
    const uint4* nodes;          // the mesh's 4-wide nodes
    const float4* tris;          // the mesh's triangle records (tri_base applied)
    const MeshDev* mesh;         // its device record (root_ref is read there: a rebuild writes it)
    const uint32_t* live_nodes;  // its BuildResult's live_nodes
    float4* mom;                 // the mesh's node slot records (node_base applied)
    float4* root;                // the mesh's root record
    uint32_t* parent; uint32_t* need; uint32_t* arrive;   // per node
    double* area;                // per child slot: the area of the subtree's triangles
    uint32_t n_tris;             // N_eff
};

#define WD_FOUR_PI 12.566370614359172
#define WD_TWO_PI 6.283185307179586

// ------------------------------------------------------------------ one candidate
// The solid angle of the triangle record {v0, e1, e2} seen from p (van Oosterom and Strackee 1983), signed by the corner order:
// a = v0 - p, b = a + e1, c = a + e2 in f32; then a, b, c are scaled by one power of two (exact: the angle does not change, and nothing
// overflows or underflows for coordinates anywhere in the f32 range), and
//   Omega = 2 atan2(det, |a||b||c| + (a.b)|c| + (a.c)|b| + (b.c)|a|),  det = a.(b x c).
// det exactly 0 (p in the plane, a degenerate record, p on a vertex) and a non-finite result (inf or NaN values) give 0.
__device__ __forceinline__ float wind_tri(f3 p, f3 v0, f3 e1, f3 e2) {
    f3 a = mk3(XSUB(v0.x, p.x), XSUB(v0.y, p.y), XSUB(v0.z, p.z));
    f3 b = mk3(XADD(a.x, e1.x), XADD(a.y, e1.y), XADD(a.z, e1.z));
    f3 c = mk3(XADD(a.x, e2.x), XADD(a.y, e2.y), XADD(a.z, e2.z));
    const float m = fmaxf(fmaxf(fmaxf(fmaxf(fabsf(a.x), fabsf(a.y)), fmaxf(fabsf(a.z), fabsf(b.x))), fmaxf(fmaxf(fabsf(b.y), fabsf(b.z)),
                          fmaxf(fabsf(c.x), fabsf(c.y)))), fabsf(c.z));
    if (!(m <= 3.40282347e+38f)) return 0.0f;                             // an infinite component (fmaxf skips NaN: caught below)
    // 2^k with the largest component scaled into [1, 2) (into [2, 4) above 2^127; a zero or subnormal m is scaled by 2^127)
    int k = 127 - (int)(__float_as_uint(m) >> 23);
    if (k < -126) k = -126;
    const float s = __uint_as_float((uint32_t)(k + 127) << 23);
    a = mk3(XMUL(a.x, s), XMUL(a.y, s), XMUL(a.z, s));
    b = mk3(XMUL(b.x, s), XMUL(b.y, s), XMUL(b.z, s));
    c = mk3(XMUL(c.x, s), XMUL(c.y, s), XMUL(c.z, s));
    const float det = dot3(a, cross3(b, c));
    if (det == 0.0f) return 0.0f;
    const float la = len3(a), lb = len3(b), lc = len3(c);
    const float den = XADD(XADD(XADD(XMUL(XMUL(la, lb), lc), XMUL(dot3(a, b), lc)), XMUL(dot3(a, c), lb)), XMUL(dot3(b, c), la));
    const float om = XMUL(2.0f, atan2f(det, den));
    return fabsf(om) <= 3.40282347e+38f ? om : 0.0f;
}

// A sphere {c, r} in halves of a full turn: 2 when d2 < r2, 1 when d2 == r2, 0 otherwise (d = p - c, d2 = (dx*dx + dy*dy) + dz*dz,
// r2 = r*r; the sign of r does not matter), and 0 for r = 0.
__device__ __forceinline__ int wind_sphere(f3 p, float4 s) {
    if (s.w == 0.0f) return 0;
    const f3 d = mk3(XSUB(p.x, s.x), XSUB(p.y, s.y), XSUB(p.z, s.z));
    const float d2 = dot3(d, d), r2 = XMUL(s.w, s.w);
    return d2 < r2 ? 2 : (d2 == r2 ? 1 : 0);
}

// ------------------------------------------------------------------ the far field
// r = c - p in f32 and its length l in f64 (no overflow or underflow anywhere in the f32 range).  The child is far from p when
// l > beta R (in f64; beta = +inf is never far, and neither is R = 0 then: the product is NaN).  u = r / l and inv = 1 / l, rounded to f32,
// are what the expansion needs.
__device__ __forceinline__ bool wind_far(f3 p, float4 m0, float beta, f3& u, float& inv) {
    const f3 r = mk3(XSUB(m0.x, p.x), XSUB(m0.y, p.y), XSUB(m0.z, p.z));
    const double l = sqrt(((double)r.x * r.x + (double)r.y * r.y) + (double)r.z * r.z);
    const double il = 1.0 / l;
    u = mk3((float)(r.x * il), (float)(r.y * il), (float)(r.z * il));
    inv = (float)il;
    return l > (double)beta * (double)m0.w;
}
// The expansion of the subtree's solid angle about c through the second derivatives of 1/|x - p| (the terms of N and T), in f32:
//   Omega ~ ((N.u) + (tr T - 3 u.T.u) inv) inv inv.   A non-finite result gives 0.
__device__ __forceinline__ float wind_expand(f3 u, float inv, float4 m1, float4 m2, float4 m3) {
    const f3 t0 = mk3(m1.w, m2.x, m2.y), t1 = mk3(m2.z, m2.w, m3.x), t2 = mk3(m3.y, m3.z, m3.w);   // rows of T
    const float utu = dot3(u, mk3(dot3(t0, u), dot3(t1, u), dot3(t2, u)));
    const float tr = XADD(XADD(m1.w, m2.w), m3.w);
    const float q = XSUB(tr, XMUL(3.0f, utu));
    const float om = XMUL(XMUL(XADD(dot3(mk3(m1.x, m1.y, m1.z), u), XMUL(q, inv)), inv), inv);
    return fabsf(om) <= 3.40282347e+38f ? om : 0.0f;
}

// ------------------------------------------------------------------ moments (float64 inside, float32 records)
// x rounded up to f32 (with a relative margin of 2^-40 for the f64 rounding of x itself).
__device__ __forceinline__ float wind_round_up(double x) {
    x = x * (1.0 + 9.094947017729282e-13);
    float f = (float)x;
    if ((double)f < x) f = nextafterf(f, __uint_as_float(0x7F800000u));
    return f;
}
struct WindMom { double c[3], N[3], T[9], area; float R; };   // a record in f64 (c and R as stored)

// The record of m: c, N and T rounded to f32; R = +inf when any of them is not finite.
__device__ __forceinline__ void wind_store(const WindMom& m, float4* rec) {
    float v[16] = {(float)m.c[0], (float)m.c[1], (float)m.c[2], m.R, (float)m.N[0], (float)m.N[1], (float)m.N[2]};
    for (int i = 0; i < 9; ++i) v[7 + i] = (float)m.T[i];
    bool fin = true;
    for (int i = 0; i < 16; ++i) fin = fin && fabsf(v[i]) <= 3.40282347e+38f;
    if (!fin) v[3] = __uint_as_float(0x7F800000u);
    for (int i = 0; i < 4; ++i) rec[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
}
__device__ __forceinline__ void wind_unused(float4* rec) {
    rec[0] = make_float4(0.0f, 0.0f, 0.0f, -1.0f);
    for (int i = 1; i < 4; ++i) rec[i] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
}
// max(R, x) with a NaN x giving +inf (fmax would skip it)
__device__ __forceinline__ double wind_max(double R, double x) { return x != x ? (double)__uint_as_float(0x7F800000u) : fmax(R, x); }
__device__ __forceinline__ double wind_len(double x, double y, double z) { return sqrt(x * x + y * y + z * z); }
// c: the area-weighted mean of the points pc[i] with weights w[i] (the plain mean when the weights sum to 0), rounded to f32.
__device__ __forceinline__ void wind_center(const double (*pc)[3], const double* w, int n, double* c) {
    double A = 0.0, s[3] = {0.0, 0.0, 0.0}, u[3] = {0.0, 0.0, 0.0};
    for (int i = 0; i < n; ++i) {
        A += w[i];
        for (int k = 0; k < 3; ++k) { s[k] += w[i] * pc[i][k]; u[k] += pc[i][k]; }
    }
    for (int k = 0; k < 3; ++k) c[k] = (double)(float)(A > 0.0 ? s[k] / A : u[k] / n);
}

// The moments of `cnt` (1..8) triangle records.
__device__ __forceinline__ void wind_leaf(const float4* __restrict__ tris, uint32_t cnt, WindMom& m) {
    double ct[8][3], w[8], Nt[8][3];
    for (uint32_t i = 0; i < cnt; ++i) {
        const float4 a = tris[3 * i], e1 = tris[3 * i + 1], e2 = tris[3 * i + 2];
        const double x1 = e1.x, y1 = e1.y, z1 = e1.z, x2 = e2.x, y2 = e2.y, z2 = e2.z;
        Nt[i][0] = 0.5 * (y1 * z2 - z1 * y2); Nt[i][1] = 0.5 * (z1 * x2 - x1 * z2); Nt[i][2] = 0.5 * (x1 * y2 - y1 * x2);
        w[i] = wind_len(Nt[i][0], Nt[i][1], Nt[i][2]);
        ct[i][0] = (double)a.x + (x1 + x2) / 3.0; ct[i][1] = (double)a.y + (y1 + y2) / 3.0; ct[i][2] = (double)a.z + (z1 + z2) / 3.0;
    }
    wind_center(ct, w, (int)cnt, m.c);
    m.area = 0.0;
    double R = 0.0;
    for (int k = 0; k < 12; ++k) (k < 3 ? m.N[k] : m.T[k - 3]) = 0.0;
    for (uint32_t i = 0; i < cnt; ++i) {
        m.area += w[i];
        for (int r = 0; r < 3; ++r) {
            m.N[r] += Nt[i][r];
            for (int c = 0; c < 3; ++c) m.T[3 * r + c] += Nt[i][r] * (ct[i][c] - m.c[c]);
        }
        const float4 a = tris[3 * i], e1 = tris[3 * i + 1], e2 = tris[3 * i + 2];
        const double v[3][3] = {{a.x, a.y, a.z}, {(double)a.x + e1.x, (double)a.y + e1.y, (double)a.z + e1.z},
                                {(double)a.x + e2.x, (double)a.y + e2.y, (double)a.z + e2.z}};
        for (int j = 0; j < 3; ++j) R = wind_max(R, wind_len(v[j][0] - m.c[0], v[j][1] - m.c[1], v[j][2] - m.c[2]));
    }
    m.R = wind_round_up(R);
}

// The merge of the used child records rec[k] (4 float4 each, R < 0: unused) with their areas: c the area-weighted mean of the children's
// c, N = sum N_k, T = sum (T_k + N_k (x) (c_k - c)) (the parallel-axis shift), R = max(|c_k - c| + R_k), rounded up.
// Returns false when no child is used.
__device__ __forceinline__ bool wind_merge(const float4 (*rec)[4], const double* area, WindMom& m) {
    double pc[4][3], w[4];
    int n = 0, idx[4];
    for (int k = 0; k < 4; ++k) {
        if (!(rec[k][0].w >= 0.0f)) continue;
        pc[n][0] = rec[k][0].x; pc[n][1] = rec[k][0].y; pc[n][2] = rec[k][0].z; w[n] = area[k]; idx[n++] = k;
    }
    if (!n) return false;
    wind_center(pc, w, n, m.c);
    m.area = 0.0;
    double R = 0.0;
    for (int k = 0; k < 12; ++k) (k < 3 ? m.N[k] : m.T[k - 3]) = 0.0;
    for (int i = 0; i < n; ++i) {
        const float4* r = rec[idx[i]];
        const double N[3] = {r[1].x, r[1].y, r[1].z};
        const double T[9] = {r[1].w, r[2].x, r[2].y, r[2].z, r[2].w, r[3].x, r[3].y, r[3].z, r[3].w};
        const double d[3] = {pc[i][0] - m.c[0], pc[i][1] - m.c[1], pc[i][2] - m.c[2]};
        m.area += w[i];
        for (int a = 0; a < 3; ++a) {
            m.N[a] += N[a];
            for (int b = 0; b < 3; ++b) m.T[3 * a + b] += T[3 * a + b] + N[a] * d[b];
        }
        R = wind_max(R, wind_len(d[0], d[1], d[2]) + (double)r[0].w);
    }
    m.R = wind_round_up(R);
    return true;
}

}  // namespace rbrt

#ifdef __CUDACC__                                                         // (not in the host build of the tests)
extern "C" {
// Enqueues the winding-number kernel on `stream`; returns a cudaError_t.
typedef int (*rbrt_wind_query_launch_fn)(const rbrt::WindQueryArgs* args, cudaStream_t stream);
// Enqueues the moment kernels of one mesh on `stream`; returns a cudaError_t.
typedef int (*rbrt_wind_moments_launch_fn)(const rbrt::WindMomentArgs* args, cudaStream_t stream);
}
#endif
