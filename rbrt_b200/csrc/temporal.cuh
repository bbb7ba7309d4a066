// temporal.cuh — temporal accumulation of a frame sequence (rbrt_gpu_temporal_accumulate*, include/rbrt_gpu.h, DESIGN.md section 15): the
// per-pixel step as a __host__ __device__ function, and the launch interface of the module that runs it (temporal.cu, built into
// librbrt_gpu_temporal.so).
//
// The functions below ARE the definition: the kernel calls tp_pixel per pixel, tests/host_device/temporal_harness.cpp compiles it with g++
// for the host, and tests/temporal_ref.py restates it in numpy.  Every operation is one IEEE f32 operation, correctly rounded (XMUL / XADD /
// XSUB / XDIV / XSQRT), a floorf, or a compare; nothing else.
#pragma once
#include "denoise.cuh"

namespace rbrt {

// Defaults of rbrt_temporal_opts (DESIGN.md section 15).
#define TP_ALPHA_MIN 0.1f              // α_min
#define TP_SIGMA_DEPTH 0.02f           // σ_z
#define TP_NORMAL_MIN 0.9f             // n_min
#define TP_MIN_WEIGHT 0.015625f        // 2^-6: a history whose consistent bilinear weights sum to less is dropped

// dot = (x*x' + y*y') + z*z', cross and length as common.cuh's dot3 / cross3 / len3 (which are device-only).
__host__ __device__ __forceinline__ float tp_dot(f3 a, f3 b) { return XADD(XADD(XMUL(a.x, b.x), XMUL(a.y, b.y)), XMUL(a.z, b.z)); }
__host__ __device__ __forceinline__ f3 tp_cross(f3 a, f3 b) {
    return mk3(XSUB(XMUL(a.y, b.z), XMUL(a.z, b.y)), XSUB(XMUL(a.z, b.x), XMUL(a.x, b.z)), XSUB(XMUL(a.x, b.y), XMUL(a.y, b.x)));
}
__host__ __device__ __forceinline__ f3 tp_sub(f3 a, f3 b) { return mk3(XSUB(a.x, b.x), XSUB(a.y, b.y), XSUB(a.z, b.z)); }
__host__ __device__ __forceinline__ f3 tp_v(const float* v) { return mk3(v[0], v[1], v[2]); }
__host__ __device__ __forceinline__ f3 tp_load3(const float* a, size_t p) { return mk3(a[3 * p], a[3 * p + 1], a[3 * p + 2]); }

// The direction of pixel (x, y)'s centre ray: camera_ray's direction (shade.cuh) with both jitter draws at 0.5, v / |v| per component.
__host__ __device__ __forceinline__ f3 tp_pixel_dir(const CamDev& c, uint32_t x, uint32_t y) {
    const float col_off = XSUB((float)x, (float)(c.width / 2));
    const float row_off = XSUB((float)y, (float)(c.height / 2));
    const float col_mm = XMUL(XSUB(XADD(col_off, 0.5f), 0.5f), c.mm_per_pix_hor);
    const float row_mm = XMUL(XSUB(XADD(row_off, 0.5f), 0.5f), c.mm_per_pix_vert);
    const float ch = XMUL(0.001f, col_mm), cv = XMUL(0.001f, row_mm);
    const f3 t = mk3(XSUB(XADD(c.center[0], XMUL(ch, c.right[0])), XMUL(cv, c.up[0])),
                     XSUB(XADD(c.center[1], XMUL(ch, c.right[1])), XMUL(cv, c.up[1])),
                     XSUB(XADD(c.center[2], XMUL(ch, c.right[2])), XMUL(cv, c.up[2])));
    const f3 v = tp_sub(t, tp_v(c.pos));
    const float l = XSQRT(tp_dot(v, v));
    return mk3(XDIV(v.x, l), XDIV(v.y, l), XDIV(v.z, l));
}

// The world point of pixel (x, y) at depth z: pos + z * d, d = tp_pixel_dir.
__host__ __device__ __forceinline__ f3 tp_world_point(const CamDev& c, uint32_t x, uint32_t y, float z) {
    const f3 d = tp_pixel_dir(c, x, y);
    return mk3(XADD(c.pos[0], XMUL(z, d.x)), XADD(c.pos[1], XMUL(z, d.y)), XADD(c.pos[2], XMUL(z, d.z)));
}

// X projected into camera c: the continuous pixel coordinates (*px, *py), integers at pixel centres.  Solves
//     pos + s * (X - pos) = center + a * right - b * up
// by Cramer's rule with D = X - pos, C = center - pos (up as stored, not assumed orthogonal to right):
//     det = D . (right x up),  s = (C . (right x up)) / det,  a = (D . (up x C)) / det,  b = (D . (right x C)) / det,
//     px = (a / 0.001) / mm_per_pix_hor + (float)(W / 2),  py = (b / 0.001) / mm_per_pix_vert + (float)(H / 2).
// Returns false when s <= 0 (or NaN): X is not in front of the camera.
__host__ __device__ __forceinline__ bool tp_project(const CamDev& c, f3 D, float* px, float* py) {
    const f3 right = tp_v(c.right), up = tp_v(c.up), C = tp_sub(tp_v(c.center), tp_v(c.pos));
    const f3 ru = tp_cross(right, up);
    const float det = tp_dot(D, ru);
    const float s = XDIV(tp_dot(C, ru), det);
    const float a = XDIV(tp_dot(D, tp_cross(up, C)), det);
    const float b = XDIV(tp_dot(D, tp_cross(right, C)), det);
    *px = XADD(XDIV(XDIV(a, 0.001f), c.mm_per_pix_hor), (float)(c.width / 2));
    *py = XADD(XDIV(XDIV(b, 0.001f), c.mm_per_pix_vert), (float)(c.height / 2));
    return s > 0.0f;
}

struct TemporalArgs {
    uint32_t W, H;
    uint32_t history;            // 0: the first frame (every h_* NULL)
    uint32_t same_cam;           // prev equals cam field for field, bit for bit: each pixel maps to itself with weight 1
    float alpha_min, sigma_z, n_min;
    CamDev prev;                 // the history's camera
    CamDev cam;                  // the current frame's camera
    const float* hdr;            // W*H*3
    const float* var;            // W*H*3 or NULL (then var_out is NULL)
    const float* depth;          // W*H
    const float* normal;         // W*H*3
    const int32_t* kind;         // W*H
    const uint32_t* elem;        // W*H
    const float* h_hdr;          // the history: W*H*3, aligned to prev
    const float* h_var;          // W*H*3; NULL when var_out is NULL (then the variance is not propagated)
    const float* h_len;          // W*H
    const float* h_depth;        // W*H
    const float* h_normal;       // W*H*3
    const int32_t* h_kind;       // W*H
    const uint32_t* h_elem;      // W*H
    float* hdr_out;              // W*H*3 or NULL
    float* var_out;              // W*H*3 or NULL
    float* len_out;              // W*H or NULL
    const float* motion;         // motion variant: W*H*2, the frame's motion pass against prev and the history's snapshot
    const float* prev_dist;      // motion variant: W*H
};

// Steps 4 and 5 for a valid pixel p with a history: the taps around (x0 + fx, y0 + fy), their consistency with depth r, and the blend.
__host__ __device__ __forceinline__ void tp_resample(const TemporalArgs& A, size_t p, f3 c, f3 v, float r, uint32_t x0, uint32_t y0, float fx,
                                                     float fy, f3* out, f3* vout, float* lout) {
    const f3 n = tp_load3(A.normal, p);
    const float ln = XSQRT(tp_dot(n, n));
    const int32_t kp = A.kind[p];
    const uint32_t ep = A.elem[p];
    const float tol = XMUL(A.sigma_z, r);
    const float gx = XSUB(1.0f, fx), gy = XSUB(1.0f, fy);
    float sw = 0.0f, s0 = 0.0f, s1 = 0.0f, s2 = 0.0f, sv0 = 0.0f, sv1 = 0.0f, sv2 = 0.0f, sl = 0.0f;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
        const uint32_t qx = x0 + (uint32_t)(t & 1), qy = y0 + (uint32_t)(t >> 1);
        const float w = XMUL((t & 1) ? fx : gx, (t >> 1) ? fy : gy);
        if (w == 0.0f || qx >= A.W || qy >= A.H) continue;
        const size_t q = (size_t)qy * A.W + qx;
        const float lq = A.h_len[q];
        if (!(lq > 0.0f) || A.h_kind[q] != kp || A.h_elem[q] != ep) continue;
        if (!(fabsf(XSUB(A.h_depth[q], r)) <= tol)) continue;
        const f3 nq = tp_load3(A.h_normal, q);
        if (!(tp_dot(n, nq) >= XMUL(A.n_min, XMUL(ln, XSQRT(tp_dot(nq, nq)))))) continue;
        const f3 cq = tp_load3(A.h_hdr, q);
        sw = XADD(sw, w);
        s0 = XADD(s0, XMUL(w, cq.x)); s1 = XADD(s1, XMUL(w, cq.y)); s2 = XADD(s2, XMUL(w, cq.z));
        sl = XADD(sl, XMUL(w, lq));
        if (A.h_var) {
            const f3 vq = tp_load3(A.h_var, q);
            const float ww = XMUL(w, w);
            sv0 = XADD(sv0, XMUL(ww, vq.x)); sv1 = XADD(sv1, XMUL(ww, vq.y)); sv2 = XADD(sv2, XMUL(ww, vq.z));
        }
    }
    if (!(sw >= TP_MIN_WEIGHT)) return;
    const float nh = XDIV(sl, sw);
    const float a1 = XDIV(1.0f, XADD(nh, 1.0f));
    const float al = a1 > A.alpha_min ? a1 : A.alpha_min;
    const f3 ch = mk3(XDIV(s0, sw), XDIV(s1, sw), XDIV(s2, sw));
    *out = mk3(XADD(ch.x, XMUL(al, XSUB(c.x, ch.x))), XADD(ch.y, XMUL(al, XSUB(c.y, ch.y))), XADD(ch.z, XMUL(al, XSUB(c.z, ch.z))));
    if (A.h_var) {
        const float sw2 = XMUL(sw, sw), om = XSUB(1.0f, al);
        const float k1 = XMUL(om, om), k2 = XMUL(al, al);
        *vout = mk3(XADD(XMUL(k1, XDIV(sv0, sw2)), XMUL(k2, v.x)), XADD(XMUL(k1, XDIV(sv1, sw2)), XMUL(k2, v.y)),
                    XADD(XMUL(k1, XDIV(sv2, sw2)), XMUL(k2, v.z)));
    }
    *lout = XADD(nh, 1.0f);
}

// Pixel (x, y):
//  1. p is VALID when its colour and depth are finite and, with a variance, each component of it is finite and >= 0 (-0 is).  An
//     invalid p gives (hdr, var, 0).
//  2. Without a history, or when the reprojection below finds none: (hdr, var, 1).
//  3. X = tp_world_point(cam, x, y, z_p); D = X - prev.pos; r = sqrt(D . D).  There is no history when r is not finite, when
//     tp_project fails or gives a non-finite coordinate, or when the point lies outside [0, W-1] x [0, H-1] (the borders are inside).
//     same_cam: (px, py) = (x, y) exactly and tp_project is not called.
//     With motion planes (rbrt_gpu_temporal_accumulate_motion*): when both components of m = motion[p] are finite, (px, py) = (x + m.x, y + m.y) and
//     r = prev_dist[p] instead, with the same tests on r and on the bounds; otherwise step 3 as above.
//  4. x0 = floor(px), fx = px - x0 (likewise y); taps (x0, y0), (x0+1, y0), (x0, y0+1), (x0+1, y0+1) in that order with the bilinear
//     weights (1-fx)*(1-fy), fx*(1-fy), (1-fx)*fy, fx*fy.  A tap q is skipped when its weight is 0, when it lies outside the image,
//     and unless it is CONSISTENT: length_q > 0, hit_kind_q == hit_kind_p, elem_idx_q == elem_idx_p, |z_q - r| <= σ_z * r and
//     n_p . n_q >= n_min * (|n_p| * |n_q|) (tp_dot, |n| = sqrt(n . n): the AOV normals are means, not unit vectors).  Σw, Σ w*c_q,
//     Σ (w*w)*v_q and Σ w*length_q are sums from +0 in tap order.  Σw < TP_MIN_WEIGHT: no history.  c_h = Σ w*c_q / Σw, v_h = Σ (w*w)*v_q / (Σw * Σw), n_h = Σ w*length_q / Σw.
//  5. α = max(1 / (n_h + 1), α_min); out = c_h + α * (c - c_h); var_out = ((1-α)*(1-α)) * v_h + (α*α) * v; len_out = n_h + 1.
// v takes part in the validity when var is given; v_h and var_out are formed only when h_var is given (var_out requested with a history).
__host__ __device__ __forceinline__ void tp_pixel(const TemporalArgs& A, uint32_t x, uint32_t y, f3* out, f3* vout, float* lout) {
    const size_t p = (size_t)y * A.W + x;
    const f3 c = tp_load3(A.hdr, p);
    const f3 v = A.var ? tp_load3(A.var, p) : mk3(0.0f, 0.0f, 0.0f);
    const float z = A.depth[p];
    *out = c;
    *vout = v;
    const bool valid = dn_finite(c.x) && dn_finite(c.y) && dn_finite(c.z) && dn_finite(z) &&
                       (!A.var || (v.x >= 0.0f && dn_finite(v.x) && v.y >= 0.0f && dn_finite(v.y) && v.z >= 0.0f && dn_finite(v.z)));
    if (!valid) { *lout = 0.0f; return; }
    *lout = 1.0f;
    if (!A.history) return;

    float r;
    uint32_t x0, y0;
    float fx, fy;
    const float mx = A.motion ? A.motion[2 * p] : 0.0f, my = A.motion ? A.motion[2 * p + 1] : 0.0f;
    if (A.motion && dn_finite(mx) && dn_finite(my)) {
        r = A.prev_dist[p];
        if (!dn_finite(r)) return;
        const float px = XADD((float)x, mx), py = XADD((float)y, my);
        if (!(px >= 0.0f && px <= (float)(A.W - 1) && py >= 0.0f && py <= (float)(A.H - 1))) return;
        const float fx0 = floorf(px), fy0 = floorf(py);
        x0 = (uint32_t)fx0; y0 = (uint32_t)fy0;
        fx = XSUB(px, fx0); fy = XSUB(py, fy0);
    } else {
        const f3 X = tp_world_point(A.cam, x, y, z);
        const f3 D = tp_sub(X, tp_v(A.prev.pos));
        r = XSQRT(tp_dot(D, D));
        if (!dn_finite(r)) return;
        if (A.same_cam) {
            x0 = x; y0 = y; fx = 0.0f; fy = 0.0f;
        } else {
            float px, py;
            if (!tp_project(A.prev, D, &px, &py)) return;
            if (!(px >= 0.0f && px <= (float)(A.W - 1) && py >= 0.0f && py <= (float)(A.H - 1))) return;   // (NaN fails too)
            const float fx0 = floorf(px), fy0 = floorf(py);
            x0 = (uint32_t)fx0; y0 = (uint32_t)fy0;
            fx = XSUB(px, fx0); fy = XSUB(py, fy0);
        }
    }
    tp_resample(A, p, c, v, r, x0, y0, fx, fy, out, vout, lout);
}

}  // namespace rbrt

#ifdef __CUDACC__                                                         // (not in the host build of the tests)
extern "C" {
// Enqueues the temporal accumulation on `stream` (one launch); returns a cudaError_t.
typedef int (*rbrt_temporal_launch_fn)(const rbrt::TemporalArgs* args, cudaStream_t stream);
}
#endif
