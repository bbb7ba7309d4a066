// variance.cuh — per-pixel variance from sample-range shards and the variance-guided à-trous filter (rbrt_gpu_render_hdr_variance*,
// rbrt_gpu_denoise_variance*, include/rbrt_gpu.h, DESIGN.md section 14): the per-pixel steps as __host__ __device__ functions, and the launch
// interface of the module that runs them (variance.cu, built into librbrt_gpu_variance.so).
//
// The functions below ARE the definition: the kernels call them per pixel, tests/host_device/variance_harness.cpp compiles them with g++ for
// the host, and tests/variance_ref.py restates them in numpy.  Every operation is one IEEE f32 operation, correctly rounded (XMUL / XADD /
// XSUB / XDIV / XSQRT), and compares; nothing else.  The filter shares the demodulation, the B3 taps, the normal and depth terms and the
// remodulation with rbrt_gpu_denoise (denoise.cuh).
#pragma once
#include "denoise.cuh"

namespace rbrt {

#define VR_MAX_SPLITS 16u
// Defaults of rbrt_denoise_opts for the variance-guided filter, chosen on the quality scenes of tests/test_gpu_variance.py (DESIGN.md
// section 14).
#define VR_DEFAULT_LEVELS 5u
#define VR_SIGMA_DEPTH 0.01f           // σ_z
#define VR_SIGMA_LUMINANCE 4.0f        // σ_l
#define VR_EPS_LUMINANCE 0.0009765625f // ε = 2^-10

// The moments of pixel p from K per-pixel sums acc[k * n + p] (k = 0..K-1, shard k's samples): the mean over all S samples, the
// arithmetic of k_sum_peers + k_finalize (((A_0 + A_1) + A_2) + ...) * (1/S), and the unbiased variance of that mean,
// Σ_k (A_k * (1/n) - mean)^2 / (K * (K - 1)), the squares summed from +0 in shard order.  inv_S = 1/S and inv_n = 1/n as f32 quotients.
__host__ __device__ __forceinline__ void vr_moments(const float4* acc, size_t n, uint32_t K, size_t p, float inv_S, float inv_n, f3* mean,
                                                    f3* var) {
    float4 a = acc[p];
    for (uint32_t k = 1; k < K; ++k) {
        const float4 b = acc[(size_t)k * n + p];
        a.x = XADD(a.x, b.x); a.y = XADD(a.y, b.y); a.z = XADD(a.z, b.z);
    }
    const float m0 = XMUL(a.x, inv_S), m1 = XMUL(a.y, inv_S), m2 = XMUL(a.z, inv_S);
    float q0 = 0.0f, q1 = 0.0f, q2 = 0.0f;
    for (uint32_t k = 0; k < K; ++k) {
        const float4 b = acc[(size_t)k * n + p];
        const float d0 = XSUB(XMUL(b.x, inv_n), m0), d1 = XSUB(XMUL(b.y, inv_n), m1), d2 = XSUB(XMUL(b.z, inv_n), m2);
        q0 = XADD(q0, XMUL(d0, d0)); q1 = XADD(q1, XMUL(d1, d1)); q2 = XADD(q2, XMUL(d2, d2));
    }
    const float kk = (float)(K * (K - 1));                                // exact: at most 240
    *mean = mk3(m0, m1, m2);
    *var = mk3(XDIV(q0, kk), XDIV(q1, kk), XDIV(q2, kk));
}

// The 3x3 prefilter weight of offset k in -1..1: {1/4, 1/2, 1/4}.
__host__ __device__ __forceinline__ float vr_k(int k) { return k == 0 ? 0.5f : 0.25f; }

// a variance component the filter can use: finite and not negative (-0 is not negative)
__host__ __device__ __forceinline__ bool vr_var_ok(float v) { return v >= 0.0f && dn_finite(v); }

// Step 1 for pixel p: rbrt_gpu_denoise's e4 = (e.rgb, l) and g4 = (n.xyz, z'), where z' is also NaN when a component of var is not finite
// or negative; *s2 = sd * sd, the variance bound of l(e):
//     sd = ((0.2126 / d_r) * sqrt(v_r) + (0.7152 / d_g) * sqrt(v_g)) + (0.0722 / d_b) * sqrt(v_b)
__host__ __device__ __forceinline__ void vr_pack(const float* c, const float* var, const float* albedo, const float* normal, const float* depth,
                                                 size_t p, float4* e4, float4* g4, float* s2) {
    dn_pack(c, albedo, normal, depth, p, e4, g4);
    const float v0 = var[3 * p], v1 = var[3 * p + 1], v2 = var[3 * p + 2];
    if (!(vr_var_ok(v0) && vr_var_ok(v1) && vr_var_ok(v2))) g4->w = __builtin_nanf("");
    const float d0 = dn_demod(albedo[3 * p]), d1 = dn_demod(albedo[3 * p + 1]), d2 = dn_demod(albedo[3 * p + 2]);
    const float sd = XADD(XADD(XMUL(XDIV(0.2126f, d0), XSQRT(v0)), XMUL(XDIV(0.7152f, d1), XSQRT(v1))), XMUL(XDIV(0.0722f, d2), XSQRT(v2)));
    *s2 = XMUL(sd, sd);
}

// Step 2, one level for the centre pixel (x, y) with step s = 2^level: e[] the previous level's (e.rgb, l), v[] its σ², g[] the guides.
//   g_p = (Σ k[dx] * k[dy] * v_q) / (Σ k[dx] * k[dy]) over the 3x3 unit-step neighbours q inside the image whose z' is finite, row-major,
//         sums from +0, k = {1/4, 1/2, 1/4} (the products are exact);
//   r'_p = 1 / (σ_l * sqrt(g_p) + ε);  x_l = (l_p - l_q) * r'_p;
//   w   = (h[dx] * h[dy] * w_n) / ((1 + x_z * x_z) * ((1 + x_l * x_l) * (1 + x_l * x_l)))
// with the taps, skips, w_n, x_z and the 9/64 centre of dn_level.  The result is (Σ w e_q.rgb) / (Σ w) and its luminance, and
// *v_out = (Σ (w * w) * v_q) / ((Σ w) * (Σ w)), sums from +0 in tap order.  A centre whose z' is not finite keeps its e and σ².
__host__ __device__ __forceinline__ float4 vr_level(const float4* e, const float4* g, const float* v, uint32_t W, uint32_t H, uint32_t x,
                                                    uint32_t y, uint32_t s, float sigma_z, float sigma_l, float* v_out) {
    const size_t p = (size_t)y * W + x;
    const float4 ep = e[p], gp = g[p];
    const float vp = v[p];
    if (!dn_finite(gp.w)) { *v_out = vp; return ep; }
    float gs = 0.0f, gw = 0.0f;
#pragma unroll
    for (int dy = -1; dy <= 1; ++dy) {
        if (dy < 0 ? y == 0 : (dy > 0 && y + 1 >= H)) continue;
        const uint32_t qy = y + (uint32_t)dy;
#pragma unroll
        for (int dx = -1; dx <= 1; ++dx) {
            if (dx < 0 ? x == 0 : (dx > 0 && x + 1 >= W)) continue;
            const size_t q = (size_t)qy * W + (x + (uint32_t)dx);
            if (!dn_finite(g[q].w)) continue;
            const float k = vr_k(dx) * vr_k(dy);                            // (exact)
            gs = XADD(gs, XMUL(k, v[q]));
            gw = XADD(gw, k);
        }
    }
    const float r_z = XDIV(1.0f, XMUL(XMUL(sigma_z, gp.w), (float)s));
    const float r_l = XDIV(1.0f, XADD(XMUL(sigma_l, XSQRT(XDIV(gs, gw))), VR_EPS_LUMINANCE));
    float sw = 0.0f, s0 = 0.0f, s1 = 0.0f, s2 = 0.0f, sv = 0.0f;
#pragma unroll
    for (int dy = -2; dy <= 2; ++dy) {
        // (x < W <= 2^31 and |dx| * s <= 256: no unsigned sum below wraps)
        if (dy < 0 ? y < (uint32_t)(-dy) * s : y + (uint32_t)dy * s >= H) continue;
        const uint32_t qy = y + (uint32_t)dy * s;
#pragma unroll
        for (int dx = -2; dx <= 2; ++dx) {
            if (dx < 0 ? x < (uint32_t)(-dx) * s : x + (uint32_t)dx * s >= W) continue;
            const uint32_t qx = x + (uint32_t)dx * s;
            float w, vq;
            float4 eq;
            if (dx == 0 && dy == 0) {
                w = 0.140625f;                                              // 9/64
                eq = ep;
                vq = vp;
            } else {
                const size_t q = (size_t)qy * W + (size_t)qx;
                const float4 gq = g[q];
                if (!dn_finite(gq.w)) continue;
                const float dot = XADD(XADD(XMUL(gp.x, gq.x), XMUL(gp.y, gq.y)), XMUL(gp.z, gq.z));
                float wn = dot > 0.0f ? dot : 0.0f;
#pragma unroll
                for (int k = 0; k < 7; ++k) wn = XMUL(wn, wn);
                if (wn == 0.0f) continue;
                eq = e[q];
                vq = v[q];
                const float xz = XMUL(fabsf(XSUB(gp.w, gq.w)), r_z);
                const float xl = XMUL(XSUB(ep.w, eq.w), r_l);
                const float dl = XADD(1.0f, XMUL(xl, xl));
                const float num = XMUL(dn_h(dx) * dn_h(dy), wn);             // (h[dx] * h[dy] is exact)
                w = XDIV(num, XMUL(XADD(1.0f, XMUL(xz, xz)), XMUL(dl, dl)));
            }
            sw = XADD(sw, w);
            s0 = XADD(s0, XMUL(w, eq.x)); s1 = XADD(s1, XMUL(w, eq.y)); s2 = XADD(s2, XMUL(w, eq.z));
            sv = XADD(sv, XMUL(XMUL(w, w), vq));
        }
    }
    const float o0 = XDIV(s0, sw), o1 = XDIV(s1, sw), o2 = XDIV(s2, sw);
    *v_out = XDIV(sv, XMUL(sw, sw));
    return make_float4(o0, o1, o2, dn_luminance(o0, o1, o2));
}

struct MomentsArgs {
    uint32_t W, H, K;            // K = splits, 2..VR_MAX_SPLITS
    float inv_S, inv_n;          // 1/S and 1/(S/K)
    const float4* acc;           // K planes of W*H float4, shard k's at acc + k * W*H
    float* hdr_out;              // W*H*3 or NULL
    float* var_out;              // W*H*3 or NULL
};

}  // namespace rbrt

#ifdef __CUDACC__                                                         // (not in the host build of the tests)
extern "C" {
// Enqueues the moments kernel on `stream` (one launch); returns a cudaError_t.
typedef int (*rbrt_variance_moments_launch_fn)(const rbrt::MomentsArgs* args, cudaStream_t stream);
// Enqueues the variance-guided filter on `stream` (1 + levels launches); args->scratch holds 3 * W*H float4 and then 2 * W*H float, var
// is the W*H*3 variance plane.  Returns a cudaError_t.
typedef int (*rbrt_variance_filter_launch_fn)(const rbrt::DenoiseArgs* args, const float* var, cudaStream_t stream);
}
#endif
