// denoise.cuh — the guided à-trous denoiser (rbrt_gpu_denoise*, include/rbrt_gpu.h, DESIGN.md section 13): the per-pixel steps as
// __host__ __device__ functions, and the launch interface of the module that runs them (denoise.cu, built into librbrt_gpu_denoise.so).
//
// The functions below ARE the definition: the kernels call them per pixel, tests/host_device/denoise_harness.cpp compiles them with g++
// for the host, and tests/denoise_ref.py restates them in numpy.  Every operation is one IEEE f32 operation, correctly rounded (XMUL / XADD
// / XSUB / XDIV: __f*_rn on the device, plain operators on a host built without contraction), and compares; nothing else.
#pragma once
#include "../../include/rbrt_gpu.h"
#include "common.cuh"

namespace rbrt {

// Defaults of rbrt_denoise_opts, chosen on the quality scenes of tests/test_gpu_denoise.py (DESIGN.md section 13).
#define DN_DEFAULT_LEVELS 4u
#define DN_MAX_LEVELS 8u
#define DN_SIGMA_DEPTH 0.01f           // σ_z
#define DN_SIGMA_LUMINANCE 0.25f       // σ_l
#define DN_EPS_LUMINANCE 0.0078125f    // ε = 2^-7
#define DN_ALBEDO_FLOOR 0.0009765625f  // 2^-10

// The B3-spline weight of tap (dx, dy), dx, dy in -2..2: h[dx] * h[dy] with h = {1/16, 1/4, 3/8, 1/4, 1/16}; exact binary fractions.
__host__ __device__ __forceinline__ float dn_h(int k) { return k == 0 ? 0.375f : (k == 1 || k == -1 ? 0.25f : 0.0625f); }

// not NaN and not +-inf
__host__ __device__ __forceinline__ bool dn_finite(float v) { return XSUB(v, v) == 0.0f; }

__host__ __device__ __forceinline__ float dn_luminance(float r, float g, float b) {
    return XADD(XADD(XMUL(0.2126f, r), XMUL(0.7152f, g)), XMUL(0.0722f, b));
}

// The demodulation divisor d_k = max(albedo_k, 2^-10); a NaN albedo gives the floor.
__host__ __device__ __forceinline__ float dn_demod(float a) { return a > DN_ALBEDO_FLOOR ? a : DN_ALBEDO_FLOOR; }

// Step 1 for pixel p: e = c / d per channel and its luminance -> *e4 = (e.rgb, l); the guide -> *g4 = (n.xyz, z'), where z' is the depth
// when c, d and z are all finite and NaN otherwise.  A NaN z' marks a pixel that is passed through as a centre and skipped as a tap: the
// three skip rules of a tap (c_q or d_q not finite, z_q not finite) are one test on z'.
__host__ __device__ __forceinline__ void dn_pack(const float* c, const float* albedo, const float* normal, const float* depth, size_t p,
                                                 float4* e4, float4* g4) {
    const float c0 = c[3 * p], c1 = c[3 * p + 1], c2 = c[3 * p + 2];
    const float d0 = dn_demod(albedo[3 * p]), d1 = dn_demod(albedo[3 * p + 1]), d2 = dn_demod(albedo[3 * p + 2]);
    const float e0 = XDIV(c0, d0), e1 = XDIV(c1, d1), e2 = XDIV(c2, d2);
    const float z = depth[p];
    const bool ok = dn_finite(c0) && dn_finite(c1) && dn_finite(c2) && dn_finite(d0) && dn_finite(d1) && dn_finite(d2) && dn_finite(z);
    *e4 = make_float4(e0, e1, e2, dn_luminance(e0, e1, e2));
    *g4 = make_float4(normal[3 * p], normal[3 * p + 1], normal[3 * p + 2], ok ? z : __builtin_nanf(""));
}

// Step 2, one level for the centre pixel (x, y) with step s = 2^level: e[] is the previous level's (e.rgb, l), g[] the guides.  Taps in
// row-major order (dy outer, dx inner), each weight
//     w = (h[dx] * h[dy] * w_n) / ((1 + x_z * x_z) * (1 + x_l * x_l))          (one division)
//     w_n = max(0, (n_p.x * n_q.x + n_p.y * n_q.y) + n_p.z * n_q.z) ^ 128       (seven squarings)
//     x_z = |z_p - z_q| * r_p,  r_p = 1 / ((σ_z * z_p) * s)
//     x_l = (l_p - l_q) * r'_p,  r'_p = 1 / (σ_l * l_p + ε)
// (products and sums left to right as written).  A tap is skipped outside the image, where z'_q is not finite, and where w_n == 0; the
// centre tap has the weight 9/64 whatever its terms.  The result is (Σ w e_q.rgb) / (Σ w), sums from +0 in tap order, and its luminance.
// A centre whose z' is not finite keeps its value.
__host__ __device__ __forceinline__ float4 dn_level(const float4* e, const float4* g, uint32_t W, uint32_t H, uint32_t x, uint32_t y,
                                                    uint32_t s, float sigma_z, float sigma_l) {
    const size_t p = (size_t)y * W + x;
    const float4 ep = e[p], gp = g[p];
    if (!dn_finite(gp.w)) return ep;
    const float r_z = XDIV(1.0f, XMUL(XMUL(sigma_z, gp.w), (float)s));
    const float r_l = XDIV(1.0f, XADD(XMUL(sigma_l, ep.w), DN_EPS_LUMINANCE));
    float sw = 0.0f, s0 = 0.0f, s1 = 0.0f, s2 = 0.0f;
#pragma unroll
    for (int dy = -2; dy <= 2; ++dy) {
        // (x < W <= 2^31 and |dx| * s <= 256: no unsigned sum below wraps)
        if (dy < 0 ? y < (uint32_t)(-dy) * s : y + (uint32_t)dy * s >= H) continue;
        const uint32_t qy = y + (uint32_t)dy * s;
#pragma unroll
        for (int dx = -2; dx <= 2; ++dx) {
            if (dx < 0 ? x < (uint32_t)(-dx) * s : x + (uint32_t)dx * s >= W) continue;
            const uint32_t qx = x + (uint32_t)dx * s;
            float w;
            float4 eq;
            if (dx == 0 && dy == 0) {
                w = 0.140625f;                                              // 9/64
                eq = ep;
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
                const float xz = XMUL(fabsf(XSUB(gp.w, gq.w)), r_z);
                const float xl = XMUL(XSUB(ep.w, eq.w), r_l);
                const float num = XMUL(dn_h(dx) * dn_h(dy), wn);             // (h[dx] * h[dy] is exact)
                w = XDIV(num, XMUL(XADD(1.0f, XMUL(xz, xz)), XADD(1.0f, XMUL(xl, xl))));
            }
            sw = XADD(sw, w);
            s0 = XADD(s0, XMUL(w, eq.x)); s1 = XADD(s1, XMUL(w, eq.y)); s2 = XADD(s2, XMUL(w, eq.z));
        }
    }
    const float o0 = XDIV(s0, sw), o1 = XDIV(s1, sw), o2 = XDIV(s2, sw);
    return make_float4(o0, o1, o2, dn_luminance(o0, o1, o2));
}

// Step 3 for pixel p: out = e_L * d per channel, or c unchanged where z' is not finite.
__host__ __device__ __forceinline__ f3 dn_remodulate(float4 eL, float4 gp, const float* c, const float* albedo, size_t p) {
    if (!dn_finite(gp.w)) return mk3(c[3 * p], c[3 * p + 1], c[3 * p + 2]);
    return mk3(XMUL(eL.x, dn_demod(albedo[3 * p])), XMUL(eL.y, dn_demod(albedo[3 * p + 1])), XMUL(eL.z, dn_demod(albedo[3 * p + 2])));
}

struct DenoiseArgs {
    uint32_t W, H, levels;       // levels 1..DN_MAX_LEVELS
    float sigma_z, sigma_l;      // resolved (> 0)
    const float* hdr;            // W*H*3
    const float* depth;          // W*H
    const float* normal;         // W*H*3
    const float* albedo;         // W*H*3
    float4* scratch;             // 3 * W*H float4: the guides and two planes of (e.rgb, l)
    float* hdr_out;              // W*H*3 or NULL
    uint8_t* rgb_out;            // W*H*3 or NULL
};

}  // namespace rbrt

#ifdef __CUDACC__                                                         // (not in the host build of the tests)
extern "C" {
// Enqueues the denoiser's kernels on `stream` (1 + levels launches); returns a cudaError_t.
typedef int (*rbrt_denoise_launch_fn)(const rbrt::DenoiseArgs* args, cudaStream_t stream);
}
#endif
