// variance_harness.cpp — TEST INFRASTRUCTURE (tests/test_variance_host.py): the per-pixel code of the variance module,
// rbrt_b200/csrc/variance.cuh, compiled for the host with the cuda_runtime.h stand-in of this directory, and driven the way variance.cu's
// kernels drive it: the moments per pixel; the filter's step 1 for every pixel, then one level at a time over the whole image, the last
// level remodulated and tonemapped with shade.cuh's as_u8.  The tests compare the results bit for bit with tests/variance_ref.py.
// Nothing under rbrt_b200/ can reach it.
#include <vector>

#include "shade.cuh"
#include "variance.cuh"

using namespace rbrt;

extern "C" {

// acc: K planes of W*H float4; hdr_out and var_out W*H*3 f32.
int hd_moments(uint32_t W, uint32_t H, uint32_t K, uint32_t S, const float* acc, float* hdr_out, float* var_out) {
    const size_t n = (size_t)W * H;
    const float inv_S = 1.0f / (float)S, inv_n = 1.0f / (float)(S / K);
    for (size_t p = 0; p < n; ++p) {
        f3 m, v;
        vr_moments((const float4*)acc, n, K, p, inv_S, inv_n, &m, &v);
        hdr_out[3 * p] = m.x; hdr_out[3 * p + 1] = m.y; hdr_out[3 * p + 2] = m.z;
        var_out[3 * p] = v.x; var_out[3 * p + 1] = v.y; var_out[3 * p + 2] = v.z;
    }
    return 0;
}

// levels 1..8 and sigmas as resolved (> 0); hdr_out W*H*3 f32 and rgb_out W*H*3 u8.
int hd_denoise_variance(uint32_t W, uint32_t H, const float* hdr, const float* var, const float* depth, const float* normal, const float* albedo,
                        uint32_t levels, float sigma_z, float sigma_l, float* hdr_out, uint8_t* rgb_out) {
    const size_t n = (size_t)W * H;
    std::vector<float4> g(n), e(n), e_next(n);
    std::vector<float> v(n), v_next(n);
    for (size_t p = 0; p < n; ++p) vr_pack(hdr, var, albedo, normal, depth, p, &e[p], &g[p], &v[p]);
    for (uint32_t i = 0; i < levels; ++i) {
        for (uint32_t y = 0; y < H; ++y)
            for (uint32_t x = 0; x < W; ++x) {
                const size_t p = (size_t)y * W + x;
                e_next[p] = vr_level(e.data(), g.data(), v.data(), W, H, x, y, 1u << i, sigma_z, sigma_l, &v_next[p]);
            }
        e.swap(e_next);
        v.swap(v_next);
    }
    for (size_t p = 0; p < n; ++p) {
        const f3 c = dn_remodulate(e[p], g[p], hdr, albedo, p);
        hdr_out[3 * p] = c.x; hdr_out[3 * p + 1] = c.y; hdr_out[3 * p + 2] = c.z;
        rgb_out[3 * p] = as_u8(XMUL(XSQRT(c.x), 256.0f));
        rgb_out[3 * p + 1] = as_u8(XMUL(XSQRT(c.y), 256.0f));
        rgb_out[3 * p + 2] = as_u8(XMUL(XSQRT(c.z), 256.0f));
    }
    return 0;
}

}  // extern "C"
