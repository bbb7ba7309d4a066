// denoise_harness.cpp — TEST INFRASTRUCTURE (tests/test_denoise_host.py): the denoiser's per-pixel code, rbrt_b200/csrc/denoise.cuh, compiled
// for the host with the cuda_runtime.h stand-in of this directory, and driven the way denoise.cu's kernels drive it: step 1 for every pixel,
// then one level at a time over the whole image, the last level remodulated and tonemapped with shade.cuh's as_u8.  The tests compare the
// result bit for bit with tests/denoise_ref.py.  Nothing under rbrt_b200/ can reach it.
#include <vector>

#include "denoise.cuh"
#include "shade.cuh"

using namespace rbrt;

extern "C" {

// levels 1..8 and sigmas as resolved (> 0); hdr_out W*H*3 f32 and rgb_out W*H*3 u8.
int hd_denoise(uint32_t W, uint32_t H, const float* hdr, const float* depth, const float* normal, const float* albedo, uint32_t levels,
               float sigma_z, float sigma_l, float* hdr_out, uint8_t* rgb_out) {
    const size_t n = (size_t)W * H;
    std::vector<float4> g(n), e(n), next(n);
    for (size_t p = 0; p < n; ++p) dn_pack(hdr, albedo, normal, depth, p, &e[p], &g[p]);
    for (uint32_t i = 0; i < levels; ++i) {
        for (uint32_t y = 0; y < H; ++y)
            for (uint32_t x = 0; x < W; ++x) next[(size_t)y * W + x] = dn_level(e.data(), g.data(), W, H, x, y, 1u << i, sigma_z, sigma_l);
        e.swap(next);
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
