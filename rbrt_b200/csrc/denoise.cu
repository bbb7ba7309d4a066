// denoise.cu — the guided à-trous denoiser (rbrt_gpu_denoise / rbrt_gpu_denoise_device): demodulate the HDR mean colour by the albedo
// AOV, filter it at 1..8 levels with edge-stopping weights from the normal, depth and luminance, remodulate and optionally tonemap.
//
// Built into its own shared object (librbrt_gpu_denoise.so), which librbrt_gpu.so loads at run time like the AOV and query modules: the
// device code of librbrt_gpu.so stays exactly the build the GPU tests verified.  The per-pixel arithmetic is denoise.cuh's, so the kernels
// and the host build of that header agree bit for bit.  One thread is one pixel, in row-major order: a warp reads 32 neighbouring 16-byte
// records per tap.  The planes of one level (2 x 16 bytes per pixel, 66 MB at 1920x1080) stay in the 126 MB L2 across a level's 25 taps.
#include "denoise.cuh"
#include "shade.cuh"

namespace rbrt {
namespace {

#define DN_THREADS 256
// (4 blocks of 256 per SM: 64 registers at most, which the level kernels need without a spill around the division's slow path)

__global__ void __launch_bounds__(DN_THREADS) k_denoise_pack(DenoiseArgs A, float4* __restrict__ e, float4* __restrict__ g) {
    const size_t p = (size_t)blockIdx.x * DN_THREADS + threadIdx.x;
    if (p >= (size_t)A.W * A.H) return;
    float4 e4, g4;
    dn_pack(A.hdr, A.albedo, A.normal, A.depth, p, &e4, &g4);
    e[p] = e4;
    g[p] = g4;
}

// LAST: remodulate, and write hdr_out / rgb_out (the tonemap of k_finalize, lib.rs:116-122) instead of the next level's plane.
template <bool LAST>
__global__ void __launch_bounds__(DN_THREADS, 4) k_denoise_level(DenoiseArgs A, const float4* __restrict__ e_in, const float4* __restrict__ g,
                                                              float4* __restrict__ e_out, uint32_t s) {
    const size_t p = (size_t)blockIdx.x * DN_THREADS + threadIdx.x;
    if (p >= (size_t)A.W * A.H) return;
    const uint32_t y = (uint32_t)(p / A.W), x = (uint32_t)(p - (size_t)y * A.W);
    const float4 o = dn_level(e_in, g, A.W, A.H, x, y, s, A.sigma_z, A.sigma_l);
    if (!LAST) { e_out[p] = o; return; }
    const f3 c = dn_remodulate(o, g[p], A.hdr, A.albedo, p);
    if (A.hdr_out) { A.hdr_out[3 * p] = c.x; A.hdr_out[3 * p + 1] = c.y; A.hdr_out[3 * p + 2] = c.z; }
    if (A.rgb_out) {
        A.rgb_out[3 * p] = as_u8(XMUL(XSQRT(c.x), 256.0f));
        A.rgb_out[3 * p + 1] = as_u8(XMUL(XSQRT(c.y), 256.0f));
        A.rgb_out[3 * p + 2] = as_u8(XMUL(XSQRT(c.z), 256.0f));
    }
}

}  // namespace
}  // namespace rbrt

extern "C" int rbrt_denoise_launch(const rbrt::DenoiseArgs* a, cudaStream_t stream) {
    const size_t n = (size_t)a->W * a->H;
    if (!n) return (int)cudaSuccess;
    const unsigned grid = (unsigned)((n + DN_THREADS - 1) / DN_THREADS);
    float4* g = a->scratch;
    float4* e[2] = {a->scratch + n, a->scratch + 2 * n};
    rbrt::k_denoise_pack<<<grid, DN_THREADS, 0, stream>>>(*a, e[0], g);
    for (uint32_t i = 0; i < a->levels; ++i) {
        if (i + 1 < a->levels) rbrt::k_denoise_level<false><<<grid, DN_THREADS, 0, stream>>>(*a, e[i & 1], g, e[(i + 1) & 1], 1u << i);
        else rbrt::k_denoise_level<true><<<grid, DN_THREADS, 0, stream>>>(*a, e[i & 1], g, nullptr, 1u << i);
    }
    return (int)cudaGetLastError();
}
