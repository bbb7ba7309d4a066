// variance.cu — per-pixel variance of a render from sample-range shards (rbrt_gpu_render_hdr_variance*) and the variance-guided à-trous
// filter (rbrt_gpu_denoise_variance*): the moments kernel turns the K shard accumulators into the mean colour and the variance of that
// mean; the filter demodulates by the albedo AOV, filters colour and variance at 1..8 levels with edge-stopping weights from the normal,
// the depth and the luminance scaled by the local standard deviation, remodulates and optionally tonemaps.
//
// Built into its own shared object (librbrt_gpu_variance.so), which librbrt_gpu.so loads at run time like the AOV, query and denoise modules:
// the device code of librbrt_gpu.so and librbrt_gpu_denoise.so stays exactly the build the GPU tests verified.  The per-pixel arithmetic
// is variance.cuh's, so the kernels and the host build of that header agree bit for bit.  One thread is one pixel, in row-major order.
#include "shade.cuh"
#include "variance.cuh"

namespace rbrt {
namespace {

#define VR_THREADS 256

__global__ void __launch_bounds__(VR_THREADS) k_variance_moments(MomentsArgs A) {
    const size_t p = (size_t)blockIdx.x * VR_THREADS + threadIdx.x;
    const size_t n = (size_t)A.W * A.H;
    if (p >= n) return;
    f3 m, v;
    vr_moments(A.acc, n, A.K, p, A.inv_S, A.inv_n, &m, &v);
    if (A.hdr_out) { A.hdr_out[3 * p] = m.x; A.hdr_out[3 * p + 1] = m.y; A.hdr_out[3 * p + 2] = m.z; }
    if (A.var_out) { A.var_out[3 * p] = v.x; A.var_out[3 * p + 1] = v.y; A.var_out[3 * p + 2] = v.z; }
}

__global__ void __launch_bounds__(VR_THREADS) k_variance_pack(DenoiseArgs A, const float* __restrict__ var, float4* __restrict__ e,
                                                             float4* __restrict__ g, float* __restrict__ v) {
    const size_t p = (size_t)blockIdx.x * VR_THREADS + threadIdx.x;
    if (p >= (size_t)A.W * A.H) return;
    float4 e4, g4;
    float s2;
    vr_pack(A.hdr, var, A.albedo, A.normal, A.depth, p, &e4, &g4, &s2);
    e[p] = e4;
    g[p] = g4;
    v[p] = s2;
}

// LAST: remodulate, and write hdr_out / rgb_out (the tonemap of k_finalize, lib.rs:116-122) instead of the next level's planes.
template <bool LAST>
__global__ void __launch_bounds__(VR_THREADS, 4) k_variance_level(DenoiseArgs A, const float4* __restrict__ e_in, const float4* __restrict__ g,
                                                                const float* __restrict__ v_in, float4* __restrict__ e_out,
                                                                float* __restrict__ v_out, uint32_t s) {
    const size_t p = (size_t)blockIdx.x * VR_THREADS + threadIdx.x;
    if (p >= (size_t)A.W * A.H) return;
    const uint32_t y = (uint32_t)(p / A.W), x = (uint32_t)(p - (size_t)y * A.W);
    float vo;
    const float4 o = vr_level(e_in, g, v_in, A.W, A.H, x, y, s, A.sigma_z, A.sigma_l, &vo);
    if (!LAST) { e_out[p] = o; v_out[p] = vo; return; }
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

extern "C" int rbrt_variance_moments_launch(const rbrt::MomentsArgs* a, cudaStream_t stream) {
    const size_t n = (size_t)a->W * a->H;
    if (!n) return (int)cudaSuccess;
    rbrt::k_variance_moments<<<(unsigned)((n + VR_THREADS - 1) / VR_THREADS), VR_THREADS, 0, stream>>>(*a);
    return (int)cudaGetLastError();
}

extern "C" int rbrt_variance_filter_launch(const rbrt::DenoiseArgs* a, const float* var, cudaStream_t stream) {
    const size_t n = (size_t)a->W * a->H;
    if (!n) return (int)cudaSuccess;
    const unsigned grid = (unsigned)((n + VR_THREADS - 1) / VR_THREADS);
    float4* g = a->scratch;
    float4* e[2] = {a->scratch + n, a->scratch + 2 * n};
    float* v[2] = {(float*)(a->scratch + 3 * n), (float*)(a->scratch + 3 * n) + n};
    rbrt::k_variance_pack<<<grid, VR_THREADS, 0, stream>>>(*a, var, e[0], g, v[0]);
    for (uint32_t i = 0; i < a->levels; ++i) {
        const uint32_t j = i & 1;
        if (i + 1 < a->levels) rbrt::k_variance_level<false><<<grid, VR_THREADS, 0, stream>>>(*a, e[j], g, v[j], e[j ^ 1], v[j ^ 1], 1u << i);
        else rbrt::k_variance_level<true><<<grid, VR_THREADS, 0, stream>>>(*a, e[j], g, v[j], nullptr, nullptr, 1u << i);
    }
    return (int)cudaGetLastError();
}
