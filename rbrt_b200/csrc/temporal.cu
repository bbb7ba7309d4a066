// temporal.cu — temporal accumulation of a frame sequence (rbrt_gpu_temporal_accumulate*): each pixel's history, aligned to the previous
// camera, is reprojected through that camera, resampled from the bilinear taps whose depth, normal and hit ids agree with the pixel, and
// blended with the current frame in colour, variance and history length.  The motion variant reprojects along the frame's per-object
// motion pass (motion.cu) where that is finite.
//
// Built into its own shared object (librbrt_gpu_temporal.so), which librbrt_gpu.so loads at run time like the other device modules: the
// device code of librbrt_gpu.so stays exactly the build the GPU tests verified.  The per-pixel arithmetic is temporal.cuh's, so the kernel
// and the host build of that header agree bit for bit.  One thread is one pixel, in row-major order.
#include "temporal.cuh"

namespace rbrt {
namespace {

#define TP_THREADS 256

__global__ void __launch_bounds__(TP_THREADS) k_temporal(TemporalArgs A) {
    const size_t p = (size_t)blockIdx.x * TP_THREADS + threadIdx.x;
    if (p >= (size_t)A.W * A.H) return;
    const uint32_t y = (uint32_t)(p / A.W), x = (uint32_t)(p - (size_t)y * A.W);
    f3 o, v;
    float l;
    tp_pixel(A, x, y, &o, &v, &l);
    if (A.hdr_out) { A.hdr_out[3 * p] = o.x; A.hdr_out[3 * p + 1] = o.y; A.hdr_out[3 * p + 2] = o.z; }
    if (A.var_out) { A.var_out[3 * p] = v.x; A.var_out[3 * p + 1] = v.y; A.var_out[3 * p + 2] = v.z; }
    if (A.len_out) A.len_out[p] = l;
}

}  // namespace
}  // namespace rbrt

extern "C" int rbrt_temporal_launch(const rbrt::TemporalArgs* a, cudaStream_t stream) {
    const size_t n = (size_t)a->W * a->H;
    if (!n) return (int)cudaSuccess;
    rbrt::k_temporal<<<(unsigned)((n + TP_THREADS - 1) / TP_THREADS), TP_THREADS, 0, stream>>>(*a);
    return (int)cudaGetLastError();
}
