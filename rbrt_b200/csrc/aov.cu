// aov.cu — first-hit AOVs (rbrt_gpu_render_aov / rbrt_gpu_render_aov_device): per pixel the mean depth, shading normal and albedo of
// the camera rays' closest hits, the share of samples that hit, and the ids of sample 0's hit.
//
// Built into its own shared object (librbrt_gpu_aov.so), which librbrt_gpu.so loads at run time: the device code of librbrt_gpu.so
// stays exactly the build the GPU tests verified.  Every value is composed from functions the renderer and the parity hooks use:
//   ray  = camera_ray (shade.cuh), the ray rbrt_gpu_primary_rays returns for (seed, sample);
//   hit  = scene_hit<false> (intersect.cuh), the closest-hit query of rbrt_gpu_trace_rays(RBRT_TRACE_BVH), bit for bit;
//   then the rules of include/rbrt_gpu.h (DESIGN.md section 11): f32 sums in sample order over the hit samples, one division.
// One warp is one 8x4-pixel tile (the renderer's tile order: neighbouring lanes trace neighbouring rays), one lane one pixel, and the
// lane runs its pixel's whole sample loop, so the order of every sum is fixed.
#include "aov.cuh"
#include "intersect.cuh"
#include "shade.cuh"

namespace rbrt {
namespace {

#define AOV_THREADS 128

template <bool STATS>
__global__ void __launch_bounds__(AOV_THREADS) k_aov(AovArgs A) {
    const uint32_t gt = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t T = gt >> 5, lane = gt & 31;
    uint32_t nan_count = 0;
    TraceCounters cnt; cnt.nodes = 0; cnt.tris = 0;
    const uint32_t ty = T / A.tiles_x, tx = T - ty * A.tiles_x;
    const uint32_t col = tx * 8 + (lane & 7), row = ty * 4 + (lane >> 3);
    if (T < A.tiles_total && col < A.cam.width && row < A.cam.height) {
        const SceneDev& S = A.S;
        const uint32_t px = row * A.cam.width + col;
        RngKey key; key.k0 = A.key0; key.k1 = A.key1;
        float depth = 0.0f;
        f3 nrm = mk3(0.0f, 0.0f, 0.0f), alb = mk3(0.0f, 0.0f, 0.0f);
        uint32_t n_hit = 0;
        int32_t kind0 = RBRT_HIT_NONE;
        uint32_t elem0 = 0, tri0 = 0;
        for (uint32_t s = 0; s < A.n_samples; ++s) {
            f3 o, d;
            camera_ray(A.cam, row, col, key, px, s, o, d);
            const Hit h = scene_hit<false>(S, o, d, STATS ? &cnt : nullptr);
            if (h.kind < 0) { if (h.kind == -2) ++nan_count; continue; }   // -2: a NaN ray (the reference panics): a miss here
            const f3 p = o + h.t * d;                                     // ray.point_at (sphere.rs:49, mesh.rs:247)
            f3 n;
            uint32_t e;
            bool basic = false;
            if (h.kind == 0) {
                basic = S.n_etris && __ldg(S.elem_kind + h.elem);
                n = element_normal(S, h.elem, p);
                if (!basic) n = norm3(n);                                 // sphere: p - c divided by len3(p - c)
                e = h.elem;
            } else {
                const float4 nn = __ldg(S.normals + S.meshes[h.elem].nrm_base + h.tri);
                n = mk3(nn.x, nn.y, nn.z);
                e = S.n_spheres + h.elem;
            }
            f3 a = mk3(1.0f, 1.0f, 1.0f);                                 // Dielectric: attenuation (1,1,1) (dielectric.rs:19)
            if (__ldg(S.mat_kind + e) != RBRT_MAT_DIELECTRIC) { const float4 m = __ldg(S.mat + e); a = mk3(m.x, m.y, m.z); }
            depth = XADD(depth, h.dist);
            nrm = nrm + n;
            alb = alb + a;
            ++n_hit;
            if (s == 0) { kind0 = h.kind == 1 ? RBRT_HIT_MESH : (basic ? RBRT_HIT_TRIANGLE : RBRT_HIT_SPHERE); elem0 = h.elem; tri0 = h.tri; }
        }
        const rbrt_aov_out& out = A.out;
        if (n_hit) {
            const float k = (float)n_hit;
            depth = XDIV(depth, k);
            nrm = mk3(XDIV(nrm.x, k), XDIV(nrm.y, k), XDIV(nrm.z, k));
            alb = mk3(XDIV(alb.x, k), XDIV(alb.y, k), XDIV(alb.z, k));
        } else {
            depth = __int_as_float(0x7F800000);                           // +inf: nothing was hit
        }
        if (out.depth) out.depth[px] = depth;
        if (out.normal) { float* q = out.normal + 3 * (size_t)px; q[0] = nrm.x; q[1] = nrm.y; q[2] = nrm.z; }
        if (out.albedo) { float* q = out.albedo + 3 * (size_t)px; q[0] = alb.x; q[1] = alb.y; q[2] = alb.z; }
        if (out.coverage) out.coverage[px] = XDIV((float)n_hit, (float)A.n_samples);
        if (out.hit_kind) out.hit_kind[px] = kind0;
        if (out.elem_idx) out.elem_idx[px] = elem0;
        if (out.tri_idx) out.tri_idx[px] = tri0;
    }
    if (STATS) {
        unsigned long long nodes = cnt.nodes, tris = cnt.tris;
        for (int off = 16; off; off >>= 1) {
            nan_count += __shfl_down_sync(0xFFFFFFFFu, nan_count, off);
            nodes += __shfl_down_sync(0xFFFFFFFFu, nodes, off);
            tris += __shfl_down_sync(0xFFFFFFFFu, tris, off);
        }
        if (lane == 0) {
            if (nan_count) atomicAdd(&A.stats[AOV_ST_NAN], (unsigned long long)nan_count);
            if (nodes) atomicAdd(&A.stats[AOV_ST_NODES], nodes);
            if (tris) atomicAdd(&A.stats[AOV_ST_TRIS], tris);
        }
    }
}

}  // namespace
}  // namespace rbrt

extern "C" int rbrt_aov_launch(const rbrt::AovArgs* a, cudaStream_t stream) {
    const uint64_t threads = 32ull * a->tiles_total;
    if (!threads) return (int)cudaSuccess;
    const unsigned grid = (unsigned)((threads + AOV_THREADS - 1) / AOV_THREADS);
    if (a->stats) rbrt::k_aov<true><<<grid, AOV_THREADS, 0, stream>>>(*a);
    else rbrt::k_aov<false><<<grid, AOV_THREADS, 0, stream>>>(*a);
    return (int)cudaGetLastError();
}
