// lbvh_harness.cu — linked with rbrt_b200/csrc/bvh_build.cu into a test-owned shared object: one mesh built by the product's
// build_begin + build_mesh into buffers the caller owns, then a synchronise.  Only this entry point is exported; the object is
// linked -Bsymbolic, so its rbrt:: symbols and static state stay its own when librbrt_gpu.so is loaded in the same process.
#include "bvh_build.cuh"

extern "C" __attribute__((visibility("default"))) int lbvh_harness_build(int device, const float* raw, uint64_t n_all, uint32_t n_eff, float pad_rel,
                                                                         uint32_t leaf_size, int sah, const void* proto, void* d_mesh, void* d_tris,
                                                                         void* d_normals, void* d_nodes, void* d_res) {
    cudaError_t e = cudaSetDevice(device);
    rbrt::BuildCtx ctx;
    if (e == cudaSuccess) e = rbrt::build_begin(device, &ctx);
    if (e == cudaSuccess)
        e = rbrt::build_mesh(ctx, raw, n_all, n_eff, pad_rel, leaf_size, sah != 0, *static_cast<const rbrt::MeshDev*>(proto), static_cast<rbrt::MeshDev*>(d_mesh),
                             static_cast<float4*>(d_tris), static_cast<float4*>(d_normals), static_cast<float4*>(d_nodes), static_cast<rbrt::BuildResult*>(d_res));
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx.build);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx.copy);
    return (int)e;
}
