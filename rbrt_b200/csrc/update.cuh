// update.cuh — the launch interface of the refit module (update.cu, built into librbrt_gpu_update.so).
// librbrt_gpu.so loads that module at run time (api.cu) and hands it raw device pointers and a stream; the module owns no state.
#pragma once
#include "bvh_build.cuh"

namespace rbrt {

// One mesh of a scene, in the scene's device block (replica 0), plus the new vertices.
struct RefitArgs {
    const float* raw;            // n_all x 9 floats, world space, original order (device memory)
    uint64_t n_all;              // real triangles (the AABB covers all of them, also those the SIMD tail rule drops)
    uint32_t n_eff;              // triangles in the tree (N_eff)
    float pad_rel;               // the scene's relative leaf-box padding (0 = none)
    MeshDev* mesh;               // the mesh's record
    float4* tris;                // its n_eff triangle records (Morton order)
    float4* normals;             // its n_eff unit normals (original order)
    uint4* nodes;                // its 4-wide nodes (n_eff - 1 slots)
    const BuildResult* res;      // its build result: live_nodes = the nodes in use
};

}  // namespace rbrt

extern "C" {
// Bytes of device scratch rbrt_update_refit needs for a mesh of n_eff triangles (256-byte aligned base).
typedef size_t (*rbrt_update_scratch_bytes_fn)(uint64_t n_eff);
// Enqueues the refit of one mesh on `stream`; returns a cudaError_t.
typedef int (*rbrt_update_refit_fn)(const rbrt::RefitArgs* args, void* scratch, cudaStream_t stream);
}
