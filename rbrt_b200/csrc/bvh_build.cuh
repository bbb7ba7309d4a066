// bvh_build.cuh — the GPU LBVH builder (bvh_build.cu): fully ASYNCHRONOUS.  A scene's meshes are uploaded on a copy stream
// and built on a build stream of the device; nothing is read back to the host on the way (the exact mesh AABB, the node
// grid and the MeshDev record are produced and consumed on the device), so rbrt_gpu_scene_create returns as soon as the
// triangle soup has left the caller's arrays, while renders of earlier frames keep the SMs busy.
#pragma once
#include "common.cuh"

namespace rbrt {

struct BuildResult { uint32_t live_nodes, depth, error, pad; };      // per mesh, written on the device when its tree is complete

struct BuildCtx {
    int device = 0, slot = 0;
    cudaStream_t copy = nullptr, build = nullptr;    // per-device streams (non-blocking): H2D uploads / build kernels
};

// Picks one of the device's two scratch slots (a create can upload while the previous scene's build is still running).
cudaError_t build_begin(int device, BuildCtx* ctx);
// One mesh: H2D of its n_all x 9 floats (HOST pointer, world space, original order) on ctx.copy, then on ctx.build the exact
// AABB over ALL of them (aabbox.rs:62-88), the MeshDev record (*d_mesh = proto + box + node grid), n_eff triangle records
// (Morton order), unit normals (ORIGINAL order), up to n_eff - 1 64-byte 4-wide nodes, and *d_res.
// sah: tree rotations during the refit (one-triangle leaves only).
// h_tris may also be a device pointer of ctx.device (rbrt_gpu_scene_update_mesh_device); src_ready: an event the copy waits for first.
cudaError_t build_mesh(BuildCtx& ctx, const float* h_tris, uint64_t n_all, uint32_t n_eff, float pad_rel, uint32_t leaf_size, bool sah,
                       const MeshDev& proto, MeshDev* d_mesh, float4* d_tris, float4* d_normals, float4* d_nodes, BuildResult* d_res,
                       cudaEvent_t src_ready = nullptr);
// The scratch slot ctx.slot for an update (rbrt_gpu_scene_update_mesh, RBRT_UPDATE_REFIT): grown to `bytes` and made to wait, on
// ctx.copy, for the last build that read it.  The caller enqueues its uploads on ctx.copy, then build_slot_uploaded (ctx.build
// waits for them; the returned event completes when the caller's arrays have been read), its kernels on ctx.build, then
// build_slot_release (the slot is busy until they are done).
cudaError_t build_slot_acquire(BuildCtx& ctx, size_t bytes, char** base);
cudaError_t build_slot_uploaded(BuildCtx& ctx, cudaEvent_t* uploaded);
cudaError_t build_slot_release(BuildCtx& ctx);
// Event recorded on ctx.copy after the last upload: once it has completed the caller's arrays are no longer read.
cudaError_t build_uploads_done(BuildCtx& ctx, cudaEvent_t ev);
void release_build_scratch();

}  // namespace rbrt
