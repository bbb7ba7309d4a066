// multi.cuh — multi-GPU behind the C-ABI: the communicator (NCCL or peer-mapped memory), scene replication and the
// collective render (per-GPU shard -> per-GPU finalise -> gather on rank 0).  See multi.cu.
#pragma once
#include <vector>
#include "engine.cuh"

namespace rbrt {

struct Comm {
    bool active = false, multi_process = false;
    int world = 1, rank = 0, local_n = 1, transport = RBRT_TRANSPORT_NCCL, nccl_version = 0;
    std::vector<int> devices;                  // local devices, index = local rank (global rank = rank + index)
    std::vector<void*> nccl;                   // ncclComm_t per local device (NCCL transport)
    std::vector<cudaStream_t> streams;         // [local rank * 4 + pool]: streams of the local GPUs other than the first
};
Comm& comm();

// api.cu
int current_device();
void set_current_device(int d);
int device_sm_count(int device, int* out);
int arena_alloc(int device, size_t bytes, char** base, size_t* got_bytes);
void destroy_scene(Scene* sc);

// multi.cu
// Enqueues, behind the build on `build_stream`, the copy of replica 0's block to the scene's other replicas / ranks and records
// every replica's `ready` event.  Each copy first waits for the reads of the scene enqueued so far on its replica's device (an
// update replicates again while frames of the old geometry may be in flight).
int replicate_scene(Scene* sc, cudaStream_t build_stream);
// The collective render (or, without a communicator, render + finalise on one GPU) with device outputs on rank 0.
int render_frames(const Scene& sc, const rbrt_camera* cams, const uint64_t* seeds, uint32_t n_frames, uint32_t spp,
                  const rbrt_render_opts* opts, uint8_t* const* d_rgb, float* const* d_hdr, cudaStream_t st, rbrt_stats* stats);
void release_dist_buffers();

}  // namespace rbrt
