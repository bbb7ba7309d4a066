// aov.cuh — the launch interface of the first-hit AOV module (aov.cu, built into librbrt_gpu_aov.so).
// librbrt_gpu.so loads that module at run time (api.cu) and hands it the scene's device view, the camera, the Philox key and raw
// device pointers of the requested passes; the module owns no state.
#pragma once
#include "../../include/rbrt_gpu.h"
#include "common.cuh"

namespace rbrt {

enum { AOV_ST_NAN = 0, AOV_ST_NODES = 1, AOV_ST_TRIS = 2, AOV_ST_COUNT = 4 };

struct AovArgs {
    SceneDev S;                  // replica 0 of the scene
    CamDev cam;
    uint32_t key0, key1;         // Philox key = the call's seed
    uint32_t n_samples;          // samples per pixel, s = 0 .. n_samples - 1
    uint32_t tiles_x, tiles_total;   // 8x4-pixel tiles of the image: one warp per tile, one lane per pixel
    rbrt_aov_out out;            // device planes; a NULL member is not written
    unsigned long long* stats;   // AOV_ST_COUNT counters, or NULL (no counting)
};

}  // namespace rbrt

extern "C" {
// Enqueues the AOV kernel on `stream`; returns a cudaError_t.
typedef int (*rbrt_aov_launch_fn)(const rbrt::AovArgs* args, cudaStream_t stream);
}
