// engine.cuh — host-side objects behind the opaque rbrt_scene handle and the wavefront state.
#pragma once
#include <mutex>
#include <string>
#include <vector>
#include "../../include/rbrt_gpu.h"
#include "common.cuh"

namespace rbrt {

// Per-iteration queue counters.  All iterations of a batch get their own slot, so one memset per
// batch resets everything and no kernel ever has to reset a counter another kernel still reads.
struct IterCtr {
    uint32_t ray_count;      // rays of this iteration = Scene::hit calls (statistics)
    uint32_t cand_count;     // rays that passed a mesh AABB and are queued for BVH traversal
    uint32_t cand_head;      // persistent-thread work cursor of the trace kernel
    uint32_t mat_count[3];   // hits queued for shading, per material kind
    uint32_t shade_head;     // persistent-thread work cursor of the shade kernel
    uint32_t pad;
};

enum { ST_RAYS = 0, ST_NAN = 1, ST_NODES = 2, ST_TRIS = 3, ST_CAND = 4, ST_TAIL_NODES = 5, ST_TAIL_TRIS = 6, ST_TAIL_CAND = 7, ST_COUNT = 8 };

// Wavefront state.  Every per-path record lives at the path's own index pid (no slot compaction): a
// path's next ray overwrites its previous one, so one ray buffer serves all bounce iterations.
struct WaveBuffers {
    uint32_t cap = 0;            // paths per batch the buffers hold
    uint32_t depth_cap = 0;      // bounce iterations the history/counter arrays hold
    uint4* rec = nullptr;        // [pid] ONE 32-byte record per path = one DRAM sector (render.cu, "path record"): a traversal candidate
                                 //   {t_sphere, sphere | first mesh, origin, direction} or a pending hit {hit point, direction, element, triangle}
    uint32_t* candq = nullptr;   // pids queued for BVH traversal
    uint32_t* matq[2][3] = {{nullptr, nullptr, nullptr}, {nullptr, nullptr, nullptr}};   // pids queued for shading, by iteration parity and material kind
                                 // (k_shade(it) reads parity it&1 while it fills parity (it+1)&1)
    float4* out = nullptr;       // [pid] final radiance of the path (written exactly once, when the path ends)
    uint16_t* hist = nullptr;    // [iteration][pid]: element scattered at (attenuation product when the path ends)
    IterCtr* ctr = nullptr;      // [depth_cap + 2]
    unsigned long long* stats = nullptr;   // ST_COUNT counters
    float4* accum = nullptr;     // internal W*H accumulation buffer for the host-pointer entry points
    size_t accum_px = 0;
    uint8_t* rgb = nullptr; float* hdr = nullptr; size_t out_px = 0;
    std::vector<cudaEvent_t> ev;   // event pool for per-kernel timing (RBRT_OPT_TIME_KERNELS)
    size_t bytes = 0;
};

// A scene's device data is ONE allocation ("arena"); every array sits at a fixed offset, so a replica on another GPU is
// the same bytes at another base address (multi.cu broadcasts the arena instead of rebuilding the LBVH on every GPU).
struct ArenaLayout { size_t nodes = 0, tris = 0, nrm = 0, sph = 0, mat = 0, kind = 0, mesh = 0, etris = 0, ekind = 0, result = 0, total = 0; };
struct Replica { int device = 0; char* arena = nullptr; size_t arena_bytes = 0; SceneDev dev{}; int sm_count = 148;
                 cudaEvent_t ready = nullptr; };   // recorded when this replica's data is complete (build / replication are asynchronous): every reader's stream waits for it
struct SceneUse { int device; cudaStream_t stream; cudaEvent_t ev; };   // last work enqueued on a stream that reads the scene

struct Scene {
    int device = 0;              // device of replica 0 (the one that uploaded and built)
    SceneDev dev{};              // = rep[0].dev
    std::vector<MeshDev> meshes_h;
    std::vector<Replica> rep;    // one per local device of the communicator the scene was created under (else one)
    ArenaLayout lay{};
    uint32_t n_elems = 0, n_meshes = 0, n_etris = 0;
    rbrt_scene_info info{};
    int sm_count = 148;
    bool collective = false;     // created under a communicator: renders with shard_count == 0 are sharded over its ranks
    mutable std::vector<SceneUse> uses;
    // scene_create does not wait for the build: per-mesh results (live nodes, depth, error) arrive in pinned host memory behind info_ev
    void* res_h = nullptr;       // BuildResult[n_meshes]
    cudaEvent_t info_ev = nullptr, t_up0 = nullptr, t_up1 = nullptr, t_b0 = nullptr, t_b1 = nullptr;
    mutable bool info_resolved = false;
    mutable int build_error = 0; // mesh index + 1 whose tree was refused (deeper than the traversal stack), 0 = none
    double ms_host_create = 0;
    // ---- what an update (rbrt_gpu_scene_update_*) needs to know about the creation
    std::vector<uint64_t> mesh_n_all;       // real triangles per mesh (the count an update must hand in)
    std::vector<uint32_t> elem_kind_h;      // RBRT_ELEM_* per element, in order
    float pad_rel = 0.0f;
    uint32_t leaf_size = 1;
    bool sah = true;
    bool replicated = false;                // replicas are copies of replica 0 (one process; or RBRT_SCENE_BROADCAST)
    cudaEvent_t upd_in = nullptr, upd_out = nullptr;   // device-pointer updates: caller's stream -> build stream -> caller's stream
    cudaEvent_t rebuild_ev = nullptr;       // RBRT_UPDATE_REBUILD: the rebuilt mesh's BuildResult has reached res_h
    mutable bool rebuild_pending = false;
    struct Staging { void* p = nullptr; size_t bytes = 0; cudaEvent_t done = nullptr; };
    Staging stage[2];                       // pinned host staging of element / material values, alternating; `done`: its copy has run
    int stage_next = 0;
};
int resolve_scene_info(const Scene& sc, bool wait);   // api.cu: fills info from the build results once they are there (wait: block for them); returns RBRT_E_* if the build refused a mesh
void wait_scene_ready(const Scene& sc, int li, cudaStream_t st);   // makes `st` wait for replica li's data
void wait_scene_uses(const Scene& sc, int device, cudaStream_t st);   // makes `st` wait for every read of the scene enqueued so far on `device` (< 0: any)

// Everything a wavefront kernel needs, passed by value (kernel parameter space).
struct WaveParams {
    SceneDev S;
    CamDev cam[RBRT_MAX_FRAMES];                 // one camera and one Philox key per FRAME of the batch (same image size)
    ShardDev sh;
    uint32_t key0[RBRT_MAX_FRAMES], key1[RBRT_MAX_FRAMES];
    uint32_t n_frames;       // frames rendered together: path id = ((f * s_count + s_local) * paths_px + j
    FastDiv fd_s_count;      // division by s_count (frame index of a path)
    uint32_t cap;            // capacity of the per-path buffers = paths of a full batch
    uint32_t paths_px;       // P_r = tiles_mine * 32: path id = s_local * paths_px + j
    FastDiv fd_paths_px;     // division by paths_px
    uint32_t s_base;         // first sample index of this batch
    uint32_t s_count;        // samples in this batch
    uint32_t max_depth;      // 50 (lib.rs:99)
    uint32_t fetch_thr;      // k_trace re-fills a warp from the queue when fewer lanes than this still traverse
    uint32_t tail_thr;       // the same for k_tail, whose "re-fill" also shades the lanes' pending hits
    uint32_t use_cull;       // k_generate skips provably missed elements of camera rays (render.cu cone_of_sphere)
    uint32_t keep_t;         // resolve() also leaves t in out[pid].x (rbrt_gpu_trace_rays reports it; a render does not need it)
    uint4* rec;
    uint32_t* candq; uint32_t* matq[2][3];
    float4* out; uint16_t* hist; IterCtr* ctr; unsigned long long* stats;
};

void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);

std::recursive_mutex& api_mutex();          // serialises every entry point (api.cu)
uint64_t pool_limit_bytes();                // rbrt_gpu_set_pool_limit
SceneDev make_scene_dev(char* base, const ArenaLayout& lay, uint32_t n_elems, uint32_t n_meshes, uint32_t n_etris);

// render.cu
// What a render left behind for its statistics (device counters, events); collect_stats() waits for the frame and reads them.
struct RenderJob {
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    WaveBuffers* wb = nullptr, *wb2 = nullptr;   // wb2: the second lane's pool (RBRT_OPT_SPLIT_BATCHES)
    ShardDev sh{};
    uint32_t P = 0, n_frames = 0, W = 0, H = 0, launches = 0, iterations = 0, batch_iters = 0, flags = 0, max_depth = 0;
    bool rendered = false;
    ~RenderJob() { if (ev0) cudaEventDestroy(ev0); if (ev1) cudaEventDestroy(ev1); }
};
int make_shard(const rbrt_render_opts& o, uint32_t W, uint32_t H, uint32_t spp, ShardDev* out);
// Renders replica `li` of the scene on that replica's device (the caller has made it current).  With `job` the call only
// enqueues and fills *job (collect_stats later); without, stats (may be NULL = enqueue only) are collected before returning.
// pool: the wavefront pool, 0..7 (4 + p: the second lane of pool p, see RBRT_OPT_SPLIT_BATCHES); -1 = the one opts->flags name.
int render_accum(const Scene& sc, int li, const rbrt_camera* cams, const uint64_t* seeds, uint32_t n_frames, uint32_t spp,
                 const rbrt_render_opts* opts, float4* const* d_accum, cudaStream_t st, rbrt_stats* stats, RenderJob* job = nullptr,
                 int pool = -1);
int collect_stats(RenderJob& job, rbrt_stats* stats);
int trace_rays_wavefront(const Scene& sc, const rbrt_ray* d_rays, uint64_t n, rbrt_hit* d_hits, unsigned long long* d_stats, cudaStream_t st);
int scatter_device(const rbrt_scatter_in* d_in, uint64_t n, uint64_t seed, rbrt_scatter_out* d_out, cudaStream_t st);
void note_scene_use(const Scene& sc, int device, cudaStream_t st);   // records the scene's last-use event on `st`
int finalize(const float4* d_accum, uint32_t W, uint32_t H, uint32_t spp, uint8_t* d_rgb, float* d_hdr, cudaStream_t st);
int trace_rays_device(const Scene& sc, const rbrt_ray* d_rays, uint64_t n, uint32_t mode, rbrt_hit* d_hits,
                      unsigned long long* d_stats, cudaStream_t st);
int primary_rays_device(const rbrt_camera& cam, uint64_t seed, uint32_t sample, rbrt_ray* d_rays, cudaStream_t st);
CamDev make_cam(const rbrt_camera& c);       // the kernels' view of a camera
void free_wave_buffers(WaveBuffers& wb);
// Per-device pool of wavefront state, shared by every scene of the process and kept between renders (allocating and
// freeing tens of GB per render would cost more than the render).  The library is single-threaded per device.
WaveBuffers& device_wave_buffers(int device, int pool = 0);
void release_device_wave_buffers();

}  // namespace rbrt
