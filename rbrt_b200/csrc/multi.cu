// multi.cu — multi-GPU inside the C-ABI.
//
// The reference's one parallelism strategy lives inside render_scene: rayon over image columns
// (rbrt_lib/src/lib.rs:84-86), no state shared between pixels.  Here the same call shards the image over the GPUs
// of one box: interleaved 8x4-pixel tiles (sky tiles are cheap, mesh tiles expensive: interleaving balances) or
// sample ranges.  There is no exchange step inside the path; what moves between GPUs is
//   * the scene, once: rank 0 uploads and builds the LBVH, the block is replicated over NVLink
//     (ncclBroadcast, or peer copies), instead of N uploads over PCIe and N builds;
//   * the result, once per frame: every GPU applies lib.rs:101,116-122 (x 1/spp, sqrt, x256, saturating u8) to ITS
//     pixels, and rank 0 gathers 3 bytes per pixel (tile shards) — or, for sample shards, the f32 accumulators are
//     summed (ncclReduce / a peer-reading sum kernel) and rank 0 finalises.
// Two transports.  NCCL (one process per GPU, or one process): grouped ncclSend/ncclRecv of each rank's slab of
// finalised pixels (shard order) + one un-tiling kernel on rank 0.  PEER (one process): the finalise kernel of every
// GPU stores its pixels straight into rank 0's image through peer-mapped memory — the compute step and its gather are
// ONE kernel, the stores travel over NVLink while the kernel runs, and rank 0 only waits for an event per GPU.
// NCCL is loaded at run time (dlopen), so a one-GPU host does not need it.
#include <dlfcn.h>
#include <nccl.h>
#include <chrono>
#include <condition_variable>
#include <cstdio>
#include <cstring>
#include <functional>
#include <string>
#include <thread>
#include "bvh_build.cuh"
#include "multi.cuh"
#include "shade.cuh"

namespace rbrt {

#define CKM(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) return cuda_fail(e_, #x); } while (0)

// ------------------------------------------------------------------ NCCL, resolved at run time
struct NcclApi {
    void* handle = nullptr;
    ncclResult_t (*GetVersion)(int*) = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Broadcast)(const void*, void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Reduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, int, ncclComm_t, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
};
static NcclApi g_nccl;

static int load_nccl() {
    if (g_nccl.handle) return RBRT_OK;
    void* h = nullptr;
    const char* env = getenv("RBRT_NCCL_LIB");
    if (env && *env) h = dlopen(env, RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);          // already in the process (e.g. brought in by torch)
    if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) { set_error("NCCL is not available (dlopen libnccl.so.2: %s); set RBRT_NCCL_LIB", dlerror()); return RBRT_E_INVALID; }
    NcclApi a; a.handle = h;
#define SYM(field, name) do { *(void**)(&a.field) = dlsym(h, name); if (!a.field) { set_error("NCCL symbol %s missing", name); return RBRT_E_INVALID; } } while (0)
    SYM(GetVersion, "ncclGetVersion"); SYM(GetUniqueId, "ncclGetUniqueId"); SYM(CommInitRank, "ncclCommInitRank"); SYM(CommInitAll, "ncclCommInitAll");
    SYM(CommDestroy, "ncclCommDestroy"); SYM(GroupStart, "ncclGroupStart"); SYM(GroupEnd, "ncclGroupEnd"); SYM(Send, "ncclSend"); SYM(Recv, "ncclRecv");
    SYM(Broadcast, "ncclBroadcast"); SYM(Reduce, "ncclReduce"); SYM(GetErrorString, "ncclGetErrorString");
#undef SYM
    g_nccl = a;
    return RBRT_OK;
}
static int nccl_fail(ncclResult_t r, const char* what) {
    set_error("NCCL error %d (%s) at %s", (int)r, g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?", what);
    return RBRT_E_CUDA;
}
#define CKN(x) do { ncclResult_t r_ = (x); if (r_ != ncclSuccess) return nccl_fail(r_, #x); } while (0)

static Comm g_comm;
Comm& comm() { return g_comm; }

// ------------------------------------------------------------------ per (pool, local rank) buffers of the collective render
struct DistBuffers {
    int device = -1;
    float4* accum[RBRT_MAX_FRAMES] = {nullptr, nullptr, nullptr, nullptr}; size_t accum_px = 0; uint32_t accum_n = 0;
    uint8_t* slab = nullptr; size_t slab_bytes = 0;          // this rank's finalised pixels in shard order (NCCL transport)
    cudaEvent_t ev_start = nullptr, ev_done = nullptr;       // fork / join of the local GPUs of a one-process render
};
static DistBuffers g_dist[4][16];
static uint8_t* g_gather[4] = {nullptr, nullptr, nullptr, nullptr};   // rank 0: the slabs of all ranks
static size_t g_gather_bytes[4] = {0, 0, 0, 0};
static int g_gather_dev[4] = {-1, -1, -1, -1};

static void free_dist(DistBuffers& d) {
    if (d.device < 0) return;
    cudaSetDevice(d.device);
    for (auto& p : d.accum) { cudaFree(p); p = nullptr; }
    cudaFree(d.slab);
    if (d.ev_start) cudaEventDestroy(d.ev_start);
    if (d.ev_done) cudaEventDestroy(d.ev_done);
    d = DistBuffers();
}
void release_dist_buffers() {
    int cur = 0; cudaGetDevice(&cur);
    for (int p = 0; p < 4; ++p) {
        for (int l = 0; l < 16; ++l) free_dist(g_dist[p][l]);
        if (g_gather[p]) { cudaSetDevice(g_gather_dev[p]); cudaFree(g_gather[p]); g_gather[p] = nullptr; g_gather_bytes[p] = 0; g_gather_dev[p] = -1; }
    }
    cudaSetDevice(cur);
}
// the caller has made `device` current
static int ensure_dist(DistBuffers& d, int device, size_t n_px, uint32_t n_frames, size_t slab_bytes) {
    if (d.device != device) { free_dist(d); cudaSetDevice(device); d.device = device; }
    // every allocated accumulator holds accum_px pixels: one added for a further frame gets the size of those already there, not
    // n_px (a smaller image), or a later, larger image with that many frames would pass the size check and not fit in it
    if (d.accum_px < n_px) { for (auto& p : d.accum) { cudaFree(p); p = nullptr; } d.accum_px = n_px; d.accum_n = 0; }
    for (uint32_t f = 0; f < n_frames; ++f)
        if (!d.accum[f]) { CKM(cudaMalloc(&d.accum[f], 16 * d.accum_px)); }
    d.accum_n = std::max(d.accum_n, n_frames);
    if (d.slab_bytes < slab_bytes) { cudaFree(d.slab); d.slab = nullptr; d.slab_bytes = 0; CKM(cudaMalloc(&d.slab, slab_bytes)); d.slab_bytes = slab_bytes; }
    if (!d.ev_start) { CKM(cudaEventCreateWithFlags(&d.ev_start, cudaEventDisableTiming)); CKM(cudaEventCreateWithFlags(&d.ev_done, cudaEventDisableTiming)); }
    return RBRT_OK;
}

// ------------------------------------------------------------------ kernels
// lib.rs:101 + lib.rs:116-122 for the pixels of ONE rank's tile shard.  DIRECT: the result goes to its place in the
// full row-major image `out` — rank 0's image, reached through peer-mapped memory on the other GPUs (the stores cross
// NVLink while the kernel runs: finalise + gather in one kernel).  Otherwise it goes to slot j of the rank's slab.
template <typename T, bool DIRECT>
__global__ void __launch_bounds__(256) k_finalize_shard(const float4* __restrict__ accum, ShardDev sh, uint32_t W, uint32_t H, uint32_t P,
                                                        float inv_spp, T* __restrict__ out) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= P) return;
    CamDev cam; cam.width = W; cam.height = H;
    uint32_t row, col;
    if (!shard_pixel(sh, cam, j, row, col)) return;
    const size_t px = (size_t)row * W + col;
    const float4 a = accum[px];
    const f3 c = mk3(a.x, a.y, a.z) * inv_spp;                            // lib.rs:101
    T* o = out + 3 * (DIRECT ? px : (size_t)j);
    if (sizeof(T) == 1) {                                                 // lib.rs:118-120
        o[0] = (T)as_u8(XMUL(XSQRT(c.x), 256.0f)); o[1] = (T)as_u8(XMUL(XSQRT(c.y), 256.0f)); o[2] = (T)as_u8(XMUL(XSQRT(c.z), 256.0f));
    } else { o[0] = (T)c.x; o[1] = (T)c.y; o[2] = (T)c.z; }
}

// rank 0: slabs of all ranks (shard order) -> row-major images.  off_px[r] = first pixel slot of rank r's slab.
struct GatherMap { uint32_t off_px[65]; uint32_t world, tiles_x, tiles_total, W, H; FastDiv fd_tiles_x, fd_world; };
struct OutPtrs { void* p[RBRT_MAX_FRAMES]; };
template <typename T>
__global__ void __launch_bounds__(256) k_untile(const T* __restrict__ gather, GatherMap g, OutPtrs out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;             // tile * 32 + lane
    const uint32_t f = blockIdx.y, n_frames = gridDim.y;
    const uint32_t tile = i >> 5, lane = i & 31;
    if (tile >= g.tiles_total) return;
    const uint32_t tj = fast_div(tile, g.fd_world), r = tile - tj * g.world;
    const uint32_t ty = fast_div(tile, g.fd_tiles_x), tx = tile - ty * g.tiles_x;
    const uint32_t col = tx * 8 + (lane & 7), row = ty * 4 + (lane >> 3);
    if (col >= g.W || row >= g.H) return;
    const uint32_t P_r = (g.off_px[r + 1] - g.off_px[r]) / n_frames;      // pixel slots of rank r per frame
    const T* src = gather + 3 * ((size_t)g.off_px[r] + (size_t)f * P_r + tj * 32 + lane);
    T* dst = (T*)out.p[f] + 3 * ((size_t)row * g.W + col);
    dst[0] = src[0]; dst[1] = src[1]; dst[2] = src[2];
}

// sample shards, PEER transport: rank 0 sums the ranks' accumulators in rank order, reading them through peer-mapped memory
struct PeerPtrs { const float4* p[16]; uint32_t n; };
__global__ void __launch_bounds__(256) k_sum_peers(float4* __restrict__ dst, PeerPtrs src, size_t n_px) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_px) return;
    float4 a = dst[i];
    for (uint32_t r = 1; r < src.n; ++r) { const float4 b = src.p[r][i]; a.x = XADD(a.x, b.x); a.y = XADD(a.y, b.y); a.z = XADD(a.z, b.z); }
    dst[i] = a;
}

// ------------------------------------------------------------------ scene replication
int replicate_scene(Scene* sc, cudaStream_t bs) {
    // Enqueued, not waited for: the build on rank 0's build stream `bs` is followed by the copy of the WHOLE block (its size is
    // known to every rank from the scene description alone; how many LBVH node slots are live is only known on the device),
    // and every replica's `ready` event is recorded behind its copy.
    Comm& C = g_comm;
    const size_t bytes = sc->lay.total;
    if (C.multi_process) {
        CKM(cudaSetDevice(C.devices[0]));
        wait_scene_uses(*sc, C.devices[0], bs);
        CKN(g_nccl.Broadcast(sc->rep[0].arena, sc->rep[0].arena, bytes, ncclChar, 0, (ncclComm_t)C.nccl[0], bs));
        CKM(cudaEventRecord(sc->rep[0].ready, bs));
        return RBRT_OK;
    }
    std::vector<cudaStream_t> s_of(C.local_n, bs);
    for (int li = 1; li < C.local_n; ++li) {
        if (C.devices[li] == C.devices[0]) continue;
        CKM(cudaSetDevice(C.devices[li]));
        BuildCtx other; cudaError_t e = build_begin(C.devices[li], &other);
        if (e != cudaSuccess) return cuda_fail(e, "build_begin");
        s_of[li] = other.build;
    }
    for (int li = 0; li < C.local_n; ++li) {                              // readers of the replica this copy overwrites
        CKM(cudaSetDevice(C.devices[li]));
        if (s_of[li] != bs) wait_scene_uses(*sc, C.devices[li], s_of[li]);
    }
    CKM(cudaSetDevice(C.devices[0]));
    wait_scene_uses(*sc, -1, bs);                                         // the peer copies below run on bs
    if (C.transport == RBRT_TRANSPORT_NCCL) {
        CKN(g_nccl.GroupStart());
        for (int li = 0; li < C.local_n; ++li)
            CKN(g_nccl.Broadcast(sc->rep[li].arena, sc->rep[li].arena, bytes, ncclChar, 0, (ncclComm_t)C.nccl[li], s_of[li]));
        CKN(g_nccl.GroupEnd());
        for (int li = 0; li < C.local_n; ++li) { CKM(cudaSetDevice(C.devices[li])); CKM(cudaEventRecord(sc->rep[li].ready, s_of[li])); }
    } else {
        for (int li = 1; li < C.local_n; ++li) {
            if (C.devices[li] == C.devices[0]) CKM(cudaMemcpyAsync(sc->rep[li].arena, sc->rep[0].arena, bytes, cudaMemcpyDeviceToDevice, bs));
            else CKM(cudaMemcpyPeerAsync(sc->rep[li].arena, C.devices[li], sc->rep[0].arena, C.devices[0], bytes, bs));
        }
        CKM(cudaEventRecord(sc->rep[0].ready, bs));                        // behind the build AND the copies
        for (int li = 1; li < C.local_n; ++li) {
            if (C.devices[li] == C.devices[0]) { CKM(cudaEventRecord(sc->rep[li].ready, bs)); continue; }
            CKM(cudaSetDevice(C.devices[li]));                             // an event is recorded on a stream of ITS device: hop over
            CKM(cudaStreamWaitEvent(s_of[li], sc->rep[0].ready, 0));
            CKM(cudaEventRecord(sc->rep[li].ready, s_of[li]));
        }
    }
    CKM(cudaSetDevice(C.devices[0]));
    return RBRT_OK;
}

// ------------------------------------------------------------------ one enqueue thread per local GPU (one process driving several GPUs)
// Kernel launches are asynchronous but not free: a frame is 28-40 launches per GPU, ~0.13 ms of host time, and one thread feeding
// eight GPUs in turn lets the last one start a millisecond late.  The threads only ENQUEUE (they hold no CUDA state of their own
// beyond the current device); the caller waits for all of them before it issues the collective part on its own thread.
struct Workers {
    std::vector<std::thread> th;
    std::mutex mu;
    std::condition_variable cv_go, cv_done;
    std::function<int(int)> job;
    std::vector<int> rc;
    std::vector<std::string> msg;
    uint64_t gen = 0;
    int pending = 0;
    bool stop = false;
};
static Workers* g_workers = nullptr;

static void worker_main(Workers* w, int li) {
    uint64_t seen = 0;
    for (;;) {
        std::function<int(int)> job;
        {
            std::unique_lock<std::mutex> lk(w->mu);
            w->cv_go.wait(lk, [&] { return w->stop || w->gen != seen; });
            if (w->stop) return;
            seen = w->gen; job = w->job;
        }
        const int rc = job(li);
        std::string m = rc ? rbrt_last_error() : "";
        std::lock_guard<std::mutex> lk(w->mu);
        w->rc[li] = rc; w->msg[li] = m;
        if (--w->pending == 0) w->cv_done.notify_all();
    }
}
static void workers_start(int n) {
    Workers* w = new Workers();
    w->rc.assign(n, 0); w->msg.assign(n, "");
    for (int li = 0; li < n; ++li) w->th.emplace_back(worker_main, w, li);
    g_workers = w;
}
static void workers_stop() {
    Workers* w = g_workers;
    if (!w) return;
    { std::lock_guard<std::mutex> lk(w->mu); w->stop = true; }
    w->cv_go.notify_all();
    for (auto& t : w->th) t.join();
    delete w; g_workers = nullptr;
}
static bool workers_ready(int n) {
    static const bool off = getenv("RBRT_NO_ENQUEUE_THREADS") != nullptr;  // A/B knob
    return !off && g_workers && (int)g_workers->th.size() == n;
}
static int workers_run(int n, const std::function<int(int)>& job) {
    Workers* w = g_workers;
    {
        std::lock_guard<std::mutex> lk(w->mu);
        w->job = job; w->pending = n; ++w->gen;
        for (int i = 0; i < n; ++i) { w->rc[i] = 0; w->msg[i].clear(); }
    }
    w->cv_go.notify_all();
    std::unique_lock<std::mutex> lk(w->mu);
    w->cv_done.wait(lk, [&] { return w->pending == 0; });
    for (int i = 0; i < n; ++i) if (w->rc[i]) { set_error("%s", w->msg[i].c_str()); return w->rc[i]; }
    return RBRT_OK;
}

// ------------------------------------------------------------------ the collective render
static void add_stats(rbrt_stats* t, const rbrt_stats& s) {
    t->rays += s.rays; t->paths += s.paths; t->nan_rays += s.nan_rays; t->node_visits += s.node_visits; t->tri_tests += s.tri_tests;
    t->traversed_rays += s.traversed_rays; t->tail_node_visits += s.tail_node_visits; t->tail_tri_tests += s.tail_tri_tests;
    t->tail_traversed_rays += s.tail_traversed_rays; t->launches += s.launches;
    t->iterations = std::max(t->iterations, s.iterations); t->ms_device = std::max(t->ms_device, s.ms_device); t->ms_trace = std::max(t->ms_trace, s.ms_trace);
}

template <typename T>
static int finalize_shard(const DistBuffers& D, uint32_t n_frames, const ShardDev& sh, uint32_t W, uint32_t H, uint32_t spp, bool direct,
                          T* const* direct_out, T* slab, cudaStream_t st) {
    const uint32_t P = sh.tiles_mine * 32;
    if (!P) return RBRT_OK;
    const float inv = 1.0f / (float)spp;                                  // lib.rs:101
    for (uint32_t f = 0; f < n_frames; ++f) {
        if (direct) k_finalize_shard<T, true><<<(P + 255) / 256, 256, 0, st>>>(D.accum[f], sh, W, H, P, inv, direct_out[f]);
        else k_finalize_shard<T, false><<<(P + 255) / 256, 256, 0, st>>>(D.accum[f], sh, W, H, P, inv, slab + 3 * (size_t)f * P);
    }
    CKM(cudaGetLastError());
    return RBRT_OK;
}

int render_frames(const Scene& sc, const rbrt_camera* cams, const uint64_t* seeds, uint32_t n_frames, uint32_t spp,
                  const rbrt_render_opts* opts, uint8_t* const* d_rgb, float* const* d_hdr, cudaStream_t st, rbrt_stats* stats) {
    rbrt_render_opts o{}; if (opts) o = *opts;
    const uint32_t W = cams[0].img_width_pix, H = cams[0].img_height_pix;
    const size_t n_px = (size_t)W * H;
    if (!n_px || !spp) { set_error("empty image or zero samples"); return RBRT_E_INVALID; }
    { int rc0 = resolve_scene_info(sc, false); if (rc0) return rc0; }     // a mesh the (asynchronous) build refused, if that is known by now
    const int pool = (int)((o.flags & RBRT_OPT_POOL_MASK) >> RBRT_OPT_POOL_SHIFT);
    Comm& C = g_comm;
    const bool sharded = sc.collective && o.shard_count == 0 && C.active && C.world > 1;
    if (!sharded) {                                                       // one GPU (or an explicit shard placed by the host)
        const int dev = sc.rep[0].device;
        CKM(cudaSetDevice(dev));
        DistBuffers& D = g_dist[pool][0];
        int rc = ensure_dist(D, dev, n_px, n_frames, 0);
        if (rc) return rc;
        rc = render_accum(sc, 0, cams, seeds, n_frames, spp, &o, D.accum, st, stats);
        if (rc) return rc;
        for (uint32_t f = 0; f < n_frames; ++f) {
            rc = finalize(D.accum[f], W, H, spp, d_rgb ? d_rgb[f] : nullptr, d_hdr ? d_hdr[f] : nullptr, st);
            if (rc) return rc;
        }
        if (stats) { stats->launches += n_frames; return resolve_scene_info(sc, true); }
        return RBRT_OK;
    }

    if (C.world > 64 || C.local_n > 16) { set_error("communicator too large"); return RBRT_E_INVALID; }
    const bool samples = o.shard_mode == RBRT_SHARD_SAMPLES;
    const bool peer = C.transport == RBRT_TRANSPORT_PEER;
    const bool i_am_root = C.rank == 0;
    const uint32_t world = (uint32_t)C.world;
    // shard geometry of every rank (tile shards): pixel slots per frame, slab offsets
    rbrt_render_opts og = o; og.shard_mode = RBRT_SHARD_TILES; og.shard_count = world; og.shard_rank = 0;
    ShardDev sh0; { int rc = make_shard(og, W, H, spp, &sh0); if (rc) return rc; }
    GatherMap gm; memset(&gm, 0, sizeof(gm));
    gm.world = world; gm.tiles_x = sh0.tiles_x; gm.tiles_total = sh0.tiles_total; gm.W = W; gm.H = H; gm.fd_tiles_x = sh0.fd_tiles_x; gm.fd_world = make_fastdiv(world);
    for (uint32_t r = 0; r < world; ++r) {
        const uint32_t mine = sh0.tiles_total > r ? (sh0.tiles_total - r + world - 1) / world : 0;
        gm.off_px[r + 1] = gm.off_px[r] + mine * 32 * n_frames;
    }
    const size_t esize = (d_rgb ? 1 : 0) + (d_hdr ? 4 : 0);               // both outputs: the u8 slabs first, then the f32 ones
    const size_t gather_total = 3ull * gm.off_px[world] * esize;
    const size_t hdr_base = d_rgb ? 3ull * gm.off_px[world] : 0;          // byte offset of the f32 part of the gather buffer (16-byte aligned: off_px are multiples of 32)

    const bool dbg = getenv("RBRT_DEBUG_MULTI") != nullptr;
    const auto t_dbg0 = std::chrono::steady_clock::now();
    auto dbg_ms = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_dbg0).count(); };
    std::vector<RenderJob> jobs(stats ? C.local_n : 0);
    rbrt_stats total; memset(&total, 0, sizeof(total));
    CKM(cudaSetDevice(C.devices[0]));
    if (!samples && !peer && i_am_root && g_gather_bytes[pool] < gather_total) {
        cudaFree(g_gather[pool]); g_gather[pool] = nullptr; g_gather_bytes[pool] = 0;
        CKM(cudaMalloc(&g_gather[pool], gather_total)); g_gather_bytes[pool] = gather_total; g_gather_dev[pool] = C.devices[0];
    }
    {
        int rc = ensure_dist(g_dist[pool][0], C.devices[0], n_px, n_frames, 0);
        if (rc) return rc;
    }
    if (C.local_n > 1) CKM(cudaEventRecord(g_dist[pool][0].ev_start, st));
    std::vector<cudaStream_t> s_of(C.local_n);
    std::vector<ShardDev> sh_of(C.local_n);
    bool any_shared = false;                                              // one-GPU emulation of N ranks: several local ranks on one device
    for (int li = 0; li < C.local_n; ++li) for (int lj = 0; lj < li; ++lj) if (C.devices[lj] == C.devices[li]) any_shared = true;
    for (int li = 0; li < C.local_n; ++li) s_of[li] = (li == 0 || C.devices[li] == C.devices[0]) ? st : C.streams[li * 4 + pool];
    std::mutex total_mu;
    // Everything ONE local rank enqueues on its GPU: shard render, finalise of its own pixels (into its slab, or straight into rank 0's
    // image through peer-mapped memory).  Runs on that GPU's enqueue thread when the local GPUs are distinct (see Workers).
    auto enqueue_rank = [&](int li) -> int {
        const int dev = C.devices[li];
        const uint32_t r = (uint32_t)(C.rank + li);
        CKM(cudaSetDevice(dev));
        cudaStream_t s = s_of[li];
        if (s != st) CKM(cudaStreamWaitEvent(s, g_dist[pool][0].ev_start, 0));
        DistBuffers& D = g_dist[pool][li];
        const uint32_t P_r = (gm.off_px[r + 1] - gm.off_px[r]) / n_frames;
        const size_t slab_bytes = (!samples && !peer && r != 0) ? 3ull * P_r * n_frames * esize : 0;
        int rc = ensure_dist(D, dev, n_px, n_frames, slab_bytes);
        if (rc) return rc;
        rbrt_render_opts ol = o;
        ol.shard_mode = samples ? RBRT_SHARD_SAMPLES : RBRT_SHARD_TILES; ol.shard_rank = r; ol.shard_count = world;
        rc = make_shard(ol, W, H, spp, &sh_of[li]);
        if (rc) return rc;
        rc = render_accum(sc, li, cams, seeds, n_frames, spp, &ol, D.accum, s, nullptr, stats ? &jobs[li] : nullptr);
        if (rc) return rc;
        bool shared_dev = false;                                          // does another local rank use this GPU?
        for (int lj = 0; lj < C.local_n; ++lj) if (lj != li && C.devices[lj] == dev) shared_dev = true;
        if (stats && shared_dev) {                                        // the ranks share the device's wavefront pool,
            rbrt_stats one; memset(&one, 0, sizeof(one));                 // so this rank's counters are read before the next rank resets them
            rc = collect_stats(jobs[li], &one); if (rc) return rc;
            std::lock_guard<std::mutex> g(total_mu);
            add_stats(&total, one); jobs[li].wb = nullptr;
        }
        if (!samples) {
            if (peer) {                                                   // finalise + gather in one kernel: stores into rank 0's image
                if (d_rgb) { rc = finalize_shard<uint8_t>(D, n_frames, sh_of[li], W, H, spp, true, d_rgb, nullptr, s); if (rc) return rc; }
                if (d_hdr) { rc = finalize_shard<float>(D, n_frames, sh_of[li], W, H, spp, true, d_hdr, nullptr, s); if (rc) return rc; }
            } else {
                uint8_t* base = r == 0 ? g_gather[pool] : D.slab;          // rank 0 finalises straight into its part of the gather buffer
                const size_t my_hdr = r == 0 ? hdr_base : (d_rgb ? 3ull * P_r * n_frames : 0);
                if (d_rgb) { rc = finalize_shard<uint8_t>(D, n_frames, sh_of[li], W, H, spp, false, nullptr, base, s); if (rc) return rc; }
                if (d_hdr) { rc = finalize_shard<float>(D, n_frames, sh_of[li], W, H, spp, false, nullptr, (float*)(base + my_hdr), s); if (rc) return rc; }
            }
        }
        if (s != st) CKM(cudaEventRecord(D.ev_done, s));
        if (dbg) fprintf(stderr, "[multi] rank %u enqueued at %.3f ms\n", r, dbg_ms());
        return RBRT_OK;
    };
    if (C.local_n > 1 && !any_shared && workers_ready(C.local_n)) {
        int rc = workers_run(C.local_n, enqueue_rank);                    // one enqueue thread per GPU: a frame is 28-40 launches per GPU,
        if (rc) return rc;                                                // 0.13 ms each from one thread = 1 ms of an 8-GPU frame of 6 ms
    } else {
        for (int li = 0; li < C.local_n; ++li) { int rc = enqueue_rank(li); if (rc) return rc; }
    }
    CKM(cudaSetDevice(C.devices[0]));
    static const bool dbg_no_gather = getenv("RBRT_DEBUG_NO_GATHER") != nullptr;   // TIMING EXPERIMENT ONLY: rank 0's image then lacks the other ranks' pixels
    if (!samples) {
        if (!peer && !dbg_no_gather) {
            CKN(g_nccl.GroupStart());
            for (int li = 0; li < C.local_n; ++li) {
                const uint32_t r = (uint32_t)(C.rank + li);
                const uint32_t P_r = (gm.off_px[r + 1] - gm.off_px[r]);   // pixel slots of all frames
                if (r == 0) {
                    for (uint32_t q = 1; q < world; ++q) {
                        const size_t slots = gm.off_px[q + 1] - gm.off_px[q];
                        if (!slots) continue;
                        if (d_rgb) CKN(g_nccl.Recv(g_gather[pool] + 3ull * gm.off_px[q], 3 * slots, ncclChar, (int)q, (ncclComm_t)C.nccl[li], s_of[li]));
                        if (d_hdr) CKN(g_nccl.Recv(g_gather[pool] + hdr_base + 12ull * gm.off_px[q], 3 * slots, ncclFloat, (int)q, (ncclComm_t)C.nccl[li], s_of[li]));
                    }
                } else if (P_r) {
                    DistBuffers& D = g_dist[pool][li];
                    if (d_rgb) CKN(g_nccl.Send(D.slab, 3ull * P_r, ncclChar, 0, (ncclComm_t)C.nccl[li], s_of[li]));
                    if (d_hdr) CKN(g_nccl.Send(D.slab + (d_rgb ? 3ull * P_r : 0), 3ull * P_r, ncclFloat, 0, (ncclComm_t)C.nccl[li], s_of[li]));
                }
            }
            CKN(g_nccl.GroupEnd());
            if (i_am_root) {
                CKM(cudaSetDevice(C.devices[0]));
                const dim3 grid((sh0.tiles_total * 32 + 255) / 256, n_frames);
                OutPtrs op;
                if (d_rgb) { for (uint32_t f = 0; f < RBRT_MAX_FRAMES; ++f) op.p[f] = d_rgb[f < n_frames ? f : 0]; k_untile<uint8_t><<<grid, 256, 0, st>>>(g_gather[pool], gm, op); }
                if (d_hdr) { for (uint32_t f = 0; f < RBRT_MAX_FRAMES; ++f) op.p[f] = d_hdr[f < n_frames ? f : 0]; k_untile<float><<<grid, 256, 0, st>>>((const float*)(g_gather[pool] + hdr_base), gm, op); }
                CKM(cudaGetLastError());
            }
        } else if (peer) {
            CKM(cudaSetDevice(C.devices[0]));
            for (int li = 1; li < C.local_n; ++li) if (s_of[li] != st) CKM(cudaStreamWaitEvent(st, g_dist[pool][li].ev_done, 0));
        }
    } else {
        if (!peer) {                                                      // sample shards: sum the f32 accumulators on rank 0 (lib.rs:96-100 across ranks)
            CKN(g_nccl.GroupStart());
            for (int li = 0; li < C.local_n; ++li)
                for (uint32_t f = 0; f < n_frames; ++f)
                    CKN(g_nccl.Reduce(g_dist[pool][li].accum[f], g_dist[pool][li].accum[f], 4 * n_px, ncclFloat, ncclSum, 0, (ncclComm_t)C.nccl[li], s_of[li]));
            CKN(g_nccl.GroupEnd());
        } else {
            CKM(cudaSetDevice(C.devices[0]));
            for (int li = 1; li < C.local_n; ++li) if (s_of[li] != st) CKM(cudaStreamWaitEvent(st, g_dist[pool][li].ev_done, 0));
            for (uint32_t f = 0; f < n_frames; ++f) {
                PeerPtrs pp; pp.n = (uint32_t)C.local_n;
                for (int li = 0; li < C.local_n; ++li) pp.p[li] = g_dist[pool][li].accum[f];
                k_sum_peers<<<(unsigned)((n_px + 255) / 256), 256, 0, st>>>(g_dist[pool][0].accum[f], pp, n_px);
            }
            CKM(cudaGetLastError());
        }
        if (i_am_root) {
            CKM(cudaSetDevice(C.devices[0]));
            for (uint32_t f = 0; f < n_frames; ++f) {
                int rc = finalize(g_dist[pool][0].accum[f], W, H, spp, d_rgb ? d_rgb[f] : nullptr, d_hdr ? d_hdr[f] : nullptr, st);
                if (rc) return rc;
            }
        }
    }
    if (dbg) fprintf(stderr, "[multi] collectives enqueued at %.3f ms\n", dbg_ms());
    if (stats) {
        for (int li = 0; li < C.local_n; ++li) {
            if (!jobs[li].wb) continue;
            CKM(cudaSetDevice(C.devices[li]));
            rbrt_stats one; memset(&one, 0, sizeof(one));
            int rc = collect_stats(jobs[li], &one); if (rc) return rc;
            add_stats(&total, one);
            if (dbg) fprintf(stderr, "[multi] local rank %d done at %.3f ms (device time %.3f ms)\n", li, dbg_ms(), one.ms_device);
        }
        CKM(cudaSetDevice(C.devices[0]));
        CKM(cudaStreamSynchronize(st));                                   // stats != NULL: the call waits for the frame (gather included)
        *stats = total;
        int rc1 = resolve_scene_info(sc, true); if (rc1) return rc1;
    }
    CKM(cudaSetDevice(C.devices[0]));
    return RBRT_OK;
}

}  // namespace rbrt

using namespace rbrt;
#define LOCK std::lock_guard<std::recursive_mutex> lock_(api_mutex())

extern "C" {

int rbrt_gpu_comm_info(rbrt_comm_info* out) {
    LOCK;
    if (!out) { set_error("null argument"); return RBRT_E_INVALID; }
    memset(out, 0, sizeof(*out));
    const Comm& C = g_comm;
    out->active = C.active ? 1 : 0; out->world = C.world; out->rank = C.rank; out->local_devices = C.local_n;
    out->transport = C.active ? C.transport : 0; out->nccl_version = C.nccl_version;
    for (int i = 0; i < C.local_n && i < 16 && i < (int)C.devices.size(); ++i) out->devices[i] = C.devices[i];
    return RBRT_OK;
}

int rbrt_gpu_comm_destroy(void) {
    LOCK;
    Comm& C = g_comm;
    if (!C.active) return RBRT_OK;
    workers_stop();
    int cur = 0; cudaGetDevice(&cur);
    for (int li = 0; li < (int)C.devices.size(); ++li) { cudaSetDevice(C.devices[li]); cudaDeviceSynchronize(); }
    for (void* c : C.nccl) if (c && g_nccl.CommDestroy) g_nccl.CommDestroy((ncclComm_t)c);
    for (size_t i = 0; i < C.streams.size(); ++i) if (C.streams[i]) { cudaSetDevice(C.devices[i / 4]); cudaStreamDestroy(C.streams[i]); }
    release_dist_buffers();
    C = Comm();
    cudaSetDevice(cur);
    return RBRT_OK;
}

int rbrt_gpu_init_multi(const int* devices, int n_devices, int transport) {
    LOCK;
    Comm& C = g_comm;
    if (C.active) { set_error("a communicator is already active; rbrt_gpu_comm_destroy() first"); return RBRT_E_INVALID; }
    if (n_devices < 1 || n_devices > 16) { set_error("n_devices must be 1..16"); return RBRT_E_INVALID; }
    if (transport < RBRT_TRANSPORT_AUTO || transport > RBRT_TRANSPORT_PEER) { set_error("unknown transport %d", transport); return RBRT_E_INVALID; }
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        set_error("no CUDA device available (%s); rbrt_b200 has no CPU fallback", e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
        cudaGetLastError();
        return RBRT_E_NODEVICE;
    }
    std::vector<int> devs(n_devices);
    bool dup = false;
    for (int i = 0; i < n_devices; ++i) {
        devs[i] = devices ? devices[i] : i;
        if (devs[i] < 0 || devs[i] >= n) { set_error("device %d out of range (0..%d)", devs[i], n - 1); return RBRT_E_INVALID; }
        for (int k = 0; k < i; ++k) if (devs[k] == devs[i]) dup = true;
    }
    bool can_peer = true;
    for (int i = 1; i < n_devices; ++i) {
        if (devs[i] == devs[0]) continue;
        int a = 0, b = 0;
        cudaDeviceCanAccessPeer(&a, devs[i], devs[0]); cudaDeviceCanAccessPeer(&b, devs[0], devs[i]);
        if (!a || !b) can_peer = false;
    }
    if (transport == RBRT_TRANSPORT_AUTO) transport = (can_peer || dup) ? RBRT_TRANSPORT_PEER : RBRT_TRANSPORT_NCCL;
    if (dup && transport != RBRT_TRANSPORT_PEER) { set_error("a device listed twice needs RBRT_TRANSPORT_PEER"); return RBRT_E_INVALID; }
    if (transport == RBRT_TRANSPORT_PEER && !can_peer) { set_error("RBRT_TRANSPORT_PEER: the GPUs cannot map each other's memory"); return RBRT_E_INVALID; }
    Comm N;
    N.world = n_devices; N.rank = 0; N.local_n = n_devices; N.transport = transport; N.devices = devs; N.multi_process = false;
    if (transport == RBRT_TRANSPORT_NCCL && n_devices > 1) {
        int rc = load_nccl(); if (rc) return rc;
        g_nccl.GetVersion(&N.nccl_version);
        std::vector<ncclComm_t> cs(n_devices);
        CKN(g_nccl.CommInitAll(cs.data(), n_devices, devs.data()));
        for (auto c : cs) N.nccl.push_back((void*)c);
    } else if (transport == RBRT_TRANSPORT_PEER) {
        for (int i = 1; i < n_devices; ++i) {
            if (devs[i] == devs[0]) continue;
            cudaSetDevice(devs[i]); e = cudaDeviceEnablePeerAccess(devs[0], 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return cuda_fail(e, "cudaDeviceEnablePeerAccess");
            cudaGetLastError();
            cudaSetDevice(devs[0]); e = cudaDeviceEnablePeerAccess(devs[i], 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return cuda_fail(e, "cudaDeviceEnablePeerAccess");
            cudaGetLastError();
        }
    }
    N.streams.assign((size_t)n_devices * 4, nullptr);
    for (int i = 1; i < n_devices; ++i) {
        if (devs[i] == devs[0]) continue;
        CKM(cudaSetDevice(devs[i]));
        for (int p = 0; p < 4; ++p) CKM(cudaStreamCreateWithFlags(&N.streams[(size_t)i * 4 + p], cudaStreamNonBlocking));
    }
    CKM(cudaSetDevice(devs[0]));
    set_current_device(devs[0]);
    N.active = true;
    C = N;
    if (n_devices > 1 && !dup) workers_start(n_devices);                  // one enqueue thread per GPU (render_frames)
    return RBRT_OK;
}

int rbrt_gpu_comm_unique_id(uint8_t id_out[RBRT_COMM_ID_BYTES]) {
    LOCK;
    if (!id_out) { set_error("null argument"); return RBRT_E_INVALID; }
    int rc = load_nccl(); if (rc) return rc;
    static_assert(sizeof(ncclUniqueId) == RBRT_COMM_ID_BYTES, "ncclUniqueId size");
    ncclUniqueId id;
    CKN(g_nccl.GetUniqueId(&id));
    memcpy(id_out, &id, sizeof(id));
    return RBRT_OK;
}

int rbrt_gpu_comm_init_rank(const uint8_t id[RBRT_COMM_ID_BYTES], int rank, int world) {
    LOCK;
    Comm& C = g_comm;
    if (C.active) { set_error("a communicator is already active; rbrt_gpu_comm_destroy() first"); return RBRT_E_INVALID; }
    if (!id || world < 1 || world > 64 || rank < 0 || rank >= world) { set_error("bad communicator arguments"); return RBRT_E_INVALID; }
    int dev = current_device();
    if (dev < 0) { int n = 0; if (cudaGetDeviceCount(&n) != cudaSuccess || !n) { cudaGetLastError(); set_error("no CUDA device available; rbrt_b200 has no CPU fallback"); return RBRT_E_NODEVICE; } dev = 0; set_current_device(0); }
    CKM(cudaSetDevice(dev));
    Comm N;
    N.world = world; N.rank = rank; N.local_n = 1; N.transport = RBRT_TRANSPORT_NCCL; N.devices = {dev}; N.multi_process = true;
    N.streams.assign(4, nullptr);
    if (world > 1) {
        int rc = load_nccl(); if (rc) return rc;
        g_nccl.GetVersion(&N.nccl_version);
        ncclUniqueId uid; memcpy(&uid, id, sizeof(uid));
        ncclComm_t c = nullptr;
        CKN(g_nccl.CommInitRank(&c, world, uid, rank));
        N.nccl.push_back((void*)c);
    }
    N.active = true;
    C = N;
    return RBRT_OK;
}

}  // extern "C"
