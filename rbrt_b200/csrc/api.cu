// api.cu — the C-ABI of include/rbrt_gpu.h: scene upload (+LBVH build) and the render entry points.
// There is NO CPU fallback: without a usable CUDA device every GPU entry point fails with
// RBRT_E_NODEVICE / RBRT_E_CUDA and a message.
// Every entry point takes the process-wide lock (api_mutex): the library keeps per-device pools (scene blocks,
// wavefront state, build scratch), and the reference's render_scene may be called from any thread.
#include <dlfcn.h>
#include <chrono>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cfloat>
#include "aov.cuh"
#include "bvh_build.cuh"
#include "denoise.cuh"
#include "engine.cuh"
#include "multi.cuh"
#include "query.cuh"
#include "update.cuh"
#include "variance.cuh"

namespace rbrt {

static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
    va_list ap; va_start(ap, fmt); vsnprintf(g_err, sizeof(g_err), fmt, ap); va_end(ap);
}
int cuda_fail(cudaError_t e, const char* what) {
    set_error("CUDA error %d (%s) at %s", (int)e, cudaGetErrorString(e), what);
    cudaGetLastError();
    return (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver) ? RBRT_E_NODEVICE : RBRT_E_CUDA;
}
std::recursive_mutex& api_mutex() { static std::recursive_mutex m; return m; }
static uint64_t g_pool_limit = 0;
uint64_t pool_limit_bytes() { return g_pool_limit; }

static int g_device = -1;
static double now_ms() {
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

#define CKA(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) return cuda_fail(e_, #x); } while (0)
#define LOCK std::lock_guard<std::recursive_mutex> lock_(api_mutex())

int current_device() { return g_device; }
void set_current_device(int d) { g_device = d; }

static int ensure_device() {
    if (g_device >= 0) { CKA(cudaSetDevice(g_device)); return RBRT_OK; }
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        set_error("no CUDA device available (%s); rbrt_b200 has no CPU fallback", e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
        cudaGetLastError();
        return RBRT_E_NODEVICE;
    }
    g_device = 0;
    CKA(cudaSetDevice(0));
    return RBRT_OK;
}

int device_sm_count(int device, int* out) {
    static int cached[64] = {0};                                           // cudaGetDeviceProperties is slow (tens of ms at times)
    if (!cached[device & 63]) {
        int smc = 0;
        cudaError_t e = cudaDeviceGetAttribute(&smc, cudaDevAttrMultiProcessorCount, device);
        if (e != cudaSuccess) return cuda_fail(e, "cudaDeviceGetAttribute");
        cached[device & 63] = smc;
    }
    *out = cached[device & 63];
    return RBRT_OK;
}

// All device buffers of a scene are carved from ONE allocation, and a destroyed scene's block is kept for the next
// scene of the same device (cudaMalloc / cudaFree synchronise the device and occasionally take tens to hundreds of ms;
// an application that re-creates its scene every frame should not pay that).  rbrt_gpu_release_cache() frees them.
// A pooled block remembers the last work that was enqueued against its scene (one event per stream): renders that were
// only ENQUEUED (stats == NULL) on non-blocking streams may still be reading it, so the block is not handed out again
// before those events have completed.
struct ArenaBlock { void* p; size_t bytes; int device; std::vector<cudaEvent_t> pending; };
static std::vector<ArenaBlock> g_arena_pool;
static void wait_block(ArenaBlock& b) {
    for (cudaEvent_t e : b.pending) { cudaEventSynchronize(e); cudaEventDestroy(e); }
    b.pending.clear();
}
static void arena_release_all() {
    int cur = 0; cudaGetDevice(&cur);
    for (auto& b : g_arena_pool) { cudaSetDevice(b.device); wait_block(b); cudaFree(b.p); }
    g_arena_pool.clear();
    cudaSetDevice(cur);
}
// the caller has made `device` current
int arena_alloc(int device, size_t bytes, char** base, size_t* got_bytes) {
    if (!bytes) bytes = 256;
    int best = -1;
    for (size_t i = 0; i < g_arena_pool.size(); ++i)
        if (g_arena_pool[i].device == device && g_arena_pool[i].bytes >= bytes && g_arena_pool[i].bytes <= bytes + bytes / 4 + (1u << 20) &&
            (best < 0 || g_arena_pool[i].bytes < g_arena_pool[best].bytes)) best = (int)i;
    void* q = nullptr; size_t got = bytes;
    if (best >= 0) {
        wait_block(g_arena_pool[best]);
        q = g_arena_pool[best].p; got = g_arena_pool[best].bytes; g_arena_pool.erase(g_arena_pool.begin() + best);
    } else {
        cudaError_t e = cudaMalloc(&q, bytes);
        if (e != cudaSuccess) { cudaGetLastError(); arena_release_all(); cudaSetDevice(device); e = cudaMalloc(&q, bytes); }
        if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc");
    }
    *base = (char*)q; *got_bytes = got;
    return RBRT_OK;
}
static inline size_t a256(size_t b) { return (b + 255) & ~(size_t)255; }

// pinned 4 KB blocks for the per-scene build results (cudaMallocHost is slow: recycled)
static std::vector<void*> g_pinned_free;
static void* pinned_get(size_t bytes) {
    if (bytes <= 4096 && !g_pinned_free.empty()) { void* p = g_pinned_free.back(); g_pinned_free.pop_back(); return p; }
    void* p = nullptr;
    if (cudaMallocHost(&p, bytes <= 4096 ? 4096 : bytes) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
static void pinned_put(void* p, size_t bytes) { if (!p) return; if (bytes <= 4096 && g_pinned_free.size() < 16) g_pinned_free.push_back(p); else cudaFreeHost(p); }

void wait_scene_ready(const Scene& sc, int li, cudaStream_t st) { if (sc.rep[li].ready) cudaStreamWaitEvent(st, sc.rep[li].ready, 0); }
void wait_scene_uses(const Scene& sc, int device, cudaStream_t st) {
    for (const SceneUse& u : sc.uses) if (u.ev && (device < 0 || u.device == device)) cudaStreamWaitEvent(st, u.ev, 0);
}

int resolve_scene_info(const Scene& sc, bool wait) {
    Scene& m = const_cast<Scene&>(sc);                                     // lazily filled cache behind the handle (under the API lock)
    if (!m.info_resolved) {
        if (!m.info_ev) { m.info_resolved = true; return RBRT_OK; }
        if (!wait && cudaEventQuery(m.info_ev) != cudaSuccess) { cudaGetLastError(); return RBRT_OK; }
        cudaError_t e = cudaEventSynchronize(m.info_ev);
        if (e != cudaSuccess) return cuda_fail(e, "scene build");
        const BuildResult* r = (const BuildResult*)m.res_h;
        uint64_t live = 0;
        for (uint32_t i = 0; i < m.n_meshes; ++i) { live += r[i].live_nodes; if (r[i].error && !m.build_error) m.build_error = (int)i + 1; }
        m.info.num_bvh_nodes = live;
        float up = 0, bu = 0;
        if (m.t_up0 && cudaEventElapsedTime(&up, m.t_up0, m.t_up1) != cudaSuccess) { cudaGetLastError(); up = 0; }
        // build = from the end of the uploads (the build stream waits for them) to the end of the build kernels
        if (m.t_b0 && cudaEventElapsedTime(&bu, m.t_up1, m.t_b1) != cudaSuccess) { cudaGetLastError(); bu = 0; }
        if (bu < 0) bu = 0;
        m.info.ms_upload = up; m.info.ms_build = bu;                       // device times: H2D of the triangle soup / build kernels
        m.info_resolved = true;
    }
    if (m.rebuild_pending && (wait || cudaEventQuery(m.rebuild_ev) == cudaSuccess)) {   // a mesh rebuilt by an update (RBRT_UPDATE_REBUILD)
        cudaGetLastError();
        cudaError_t e = cudaEventSynchronize(m.rebuild_ev);
        if (e != cudaSuccess) return cuda_fail(e, "scene update");
        const BuildResult* r = (const BuildResult*)m.res_h;
        for (uint32_t i = 0; i < m.n_meshes; ++i) if (r[i].error && !m.build_error) m.build_error = (int)i + 1;
        m.rebuild_pending = false;
    }
    if (m.build_error) { set_error("mesh %d: BVH deeper than the traversal stack allows (the mesh was left out of the scene)", m.build_error - 1); return RBRT_E_INVALID; }
    return RBRT_OK;
}

void destroy_scene(Scene* sc) {
    if (!sc) return;
    int cur = 0; cudaGetDevice(&cur);
    for (cudaEvent_t* e : {&sc->info_ev, &sc->t_up0, &sc->t_up1, &sc->t_b0, &sc->t_b1, &sc->upd_in, &sc->upd_out, &sc->rebuild_ev})
        if (*e) { cudaEventSynchronize(*e); cudaEventDestroy(*e); *e = nullptr; }
    for (Scene::Staging& s : sc->stage) {
        if (s.done) { cudaEventSynchronize(s.done); cudaEventDestroy(s.done); }
        if (s.p) cudaFreeHost(s.p);
        s = Scene::Staging();
    }
    pinned_put(sc->res_h, 16ull * sc->n_meshes); sc->res_h = nullptr;
    for (Replica& r : sc->rep) {
        if (!r.arena) { if (r.ready) cudaEventDestroy(r.ready); continue; }
        ArenaBlock b{r.arena, r.arena_bytes, r.device, {}};
        if (r.ready) { b.pending.push_back(r.ready); r.ready = nullptr; }  // the build / replication that writes the block
        for (SceneUse& u : sc->uses) if (u.device == r.device && u.ev) { b.pending.push_back(u.ev); u.ev = nullptr; }
        size_t pooled = 0;
        for (auto& g : g_arena_pool) if (g.device == r.device) ++pooled;
        if (pooled < 4) g_arena_pool.push_back(std::move(b));
        else { cudaSetDevice(r.device); wait_block(b); cudaFree(b.p); }
    }
    for (SceneUse& u : sc->uses) if (u.ev) cudaEventDestroy(u.ev);
    cudaSetDevice(cur);
    delete sc;
}

SceneDev make_scene_dev(char* base, const ArenaLayout& lay, uint32_t n_elems, uint32_t n_meshes, uint32_t n_etris) {
    SceneDev d;
    d.spheres = (const float4*)(base + lay.sph); d.etris = (const float4*)(base + lay.etris); d.elem_kind = (const uint32_t*)(base + lay.ekind);
    d.tris = (const float4*)(base + lay.tris); d.nodes = (const float4*)(base + lay.nodes); d.normals = (const float4*)(base + lay.nrm);
    d.mat = (const float4*)(base + lay.mat); d.mat_kind = (const uint32_t*)(base + lay.kind); d.meshes = (const MeshDev*)(base + lay.mesh);
    d.n_spheres = n_elems; d.n_meshes = n_meshes; d.n_etris = n_etris;
    return d;
}

// N_eff of the reference's SIMD sweep: padding appends N % lanes copies (mesh.rs:136-144) and the
// sweep runs chunks_exact(lanes) (triangle.rs:167,296), so the last N % lanes triangles are never
// tested when 2*(N % lanes) < lanes.
static uint64_t tested_triangles(uint64_t n, uint32_t lanes) {
    uint64_t r = n % lanes, total = n + r, tested = (total / lanes) * lanes;
    return tested < n ? tested : n;
}

// Scene.elements -> the block's element arrays: per element a sphere record or {bits(index into etris)}, its material and kind; per
// BasicTriangle four etris records.  mat / kind / ekind hold at least ns entries (the mesh materials follow in mat / kind).
static void pack_elements(const rbrt_element_ref* order, uint32_t ns, const rbrt_sphere_desc* spheres, const rbrt_triangle_desc* triangles,
                          std::vector<float4>& sph, std::vector<float4>& etris, std::vector<float4>& mat, std::vector<uint32_t>& kind,
                          std::vector<uint32_t>& ekind) {
    for (uint32_t i = 0; i < ns; ++i) {
        rbrt_material m;
        if (order[i].kind == RBRT_ELEM_SPHERE) {
            const rbrt_sphere_desc& sp = spheres[order[i].index];
            sph[i] = make_float4(sp.center.x, sp.center.y, sp.center.z, sp.radius);
            m = sp.material; ekind[i] = RBRT_ELEM_SPHERE;
        } else {                                                          // BasicTriangle::new (triangle.rs:19-27), host f32, no contraction
            const rbrt_triangle_desc& t = triangles[order[i].index];
            const rbrt_vec3 &a = t.corners[0], &b = t.corners[1], &c = t.corners[2];
            float e1[3] = {b.x - a.x, b.y - a.y, b.z - a.z}, e2[3] = {c.x - a.x, c.y - a.y, c.z - a.z};
            float cx = e1[1] * e2[2] - e1[2] * e2[1], cy = e1[2] * e2[0] - e1[0] * e2[2], cz = e1[0] * e2[1] - e1[1] * e2[0];
            float len = sqrtf(cx * cx + cy * cy + cz * cz);
            uint32_t ti = (uint32_t)(etris.size() / 4);
            float tif; memcpy(&tif, &ti, 4);
            sph[i] = make_float4(tif, 0.0f, 0.0f, 0.0f);
            etris.push_back(make_float4(a.x, a.y, a.z, 0.0f)); etris.push_back(make_float4(e1[0], e1[1], e1[2], 0.0f));
            etris.push_back(make_float4(e2[0], e2[1], e2[2], 0.0f)); etris.push_back(make_float4(cx / len, cy / len, cz / len, 0.0f));
            m = t.material; ekind[i] = RBRT_ELEM_TRIANGLE;
        }
        mat[i] = make_float4(m.albedo.x, m.albedo.y, m.albedo.z, m.param);
        kind[i] = m.kind;
    }
}

// ------------------------------------------------------------------ device modules
// The refit kernels (librbrt_gpu_update.so), the AOV kernel (librbrt_gpu_aov.so), the ray queries (librbrt_gpu_query.so), the denoiser
// (librbrt_gpu_denoise.so) and the variance kernels (librbrt_gpu_variance.so) live in their own device modules, loaded from this library's
// directory (or the path in the module's environment variable) on first use.  Without a module its calls are refused: there is no other
// implementation.
// Path of a device module shipped next to this library (`file`), or the value of the environment variable `env` if that is set.
static int module_path(const char* env, const char* file, std::string* path) {
    const char* e = getenv(env);
    if (e && *e) { *path = e; return RBRT_OK; }
    Dl_info di;
    if (!dladdr((void*)&module_path, &di) || !di.dli_fname) { set_error("cannot locate librbrt_gpu.so to find %s", file); return RBRT_E_CUDA; }
    *path = di.dli_fname;
    const size_t slash = path->find_last_of('/');
    *path = (slash == std::string::npos ? std::string(".") : path->substr(0, slash)) + "/" + file;
    return RBRT_OK;
}

// `what` names the module in messages; `h` is its handle once opened.
struct Module { const char* env; const char* file; const char* what; void* h; };
static Module g_update_module = {"RBRT_GPU_UPDATE_LIB", "librbrt_gpu_update.so", "refit", nullptr};
static Module g_aov_module = {"RBRT_GPU_AOV_LIB", "librbrt_gpu_aov.so", "AOV", nullptr};
static Module g_query_module = {"RBRT_GPU_QUERY_LIB", "librbrt_gpu_query.so", "query", nullptr};
static Module g_denoise_module = {"RBRT_GPU_DENOISE_LIB", "librbrt_gpu_denoise.so", "denoise", nullptr};
static Module g_variance_module = {"RBRT_GPU_VARIANCE_LIB", "librbrt_gpu_variance.so", "variance", nullptr};
// The entry point `symbol` of module m, which is opened on first use.  A failed dlopen is not remembered: the next call tries again.
template <class F> static int module_entry(Module& m, const char* symbol, F* fn) {
    if (!m.h) {
        std::string path;
        { int rc = module_path(m.env, m.file, &path); if (rc) return rc; }
        m.h = dlopen(path.c_str(), RTLD_NOW | RTLD_LOCAL);
        if (!m.h) { set_error("the %s module is missing (dlopen %s: %s); build it with make -C rbrt_b200/csrc", m.what, path.c_str(), dlerror()); return RBRT_E_CUDA; }
    }
    void* p = dlsym(m.h, symbol);
    if (!p) { set_error("the %s module lacks the entry point %s; rebuild it with make -C rbrt_b200/csrc", m.what, symbol); return RBRT_E_CUDA; }
    *fn = reinterpret_cast<F>(p);
    return RBRT_OK;
}

// ------------------------------------------------------------------ scene updates (rbrt_gpu_scene_update_*)
// Opens an update: the device's build stream, made to wait for every read of the scene enqueued so far on replica 0's device.
// Every write of the update is enqueued on ctx->build after this.
static int update_begin(Scene* sc, BuildCtx* ctx) {
    CKA(cudaSetDevice(sc->rep[0].device));
    CKA(build_begin(sc->rep[0].device, ctx));
    wait_scene_uses(*sc, sc->rep[0].device, ctx->build);
    return RBRT_OK;
}
// Publishes it: the other replicas are copied again (each behind its own readers), and every replica's `ready` is recorded
// behind the writes, so that reads enqueued from now on see the new values.
static int update_end(Scene* sc, BuildCtx& ctx) {
    if (sc->replicated) return replicate_scene(sc, ctx.build);
    CKA(cudaEventRecord(sc->rep[0].ready, ctx.build));
    return RBRT_OK;
}
// Pinned host staging for `bytes` of element / material values (copied to the block on the build stream, behind the scene's readers):
// one of two alternating buffers, once its previous copy has run.  The caller records s->done behind its copies.
static int stage_get(Scene* sc, size_t bytes, Scene::Staging** out) {
    Scene::Staging& s = sc->stage[sc->stage_next];
    sc->stage_next ^= 1;
    if (s.done) CKA(cudaEventSynchronize(s.done));
    else CKA(cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming));
    if (s.bytes < bytes) {
        if (s.p) cudaFreeHost(s.p);
        s.p = nullptr; s.bytes = 0;
        CKA(cudaMallocHost(&s.p, bytes < 4096 ? 4096 : bytes)); s.bytes = bytes < 4096 ? 4096 : bytes;
    }
    *out = &s;
    return RBRT_OK;
}
static int ensure_event(cudaEvent_t* e) { if (!*e) CKA(cudaEventCreateWithFlags(e, cudaEventDisableTiming)); return RBRT_OK; }

// rbrt_gpu_scene_update_mesh(_device).  `user_st` is the caller's stream for device vertices (on_device), unused otherwise.
static int update_mesh(rbrt_scene* scene, uint32_t mi, const float* verts, bool on_device, uint64_t n, const rbrt_material* mat,
                       uint32_t flags, cudaStream_t user_st) {
    if (!scene) { set_error("null argument"); return RBRT_E_INVALID; }
    Scene* sc = reinterpret_cast<Scene*>(scene);
    if (flags > RBRT_UPDATE_REBUILD) { set_error("unknown update flags %u", flags); return RBRT_E_INVALID; }
    if (mi >= sc->n_meshes) { set_error("mesh index %u out of range (the scene has %u meshes)", mi, sc->n_meshes); return RBRT_E_INVALID; }
    if (n != sc->mesh_n_all[mi]) {
        set_error("mesh %u: %llu triangles, created with %llu (an update keeps the count)", mi, (unsigned long long)n, (unsigned long long)sc->mesh_n_all[mi]);
        return RBRT_E_INVALID;
    }
    if (mat && mat->kind > 2) { set_error("mesh %u: unknown material kind", mi); return RBRT_E_INVALID; }
    const bool receiver = sc->replicated && comm().multi_process && comm().rank != 0;   // RBRT_SCENE_BROADCAST: rank 0's update arrives by broadcast
    if (n && !verts && !receiver) { set_error("mesh %u: null tri_vertices", mi); return RBRT_E_INVALID; }
    {   // a mesh whose tree was refused (too deep) is out of the scene: nothing to update
        int rc = resolve_scene_info(*sc, true);
        if (rc) return rc;
    }
    rbrt_update_scratch_bytes_fn scratch_bytes = nullptr;
    rbrt_update_refit_fn refit = nullptr;
    if (flags == RBRT_UPDATE_REFIT && !receiver) {
        int rc = module_entry(g_update_module, "rbrt_update_scratch_bytes", &scratch_bytes);
        if (!rc) rc = module_entry(g_update_module, "rbrt_update_refit", &refit);
        if (rc) return rc;
    }

    BuildCtx ctx;
    { int rc = update_begin(sc, &ctx); if (rc) return rc; }
    if (on_device && !receiver) {
        { int rc = ensure_event(&sc->upd_in); if (rc) return rc; }
        CKA(cudaEventRecord(sc->upd_in, user_st));                      // the vertices are ready in stream order on the caller's stream
    }
    cudaEvent_t uploaded = nullptr;                                       // host vertices: completes when they have been read
    if (!receiver) {
        const MeshDev& md = sc->meshes_h[mi];
        const uint32_t n_eff = md.n_tris;
        char* const base = sc->rep[0].arena;
        MeshDev* d_mesh = (MeshDev*)(base + sc->lay.mesh) + mi;
        float4* d_tris = (float4*)(base + sc->lay.tris) + 3ull * md.tri_base;
        float4* d_normals = (float4*)(base + sc->lay.nrm) + md.nrm_base;
        float4* d_nodes = (float4*)(base + sc->lay.nodes) + 4ull * md.node_base;
        BuildResult* d_res = (BuildResult*)(base + sc->lay.result) + mi;
        if (mat) {
            Scene::Staging* sg = nullptr;
            { int rc = stage_get(sc, 32, &sg); if (rc) return rc; }
            const float4 m4 = make_float4(mat->albedo.x, mat->albedo.y, mat->albedo.z, mat->param);
            memcpy(sg->p, &m4, 16); memcpy((char*)sg->p + 16, &mat->kind, 4);
            const size_t e = sc->n_elems + mi;
            CKA(cudaMemcpyAsync(base + sc->lay.mat + 16 * e, sg->p, 16, cudaMemcpyHostToDevice, ctx.build));
            CKA(cudaMemcpyAsync(base + sc->lay.kind + 4 * e, (char*)sg->p + 16, 4, cudaMemcpyHostToDevice, ctx.build));
            CKA(cudaEventRecord(sg->done, ctx.build));
        }
        if (flags == RBRT_UPDATE_REBUILD) {                               // the creation's build into the mesh's own slots (<= n_eff - 1 nodes)
            CKA(build_mesh(ctx, verts, n, n_eff, sc->pad_rel, sc->leaf_size, sc->sah, md, d_mesh, d_tris, d_normals, d_nodes, d_res,
                           on_device ? sc->upd_in : nullptr));
            if (!on_device) {
                { int rc = ensure_event(&sc->t_up1); if (rc) return rc; }
                CKA(build_uploads_done(ctx, sc->t_up1)); uploaded = sc->t_up1;
            }
            { int rc = ensure_event(&sc->rebuild_ev); if (rc) return rc; }   // a too-deep tree is reported like the creation's (resolve_scene_info)
            CKA(cudaMemcpyAsync((BuildResult*)sc->res_h + mi, d_res, sizeof(BuildResult), cudaMemcpyDeviceToHost, ctx.build));
            CKA(cudaEventRecord(sc->rebuild_ev, ctx.build));
            sc->rebuild_pending = true;
        } else {
            const size_t raw_bytes = on_device ? 0 : (36ull * n + 255) & ~255ull;
            char* sbase = nullptr;
            CKA(build_slot_acquire(ctx, raw_bytes + scratch_bytes(n_eff), &sbase));
            if (!on_device && n) CKA(cudaMemcpyAsync(sbase, verts, 36ull * n, cudaMemcpyHostToDevice, ctx.copy));
            CKA(build_slot_uploaded(ctx, &uploaded));
            if (on_device) CKA(cudaStreamWaitEvent(ctx.build, sc->upd_in, 0));
            RefitArgs a;
            a.raw = on_device ? verts : (const float*)sbase; a.n_all = n; a.n_eff = n_eff; a.pad_rel = sc->pad_rel;
            a.mesh = d_mesh; a.tris = d_tris; a.normals = d_normals; a.nodes = reinterpret_cast<uint4*>(d_nodes); a.res = d_res;
            CKA((cudaError_t)refit(&a, sbase + raw_bytes, ctx.build));
            CKA(build_slot_release(ctx));
            if (on_device) uploaded = nullptr;
        }
    }
    { int rc = update_end(sc, ctx); if (rc) return rc; }
    if (on_device && !receiver) {                                         // the caller's stream continues behind the update
        { int rc = ensure_event(&sc->upd_out); if (rc) return rc; }
        CKA(cudaEventRecord(sc->upd_out, ctx.build));
        CKA(cudaStreamWaitEvent(user_st, sc->upd_out, 0));
    }
    if (uploaded) CKA(cudaEventSynchronize(uploaded));                    // the caller's array has been read (copy engine: no wait for busy SMs)
    return RBRT_OK;
}

// ------------------------------------------------------------------ per-device state of the calls into the device modules
// Created on first use, freed by rbrt_gpu_release_cache.
//  - The staging block that the host-pointer AOV and denoise calls carve their device planes from (grown, never shrunk).  One block
//    serves both: each such call runs on the legacy default stream and synchronises it before returning.
//  - The timing events of calls with stats (AOV, query, denoise, variance).  Each such call waits for `e1` or its stream before returning.
//  - The AOV counters, used by calls with stats.
//  - The query ring: QRY_RING counter blocks (the ray cursor of the persistent kernel and the stats counters).  Each call takes the next
//    block, zeroes it on its own stream and records `qry_used` behind its kernel, so calls on different streams never share a cursor.  A
//    block is reused QRY_RING calls later; the host waits for its previous call only if that one has still not run by then.
//  - The variance lane: an internal stream and the events that fork a call's shards onto it and join them back (render_variance).
//    Calls without stats return before their shards run, so the lane is ordered by those events, not by the host.
#define QRY_RING 256
struct DeviceCache {
    char* buf = nullptr; size_t bytes = 0;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    unsigned long long* aov_ctr = nullptr;
    unsigned long long* qry_ctr = nullptr; cudaEvent_t qry_used[QRY_RING] = {}; uint32_t qry_next = 0;
    cudaStream_t aux = nullptr; cudaEvent_t fork = nullptr, join = nullptr;
};
static DeviceCache g_cache[64];
static void cache_release_all() {
    int cur = 0; cudaGetDevice(&cur);
    for (int d = 0; d < 64; ++d) {
        DeviceCache& c = g_cache[d];
        if (!c.buf && !c.e0 && !c.e1 && !c.aov_ctr && !c.qry_ctr && !c.aux) continue;
        cudaSetDevice(d);
        for (cudaEvent_t& e : c.qry_used) if (e) { cudaEventSynchronize(e); cudaEventDestroy(e); }
        if (c.aux) { cudaStreamSynchronize(c.aux); cudaStreamDestroy(c.aux); }
        for (cudaEvent_t e : {c.e0, c.e1, c.fork, c.join}) if (e) cudaEventDestroy(e);
        cudaFree(c.buf); cudaFree(c.aov_ctr); cudaFree(c.qry_ctr);
        c = DeviceCache();
    }
    cudaSetDevice(cur);
}
// The device's staging block, grown to at least `need` bytes.
static int staging_block(DeviceCache& c, size_t need, char** out) {
    if (c.bytes < need) {
        cudaFree(c.buf); c.buf = nullptr; c.bytes = 0;
        CKA(cudaMalloc(&c.buf, need)); c.bytes = need;
    }
    *out = c.buf;
    return RBRT_OK;
}
static int timing_events(DeviceCache& c) {
    if (!c.e0) CKA(cudaEventCreate(&c.e0));
    if (!c.e1) CKA(cudaEventCreate(&c.e1));
    return RBRT_OK;
}

// Device memory on `device` (or managed / registered host memory the device can read)?  Unregistered host memory or another device's
// memory would fault in the kernel.
static bool usable_on(const void* p, int device) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    if (a.type == cudaMemoryTypeDevice) return a.device == device;
    return a.type == cudaMemoryTypeManaged || (a.type == cudaMemoryTypeHost && a.devicePointer == p);
}
// RBRT_E_INVALID with the message `msg` (formatted with the device) unless every non-NULL pointer of `ptrs` is usable on `device`.
static int check_usable_on(std::initializer_list<const void*> ptrs, int device, const char* msg) {
    for (const void* p : ptrs)
        if (p && !usable_on(p, device)) { set_error(msg, device); return RBRT_E_INVALID; }
    return RBRT_OK;
}

// ------------------------------------------------------------------ first-hit AOVs (rbrt_gpu_render_aov*)
static int render_aov(const rbrt_scene* scene, const rbrt_camera* cam, uint32_t spp, uint64_t seed, const rbrt_aov_out* out, bool host,
                      cudaStream_t st, rbrt_stats* stats) {
    if (!scene || !cam || !out) { set_error("null argument"); return RBRT_E_INVALID; }
    if (!out->depth && !out->normal && !out->albedo && !out->coverage && !out->hit_kind && !out->elem_idx && !out->tri_idx) {
        set_error("no AOV requested (every member of the output is NULL)"); return RBRT_E_INVALID;
    }
    const uint64_t n = (uint64_t)cam->img_width_pix * cam->img_height_pix;
    if (!n || !spp) { set_error("empty image or zero samples"); return RBRT_E_INVALID; }
    if (n > 0xFFFFFFFFull) { set_error("more than 2^32 - 1 pixels"); return RBRT_E_INVALID; }
    const Scene& sc = *reinterpret_cast<const Scene*>(scene);
    const Replica& rp = sc.rep[0];                                        // under a communicator: this process's first device, whole image
    CKA(cudaSetDevice(rp.device));
    const double t0 = now_ms();
    if (stats) memset(stats, 0, sizeof(*stats));
    { int rc = resolve_scene_info(sc, true); if (rc) return rc; }         // a refused mesh is known before anything is written
    rbrt_aov_launch_fn launch = nullptr;
    { int rc = module_entry(g_aov_module, "rbrt_aov_launch", &launch); if (rc) return rc; }

    DeviceCache& c = g_cache[rp.device & 63];
    AovArgs a;
    memset(&a, 0, sizeof(a));
    a.S = rp.dev; a.cam = make_cam(*cam); a.key0 = (uint32_t)seed; a.key1 = (uint32_t)(seed >> 32); a.n_samples = spp;
    a.tiles_x = (cam->img_width_pix + 7) / 8; a.tiles_total = a.tiles_x * ((cam->img_height_pix + 3) / 4);
    a.out = *out;
    if (host) {                                                           // the requested planes, carved from the staging block
        const size_t b1 = a256(4 * n), b3 = a256(12 * n);
        const size_t need = (out->depth ? b1 : 0) + (out->normal ? b3 : 0) + (out->albedo ? b3 : 0) + (out->coverage ? b1 : 0) +
                            (out->hit_kind ? b1 : 0) + (out->elem_idx ? b1 : 0) + (out->tri_idx ? b1 : 0);
        char* p = nullptr;
        { int rc = staging_block(c, need, &p); if (rc) return rc; }
        auto take = [&](const void* want, size_t b) -> char* { if (!want) return nullptr; char* q = p; p += b; return q; };
        a.out.depth = (float*)take(out->depth, b1); a.out.normal = (float*)take(out->normal, b3); a.out.albedo = (float*)take(out->albedo, b3);
        a.out.coverage = (float*)take(out->coverage, b1); a.out.hit_kind = (int32_t*)take(out->hit_kind, b1);
        a.out.elem_idx = (uint32_t*)take(out->elem_idx, b1); a.out.tri_idx = (uint32_t*)take(out->tri_idx, b1);
    }
    if (stats) {
        if (!c.aov_ctr) CKA(cudaMalloc(&c.aov_ctr, 8 * AOV_ST_COUNT));
        { int rc = timing_events(c); if (rc) return rc; }
        a.stats = c.aov_ctr;
    }
    wait_scene_ready(sc, 0, st);                                          // behind the scene's build and every update enqueued so far
    if (stats) { CKA(cudaMemsetAsync(c.aov_ctr, 0, 8 * AOV_ST_COUNT, st)); CKA(cudaEventRecord(c.e0, st)); }
    CKA((cudaError_t)launch(&a, st));
    if (stats) CKA(cudaEventRecord(c.e1, st));
    note_scene_use(sc, rp.device, st);                                    // later updates wait for this read
    if (!host && !stats) return RBRT_OK;                                  // enqueue only

    if (stats) CKA(cudaEventSynchronize(c.e1));
    const double t1 = now_ms();
    if (host) {
        if (out->depth) CKA(cudaMemcpyAsync(out->depth, a.out.depth, 4 * n, cudaMemcpyDeviceToHost, st));
        if (out->normal) CKA(cudaMemcpyAsync(out->normal, a.out.normal, 12 * n, cudaMemcpyDeviceToHost, st));
        if (out->albedo) CKA(cudaMemcpyAsync(out->albedo, a.out.albedo, 12 * n, cudaMemcpyDeviceToHost, st));
        if (out->coverage) CKA(cudaMemcpyAsync(out->coverage, a.out.coverage, 4 * n, cudaMemcpyDeviceToHost, st));
        if (out->hit_kind) CKA(cudaMemcpyAsync(out->hit_kind, a.out.hit_kind, 4 * n, cudaMemcpyDeviceToHost, st));
        if (out->elem_idx) CKA(cudaMemcpyAsync(out->elem_idx, a.out.elem_idx, 4 * n, cudaMemcpyDeviceToHost, st));
        if (out->tri_idx) CKA(cudaMemcpyAsync(out->tri_idx, a.out.tri_idx, 4 * n, cudaMemcpyDeviceToHost, st));
        CKA(cudaStreamSynchronize(st));
    }
    const double t2 = now_ms();
    if (stats) {
        unsigned long long h[AOV_ST_COUNT];
        CKA(cudaMemcpyAsync(h, c.aov_ctr, sizeof(h), cudaMemcpyDeviceToHost, st));
        CKA(cudaStreamSynchronize(st));
        float ms = 0; CKA(cudaEventElapsedTime(&ms, c.e0, c.e1));
        stats->rays = n * spp; stats->paths = n * spp; stats->nan_rays = h[AOV_ST_NAN];
        stats->node_visits = h[AOV_ST_NODES]; stats->tri_tests = h[AOV_ST_TRIS];
        stats->ms_device = ms; stats->ms_d2h = host ? t2 - t1 : 0.0; stats->launches = 1;
        stats->ms_total = now_ms() - t0;
    }
    return RBRT_OK;
}

// ------------------------------------------------------------------ ray queries on device memory (rbrt_gpu_query_*_device)
// occ: an occlusion query into occluded[]; else a closest query into *out.
static int query(const rbrt_scene* scene, const rbrt_ray* rays, uint64_t n, bool occ, const rbrt_query_out* out, const float* max_dist,
                 uint8_t* occluded, cudaStream_t st, rbrt_stats* stats) {
    if (stats) memset(stats, 0, sizeof(*stats));
    if (!n) return RBRT_OK;
    if (!scene || !rays || (occ ? !occluded : !out)) { set_error("null argument"); return RBRT_E_INVALID; }
    if (!occ && !out->t && !out->dist && !out->kind && !out->elem_idx && !out->tri_idx && !out->point && !out->normal) {
        set_error("no output requested (every plane of the output is NULL)"); return RBRT_E_INVALID;
    }
    if (n > 0xFFFFFFFFull) { set_error("more than 2^32 - 1 rays"); return RBRT_E_INVALID; }
    const Scene& sc = *reinterpret_cast<const Scene*>(scene);
    const Replica& rp = sc.rep[0];                                        // under a communicator: this process's first device
    CKA(cudaSetDevice(rp.device));
    const double t0 = now_ms();
    const rbrt_query_out o = occ ? rbrt_query_out{} : *out;
    { int rc = check_usable_on({rays, max_dist, occluded, o.t, o.dist, o.kind, o.elem_idx, o.tri_idx, o.point, o.normal}, rp.device,
                               "rays and outputs must be device memory on the scene's device %d"); if (rc) return rc; }
    { int rc = resolve_scene_info(sc, true); if (rc) return rc; }         // a refused mesh is known before anything is written
    rbrt_query_launch_fn launch = nullptr;
    { int rc = module_entry(g_query_module, "rbrt_query_launch", &launch); if (rc) return rc; }

    DeviceCache& c = g_cache[rp.device & 63];
    if (!c.qry_ctr) CKA(cudaMalloc(&c.qry_ctr, 8ull * QRY_ST_COUNT * QRY_RING));
    const uint32_t slot = c.qry_next++ % QRY_RING;
    cudaEvent_t& used = c.qry_used[slot];
    if (used) CKA(cudaEventSynchronize(used));
    else CKA(cudaEventCreateWithFlags(&used, cudaEventDisableTiming));
    if (stats) { int rc = timing_events(c); if (rc) return rc; }

    QueryArgs a;
    memset(&a, 0, sizeof(a));
    a.S = rp.dev; a.rays = rays; a.n = n; a.max_dist = max_dist; a.occluded = occluded; a.ctr = c.qry_ctr + QRY_ST_COUNT * slot;
    a.out = o;
    a.count = stats != nullptr;
    {
        const uint64_t blocks = (n + 127) / 128;                          // persistent: at most the resident blocks (8 per SM, query.cu)
        const uint64_t resident = 8ull * (uint64_t)rp.sm_count;
        a.blocks = (uint32_t)(blocks < resident ? blocks : resident);
    }
    wait_scene_ready(sc, 0, st);                                          // behind the scene's build and every update enqueued so far
    CKA(cudaMemsetAsync(a.ctr, 0, 8 * QRY_ST_COUNT, st));
    if (stats) CKA(cudaEventRecord(c.e0, st));
    CKA((cudaError_t)launch(&a, st));
    if (stats) CKA(cudaEventRecord(c.e1, st));
    CKA(cudaEventRecord(used, st));
    note_scene_use(sc, rp.device, st);                                    // later updates wait for this read
    if (!stats) return RBRT_OK;                                           // enqueue only

    unsigned long long h[QRY_ST_COUNT];
    CKA(cudaMemcpyAsync(h, a.ctr, sizeof(h), cudaMemcpyDeviceToHost, st));
    CKA(cudaStreamSynchronize(st));
    float ms = 0; CKA(cudaEventElapsedTime(&ms, c.e0, c.e1));
    stats->rays = n; stats->nan_rays = h[QRY_ST_NAN]; stats->node_visits = h[QRY_ST_NODES]; stats->tri_tests = h[QRY_ST_TRIS];
    stats->ms_device = ms; stats->launches = 1;
    stats->ms_total = now_ms() - t0;
    return RBRT_OK;
}

// ------------------------------------------------------------------ guided denoising (rbrt_gpu_denoise*, rbrt_gpu_denoise_variance*)
// The host-pointer variant copies its planes into the device's staging block and carves its scratch from it.  The device variant takes
// its scratch from the stream-ordered allocator on the call's stream instead, so calls in flight never share it.
static bool overlap(const void* a, size_t na, const void* b, size_t nb) {
    if (!a || !b) return false;
    const uintptr_t x = (uintptr_t)a, y = (uintptr_t)b;
    return x < y + nb && y < x + na;
}

// var: the variance-guided filter of librbrt_gpu_variance.so with that variance plane; NULL: rbrt_gpu_denoise's filter.
static int denoise(uint32_t W, uint32_t H, const float* hdr, const float* var, const rbrt_aov_out* guides, const rbrt_denoise_opts* opts,
                   float* hdr_out, uint8_t* rgb_out, bool with_var, bool host, cudaStream_t st, rbrt_stats* stats) {
    if (stats) memset(stats, 0, sizeof(*stats));
    if (!hdr || !guides || (with_var && !var)) { set_error("null argument"); return RBRT_E_INVALID; }
    if (!guides->depth || !guides->normal || !guides->albedo) { set_error("null guide plane: depth, normal and albedo are read"); return RBRT_E_INVALID; }
    if (!hdr_out && !rgb_out) { set_error("no output requested (hdr_out and rgb_out are both NULL)"); return RBRT_E_INVALID; }
    if (!W || !H) { set_error("empty image"); return RBRT_E_INVALID; }
    const size_t n = (size_t)W * H;
    if (n > 0x7FFFFFFFull) { set_error("image too large"); return RBRT_E_INVALID; }
    DenoiseArgs a;
    memset(&a, 0, sizeof(a));
    a.W = W; a.H = H;
    a.levels = opts && opts->levels ? opts->levels : (with_var ? VR_DEFAULT_LEVELS : DN_DEFAULT_LEVELS);
    if (a.levels > DN_MAX_LEVELS) { set_error("levels must be at most %u", DN_MAX_LEVELS); return RBRT_E_INVALID; }
    const float sz = opts ? opts->sigma_depth : 0.0f, sl = opts ? opts->sigma_luminance : 0.0f;
    if (!(sz >= 0.0f && sz <= FLT_MAX) || !(sl >= 0.0f && sl <= FLT_MAX)) { set_error("a sigma must be finite and >= 0 (0 = default)"); return RBRT_E_INVALID; }
    a.sigma_z = sz > 0.0f ? sz : (with_var ? VR_SIGMA_DEPTH : DN_SIGMA_DEPTH);
    a.sigma_l = sl > 0.0f ? sl : (with_var ? VR_SIGMA_LUMINANCE : DN_SIGMA_LUMINANCE);
    {
        const struct { const void* p; size_t b; } in[5] = {{hdr, 12 * n}, {guides->depth, 4 * n}, {guides->normal, 12 * n}, {guides->albedo, 12 * n},
                                                           {var, 12 * n}};
        for (const auto& i : in) {
            if (overlap(hdr_out, 12 * n, i.p, i.b) || overlap(rgb_out, 3 * n, i.p, i.b)) { set_error("an output overlaps an input"); return RBRT_E_INVALID; }
        }
        if (overlap(hdr_out, 12 * n, rgb_out, 3 * n)) { set_error("hdr_out and rgb_out overlap"); return RBRT_E_INVALID; }
    }
    { int rc = ensure_device(); if (rc) return rc; }
    const int dev = g_device;
    if (!host) {
        int rc = check_usable_on({hdr, guides->depth, guides->normal, guides->albedo, hdr_out, rgb_out, var}, dev,
                                 "planes must be device memory on the current device %d");
        if (rc) return rc;
    }
    rbrt_denoise_launch_fn launch = nullptr;
    rbrt_variance_filter_launch_fn vlaunch = nullptr;
    {
        int rc = with_var ? module_entry(g_variance_module, "rbrt_variance_filter_launch", &vlaunch)
                          : module_entry(g_denoise_module, "rbrt_denoise_launch", &launch);
        if (rc) return rc;
    }
    const size_t scratch = (with_var ? 56 : 48) * n;                      // guides and two planes of (e.rgb, l); with var two planes of σ²
    const double t0 = now_ms();

    DeviceCache& c = g_cache[dev & 63];
    if (stats) { int rc = timing_events(c); if (rc) return rc; }
    a.hdr = hdr; a.depth = guides->depth; a.normal = guides->normal; a.albedo = guides->albedo; a.hdr_out = hdr_out; a.rgb_out = rgb_out;
    if (host) {                                                           // inputs, outputs and scratch carved from the staging block
        const size_t b1 = a256(4 * n), b3 = a256(12 * n), bs = a256(scratch);
        const size_t need = bs + 3 * b3 + b1 + (with_var ? b3 : 0) + (hdr_out ? b3 : 0) + (rgb_out ? a256(3 * n) : 0);
        char* p = nullptr;
        { int rc = staging_block(c, need, &p); if (rc) return rc; }
        a.scratch = (float4*)p; p += bs;
        float* d_hdr = (float*)p; p += b3;
        float* d_nrm = (float*)p; p += b3;
        float* d_alb = (float*)p; p += b3;
        float* d_dep = (float*)p; p += b1;
        CKA(cudaMemcpyAsync(d_hdr, hdr, 12 * n, cudaMemcpyHostToDevice, st));
        CKA(cudaMemcpyAsync(d_nrm, guides->normal, 12 * n, cudaMemcpyHostToDevice, st));
        CKA(cudaMemcpyAsync(d_alb, guides->albedo, 12 * n, cudaMemcpyHostToDevice, st));
        CKA(cudaMemcpyAsync(d_dep, guides->depth, 4 * n, cudaMemcpyHostToDevice, st));
        a.hdr = d_hdr; a.normal = d_nrm; a.albedo = d_alb; a.depth = d_dep;
        if (with_var) {
            float* d_var = (float*)p; p += b3;
            CKA(cudaMemcpyAsync(d_var, var, 12 * n, cudaMemcpyHostToDevice, st));
            var = d_var;
        }
        if (hdr_out) { a.hdr_out = (float*)p; p += b3; }
        if (rgb_out) a.rgb_out = (uint8_t*)p;
    } else {
        CKA(cudaMallocAsync((void**)&a.scratch, scratch, st));
    }
    if (stats) {
        cudaError_t e = cudaEventRecord(c.e0, st);
        if (e != cudaSuccess) { if (!host) cudaFreeAsync(a.scratch, st); return cuda_fail(e, "cudaEventRecord"); }
    }
    {
        cudaError_t e = (cudaError_t)(with_var ? vlaunch(&a, var, st) : launch(&a, st));
        if (e == cudaSuccess && stats) e = cudaEventRecord(c.e1, st);
        if (!host) { cudaError_t f = cudaFreeAsync(a.scratch, st); if (e == cudaSuccess) e = f; }
        if (e != cudaSuccess) return cuda_fail(e, with_var ? "rbrt_variance_filter_launch" : "rbrt_denoise_launch");
    }
    if (host) {
        if (hdr_out) CKA(cudaMemcpyAsync(hdr_out, a.hdr_out, 12 * n, cudaMemcpyDeviceToHost, st));
        if (rgb_out) CKA(cudaMemcpyAsync(rgb_out, a.rgb_out, 3 * n, cudaMemcpyDeviceToHost, st));
        CKA(cudaStreamSynchronize(st));
    } else if (!stats) {
        return RBRT_OK;                                                   // enqueue only
    }
    if (stats) {
        CKA(cudaEventSynchronize(c.e1));
        float ms = 0; CKA(cudaEventElapsedTime(&ms, c.e0, c.e1));
        stats->ms_device = ms; stats->launches = 1 + a.levels;
        stats->ms_total = now_ms() - t0;
    }
    return RBRT_OK;
}

// ------------------------------------------------------------------ variance of a render from sample shards (rbrt_gpu_render_hdr_variance*)
// Shard k renders samples [k*n, (k+1)*n) into its own accumulator.  The shards alternate between two lanes: the caller's stream with the
// wavefront pool p of opts->flags, and an internal stream of the device with pool 4 + p (the second lane of RBRT_OPT_SPLIT_BATCHES).  No
// shard waits for another (each has its own accumulator), so the sparse last bounces of one shard run under the dense first bounces of the
// shard on the other lane.  The moments kernel then runs on the caller's stream behind both lanes.
static int render_variance(const rbrt_scene* scene, const rbrt_camera* cam, uint32_t S, uint32_t K, const rbrt_render_opts* opts,
                           float* hdr_out, float* var_out, bool host, cudaStream_t st, rbrt_stats* stats) {
    if (stats) memset(stats, 0, sizeof(*stats));
    if (!scene || !cam) { set_error("null argument"); return RBRT_E_INVALID; }
    if (!hdr_out && !var_out) { set_error("no output requested (hdr_out and var_out are both NULL)"); return RBRT_E_INVALID; }
    if (K < 2 || K > VR_MAX_SPLITS) { set_error("splits must be 2..%u", VR_MAX_SPLITS); return RBRT_E_INVALID; }
    if (!S || S % K) { set_error("num_samples must be a positive multiple of splits"); return RBRT_E_INVALID; }
    rbrt_render_opts o{}; if (opts) o = *opts;
    if (o.shard_count > 1) { set_error("shard_count > 1: the call shards the samples itself"); return RBRT_E_INVALID; }
    const size_t n = (size_t)cam->img_width_pix * cam->img_height_pix;
    if (!n) { set_error("empty image"); return RBRT_E_INVALID; }
    if (n > 0x7FFFFFFFull) { set_error("image too large"); return RBRT_E_INVALID; }
    if (overlap(hdr_out, 12 * n, var_out, 12 * n)) { set_error("hdr_out and var_out overlap"); return RBRT_E_INVALID; }
    const Scene& sc = *reinterpret_cast<const Scene*>(scene);
    const Replica& rp = sc.rep[0];                                        // under a communicator: this process's first device, whole image
    CKA(cudaSetDevice(rp.device));
    if (!host) {
        int rc = check_usable_on({hdr_out, var_out}, rp.device, "outputs must be device memory on the scene's device %d");
        if (rc) return rc;
    }
    const double t0 = now_ms();
    { int rc = resolve_scene_info(sc, true); if (rc) return rc; }         // a refused mesh is known before anything is written
    rbrt_variance_moments_launch_fn launch = nullptr;
    { int rc = module_entry(g_variance_module, "rbrt_variance_moments_launch", &launch); if (rc) return rc; }
    DeviceCache& c = g_cache[rp.device & 63];
    if (!c.aux) {
        CKA(cudaStreamCreateWithFlags(&c.aux, cudaStreamNonBlocking));
        CKA(cudaEventCreateWithFlags(&c.fork, cudaEventDisableTiming)); CKA(cudaEventCreateWithFlags(&c.join, cudaEventDisableTiming));
    }
    if (stats) { int rc = timing_events(c); if (rc) return rc; }
    const uint32_t pool = (o.flags & RBRT_OPT_POOL_MASK) >> RBRT_OPT_POOL_SHIFT;
    o.flags &= ~(uint32_t)RBRT_OPT_SPLIT_BATCHES;                         // the two lanes are the shards'
    o.shard_mode = RBRT_SHARD_SAMPLES; o.shard_count = K;

    // K accumulators, then (host variant) the two output planes, from the stream-ordered allocator on the call's stream
    const size_t b_acc = 16 * n * K, b3 = a256(12 * n);
    char* block = nullptr;
    CKA(cudaMallocAsync((void**)&block, b_acc + (host ? 2 * b3 : 0), st));
    MomentsArgs m;
    memset(&m, 0, sizeof(m));
    m.W = cam->img_width_pix; m.H = cam->img_height_pix; m.K = K;
    m.inv_S = 1.0f / (float)S; m.inv_n = 1.0f / (float)(S / K);
    m.acc = (const float4*)block;
    m.hdr_out = hdr_out ? (host ? (float*)(block + b_acc) : hdr_out) : nullptr;
    m.var_out = var_out ? (host ? (float*)(block + b_acc + b3) : var_out) : nullptr;
    std::vector<RenderJob> jobs(stats ? K : 0);
    uint32_t launches = 0;
    cudaError_t e = cudaSuccess;
    int rc = RBRT_OK;
    if (stats) e = cudaEventRecord(c.e0, st);
    if (e == cudaSuccess) e = cudaEventRecord(c.fork, st);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(c.aux, c.fork, 0);
    for (uint32_t k = 0; k < K && e == cudaSuccess && !rc; ++k) {
        const int lane = (int)(k & 1);
        o.shard_rank = k;
        float4* acc1[1] = {(float4*)(block + 16 * n * k)};
        rc = render_accum(sc, 0, cam, nullptr, 1, S, &o, acc1, lane ? c.aux : st, nullptr, stats ? &jobs[k] : nullptr, (int)pool + 4 * lane);
        if (rc || !stats || (lane == 0 && k + 1 < K)) continue;
        for (uint32_t j = k - lane; j <= k && !rc; ++j) {                 // this round's counters, before the next round resets its pools
            rbrt_stats one; memset(&one, 0, sizeof(one));
            rc = collect_stats(jobs[j], &one);
            stats->rays += one.rays; stats->paths += one.paths; stats->nan_rays += one.nan_rays; launches += one.launches;
        }
    }
    if (e == cudaSuccess) e = cudaEventRecord(c.join, c.aux);           // (also when a shard was refused: the block is freed behind both lanes)
    if (e == cudaSuccess) e = cudaStreamWaitEvent(st, c.join, 0);
    if (e == cudaSuccess && !rc) e = (cudaError_t)launch(&m, st);
    if (e == cudaSuccess && !rc && stats) e = cudaEventRecord(c.e1, st);
    if (e == cudaSuccess && !rc && host) {
        if (hdr_out) e = cudaMemcpyAsync(hdr_out, m.hdr_out, 12 * n, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess && var_out) e = cudaMemcpyAsync(var_out, m.var_out, 12 * n, cudaMemcpyDeviceToHost, st);
    }
    {
        const cudaError_t f = cudaFreeAsync(block, st);
        if (e == cudaSuccess) e = f;
    }
    if (rc) return rc;
    if (e != cudaSuccess) return cuda_fail(e, "rbrt_gpu_render_hdr_variance");
    if (host) CKA(cudaStreamSynchronize(st));
    if (stats) {
        CKA(cudaEventSynchronize(c.e1));
        float ms = 0; CKA(cudaEventElapsedTime(&ms, c.e0, c.e1));
        stats->ms_device = ms; stats->launches = launches + 1;
        stats->ms_total = now_ms() - t0;
        return resolve_scene_info(sc, true);
    }
    return RBRT_OK;
}

}  // namespace rbrt

using namespace rbrt;

extern "C" {

const char* rbrt_last_error(void) { return g_err; }
const char* rbrt_gpu_version(void) { return "rbrt_b200 0.2.0 sm_100a"; }

int rbrt_gpu_init(int device) {
    LOCK;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        set_error("no CUDA device available (%s); rbrt_b200 has no CPU fallback", e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
        cudaGetLastError();
        return RBRT_E_NODEVICE;
    }
    if (device < 0 || device >= n) { set_error("device %d out of range (0..%d)", device, n - 1); return RBRT_E_INVALID; }
    if (comm().active && comm().devices[0] != device) { set_error("a communicator is active on device %d; rbrt_gpu_comm_destroy() first", comm().devices[0]); return RBRT_E_INVALID; }
    CKA(cudaSetDevice(device));
    g_device = device;
    return RBRT_OK;
}

int rbrt_gpu_set_pool_limit(uint64_t max_bytes_per_pool) { LOCK; g_pool_limit = max_bytes_per_pool; return RBRT_OK; }

int rbrt_gpu_scene_create(const rbrt_sphere_desc* spheres, uint32_t ns, const rbrt_mesh_desc* meshes, uint32_t nm,
                          const rbrt_scene_opts* opts, rbrt_scene** out) {
    if (!out || (ns && !spheres) || (nm && !meshes)) { set_error("null argument"); return RBRT_E_INVALID; }
    std::vector<rbrt_element_ref> order(ns);
    for (uint32_t i = 0; i < ns; ++i) order[i] = rbrt_element_ref{RBRT_ELEM_SPHERE, i};
    return rbrt_gpu_scene_create_elements(order.data(), ns, spheres, ns, nullptr, 0, meshes, nm, opts, out);
}

int rbrt_gpu_scene_create_elements(const rbrt_element_ref* order, uint32_t ne, const rbrt_sphere_desc* spheres, uint32_t n_sph,
                                   const rbrt_triangle_desc* triangles, uint32_t n_bt, const rbrt_mesh_desc* meshes, uint32_t nm,
                                   const rbrt_scene_opts* opts, rbrt_scene** out) {
    LOCK;
    if (!out || (ne && !order) || (n_sph && !spheres) || (n_bt && !triangles) || (nm && !meshes)) { set_error("null argument"); return RBRT_E_INVALID; }
    uint32_t n_et = 0;
    for (uint32_t i = 0; i < ne; ++i) {
        if (order[i].kind == RBRT_ELEM_SPHERE ? order[i].index >= n_sph : (order[i].kind == RBRT_ELEM_TRIANGLE ? order[i].index >= n_bt : true)) {
            set_error("element %u: bad kind or index", i); return RBRT_E_INVALID;
        }
        const rbrt_material& m = order[i].kind == RBRT_ELEM_SPHERE ? spheres[order[i].index].material : triangles[order[i].index].material;
        if (m.kind > 2) { set_error("element %u: unknown material kind", i); return RBRT_E_INVALID; }
        if (order[i].kind == RBRT_ELEM_TRIANGLE) ++n_et;
    }
    const uint32_t ns = ne;                                               // below, `ns` counts ELEMENTS (spheres + basic triangles)
    *out = nullptr;
    uint32_t lanes = (opts && opts->simd_lanes) ? opts->simd_lanes : 8;
    if (lanes != 8 && lanes != 4) { set_error("simd_lanes must be 8 (AVX) or 4 (SSE)"); return RBRT_E_INVALID; }
    uint32_t leaf_size = (opts && opts->leaf_size) ? opts->leaf_size : 1;   // swept 1..8 on C3 (profiles/): a triangle test costs a warp step like a node visit, so fewer tests win
    if (leaf_size > 8) { set_error("leaf_size must be <= 8"); return RBRT_E_INVALID; }
    const uint32_t sflags = opts ? opts->flags : 0;
    float pad_rel = 2e-5f;
    if (opts && opts->box_pad_rel > 0.0f) pad_rel = opts->box_pad_rel;
    else if (opts && opts->box_pad_rel < 0.0f) pad_rel = 0.0f;
    if ((uint64_t)ns + nm > 65535) { set_error("more than 65535 scene elements"); return RBRT_E_INVALID; }
    int rc = ensure_device();
    if (rc) return rc;
    const bool collective = comm().active && comm().world > 1 && !(sflags & RBRT_SCENE_LOCAL);
    // replicas: one process -> built once, copied device to device; process per GPU -> every rank builds its own (default) or
    // rank 0 builds and broadcasts (RBRT_SCENE_BROADCAST)
    const bool replicate = collective && (!comm().multi_process || (sflags & RBRT_SCENE_BROADCAST));
    const bool is_root = !replicate || comm().rank == 0;                  // this process uploads and builds
    uint64_t total_tris = 0, total_eff = 0;
    for (uint32_t i = 0; i < nm; ++i) {
        if (meshes[i].material.kind > 2) { set_error("mesh %u: unknown material kind", i); return RBRT_E_INVALID; }
        if (meshes[i].num_triangles && !meshes[i].tri_vertices && is_root) { set_error("mesh %u: null tri_vertices", i); return RBRT_E_INVALID; }
        if (meshes[i].num_triangles > (1ull << 28)) { set_error("mesh %u: more than 2^28 triangles", i); return RBRT_E_INVALID; }
        total_tris += meshes[i].num_triangles;
        total_eff += tested_triangles(meshes[i].num_triangles, lanes);
    }
    if (total_eff > (1ull << 28)) { set_error("more than 2^28 triangles in the scene"); return RBRT_E_INVALID; }

    Scene* sc = new Scene();
    sc->device = g_device;
    sc->collective = collective;
    sc->n_elems = ns; sc->n_meshes = nm; sc->n_etris = n_et;
    sc->info.num_spheres = ns; sc->info.num_meshes = nm;
    sc->info.num_triangles = total_tris; sc->info.num_triangles_tested = total_eff;
    sc->pad_rel = pad_rel; sc->leaf_size = leaf_size; sc->sah = !(sflags & RBRT_SCENE_NO_SAH); sc->replicated = replicate;
    sc->mesh_n_all.resize(nm);
    for (uint32_t i = 0; i < nm; ++i) sc->mesh_n_all[i] = meshes[i].num_triangles;
    sc->elem_kind_h.resize(ns);
    for (uint32_t i = 0; i < ns; ++i) sc->elem_kind_h[i] = order[i].kind;
    double t0 = now_ms();

#define CKS(x) do { int rc_ = (x); if (rc_) { destroy_scene(sc); return rc_; } } while (0)
#define CKSC(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { int rc_ = cuda_fail(e_, #x); destroy_scene(sc); return rc_; } } while (0)

    // ---- the scene's device block.  The LBVH nodes come LAST: only the live ones (about N/3 of the N slots) are
    //      replicated to other GPUs.
    {
        ArenaLayout& L = sc->lay; size_t off = 0;
        L.tris = off; off += a256(48ull * total_eff);
        L.nrm = off; off += a256(16ull * total_eff);
        L.sph = off; off += a256(16ull * ns);
        L.mat = off; off += a256(16ull * (ns + nm));
        L.kind = off; off += a256(4ull * (ns + nm));
        L.mesh = off; off += a256(sizeof(MeshDev) * nm);
        L.etris = off; off += a256(64ull * n_et);
        L.ekind = off; off += a256(4ull * ns);
        L.result = off; off += a256(sizeof(BuildResult) * (nm ? nm : 1));
        L.nodes = off; off += a256(64ull * total_eff);
        L.total = off;
    }
    const int n_local = collective ? comm().local_n : 1;
    sc->rep.resize(n_local);
    for (int li = 0; li < n_local; ++li) {
        Replica& r = sc->rep[li];
        r.device = collective ? comm().devices[li] : g_device;
        CKSC(cudaSetDevice(r.device));
        CKS(device_sm_count(r.device, &r.sm_count));
        CKS(arena_alloc(r.device, sc->lay.total, &r.arena, &r.arena_bytes));
        r.dev = make_scene_dev(r.arena, sc->lay, ns, nm, n_et);
        sc->info.device_bytes += sc->lay.total;
    }
    CKSC(cudaSetDevice(sc->rep[0].device));
    sc->dev = sc->rep[0].dev; sc->sm_count = sc->rep[0].sm_count;
    char* const base = sc->rep[0].arena;
    sc->meshes_h.resize(nm);
    for (Replica& r : sc->rep) { CKSC(cudaSetDevice(r.device)); CKSC(cudaEventCreateWithFlags(&r.ready, cudaEventDisableTiming)); }
    CKSC(cudaSetDevice(sc->rep[0].device));
    sc->res_h = pinned_get(sizeof(BuildResult) * (nm ? nm : 1));
    if (!sc->res_h) { set_error("out of pinned host memory"); destroy_scene(sc); return RBRT_E_ALLOC; }
    memset(sc->res_h, 0, sizeof(BuildResult) * (nm ? nm : 1));
    CKSC(cudaEventCreate(&sc->info_ev));

    // Everything below is ENQUEUED: uploads on the device's copy stream, kernels on its build stream (bvh_build.cu).  The call
    // returns when the caller's arrays have been read; readers of the scene wait for Replica::ready on their own streams.
    BuildCtx ctx;
    CKSC(build_begin(sc->rep[0].device, &ctx));
    if (is_root) {
        CKSC(cudaEventCreate(&sc->t_up0)); CKSC(cudaEventCreate(&sc->t_up1)); CKSC(cudaEventCreate(&sc->t_b0)); CKSC(cudaEventCreate(&sc->t_b1));
        CKSC(cudaEventRecord(sc->t_up0, ctx.copy)); CKSC(cudaEventRecord(sc->t_b0, ctx.build));
        // ---- elements: spheres + per-element materials (flattened SoA, 16-byte records)
        std::vector<float4> sph(ns), mat(ns + nm), etris;
        std::vector<uint32_t> kind(ns + nm), ekind(ns);
        pack_elements(order, ns, spheres, triangles, sph, etris, mat, kind, ekind);
        for (uint32_t i = 0; i < nm; ++i) {
            mat[ns + i] = make_float4(meshes[i].material.albedo.x, meshes[i].material.albedo.y, meshes[i].material.albedo.z, meshes[i].material.param);
            kind[ns + i] = meshes[i].material.kind;
        }
        // small pageable arrays: cudaMemcpyAsync stages them before it returns, so the vectors may die at the end of this block
        if (ns) CKSC(cudaMemcpyAsync(base + sc->lay.sph, sph.data(), 16ull * ns, cudaMemcpyHostToDevice, ctx.copy));
        if (!etris.empty()) {
            CKSC(cudaMemcpyAsync(base + sc->lay.etris, etris.data(), 16ull * etris.size(), cudaMemcpyHostToDevice, ctx.copy));
            CKSC(cudaMemcpyAsync(base + sc->lay.ekind, ekind.data(), 4ull * ns, cudaMemcpyHostToDevice, ctx.copy));
        }
        if (ns + nm) {
            CKSC(cudaMemcpyAsync(base + sc->lay.mat, mat.data(), 16ull * (ns + nm), cudaMemcpyHostToDevice, ctx.copy));
            CKSC(cudaMemcpyAsync(base + sc->lay.kind, kind.data(), 4ull * (ns + nm), cudaMemcpyHostToDevice, ctx.copy));
        }
        CKSC(cudaStreamSynchronize(ctx.copy));                            // (these few KB only; keeps the staging assumption out of the contract)

        // ---- meshes: upload, exact AABB (aabbox.rs:62-88, over ALL real triangles), MeshDev record and LBVH, all on the device
        float4* d_tris = (float4*)(base + sc->lay.tris); float4* d_normals = (float4*)(base + sc->lay.nrm); float4* d_nodes = (float4*)(base + sc->lay.nodes);
        MeshDev* d_meshes = (MeshDev*)(base + sc->lay.mesh); BuildResult* d_res = (BuildResult*)(base + sc->lay.result);
        uint64_t tri_off = 0;
        for (uint32_t i = 0; i < nm; ++i) {
            const rbrt_mesh_desc& m = meshes[i];
            MeshDev md; memset(&md, 0, sizeof(md));
            const uint64_t n_eff = tested_triangles(m.num_triangles, lanes);
            md.tri_base = (uint32_t)tri_off; md.n_tris = (uint32_t)n_eff; md.node_base = (uint32_t)tri_off;
            md.nrm_base = (uint32_t)tri_off; md.elem = ns + i; md.root_ref = make_leaf_ref(0, 1);
            cudaError_t ce = build_mesh(ctx, m.tri_vertices, m.num_triangles, (uint32_t)n_eff, pad_rel, leaf_size, !(sflags & RBRT_SCENE_NO_SAH), md, d_meshes + i,
                                        d_tris + 3 * tri_off, d_normals + tri_off, d_nodes + 4 * tri_off, d_res + i);
            if (ce != cudaSuccess) { int rc_ = cuda_fail(ce, "build_mesh"); destroy_scene(sc); return rc_; }
            sc->meshes_h[i] = md;
            tri_off += n_eff;
        }
        CKSC(cudaEventRecord(sc->t_up1, ctx.copy));
        CKSC(cudaEventRecord(sc->t_b1, ctx.build));
    }
    if (replicate) CKS(replicate_scene(sc, ctx.build));                   // replicas on the other GPUs (multi.cu): NCCL broadcast / peer copies, enqueued behind the build
    else CKSC(cudaEventRecord(sc->rep[0].ready, ctx.build));
    // the per-mesh results: device -> pinned host, behind everything else on the build stream
    if (nm) CKSC(cudaMemcpyAsync(sc->res_h, base + sc->lay.result, sizeof(BuildResult) * nm, cudaMemcpyDeviceToHost, ctx.build));
    CKSC(cudaEventRecord(sc->info_ev, ctx.build));
    if (is_root) CKSC(cudaEventSynchronize(sc->t_up1));                   // the caller's triangle arrays have been read (copy engine: does not wait for busy SMs)
    sc->ms_host_create = now_ms() - t0;
    CKSC(cudaSetDevice(sc->rep[0].device));
    *out = reinterpret_cast<rbrt_scene*>(sc);
    return RBRT_OK;
#undef CKS
#undef CKSC
}

int rbrt_gpu_scene_info(const rbrt_scene* scene, rbrt_scene_info* out) {
    LOCK;
    if (!scene || !out) { set_error("null argument"); return RBRT_E_INVALID; }
    const Scene& sc = *reinterpret_cast<const Scene*>(scene);
    int rc = resolve_scene_info(sc, true);                                // waits for the (asynchronous) build; reports a refused mesh
    *out = sc.info;
    return rc;
}

int rbrt_gpu_scene_destroy(rbrt_scene* scene) {
    LOCK;
    if (!scene) return RBRT_OK;
    destroy_scene(reinterpret_cast<Scene*>(scene));
    return RBRT_OK;
}

int rbrt_gpu_scene_update_mesh(rbrt_scene* scene, uint32_t mesh_index, const float* tri_vertices, uint64_t num_triangles,
                               const rbrt_material* material, uint32_t flags) {
    LOCK;
    return update_mesh(scene, mesh_index, tri_vertices, false, num_triangles, material, flags, nullptr);
}

int rbrt_gpu_scene_update_mesh_device(rbrt_scene* scene, uint32_t mesh_index, const void* d_tri_vertices, uint64_t num_triangles,
                                      const rbrt_material* material, uint32_t flags, void* cuda_stream) {
    LOCK;
    return update_mesh(scene, mesh_index, (const float*)d_tri_vertices, true, num_triangles, material, flags, (cudaStream_t)cuda_stream);
}

int rbrt_gpu_scene_update_elements(rbrt_scene* scene, const rbrt_element_ref* order, uint32_t ne, const rbrt_sphere_desc* spheres,
                                   uint32_t n_sph, const rbrt_triangle_desc* triangles, uint32_t n_bt) {
    LOCK;
    if (!scene) { set_error("null argument"); return RBRT_E_INVALID; }
    Scene* sc = reinterpret_cast<Scene*>(scene);
    const bool receiver = sc->replicated && comm().multi_process && comm().rank != 0;   // RBRT_SCENE_BROADCAST: rank 0's values arrive by broadcast
    if (ne != sc->n_elems) { set_error("%u elements, the scene was created with %u (an update keeps them)", ne, sc->n_elems); return RBRT_E_INVALID; }
    const bool have = !receiver || order;
    if (have) {
        if ((ne && !order) || (n_sph && !spheres) || (n_bt && !triangles)) { set_error("null argument"); return RBRT_E_INVALID; }
        for (uint32_t i = 0; i < ne; ++i) {
            if (order[i].kind != sc->elem_kind_h[i]) { set_error("element %u: kind %u, created as %u (an update keeps the kinds)", i, order[i].kind, sc->elem_kind_h[i]); return RBRT_E_INVALID; }
            if (order[i].kind == RBRT_ELEM_SPHERE ? order[i].index >= n_sph : order[i].index >= n_bt) { set_error("element %u: bad index", i); return RBRT_E_INVALID; }
            const rbrt_material& m = order[i].kind == RBRT_ELEM_SPHERE ? spheres[order[i].index].material : triangles[order[i].index].material;
            if (m.kind > 2) { set_error("element %u: unknown material kind", i); return RBRT_E_INVALID; }
        }
    }
    BuildCtx ctx;
    { int rc = update_begin(sc, &ctx); if (rc) return rc; }
    if (have && ne) {
        std::vector<float4> sph(ne), mat(ne), etris;
        std::vector<uint32_t> kind(ne), ekind(ne);
        pack_elements(order, ne, spheres, triangles, sph, etris, mat, kind, ekind);
        const size_t b_sph = 16ull * ne, b_et = 16ull * etris.size(), b_mat = 16ull * ne, b_kind = 4ull * ne;
        Scene::Staging* sg = nullptr;
        { int rc = stage_get(sc, b_sph + b_et + b_mat + b_kind, &sg); if (rc) return rc; }
        char* h = (char*)sg->p;
        memcpy(h, sph.data(), b_sph); memcpy(h + b_sph, etris.data(), b_et);
        memcpy(h + b_sph + b_et, mat.data(), b_mat); memcpy(h + b_sph + b_et + b_mat, kind.data(), b_kind);
        char* const base = sc->rep[0].arena;
        CKA(cudaMemcpyAsync(base + sc->lay.sph, h, b_sph, cudaMemcpyHostToDevice, ctx.build));
        if (b_et) CKA(cudaMemcpyAsync(base + sc->lay.etris, h + b_sph, b_et, cudaMemcpyHostToDevice, ctx.build));
        CKA(cudaMemcpyAsync(base + sc->lay.mat, h + b_sph + b_et, b_mat, cudaMemcpyHostToDevice, ctx.build));
        CKA(cudaMemcpyAsync(base + sc->lay.kind, h + b_sph + b_et + b_mat, b_kind, cudaMemcpyHostToDevice, ctx.build));
        CKA(cudaEventRecord(sg->done, ctx.build));
    }
    return update_end(sc, ctx);
}

int rbrt_gpu_render_accum_device(const rbrt_scene* scene, const rbrt_camera* cam, uint32_t spp, const rbrt_render_opts* opts,
                                 void* d_accum, void* stream, rbrt_stats* stats) {
    LOCK;
    if (!scene || !cam || !d_accum) { set_error("null argument"); return RBRT_E_INVALID; }
    const Scene& sc = *reinterpret_cast<const Scene*>(scene);
    CKA(cudaSetDevice(sc.device));
    double t0 = now_ms();
    if (stats) memset(stats, 0, sizeof(*stats));
    float4* acc1[1] = {(float4*)d_accum};
    int rc = resolve_scene_info(sc, false);
    if (!rc) rc = render_accum(sc, 0, cam, nullptr, 1, spp, opts, acc1, (cudaStream_t)stream, stats);
    if (rc) return rc;
    if (stats) { stats->ms_total = now_ms() - t0; return resolve_scene_info(sc, true); }
    return RBRT_OK;
}

int rbrt_gpu_render_accum_device_frames(const rbrt_scene* scene, const rbrt_camera* cams, const uint64_t* seeds, uint32_t n_frames,
                                        uint32_t spp, const rbrt_render_opts* opts, void* const* d_accum, void* stream, rbrt_stats* stats) {
    LOCK;
    if (!scene || !cams || !seeds || !d_accum) { set_error("null argument"); return RBRT_E_INVALID; }
    if (!n_frames || n_frames > RBRT_MAX_FRAMES) { set_error("n_frames must be 1..%d", RBRT_MAX_FRAMES); return RBRT_E_INVALID; }
    float4* acc[RBRT_MAX_FRAMES];
    for (uint32_t f = 0; f < n_frames; ++f) { if (!d_accum[f]) { set_error("null accumulation buffer"); return RBRT_E_INVALID; } acc[f] = (float4*)d_accum[f]; }
    const Scene& sc = *reinterpret_cast<const Scene*>(scene);
    CKA(cudaSetDevice(sc.device));
    double t0 = now_ms();
    if (stats) memset(stats, 0, sizeof(*stats));
    int rc = resolve_scene_info(sc, false);
    if (!rc) rc = render_accum(sc, 0, cams, seeds, n_frames, spp, opts, acc, (cudaStream_t)stream, stats);
    if (rc) return rc;
    if (stats) { stats->ms_total = now_ms() - t0; return resolve_scene_info(sc, true); }
    return RBRT_OK;
}

int rbrt_gpu_release_cache(void) {
    LOCK;
    release_device_wave_buffers();
    release_dist_buffers();
    release_build_scratch();
    cache_release_all();
    arena_release_all();
    for (void* p : g_pinned_free) cudaFreeHost(p);
    g_pinned_free.clear();
    return RBRT_OK;
}

int rbrt_gpu_finalize_device(const void* d_accum, uint32_t W, uint32_t H, uint32_t spp, void* d_rgb, void* d_hdr, void* stream) {
    LOCK;
    if (!d_accum) { set_error("null argument"); return RBRT_E_INVALID; }
    int rc = ensure_device();
    if (rc) return rc;
    return finalize((const float4*)d_accum, W, H, spp, (uint8_t*)d_rgb, (float*)d_hdr, (cudaStream_t)stream);
}

int rbrt_gpu_render_frames_device(const rbrt_scene* scene, const rbrt_camera* cams, const uint64_t* seeds, uint32_t n_frames,
                                  uint32_t spp, const rbrt_render_opts* opts, void* const* d_rgb, void* const* d_hdr, void* stream, rbrt_stats* stats) {
    LOCK;
    if (!scene || !cams || !seeds) { set_error("null argument"); return RBRT_E_INVALID; }
    if (!n_frames || n_frames > RBRT_MAX_FRAMES) { set_error("n_frames must be 1..%d", RBRT_MAX_FRAMES); return RBRT_E_INVALID; }
    const Scene& sc = *reinterpret_cast<const Scene*>(scene);
    CKA(cudaSetDevice(sc.device));
    double t0 = now_ms();
    if (stats) memset(stats, 0, sizeof(*stats));
    int rc = render_frames(sc, cams, seeds, n_frames, spp, opts, (uint8_t* const*)d_rgb, (float* const*)d_hdr, (cudaStream_t)stream, stats);
    cudaSetDevice(sc.device);
    if (rc) return rc;
    if (stats) stats->ms_total = now_ms() - t0;
    return RBRT_OK;
}

// render_scene with HOST output: the collective render into the pool's own device image, then one copy to the host
static int render_host(const rbrt_scene* scene, const rbrt_camera* cam, uint32_t spp, const rbrt_render_opts* opts,
                       uint8_t* rgb_out, float* hdr_out, rbrt_stats* stats) {
    LOCK;
    if (!scene || !cam) { set_error("null argument"); return RBRT_E_INVALID; }
    const Scene& sc = *reinterpret_cast<const Scene*>(scene);
    rbrt_render_opts ro{}; if (opts) ro = *opts;
    opts = &ro;
    const bool sharded = sc.collective && opts->shard_count == 0;
    {   // a lone, blocking frame with enough paths per GPU (measured: pays from ~2^26 on, costs a few % below): two lanes (render.cu)
        const uint64_t share = (uint64_t)cam->img_width_pix * cam->img_height_pix * spp / (uint64_t)(sharded ? comm().world : (ro.shard_count > 1 ? ro.shard_count : 1));
        if (!(ro.flags & RBRT_OPT_TIME_KERNELS) && share >= (1ull << 26)) ro.flags |= RBRT_OPT_SPLIT_BATCHES;
    }
    const bool root = !sharded || comm().rank == 0;
    if (root && !rgb_out && !hdr_out) { set_error("null output"); return RBRT_E_INVALID; }
    CKA(cudaSetDevice(sc.device));
    double t0 = now_ms();
    size_t n = (size_t)cam->img_width_pix * cam->img_height_pix;
    if (!n || !spp) { set_error("empty image or zero samples"); return RBRT_E_INVALID; }
    WaveBuffers& wb = device_wave_buffers(sc.device, (int)((opts->flags & RBRT_OPT_POOL_MASK) >> RBRT_OPT_POOL_SHIFT));
    if (wb.out_px < n) {
        cudaFree(wb.rgb); cudaFree(wb.hdr); wb.rgb = nullptr; wb.hdr = nullptr; wb.out_px = 0;
        CKA(cudaMalloc(&wb.rgb, 3 * n)); CKA(cudaMalloc(&wb.hdr, 12 * n)); wb.out_px = n;
    }
    if (stats) memset(stats, 0, sizeof(*stats));
    rbrt_stats local; memset(&local, 0, sizeof(local));
    const uint64_t seed = opts->seed;
    uint8_t* rgb1[1] = {wb.rgb}; float* hdr1[1] = {wb.hdr};
    const bool want_rgb = rgb_out || (!root && !hdr_out), want_hdr = hdr_out != nullptr;    // every rank must make the same choice: see below
    int rc = render_frames(sc, cam, &seed, 1, spp, opts, want_rgb ? rgb1 : nullptr, want_hdr ? hdr1 : nullptr, 0, &local);
    cudaSetDevice(sc.device);
    if (rc) return rc;
    double t1 = now_ms();
    if (root && rgb_out) CKA(cudaMemcpy(rgb_out, wb.rgb, 3 * n, cudaMemcpyDeviceToHost));
    if (root && hdr_out) CKA(cudaMemcpy(hdr_out, wb.hdr, 12 * n, cudaMemcpyDeviceToHost));
    double t2 = now_ms();
    if (stats) { *stats = local; stats->ms_d2h = t2 - t1; stats->ms_total = t2 - t0; }
    return RBRT_OK;
}

int rbrt_gpu_render(const rbrt_scene* scene, const rbrt_camera* cam, uint32_t spp, const rbrt_render_opts* opts,
                    uint8_t* rgb_out, rbrt_stats* stats) {
    LOCK;                                                                 // (recursive: render_host takes it again; comm() is read under it)
    // non-root ranks of a collective render may pass NULL; the root must not
    if (!rgb_out && !(scene && reinterpret_cast<const Scene*>(scene)->collective && comm().rank != 0 && (!opts || opts->shard_count == 0))) {
        set_error("null rgb_out"); return RBRT_E_INVALID;
    }
    return render_host(scene, cam, spp, opts, rgb_out, nullptr, stats);
}

int rbrt_gpu_render_hdr(const rbrt_scene* scene, const rbrt_camera* cam, uint32_t spp, const rbrt_render_opts* opts,
                        float* hdr_out, rbrt_stats* stats) {
    LOCK;
    static float dummy;                                                   // non-root ranks: "an HDR render", without a buffer
    const bool nonroot = scene && reinterpret_cast<const Scene*>(scene)->collective && comm().rank != 0 && (!opts || opts->shard_count == 0);
    if (!hdr_out && !nonroot) { set_error("null rgb_f32_out"); return RBRT_E_INVALID; }
    return render_host(scene, cam, spp, opts, nullptr, hdr_out ? hdr_out : (nonroot ? &dummy : nullptr), stats);
}

int rbrt_gpu_trace_rays(const rbrt_scene* scene, const rbrt_ray* rays, uint64_t n, uint32_t mode, rbrt_hit* hits, rbrt_stats* stats) {
    LOCK;
    if (!scene || (n && (!rays || !hits))) { set_error("null argument"); return RBRT_E_INVALID; }
    if (mode > RBRT_TRACE_WAVEFRONT) { set_error("unknown trace_mode %u", mode); return RBRT_E_INVALID; }
    const Scene& sc = *reinterpret_cast<const Scene*>(scene);
    CKA(cudaSetDevice(sc.device));
    if (stats) memset(stats, 0, sizeof(*stats));
    { int rc = resolve_scene_info(sc, true); if (rc) return rc; }         // a refused mesh: the hits would not be Scene::hit's
    if (!n) return RBRT_OK;
    double t0 = now_ms();
    rbrt_ray* d_rays = nullptr; rbrt_hit* d_hits = nullptr; unsigned long long* d_stats = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    int rc = RBRT_OK;
    cudaError_t ce;
#define CKT(x) do { ce = (x); if (ce != cudaSuccess) { rc = cuda_fail(ce, #x); goto done; } } while (0)
    CKT(cudaMalloc(&d_rays, sizeof(rbrt_ray) * n)); CKT(cudaMalloc(&d_hits, sizeof(rbrt_hit) * n));
    CKT(cudaMalloc(&d_stats, 8 * ST_COUNT)); CKT(cudaMemset(d_stats, 0, 8 * ST_COUNT));
    CKT(cudaEventCreate(&e0)); CKT(cudaEventCreate(&e1));
    {
        double t1 = now_ms();
        CKT(cudaMemcpy(d_rays, rays, sizeof(rbrt_ray) * n, cudaMemcpyHostToDevice));
        double t2 = now_ms();
        CKT(cudaEventRecord(e0, 0));
        rc = mode == RBRT_TRACE_WAVEFRONT ? trace_rays_wavefront(sc, d_rays, n, d_hits, stats ? d_stats : nullptr, 0)
                                          : trace_rays_device(sc, d_rays, n, mode, d_hits, stats ? d_stats : nullptr, 0);
        if (rc) goto done;
        CKT(cudaEventRecord(e1, 0));
        CKT(cudaEventSynchronize(e1));
        double t3 = now_ms();
        CKT(cudaMemcpy(hits, d_hits, sizeof(rbrt_hit) * n, cudaMemcpyDeviceToHost));
        double t4 = now_ms();
        if (stats) {
            unsigned long long h[ST_COUNT];
            CKT(cudaMemcpy(h, d_stats, sizeof(h), cudaMemcpyDeviceToHost));
            float ms = 0; CKT(cudaEventElapsedTime(&ms, e0, e1));
            stats->rays = n; stats->nan_rays = h[ST_NAN]; stats->node_visits = h[ST_NODES]; stats->tri_tests = h[ST_TRIS]; stats->traversed_rays = h[ST_CAND];
            stats->ms_device = ms; stats->ms_trace = ms; stats->ms_h2d = t2 - t1; stats->ms_d2h = t4 - t3; stats->launches = mode == RBRT_TRACE_WAVEFRONT ? 3 : 1;
            stats->ms_total = now_ms() - t0;
        }
    }
done:
#undef CKT
    if (e0) cudaEventDestroy(e0);
    if (e1) cudaEventDestroy(e1);
    cudaFree(d_rays); cudaFree(d_hits); cudaFree(d_stats);
    return rc;
}

int rbrt_gpu_render_aov(const rbrt_scene* scene, const rbrt_camera* cam, uint32_t num_samples, uint64_t seed, const rbrt_aov_out* out,
                        rbrt_stats* stats) {
    LOCK;
    return render_aov(scene, cam, num_samples, seed, out, true, 0, stats);
}

int rbrt_gpu_render_aov_device(const rbrt_scene* scene, const rbrt_camera* cam, uint32_t num_samples, uint64_t seed, const rbrt_aov_out* d_out,
                               void* cuda_stream, rbrt_stats* stats) {
    LOCK;
    return render_aov(scene, cam, num_samples, seed, d_out, false, (cudaStream_t)cuda_stream, stats);
}

int rbrt_gpu_query_closest_device(const rbrt_scene* scene, const rbrt_ray* d_rays, uint64_t n, const rbrt_query_out* d_out, void* cuda_stream,
                                  rbrt_stats* stats) {
    LOCK;
    return query(scene, d_rays, n, false, d_out, nullptr, nullptr, (cudaStream_t)cuda_stream, stats);
}

int rbrt_gpu_query_occluded_device(const rbrt_scene* scene, const rbrt_ray* d_rays, uint64_t n, const float* d_max_dist, uint8_t* d_occluded,
                                   void* cuda_stream, rbrt_stats* stats) {
    LOCK;
    return query(scene, d_rays, n, true, nullptr, d_max_dist, d_occluded, (cudaStream_t)cuda_stream, stats);
}

int rbrt_gpu_denoise(uint32_t width, uint32_t height, const float* hdr, const rbrt_aov_out* guides, const rbrt_denoise_opts* opts,
                     float* hdr_out, uint8_t* rgb_out, rbrt_stats* stats) {
    LOCK;
    return denoise(width, height, hdr, nullptr, guides, opts, hdr_out, rgb_out, false, true, 0, stats);
}

int rbrt_gpu_denoise_device(uint32_t width, uint32_t height, const float* d_hdr, const rbrt_aov_out* d_guides, const rbrt_denoise_opts* opts,
                            float* d_hdr_out, uint8_t* d_rgb_out, void* cuda_stream, rbrt_stats* stats) {
    LOCK;
    return denoise(width, height, d_hdr, nullptr, d_guides, opts, d_hdr_out, d_rgb_out, false, false, (cudaStream_t)cuda_stream, stats);
}

int rbrt_gpu_render_hdr_variance(const rbrt_scene* scene, const rbrt_camera* cam, uint32_t num_samples, uint32_t splits,
                                 const rbrt_render_opts* opts, float* hdr_out, float* var_out, rbrt_stats* stats) {
    LOCK;
    return render_variance(scene, cam, num_samples, splits, opts, hdr_out, var_out, true, 0, stats);
}

int rbrt_gpu_render_hdr_variance_device(const rbrt_scene* scene, const rbrt_camera* cam, uint32_t num_samples, uint32_t splits,
                                        const rbrt_render_opts* opts, float* d_hdr_out, float* d_var_out, void* cuda_stream, rbrt_stats* stats) {
    LOCK;
    return render_variance(scene, cam, num_samples, splits, opts, d_hdr_out, d_var_out, false, (cudaStream_t)cuda_stream, stats);
}

int rbrt_gpu_denoise_variance(uint32_t width, uint32_t height, const float* hdr, const float* var, const rbrt_aov_out* guides,
                              const rbrt_denoise_opts* opts, float* hdr_out, uint8_t* rgb_out, rbrt_stats* stats) {
    LOCK;
    return denoise(width, height, hdr, var, guides, opts, hdr_out, rgb_out, true, true, 0, stats);
}

int rbrt_gpu_denoise_variance_device(uint32_t width, uint32_t height, const float* d_hdr, const float* d_var, const rbrt_aov_out* d_guides,
                                     const rbrt_denoise_opts* opts, float* d_hdr_out, uint8_t* d_rgb_out, void* cuda_stream, rbrt_stats* stats) {
    LOCK;
    return denoise(width, height, d_hdr, d_var, d_guides, opts, d_hdr_out, d_rgb_out, true, false, (cudaStream_t)cuda_stream, stats);
}

int rbrt_gpu_scatter(const rbrt_scatter_in* items, uint64_t n, uint64_t seed, rbrt_scatter_out* out) {
    LOCK;
    if (n && (!items || !out)) { set_error("null argument"); return RBRT_E_INVALID; }
    int rc = ensure_device();
    if (rc) return rc;
    if (!n) return RBRT_OK;
    for (uint64_t i = 0; i < n; ++i) if (items[i].material.kind > 2) { set_error("item %llu: unknown material kind", (unsigned long long)i); return RBRT_E_INVALID; }
    rbrt_scatter_in* d_in = nullptr; rbrt_scatter_out* d_out = nullptr;
    cudaError_t ce = cudaMalloc(&d_in, sizeof(rbrt_scatter_in) * n);
    if (ce == cudaSuccess) ce = cudaMalloc(&d_out, sizeof(rbrt_scatter_out) * n);
    if (ce == cudaSuccess) ce = cudaMemcpy(d_in, items, sizeof(rbrt_scatter_in) * n, cudaMemcpyHostToDevice);
    if (ce == cudaSuccess) { rc = scatter_device(d_in, n, seed, d_out, 0); if (!rc) ce = cudaMemcpy(out, d_out, sizeof(rbrt_scatter_out) * n, cudaMemcpyDeviceToHost); }
    cudaFree(d_in); cudaFree(d_out);
    if (ce != cudaSuccess) return cuda_fail(ce, "rbrt_gpu_scatter");
    return rc;
}

int rbrt_gpu_primary_rays(const rbrt_camera* cam, uint64_t seed, uint32_t sample, rbrt_ray* rays_out) {
    LOCK;
    if (!cam || !rays_out) { set_error("null argument"); return RBRT_E_INVALID; }
    int rc = ensure_device();
    if (rc) return rc;
    size_t n = (size_t)cam->img_width_pix * cam->img_height_pix;
    if (!n) return RBRT_OK;
    rbrt_ray* d = nullptr;
    CKA(cudaMalloc(&d, sizeof(rbrt_ray) * n));
    rc = primary_rays_device(*cam, seed, sample, d, 0);
    if (!rc) { cudaError_t e = cudaMemcpy(rays_out, d, sizeof(rbrt_ray) * n, cudaMemcpyDeviceToHost); if (e != cudaSuccess) rc = cuda_fail(e, "cudaMemcpy"); }
    cudaFree(d);
    return rc;
}

}  // extern "C"
