/*
 * rbrt_gpu.h — C-ABI boundary of the B200 path tracer that replaces rbrt_lib's hot path.
 *
 * rbrt (the reference, Rust) has no FFI today: the hot path sits behind the library call
 *     pub fn render_scene(cam: Camera, num_samples: u32, scene: Scene) -> ImageBuffer<Rgb<u8>>
 *                                                           (rbrt_lib/src/lib.rs:75-79)
 * whose only caller is src/main.rs:82.  `Scene` holds type-erased `Box<dyn Intersectable>` /
 * `Box<dyn RayScattering>` objects (rbrt_lib/src/scene.rs:12-16), so a GPU scene cannot be
 * recovered from a built `Scene`; the boundary therefore hooks at the blueprint level
 * (rbrt_lib/src/blueprints.rs:132 create_scene_from_scene_blueprint): plain-old-data sphere,
 * mesh and material descriptions in, opaque scene handle out.
 *
 * Every entry point is `extern "C"`, takes plain pointers and sizes, never unwinds, returns
 * 0 on success and a non-zero RBRT_E_* code on failure (message via rbrt_last_error()).
 * The CPU checker used by the tests mirrors these shapes (see DESIGN.md); it is never linked here.
 *
 * Multi-GPU is INSIDE this boundary, like the reference's one parallelism strategy is inside render_scene
 * (rayon over columns, rbrt_lib/src/lib.rs:84-86).  Two set-ups, same entry points afterwards:
 *   - one process, N GPUs:     rbrt_gpu_init_multi(devices, N, transport)
 *   - one process per GPU:     rbrt_gpu_init(device); rank 0: rbrt_gpu_comm_unique_id(id); every rank:
 *                              rbrt_gpu_comm_init_rank(id, rank, world)   (id travels over any side channel)
 * Under a communicator rbrt_gpu_scene_create makes one replica of the scene per GPU — one process: built once, copied
 * device to device over NVLink (NCCL broadcast / peer copies); process per GPU: built by every rank from its own arrays,
 * or by rank 0 alone + ncclBroadcast (RBRT_SCENE_BROADCAST) — and rbrt_gpu_render shards the image by
 * interleaved 8x4-pixel tiles (or by sample range), every GPU finalises its own pixels and rank 0 gathers them.
 * The explicit building blocks (rbrt_render_opts.shard_*, rbrt_gpu_render_accum_device) remain for hosts that
 * place shards themselves.
 */
#ifndef RBRT_GPU_H
#define RBRT_GPU_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- plain data mirrored from the reference ------------------------------------------ */

/* = rbrt_lib::vec3::Vec3 (rbrt_lib/src/vec3.rs:6-10), 12 bytes */
typedef struct rbrt_vec3 { float x, y, z; } rbrt_vec3;

/* = rbrt_lib::ray::Ray (rbrt_lib/src/ray.rs:4-7), 24 bytes */
typedef struct rbrt_ray { rbrt_vec3 origin, direction; } rbrt_ray;

/* = rbrt_lib::cam::Camera, the 14 pub fields in declaration order (rbrt_lib/src/cam.rs:4-19) */
typedef struct rbrt_camera {
    float     hor_fov_rad;
    uint32_t  img_width_pix;
    float     img_height_mm;
    float     vert_fov_rad;
    uint32_t  img_height_pix;
    float     img_width_mm;
    rbrt_vec3 position;
    float     focal_len_mm;
    rbrt_vec3 look_at;
    rbrt_vec3 up;
    rbrt_vec3 right;
    rbrt_vec3 img_center_point;
    float     mm_per_pix_hor;
    float     mm_per_pix_vert;
} rbrt_camera;

/* material kinds = the three RayScattering impls (lambertian.rs:6, metal.rs:6, dielectric.rs:6) */
enum { RBRT_MAT_LAMBERTIAN = 0, RBRT_MAT_METAL = 1, RBRT_MAT_DIELECTRIC = 2 };

/* albedo: Lambertian/Metal; param: Metal roughness or Dielectric ref_idx
 * (blueprints.rs:50-74 create_material_from_description) */
typedef struct rbrt_material { uint32_t kind; rbrt_vec3 albedo; float param; } rbrt_material;

/* = rbrt_lib::sphere::Sphere (sphere.rs:6-10) */
typedef struct rbrt_sphere_desc { rbrt_vec3 center; float radius; rbrt_material material; } rbrt_sphere_desc;

/* = rbrt_lib::triangle::BasicTriangle::new(corners, material) (triangle.rs:9-28): a single triangle as a scene ELEMENT
 * (an `Intersectable` pushed into Scene.elements next to the spheres; unreachable from the YAML/CLI path).  Counter-clockwise
 * corners; tested by basic_triangle_intersect_w_ray (triangle.rs:92-130): same Moeller-Trumbore arithmetic as the mesh
 * sweep but `u` must lie IN [0,1] (NaN rejects), there is no upper cap on t, and dist is accepted in [min_dist, max_dist]. */
typedef struct rbrt_triangle_desc { rbrt_vec3 corners[3]; rbrt_material material; } rbrt_triangle_desc;

/* One entry of Scene.elements (scene.rs:13), in iteration order: kind RBRT_ELEM_SPHERE -> spheres[index],
 * RBRT_ELEM_TRIANGLE -> triangles[index].  Order matters: the earlier element wins exact distance ties (scene.rs:23-31). */
enum { RBRT_ELEM_SPHERE = 0, RBRT_ELEM_TRIANGLE = 1 };
typedef struct rbrt_element_ref { uint32_t kind; uint32_t index; } rbrt_element_ref;

/* = what TriangleMesh::new (mesh.rs:41-74) holds after load_mesh_vertices_from_file
 * (mesh.rs:78-121): world-space triangle soup, 9 floats per triangle (v0 v1 v2), already
 * scale -> rotate_point -> translate'd in f32.  One material per mesh (mesh.rs:24).
 * Coordinates: any f32 value, inf and NaN included; hits are the reference's at every extent.  The BVH culls on an axis only while
 * its node grid step, (padded extent) / 65 500, is at most 2e6, i.e. up to a padded extent of about 1.3e11 on that axis (the padding is
 * 2e-5 of the mesh's largest coordinate).  Beyond that the axis is not culled; from a largest coordinate or extent of about 3.3e15 on
 * the padding alone exceeds it on every axis and the mesh is traversed like a brute-force sweep: exact, but slow. */
typedef struct rbrt_mesh_desc {
    const float*  tri_vertices;   /* num_triangles * 9 floats, caller keeps ownership */
    uint64_t      num_triangles;
    rbrt_material material;
} rbrt_mesh_desc;

/* Result of one closest-hit query = what Scene::hit (scene.rs:19-43) returns, plus ids. */
enum { RBRT_HIT_NONE = -1, RBRT_HIT_SPHERE = 0, RBRT_HIT_MESH = 1, RBRT_HIT_TRIANGLE = 2 /* a BasicTriangle element */ };
typedef struct rbrt_hit {
    int32_t   kind;       /* RBRT_HIT_* */
    uint32_t  elem_idx;   /* position in Scene.elements (spheres / basic triangles), or mesh index, in creation order */
    uint32_t  tri_idx;    /* original triangle index inside the mesh (0 for spheres) */
    float     t;          /* ray parameter */
    float     dist;       /* dist_from_ray_orig (lib.rs:35) */
    rbrt_vec3 point;      /* hit_point */
    rbrt_vec3 normal;     /* hit_normal: unit for meshes, un-normalised for spheres (sphere.rs:56) */
} rbrt_hit;

/* ---- options -------------------------------------------------------------------------- */

/* How triangle meshes are padded / truncated for SIMD.  The reference picks this at run time
 * (mesh.rs:27-39 determine_num_vector_lanes); AVX (8) is the baseline build. */
enum { RBRT_LANES_AVX = 8, RBRT_LANES_SSE = 4 };

enum { RBRT_SHARD_NONE = 0, RBRT_SHARD_TILES = 1, RBRT_SHARD_SAMPLES = 2 };
enum {
    RBRT_TRACE_BVH = 0,        /* per-mesh LBVH (render: the wavefront kernels; rbrt_gpu_trace_rays: a plain one-lane-one-ray traversal) */
    RBRT_TRACE_BRUTE = 1,      /* every triangle, the reference's own loop (triangle.rs:163-262) */
    RBRT_TRACE_WAVEFRONT = 2   /* rbrt_gpu_trace_rays only: the caller's rays go through the RENDERER's own kernels — stage A
                                  (spheres + mesh-AABB pre-test) and k_trace (persistent warps, warp-voted traversal, dynamic fetch) */
};
#define RBRT_MAX_FRAMES 4      /* frames one wavefront batch can hold (rbrt_gpu_render_accum_device_frames) */
enum {
    RBRT_OPT_COUNT_VISITS = 1,   /* fill rbrt_stats.node_visits / tri_tests (instrumented kernels, slower) */
    RBRT_OPT_TIME_KERNELS = 2,   /* bracket every trace launch with CUDA events -> rbrt_stats.ms_trace */
    RBRT_OPT_NO_TAIL_KERNEL = 4, /* run all 51 bounce iterations as wavefront launches (no single-launch tail) */
    RBRT_OPT_POOL_SHIFT = 3,     /* bits 3-4: which of the device's FOUR pools of wavefront state the call uses (0 = default), so that
                                    up to four renders can be in flight on four streams (rbrt_gpu_render_accum_device with
                                    stats = NULL returns without synchronising): the sparse last bounces of one frame then
                                    overlap the dense first bounces of the next */
    RBRT_OPT_POOL_MASK = 24,
    RBRT_OPT_SPLIT_BATCHES = 32  /* render the frame's samples as (at least) two batches on two internal lanes, so that the sparse, latency-bound
                                    end of one batch runs under the dense start of the next: shortens a LONE, LARGE frame (rbrt_gpu_render and
                                    rbrt_gpu_render_hdr set it themselves from 2^26 paths per GPU; smaller frames lose a few %).  Leave it off
                                    when several frames are in flight anyway.  Images do not depend on it. */
};

enum {
    RBRT_SCENE_LOCAL = 1,     /* under a communicator: build on THIS rank only, no replication (renders of it are not auto-sharded) */
    RBRT_SCENE_NO_SAH = 2,    /* skip the SAH pass over the LBVH (tree rotations during the refit): the plain Morton-order tree */
    RBRT_SCENE_BROADCAST = 4  /* one process per GPU only: rank 0 alone uploads and builds, the other ranks receive the scene's device block by
                                 ncclBroadcast (they may pass tri_vertices = NULL).  Default there: EVERY rank uploads and builds from its own
                                 (identical) arrays — no rank waits for another, measured faster (DESIGN.md section 7).  One process driving
                                 several GPUs always builds once and copies device to device. */
};
typedef struct rbrt_scene_opts {
    uint32_t simd_lanes;     /* RBRT_LANES_*; 0 = 8 */
    uint32_t leaf_size;      /* max triangles per BVH leaf; 0 = default */
    float    box_pad_rel;    /* conservative padding of BVH boxes relative to the mesh's largest coordinate; 0 = default (2e-5, and never less
                              * than 2^-21 * (that coordinate + 1000): rays may start 1000 units away), <0 = none */
    uint32_t flags;          /* RBRT_SCENE_* */
} rbrt_scene_opts;

typedef struct rbrt_render_opts {
    uint64_t seed;           /* Philox key */
    uint32_t max_depth;      /* 0 = 50 (lib.rs:99) */
    uint32_t trace_mode;     /* RBRT_TRACE_* */
    uint32_t shard_mode;     /* RBRT_SHARD_* */
    uint32_t shard_rank;
    uint32_t shard_count;    /* 0 = automatic: unsharded, or - for a scene created under a communicator - sharded over its GPUs with the
                                gather on rank 0 inside the call; 1 = this GPU renders everything; > 1 = the host places shard_rank of
                                shard_count itself (no collective) */
    uint32_t batch_paths;    /* paths in flight per wavefront batch; 0 = as many as fit (<= 2^27, <= half of free HBM) */
    uint32_t integrator;     /* 0 = wavefront (default); other values are rejected */
    uint32_t flags;          /* RBRT_OPT_* */
} rbrt_render_opts;

typedef struct rbrt_stats {
    uint64_t rays;           /* closest-hit queries (= calls to Scene::hit): primary + bounces */
    uint64_t paths;          /* samples rendered = pixels_in_shard * spp_in_shard */
    uint64_t nan_rays;       /* rays the reference would have panicked on (sphere.rs:33) */
    uint64_t node_visits;    /* BVH node visits (only when counters are compiled in / enabled) */
    uint64_t tri_tests;
    double   ms_total;       /* whole call, host clock */
    double   ms_device;      /* device time of the render proper (CUDA events) */
    double   ms_trace;       /* device time inside trace kernels (events, wavefront only) */
    double   ms_h2d;
    double   ms_d2h;
    uint32_t launches;       /* kernels launched by this call */
    uint32_t iterations;     /* wavefront bounce iterations executed */
    uint64_t traversed_rays; /* rays that entered a mesh AABB and were traversed through the LBVH (RBRT_OPT_COUNT_VISITS) */
    uint64_t tail_node_visits, tail_tri_tests, tail_traversed_rays;   /* the part of the three counters above done by the tail kernel */
} rbrt_stats;

typedef struct rbrt_scene_info {
    uint32_t num_spheres, num_meshes;
    uint64_t num_triangles;        /* real triangles handed in */
    uint64_t num_triangles_tested; /* N_eff after the reference's SIMD tail rule */
    uint64_t num_bvh_nodes;
    uint64_t device_bytes;
    double   ms_upload, ms_build;
} rbrt_scene_info;

typedef struct rbrt_scene rbrt_scene;   /* opaque */

/* ---- error codes ---------------------------------------------------------------------- */
enum {
    RBRT_OK = 0,
    RBRT_E_INVALID = 1,      /* bad argument */
    RBRT_E_CUDA = 2,         /* CUDA runtime error */
    RBRT_E_NODEVICE = 3,     /* no usable GPU: there is NO CPU fallback */
    RBRT_E_ALLOC = 4
};

/* ---- host-side helpers (pure f32 arithmetic, no GPU) ------------------------------------ */

/* = Camera::new(position, look_at, up, img_height_pix, img_width_pix, focal_len_mm)
 *   (cam.rs:22-62).  NOTE the reference's argument order: height before width. */
int rbrt_camera_new(rbrt_vec3 position, rbrt_vec3 look_at, rbrt_vec3 up,
                    uint32_t img_height_pix, uint32_t img_width_pix, float focal_len_mm,
                    rbrt_camera* out);

/* = the per-vertex transform of load_mesh_vertices_from_file (mesh.rs:102-112):
 *   v*scale -> Vec3::rotate_point(rotation) (vec3.rs:139-155) -> + translation, in place on
 *   n_vertices xyz triples. */
int rbrt_transform_vertices(float* xyz, uint64_t n_vertices, float scale,
                            rbrt_vec3 rotation_rad, rbrt_vec3 translation);

/* = load_mesh_vertices_from_file(filepath, translation, rotation, scale) (mesh.rs:78-121): reads the
 *   .obj the way the reference consumes tobj 4's default output (every model's position indices cut
 *   into triples; `f` and `l` records, `o` / `g` / `usemtl` model boundaries, relative indices; see
 *   csrc/obj_loader.cpp), applies the transform above to every corner and returns a malloc'ed
 *   num_triangles x 9 f32 soup (*tri_vertices_out = NULL for none) — what rbrt_mesh_desc.tri_vertices
 *   takes.  Free it with rbrt_mesh_free.  Where the reference panics (`assert!(loaded_mesh.is_ok())`,
 *   mesh.rs:89: unreadable file, malformed record, index out of bounds) this returns RBRT_E_INVALID
 *   and rbrt_last_error() names the line.  Parses on all host threads (RBRT_HOST_THREADS caps them). */
int rbrt_mesh_load_obj(const char* filepath, rbrt_vec3 translation, rbrt_vec3 rotation_rad, float scale,
                       float** tri_vertices_out, uint64_t* num_triangles_out);
void rbrt_mesh_free(float* tri_vertices);

/* ---- GPU entry points ------------------------------------------------------------------- */

/* Select the CUDA device this process renders on (one process per GPU). */
int rbrt_gpu_init(int device);

/* ---- multi-GPU set-up (see the head of this file) ---------------------------------------- */
#define RBRT_COMM_ID_BYTES 128           /* = sizeof(ncclUniqueId) */
enum {
    RBRT_TRANSPORT_AUTO = 0,             /* one process: PEER when every GPU can map GPU 0's memory, else NCCL; process per GPU: NCCL */
    RBRT_TRANSPORT_NCCL = 1,             /* NCCL broadcast / send-recv gather / reduce over NVLink */
    RBRT_TRANSPORT_PEER = 2              /* one process only: the finalise kernel of every GPU stores its pixels straight into rank 0's
                                            image through peer-mapped memory (compute + gather in ONE kernel), scene replicas by peer copies */
};
typedef struct rbrt_comm_info {
    int32_t  active, world, rank, local_devices;   /* rank = global rank of this process's first device */
    int32_t  transport;                            /* RBRT_TRANSPORT_* in use */
    int32_t  nccl_version;                         /* of the library loaded at run time, 0 if none */
    int32_t  devices[16];
} rbrt_comm_info;
/* One process, n_devices GPUs (devices == NULL: 0..n_devices-1).  The same device may be listed several times with
 * RBRT_TRANSPORT_PEER (a one-GPU emulation of N ranks, used by the tests). */
int rbrt_gpu_init_multi(const int* devices, int n_devices, int transport);
int rbrt_gpu_comm_unique_id(uint8_t id_out[RBRT_COMM_ID_BYTES]);
int rbrt_gpu_comm_init_rank(const uint8_t id[RBRT_COMM_ID_BYTES], int rank, int world);
int rbrt_gpu_comm_info(rbrt_comm_info* out);
int rbrt_gpu_comm_destroy(void);

/* = create_scene_from_scene_blueprint (blueprints.rs:132-158) after material parsing: copies
 *   the inputs to 16-byte-aligned SoA device buffers, applies the reference's SIMD tail rule
 *   (mesh.rs:136-144 + triangle.rs:167), computes edges / unit normals / exact mesh AABB
 *   (mesh.rs:50-61, triangle.rs:30-34, aabbox.rs:62-88) and builds one LBVH per mesh on the GPU.
 *   opts may be NULL. */
int rbrt_gpu_scene_create(const rbrt_sphere_desc* spheres, uint32_t num_spheres,
                          const rbrt_mesh_desc* meshes, uint32_t num_meshes,
                          const rbrt_scene_opts* opts, rbrt_scene** out);
/* Same, with Scene.elements given explicitly as an ordered mix of spheres and BasicTriangles (`order`, num_elements entries);
 *   rbrt_gpu_scene_create(...) == this with order = every sphere in array order. */
int rbrt_gpu_scene_create_elements(const rbrt_element_ref* order, uint32_t num_elements,
                                   const rbrt_sphere_desc* spheres, uint32_t num_spheres,
                                   const rbrt_triangle_desc* triangles, uint32_t num_triangles,
                                   const rbrt_mesh_desc* meshes, uint32_t num_meshes,
                                   const rbrt_scene_opts* opts, rbrt_scene** out);
int rbrt_gpu_scene_info(const rbrt_scene* scene, rbrt_scene_info* out);
int rbrt_gpu_scene_destroy(rbrt_scene* scene);

/* ---- updating a scene in place (animation) ------------------------------------------------
 * New vertices for a mesh, new values for Scene.elements, without creating the scene again.  The scene keeps its counts, its element
 * kinds, its device block and, by default, each mesh's tree topology.  Every update is ordered after every render / trace already
 * enqueued against the scene (on any stream, any replica) and before every one enqueued afterwards; replicas under a communicator
 * are updated too (one process: replica 0 is updated and copied again; process per GPU: the call is collective like the creation,
 * every rank updates its own replica from its own arrays, or with RBRT_SCENE_BROADCAST rank 0 updates and broadcasts and the other
 * ranks may pass NULL data).  rbrt_scene_info keeps describing the creation.  Images and hits are bit-exact for the new geometry
 * whatever the tree's shape (DESIGN.md section 10); a refit tree may only be slower to traverse.
 * Refused with RBRT_E_INVALID, the scene untouched: a triangle or element count, or element kinds, that differ from the creation,
 * a bad mesh index, an unknown material kind, NULL data, a scene with a mesh whose tree was refused as too deep. */
enum {
    RBRT_UPDATE_REFIT = 0,     /* keep the mesh's tree topology, recompute every box on the device (default; librbrt_gpu_update.so) */
    RBRT_UPDATE_REBUILD = 1    /* full LBVH build of the new vertices into the same slots (the creation's build) */
};
/* New world-space positions for mesh `mesh_index`: num_triangles * 9 floats in the creation's triangle order, num_triangles equal to
 * the count it was created with (the SIMD tail rule, N_eff, the block layout and the triangle order do not change); material NULL =
 * keep.  HOST pointer: returns once it has been read. */
int rbrt_gpu_scene_update_mesh(rbrt_scene* scene, uint32_t mesh_index, const float* tri_vertices, uint64_t num_triangles,
                               const rbrt_material* material, uint32_t flags);
/* The same with a DEVICE pointer on the scene's first device, read in stream order on cuda_stream; cuda_stream then waits for the
 * update, so the caller may overwrite the buffer with work enqueued later on that stream.  Returns without synchronising. */
int rbrt_gpu_scene_update_mesh_device(rbrt_scene* scene, uint32_t mesh_index, const void* d_tri_vertices, uint64_t num_triangles,
                                      const rbrt_material* material, uint32_t flags, void* cuda_stream);
/* New values for Scene.elements: the same count and the same kinds in the same order as at creation (centres, radii, corners and
 * materials may change, material kinds included).  HOST pointers: returns once they have been read. */
int rbrt_gpu_scene_update_elements(rbrt_scene* scene, const rbrt_element_ref* order, uint32_t num_elements,
                                   const rbrt_sphere_desc* spheres, uint32_t num_spheres,
                                   const rbrt_triangle_desc* triangles, uint32_t num_triangles);

/* = render_scene (lib.rs:75-124).  rgb_out: caller-allocated W*H*3 bytes, row-major RGB8 =
 *   the layout of image::ImageBuffer<Rgb<u8>>.  opts / stats may be NULL.  HOST pointers.
 *   Under a communicator (scene created collectively, opts->shard_count == 0) the call is collective: every rank makes
 *   it, the image is sharded over all GPUs (opts->shard_mode: tiles by default, RBRT_SHARD_SAMPLES for sample ranges),
 *   rank 0 receives the image (rgb_out may be NULL on the other ranks); stats are this process's own GPUs'. */
int rbrt_gpu_render(const rbrt_scene* scene, const rbrt_camera* cam, uint32_t num_samples,
                    const rbrt_render_opts* opts, uint8_t* rgb_out, rbrt_stats* stats);

/* Same render, but returns the pre-gamma mean colour (`color * (1.0/spp)`, lib.rs:101) as
 * W*H*3 f32, row-major.  HOST pointer. */
int rbrt_gpu_render_hdr(const rbrt_scene* scene, const rbrt_camera* cam, uint32_t num_samples,
                        const rbrt_render_opts* opts, float* rgb_f32_out, rbrt_stats* stats);

/* Multi-GPU building block: renders this rank's shard and leaves the per-pixel SUM over its
 * samples (lib.rs:95-100, before the 1/spp scale) in a DEVICE buffer of W*H*4 f32 (rgb + pad),
 * zero outside the shard, on the given CUDA stream (0 = default stream).  Ranks then sum these
 * buffers (NCCL reduce) and rank 0 calls rbrt_gpu_finalize_device.
 * With stats == NULL the call only ENQUEUES the frame on cuda_stream and returns (with stats it waits for the frame
 * and fills the counters).  Frames in flight at the same time must use different streams, different accumulation
 * buffers and different wavefront pools (opts->flags, RBRT_OPT_POOL_*); the scene must outlive them. */
int rbrt_gpu_render_accum_device(const rbrt_scene* scene, const rbrt_camera* cam,
                                 uint32_t num_samples, const rbrt_render_opts* opts,
                                 void* d_accum_rgba_f32, void* cuda_stream, rbrt_stats* stats);

/* The same for n_frames (1..4) frames of ONE scene rendered TOGETHER in the same wavefront batches: one camera, one
 * seed (Philox key) and one accumulation buffer per frame, all cameras with the same image size, the same sample count
 * and options for all (opts->seed is ignored).  Each image is bit-identical to what rbrt_gpu_render_accum_device gives
 * for that camera and seed alone; the point is kernel size: a rank's share of a frame on 8 GPUs is small, and two or
 * four frames per batch restore the efficiency the kernels have on larger shards (DESIGN.md section 7). */
int rbrt_gpu_render_accum_device_frames(const rbrt_scene* scene, const rbrt_camera* cams, const uint64_t* seeds,
                                        uint32_t n_frames, uint32_t num_samples, const rbrt_render_opts* opts,
                                        void* const* d_accum_rgba_f32, void* cuda_stream, rbrt_stats* stats);

/* The collective render with DEVICE outputs, enqueue-only when stats == NULL: n_frames (1..RBRT_MAX_FRAMES) frames of one scene
 * (a camera and a seed each) -> per GPU: render its shard, finalise its own pixels -> gather on rank 0 into
 * d_rgb_u8[f] (W*H*3 u8) and / or d_hdr_f32[f] (W*H*3 f32), device pointers on rank 0's GPU (ignored elsewhere; either
 * array may be NULL).  Everything is ordered on cuda_stream (a stream of this process's first device).  Without a
 * communicator this is render + finalise on one GPU.  Frames in flight at the same time use different streams and
 * different pools (opts->flags, RBRT_OPT_POOL_*); every rank must issue its calls in the same order. */
int rbrt_gpu_render_frames_device(const rbrt_scene* scene, const rbrt_camera* cams, const uint64_t* seeds, uint32_t n_frames,
                                  uint32_t num_samples, const rbrt_render_opts* opts, void* const* d_rgb_u8,
                                  void* const* d_hdr_f32, void* cuda_stream, rbrt_stats* stats);

/* = lib.rs:101 + lib.rs:116-122: colour *= 1/spp; (sqrt(c)*256) as u8 (saturating).
 *   d_rgb_u8 (W*H*3) and d_hdr_f32 (W*H*3) are DEVICE pointers; either may be NULL. */
int rbrt_gpu_finalize_device(const void* d_accum_rgba_f32, uint32_t width, uint32_t height,
                             uint32_t num_samples, void* d_rgb_u8, void* d_hdr_f32,
                             void* cuda_stream);

/* Parity hook = Scene::hit (scene.rs:19-43) for caller-supplied rays; the reference's nearest
 * public analogue is do_intersection_soa (mesh.rs:183-190).  HOST pointers.
 * trace_mode: RBRT_TRACE_BVH or RBRT_TRACE_BRUTE (every triangle, the reference's own loop).
 * Refused with RBRT_E_INVALID, nothing written: a scene with a mesh whose tree was refused as too deep (the call waits for the
 * scene's build to know). */
int rbrt_gpu_trace_rays(const rbrt_scene* scene, const rbrt_ray* rays, uint64_t n,
                        uint32_t trace_mode, rbrt_hit* hits_out, rbrt_stats* stats);

/* Parity hook = RayScattering::scatter (materials.rs:4-12; lambertian.rs:11-24, metal.rs:12-25, dielectric.rs:11-60) for
 * caller-supplied hits: item i scatters in_ray at (hit_point, hit_normal) off `material`, drawing from the Philox stream the
 * renderer would use at (seed, pixel, sample, bounce).  out[i].scattered = scatter()'s return value; attenuation and out_ray as
 * the reference leaves them (out_ray.origin = hit_point).  HOST pointers. */
typedef struct rbrt_scatter_in {
    rbrt_material material;
    rbrt_ray      in_ray;
    rbrt_vec3     hit_point, hit_normal;
    uint32_t      pixel, sample, bounce;
} rbrt_scatter_in;
typedef struct rbrt_scatter_out { int32_t scattered; rbrt_vec3 attenuation; rbrt_ray out_ray; } rbrt_scatter_out;
int rbrt_gpu_scatter(const rbrt_scatter_in* items, uint64_t n, uint64_t seed, rbrt_scatter_out* out);

/* Primary rays exactly as the renderer generates them (cam.rs:64-82 with the Philox stream of
 * sample `sample_idx`), one per pixel, row-major.  HOST pointer, W*H rays. */
int rbrt_gpu_primary_rays(const rbrt_camera* cam, uint64_t seed, uint32_t sample_idx,
                          rbrt_ray* rays_out);

/* ---- first-hit AOVs (DESIGN.md section 11) -------------------------------------------------
 * Geometric passes of the render's own camera rays: depth, shading normal, albedo, coverage and the ids of what each pixel sees.
 * For pixel px = row*W + col and samples s = 0 .. num_samples-1 (S = num_samples):
 *   r[px,s] = the camera ray rbrt_gpu_primary_rays(cam, seed, s) returns for px, bit for bit;
 *   h[px,s] = Scene::hit(r), bit for bit what rbrt_gpu_trace_rays reports for that ray with RBRT_TRACE_BVH.
 * A sample hits when h.kind != RBRT_HIT_NONE; a NaN ray, where the reference panics, is a miss and is counted in stats->nan_rays.
 * With n_hit hit samples, every sum below is an f32 sum starting from +0, left to right in sample order over the hit samples only,
 * followed by ONE IEEE division by the float n_hit:
 *   coverage = n_hit / S (both as float);
 *   depth    = sum of h.dist / n_hit, +inf when n_hit = 0;
 *   normal   = sum of n / n_hit per component, 0 when n_hit = 0.  Mesh and BasicTriangle normals as stored (unit); a sphere's normal
 *              p - c is divided per component by its length sqrt((x*x + y*y) + z*z).  No normal is flipped toward the ray, and the
 *              mean is not renormalised;
 *   albedo   = sum of a / n_hit per component, 0 when n_hit = 0: the hit element's material albedo for Lambertian and Metal (a mesh's
 *              material for a mesh hit), (1,1,1) for Dielectric, the attenuation rbrt_gpu_scatter reports;
 *   hit_kind, elem_idx, tri_idx = sample 0's hit as rbrt_hit reports it (RBRT_HIT_NONE, 0, 0 for a miss).
 * The planes are row-major, W*H values (W*H*3 for normal and albedo, xyz per pixel).  A NULL member is not produced and not written. */
typedef struct rbrt_aov_out {
    float*    depth;      /* W*H */
    float*    normal;     /* W*H*3 */
    float*    albedo;     /* W*H*3 */
    float*    coverage;   /* W*H */
    int32_t*  hit_kind;   /* W*H, sample 0: RBRT_HIT_* */
    uint32_t* elem_idx;   /* W*H, sample 0 */
    uint32_t* tri_idx;    /* W*H, sample 0 */
} rbrt_aov_out;
/* HOST pointers; blocks until the passes are on the host.  The kernel lives in librbrt_gpu_aov.so, loaded at run time from this
 * library's directory (RBRT_GPU_AOV_LIB: another path); without it the call fails with RBRT_E_CUDA and a message.
 * Refused with RBRT_E_INVALID, nothing written: a NULL scene, camera or out, every member of out NULL, num_samples = 0, an empty image,
 * a scene with a mesh whose tree was refused as too deep (the call waits for the scene's build to know).
 * Ordered like a render: the call sees every update of the scene enqueued before it, and every later update waits for it.
 * stats may be NULL; it reports rays = W*H*S, nan_rays, node_visits / tri_tests, ms_device, ms_d2h, ms_total and launches.
 * Under a communicator the call is NOT collective: it runs on this process's first device (replica 0) over the whole image;
 * AOVs are not sharded over GPUs. */
int rbrt_gpu_render_aov(const rbrt_scene* scene, const rbrt_camera* cam, uint32_t num_samples, uint64_t seed,
                        const rbrt_aov_out* out, rbrt_stats* stats);
/* The same with DEVICE pointers on the scene's first device, enqueued on cuda_stream (0 = default stream).  stats == NULL: enqueue
 * only, no synchronisation; with stats the call waits for the kernel and fills them. */
int rbrt_gpu_render_aov_device(const rbrt_scene* scene, const rbrt_camera* cam, uint32_t num_samples, uint64_t seed,
                               const rbrt_aov_out* d_out, void* cuda_stream, rbrt_stats* stats);

/* ---- ray queries on device memory (DESIGN.md section 12) -----------------------------------
 * Scene::hit for rays the caller made, with rays and results in device memory, enqueued on the caller's stream.  Let h[i] be what
 * rbrt_gpu_trace_rays(scene, rays, n, RBRT_TRACE_BVH, ...) reports for ray i.
 *   closest:  each requested plane holds, bit for bit, the matching field of h[i] (kind RBRT_HIT_*, the sphere normal un-normalised,
 *             zeros and RBRT_HIT_NONE for a miss).  A NaN ray (a NaN sphere discriminant, where the reference panics) is a miss and
 *             is counted in stats->nan_rays.
 *   occluded: d_occluded[i] = 1 when h[i] is a hit and h[i].dist < max_dist[i] (strict; a NaN max_dist gives 0), 2 when ray i is a NaN
 *             ray whatever else it hits, 0 otherwise.  The traversal may stop at the first triangle that proves it.
 * Rays, bounds and planes are DEVICE memory on the scene's first device.  Both calls are enqueued on cuda_stream (0 = default stream):
 * stats == NULL returns without synchronising; with stats the call waits and fills rays, nan_rays, node_visits, tri_tests, ms_device,
 * ms_total and launches.  Ordered like a render: a call sees every update of the scene enqueued before it, and every later update waits
 * for it.  Under a communicator the call runs on replica 0 and is not collective.  n = 0 returns RBRT_OK, nothing written.
 * The kernels live in librbrt_gpu_query.so, loaded at run time from this library's directory (RBRT_GPU_QUERY_LIB: another path); without
 * it the call fails with RBRT_E_CUDA and a message.
 * Refused with RBRT_E_INVALID, nothing written: a NULL scene, rays or output with n > 0, every plane of the output NULL, n > 2^32 - 1,
 * rays or outputs in another device's memory or in unregistered host memory, a scene with a mesh whose tree was refused as too deep. */
typedef struct rbrt_query_out {      /* device planes, n entries each (point / normal: n*3); NULL = not produced, not written */
    float*    t;
    float*    dist;
    int32_t*  kind;                  /* RBRT_HIT_* */
    uint32_t* elem_idx;
    uint32_t* tri_idx;
    float*    point;
    float*    normal;
} rbrt_query_out;
int rbrt_gpu_query_closest_device(const rbrt_scene* scene, const rbrt_ray* d_rays, uint64_t n,
                                  const rbrt_query_out* d_out, void* cuda_stream, rbrt_stats* stats);
/* d_max_dist: n values, or NULL = +inf for every ray.  d_occluded[i]: one of */
enum { RBRT_QUERY_CLEAR = 0, RBRT_QUERY_OCCLUDED = 1, RBRT_QUERY_NAN_RAY = 2 };
int rbrt_gpu_query_occluded_device(const rbrt_scene* scene, const rbrt_ray* d_rays, uint64_t n,
                                   const float* d_max_dist,
                                   uint8_t* d_occluded, void* cuda_stream, rbrt_stats* stats);

/* ---- guided denoising (DESIGN.md section 13) -----------------------------------------------
 * An edge-aware à-trous filter of the HDR mean colour, guided by the first-hit AOVs of the same camera and seed (the spatial filter of
 * SVGF, Schied et al. 2017, without variance or temporal terms).  Inputs are row-major W x H planes: c = hdr (W*H*3, what
 * rbrt_gpu_render_hdr returns), and from `guides` the depth z (W*H), normal n and albedo a (W*H*3) as rbrt_gpu_render_aov fills them.
 * Every operation below is one IEEE f32 operation, correctly rounded, products and sums left to right as written; rbrt_b200/csrc/denoise.cuh
 * holds the per-pixel code.  Per pixel p:
 *   1. d = max(a, 2^-10) per component (a NaN albedo gives 2^-10); e = c / d; l(e) = (0.2126 e.r + 0.7152 e.g) + 0.0722 e.b.
 *      p is VALID when c, d and z are all finite (not NaN, not +-inf).
 *   2. levels L (default 4), level i = 0 .. L-1 with step s = 2^i, filters the previous level's e (level 0: step 1's).  For a valid p,
 *      over the 5x5 taps q = p + (dx*s, dy*s), dx, dy in -2..2, in row-major order (dy outer, dx inner):
 *        skipped: q outside the image; q not valid; w_n == 0;
 *        centre (dx = dy = 0): w = 9/64;
 *        other:  w_n = max(0, (n_p.x*n_q.x + n_p.y*n_q.y) + n_p.z*n_q.z) ^ 128, by seven squarings (a NaN dot gives 0);
 *                x_z = |z_p - z_q| * r_p,          r_p  = 1 / ((σ_z * z_p) * s),        σ_z = sigma_depth     (default 0.01)
 *                x_l = (l_p - l_q) * r'_p,         r'_p = 1 / (σ_l * l_p + 2^-7),       σ_l = sigma_luminance (default 0.25)
 *                w   = (h[dx]*h[dy] * w_n) / ((1 + x_z*x_z) * (1 + x_l*x_l)),   h = {1/16, 1/4, 3/8, 1/4, 1/16}  (h[dx]*h[dy] exact)
 *      with l_p, l_q the luminances of this level's input.  Σw and Σ w*e_q (per channel) are f32 sums from +0 in tap order; the
 *      output is e' = Σ w*e_q / Σw (one division per channel).  An invalid p keeps its e.
 *   3. hdr_out = e_L * d per channel for a valid p, c unchanged for an invalid one; rgb_out = (sqrt(hdr_out) * 256) as u8, saturating
 *      (NaN -> 0): the tonemap of rbrt_gpu_finalize_device.
 * A miss has depth +inf and normal 0, so it is passed through and never mixes with anything.  The guides line up with the colour when
 * they come from the same camera and seed with at most as many samples (section 11: their samples are the colour's first camera rays). */
typedef struct rbrt_denoise_opts {
    uint32_t levels;           /* à-trous levels, steps 1, 2, 4, ...; 0 = default (4); at most 8 */
    float    sigma_depth;      /* σ_z; 0 = default */
    float    sigma_luminance;  /* σ_l; 0 = default */
} rbrt_denoise_opts;
/* guides: an rbrt_aov_out as rbrt_gpu_render_aov* filled it; depth, normal and albedo are read, the other members are ignored.  opts may
 * be NULL.  Outputs: hdr_out (W*H*3 f32) and / or rgb_out (W*H*3 u8); either may be NULL, not both.
 * The calls run on this process's current render device (rbrt_gpu_init; under a communicator its first device) and are not collective.
 * The kernels live in librbrt_gpu_denoise.so, loaded at run time from this library's directory (RBRT_GPU_DENOISE_LIB: another path);
 * without it the call fails with RBRT_E_CUDA and a message.
 * Refused with RBRT_E_INVALID, nothing written: a NULL hdr, guides, guide depth, normal or albedo; both outputs NULL; W or H = 0 or
 * W*H > 2^31 - 1 (as rbrt_gpu_render_hdr); levels > 8; a negative, NaN or infinite sigma; an output that overlaps an input or the
 * other output.
 * stats may be NULL; it reports ms_device, ms_total and launches (1 + levels). */
/* HOST pointers; blocks until the outputs are on the host. */
int rbrt_gpu_denoise(uint32_t width, uint32_t height, const float* hdr, const rbrt_aov_out* guides, const rbrt_denoise_opts* opts,
                     float* hdr_out, uint8_t* rgb_out, rbrt_stats* stats);
/* DEVICE pointers on the current render device, enqueued on cuda_stream (0 = default stream); the scratch (48 bytes per pixel) is
 * allocated and freed in stream order on that stream, so calls in flight on different streams never share it.  stats == NULL: enqueue
 * only, no synchronisation; with stats the call waits for its kernels and fills them.  Also refused: inputs or outputs in another
 * device's memory or in unregistered host memory. */
int rbrt_gpu_denoise_device(uint32_t width, uint32_t height, const float* d_hdr, const rbrt_aov_out* d_guides, const rbrt_denoise_opts* opts,
                            float* d_hdr_out, uint8_t* d_rgb_out, void* cuda_stream, rbrt_stats* stats);

/* ---- per-pixel variance and variance-guided denoising (DESIGN.md section 14) ------------------
 * VARIANCE OF A RENDER.  S = num_samples, K = splits, n = S / K.  The call renders shard k = 0 .. K-1 as rbrt_gpu_render_accum_device
 * does with shard_mode = RBRT_SHARD_SAMPLES, shard_rank = k, shard_count = K: samples [k*n, (k+1)*n) of the frame's Philox stream into
 * a per-pixel sum A_k.  K shards of one seed are K independent estimates of each pixel's mean.  Per pixel and channel, in f32, each
 * operation correctly rounded, sums from +0 in shard order (rbrt_b200/csrc/variance.cuh holds the code):
 *   hdr_out = (((A_0 + A_1) + A_2) + ... + A_{K-1}) * (1.0f / (float)S)
 *             — the arithmetic of the PEER sample-sharded rbrt_gpu_render_hdr on K ranks (rank order sum, then the finalise), and the
 *             same bits; within 1e-5 relative of the unsharded rbrt_gpu_render_hdr, whose per-pixel sum runs over the samples in one chain;
 *   m_k     = A_k * (1.0f / (float)n);
 *   var_out = (Σ_k (m_k - hdr_out) * (m_k - hdr_out)) / (float)(K * (K - 1))
 *             — the unbiased variance of the mean hdr_out (the K-buffer estimate: its expectation is the pixel's sample variance / S).
 * Outputs W*H*3 f32 each, row-major; either may be NULL, not both.  opts as a render (seed, max_depth, trace_mode, batch_paths, pool).
 * Refused with RBRT_E_INVALID, nothing written: splits < 2 or > 16; num_samples = 0 or not a multiple of splits; opts->shard_count > 1
 * (the call shards by itself); a NULL scene or camera; both outputs NULL; an empty image or W*H > 2^31 - 1; the outputs overlapping;
 * a scene with a mesh whose tree was refused as too deep (the call waits for the scene's build to know); opts a render refuses.
 * Ordered against scene updates like a render.  Under a communicator the call is not collective: it runs on this process's first
 * device (replica 0).  The shards alternate between two lanes: the calling stream with the wavefront pool of opts->flags (p), and an
 * internal stream of the device with pool 4 + p (the second lane of RBRT_OPT_SPLIT_BATCHES, which the call does not use otherwise);
 * calls in flight at the same time use different pools.  The K accumulators (16 bytes per pixel each) are allocated and freed in stream
 * order on the calling stream.  The kernel that forms the moments lives in librbrt_gpu_variance.so (RBRT_GPU_VARIANCE_LIB: another path).
 * stats may be NULL; it reports rays, paths and nan_rays summed over the shards, ms_device (all shards and the moments), ms_total and
 * launches; with stats the call also waits after each pair of shards to read their counters. */
/* HOST pointers; blocks until the outputs are on the host. */
int rbrt_gpu_render_hdr_variance(const rbrt_scene* scene, const rbrt_camera* cam, uint32_t num_samples, uint32_t splits,
                                 const rbrt_render_opts* opts, float* hdr_out, float* var_out, rbrt_stats* stats);
/* DEVICE pointers on the scene's first device, enqueued on cuda_stream (0 = default stream); stats == NULL: enqueue only, no
 * synchronisation.  Also refused: outputs in another device's memory or in unregistered host memory. */
int rbrt_gpu_render_hdr_variance_device(const rbrt_scene* scene, const rbrt_camera* cam, uint32_t num_samples, uint32_t splits,
                                        const rbrt_render_opts* opts, float* d_hdr_out, float* d_var_out, void* cuda_stream,
                                        rbrt_stats* stats);

/* VARIANCE-GUIDED FILTER: rbrt_gpu_denoise with the variance of the colour steering the luminance term (the spatial filter of SVGF with
 * its variance estimate and propagation, Schied et al. 2017, without temporal terms).  Inputs as rbrt_gpu_denoise, plus var (W*H*3, as
 * var_out above).  rbrt_denoise_opts is read with this filter's defaults: levels 5, σ_z = 0.01, σ_l = 4.  Per pixel p, each operation one
 * correctly rounded f32 operation, products and sums left to right as written:
 *   1. d, e, l and validity as rbrt_gpu_denoise step 1; p is also INVALID when a component of var is NaN, +-inf or negative (-0 is not).
 *      σ² = sd * sd with sd = ((0.2126 / d.r) * sqrt(v.r) + (0.7152 / d.g) * sqrt(v.g)) + (0.0722 / d.b) * sqrt(v.b).  This adds the
 *      channels' standard deviations: an upper bound of the deviation of l(e) (Cauchy-Schwarz), exact for fully correlated channels, as
 *      path-tracing noise mostly is.  Per-channel variances cannot give the covariances that the exact value needs.
 *   2. levels L, level i = 0 .. L-1 with step s = 2^i, filters the previous level's e and σ² (level 0: step 1's).  For a valid p:
 *        g_p  = (Σ k[dx]*k[dy] * σ²_q) / (Σ k[dx]*k[dy]) over the 3x3 neighbours q = p + (dx, dy), dx, dy in -1..1, inside the image and
 *               valid, row-major, sums from +0, k = {1/4, 1/2, 1/4} (products exact);
 *        r'_p = 1 / (σ_l * sqrt(g_p) + 2^-10);  x_l = (l_p - l_q) * r'_p;
 *        taps, skips, w_n, x_z, r_p and the centre weight 9/64 as rbrt_gpu_denoise step 2, and for a tap other than the centre
 *        w    = (h[dx]*h[dy] * w_n) / ((1 + x_z*x_z) * ((1 + x_l*x_l) * (1 + x_l*x_l)));
 *        e'   = Σ w*e_q / Σw per channel;  σ²' = (Σ (w*w) * σ²_q) / (Σw * Σw), sums from +0 in tap order.
 *      An invalid p keeps its e and σ².
 *   3. hdr_out and rgb_out as rbrt_gpu_denoise step 3.
 * A pixel whose variance is 0 (a converged or constant region) takes no tap whose luminance differs: a well-sampled frame is not blurred.
 * Refusals, devices, stats and the scratch's stream-ordered allocation as rbrt_gpu_denoise*, plus a NULL var and an output that overlaps
 * var; the scratch is 56 bytes per pixel.  The kernels live in librbrt_gpu_variance.so (RBRT_GPU_VARIANCE_LIB: another path). */
/* HOST pointers; blocks until the outputs are on the host. */
int rbrt_gpu_denoise_variance(uint32_t width, uint32_t height, const float* hdr, const float* var, const rbrt_aov_out* guides,
                              const rbrt_denoise_opts* opts, float* hdr_out, uint8_t* rgb_out, rbrt_stats* stats);
/* DEVICE pointers on the current render device, enqueued on cuda_stream; stats == NULL: enqueue only. */
int rbrt_gpu_denoise_variance_device(uint32_t width, uint32_t height, const float* d_hdr, const float* d_var, const rbrt_aov_out* d_guides,
                                     const rbrt_denoise_opts* opts, float* d_hdr_out, uint8_t* d_rgb_out, void* cuda_stream,
                                     rbrt_stats* stats);

/* The wavefront state (ray / hit / queue buffers, tens of GB at full batch size) is pooled per device and kept
 * between renders and across scenes; this releases it (and the pooled scene blocks, the build scratch, the query counters, the
 * denoiser's host-call block and the variance call's internal stream). */
int rbrt_gpu_release_cache(void);

/* Upper bound, in bytes, of ONE pool of wavefront state (there are up to four per device, one per frame in flight).
 * 0 = default: as many paths as fit, <= 2^27 paths (24.7 GB at depth 50) and <= half of the free HBM.  A host that
 * embeds the library next to other users of the GPU sets this; smaller pools mean more, smaller wavefront batches. */
int rbrt_gpu_set_pool_limit(uint64_t max_bytes_per_pool);

/* Threading: every entry point may be called from any thread; calls are serialised by one process-wide lock (the
 * library keeps per-device pools).  Calls that only ENQUEUE work (stats == NULL) hold it for microseconds. */

/* Thread-local message of the last failing call on this thread. */
const char* rbrt_last_error(void);

/* Library identification: "rbrt_b200 <version> sm_100a". */
const char* rbrt_gpu_version(void);

#ifdef __cplusplus
}
#endif
#endif /* RBRT_GPU_H */
