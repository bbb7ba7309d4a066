//! Raw bindings of include/rbrt_gpu.h (SOURCE ONLY, uncompiled: see Cargo.toml) plus the safe twins of
//! `create_scene_from_scene_blueprint` (rbrt_lib/src/blueprints.rs:132) and `render_scene` (rbrt_lib/src/lib.rs:75)
//! that `rbrt_lib` would re-export.  Struct layouts are `#[repr(C)]` mirrors of the header; `RbrtCamera` has the field
//! order of `rbrt_lib::cam::Camera` (cam.rs:4-19).
use std::ffi::CStr;
use std::os::raw::{c_char, c_int, c_void};

#[repr(C)] #[derive(Copy, Clone, Debug, Default)] pub struct RbrtVec3 { pub x: f32, pub y: f32, pub z: f32 }
#[repr(C)] #[derive(Copy, Clone, Debug)] pub struct RbrtRay { pub origin: RbrtVec3, pub direction: RbrtVec3 }
#[repr(C)] #[derive(Copy, Clone, Debug)]
pub struct RbrtCamera {
    pub hor_fov_rad: f32, pub img_width_pix: u32, pub img_height_mm: f32, pub vert_fov_rad: f32,
    pub img_height_pix: u32, pub img_width_mm: f32, pub position: RbrtVec3, pub focal_len_mm: f32,
    pub look_at: RbrtVec3, pub up: RbrtVec3, pub right: RbrtVec3, pub img_center_point: RbrtVec3,
    pub mm_per_pix_hor: f32, pub mm_per_pix_vert: f32,
}
pub const RBRT_MAT_LAMBERTIAN: u32 = 0;
pub const RBRT_MAT_METAL: u32 = 1;
pub const RBRT_MAT_DIELECTRIC: u32 = 2;
#[repr(C)] #[derive(Copy, Clone, Debug)] pub struct RbrtMaterial { pub kind: u32, pub albedo: RbrtVec3, pub param: f32 }
#[repr(C)] #[derive(Copy, Clone, Debug)] pub struct RbrtSphereDesc { pub center: RbrtVec3, pub radius: f32, pub material: RbrtMaterial }
#[repr(C)] #[derive(Copy, Clone, Debug)] pub struct RbrtTriangleDesc { pub corners: [RbrtVec3; 3], pub material: RbrtMaterial }
#[repr(C)] #[derive(Copy, Clone, Debug)] pub struct RbrtElementRef { pub kind: u32, pub index: u32 }   // 0 sphere, 1 BasicTriangle
/// A triangle soup, 9 f32 per triangle.  Any coordinate value is accepted (inf and NaN too) and hits stay exact; the BVH culls on an
/// axis only while the padded extent there is at most about 1.3e11 (grid step 2e6), beyond that the axis is not culled (slower).
#[repr(C)] #[derive(Copy, Clone, Debug)] pub struct RbrtMeshDesc { pub tri_vertices: *const f32, pub num_triangles: u64, pub material: RbrtMaterial }
#[repr(C)] #[derive(Copy, Clone, Debug, Default)]
pub struct RbrtRenderOpts { pub seed: u64, pub max_depth: u32, pub trace_mode: u32, pub shard_mode: u32, pub shard_rank: u32,
                            pub shard_count: u32, pub batch_paths: u32, pub integrator: u32, pub flags: u32 }
#[repr(C)] #[derive(Copy, Clone, Debug, Default)]
pub struct RbrtStats { pub rays: u64, pub paths: u64, pub nan_rays: u64, pub node_visits: u64, pub tri_tests: u64, pub ms_total: f64,
                       pub ms_device: f64, pub ms_trace: f64, pub ms_h2d: f64, pub ms_d2h: f64, pub launches: u32, pub iterations: u32,
                       pub traversed_rays: u64, pub tail_node_visits: u64, pub tail_tri_tests: u64, pub tail_traversed_rays: u64 }
#[repr(C)] #[derive(Copy, Clone, Debug, Default)]
pub struct RbrtSceneOpts { pub simd_lanes: u32, pub leaf_size: u32, pub box_pad_rel: f32, pub flags: u32 }
#[repr(C)] #[derive(Copy, Clone, Debug, Default)]
pub struct RbrtCommInfo { pub active: i32, pub world: i32, pub rank: i32, pub local_devices: i32, pub transport: i32, pub nccl_version: i32,
                          pub devices: [i32; 16] }
/// First-hit AOV planes (row-major, W*H values; W*H*3 for normal and albedo); a null member is not produced.
#[repr(C)] #[derive(Copy, Clone, Debug)]
pub struct RbrtAovOut { pub depth: *mut f32, pub normal: *mut f32, pub albedo: *mut f32, pub coverage: *mut f32, pub hit_kind: *mut i32,
                        pub elem_idx: *mut u32, pub tri_idx: *mut u32 }
/// Ray-query planes in device memory (n values each; n*3 for point and normal); a null member is not produced.
#[repr(C)] #[derive(Copy, Clone, Debug)]
pub struct RbrtQueryOut { pub t: *mut f32, pub dist: *mut f32, pub kind: *mut i32, pub elem_idx: *mut u32, pub tri_idx: *mut u32,
                          pub point: *mut f32, pub normal: *mut f32 }
/// Nearest-surface planes in device memory (n values each; n*3 for point and normal, n*2 for uv); a null member is not produced.
#[repr(C)] #[derive(Copy, Clone, Debug)]
pub struct RbrtNearestOut { pub dist: *mut f32, pub kind: *mut i32, pub elem_idx: *mut u32, pub tri_idx: *mut u32, pub point: *mut f32,
                            pub normal: *mut f32, pub uv: *mut f32 }
/// Options of the winding-number query (rbrt_gpu_query_winding_device): beta 0 = the default 2.0, +inf = the exact sum, else > 1.
#[repr(C)] #[derive(Copy, Clone, Debug, Default)]
pub struct RbrtWindingOpts { pub beta: f32 }
/// Winding-number planes in device memory (n values each); a null member is not produced.
#[repr(C)] #[derive(Copy, Clone, Debug)]
pub struct RbrtWindingOut { pub winding: *mut f32, pub inside: *mut u8 }
/// Options of the guided denoiser (rbrt_gpu_denoise*); 0 = default (4 levels, at most 8).
#[repr(C)] #[derive(Copy, Clone, Debug, Default)]
pub struct RbrtDenoiseOpts { pub levels: u32, pub sigma_depth: f32, pub sigma_luminance: f32 }
/// Options of the temporal accumulation, every member used as given (a null pointer gives 0.1, 0.02, 0.9).
#[repr(C)] #[derive(Copy, Clone, Debug)]
pub struct RbrtTemporalOpts { pub alpha_min: f32, pub sigma_depth: f32, pub normal_min: f32 }
/// The previous temporal call's outputs (hdr, var, length), aligned to `cam`, and that frame's guides.
#[repr(C)] #[derive(Copy, Clone, Debug)]
pub struct RbrtTemporalHistory { pub cam: RbrtCamera, pub hdr: *const f32, pub var: *const f32, pub length: *const f32, pub guides: RbrtAovOut }
/// Planes of the motion pass (rbrt_gpu_render_motion*): motion W*H*2 (x, y per pixel), prev_dist W*H; a null member is not produced.
#[repr(C)] #[derive(Copy, Clone, Debug)]
pub struct RbrtMotionOut { pub motion: *mut f32, pub prev_dist: *mut f32 }
pub enum RbrtScene {}
/// `kind` of a hit (rbrt_hit, rbrt_query_out)
pub const RBRT_HIT_NONE: i32 = -1;
pub const RBRT_HIT_SPHERE: i32 = 0;
pub const RBRT_HIT_MESH: i32 = 1;
pub const RBRT_HIT_TRIANGLE: i32 = 2;
/// values of rbrt_gpu_query_occluded_device's output
pub const RBRT_QUERY_CLEAR: u8 = 0;
pub const RBRT_QUERY_OCCLUDED: u8 = 1;
pub const RBRT_QUERY_NAN_RAY: u8 = 2;
pub const RBRT_MAX_FRAMES: u32 = 4;
pub const RBRT_COMM_ID_BYTES: usize = 128;
pub const RBRT_TRANSPORT_AUTO: c_int = 0;
pub const RBRT_TRANSPORT_NCCL: c_int = 1;
pub const RBRT_TRANSPORT_PEER: c_int = 2;
pub const RBRT_SCENE_LOCAL: u32 = 1;
pub const RBRT_SCENE_NO_SAH: u32 = 2;
pub const RBRT_UPDATE_REFIT: u32 = 0;
pub const RBRT_UPDATE_REBUILD: u32 = 1;
pub const RBRT_SCENE_BROADCAST: u32 = 4;
pub const RBRT_OPT_COUNT_VISITS: u32 = 1;
pub const RBRT_OPT_TIME_KERNELS: u32 = 2;
pub const RBRT_OPT_NO_TAIL_KERNEL: u32 = 4;
pub const RBRT_OPT_POOL_SHIFT: u32 = 3;    // flags |= slot << RBRT_OPT_POOL_SHIFT, slot in 0..4: the wavefront pool of a frame in flight
pub const RBRT_OPT_POOL_MASK: u32 = 24;
pub const RBRT_OPT_SPLIT_BATCHES: u32 = 32;

extern "C" {
    pub fn rbrt_camera_new(position: RbrtVec3, look_at: RbrtVec3, up: RbrtVec3, img_height_pix: u32, img_width_pix: u32,
                           focal_len_mm: f32, out: *mut RbrtCamera) -> c_int;
    pub fn rbrt_transform_vertices(xyz: *mut f32, n_vertices: u64, scale: f32, rotation_rad: RbrtVec3, translation: RbrtVec3) -> c_int;
    /// = load_mesh_vertices_from_file (mesh.rs:78-121): .obj -> transformed triangle soup (num_triangles x 9 f32, malloc'ed; rbrt_mesh_free).
    pub fn rbrt_mesh_load_obj(filepath: *const c_char, translation: RbrtVec3, rotation_rad: RbrtVec3, scale: f32,
                              tri_vertices_out: *mut *mut f32, num_triangles_out: *mut u64) -> c_int;
    pub fn rbrt_mesh_free(tri_vertices: *mut f32);
    pub fn rbrt_gpu_init(device: c_int) -> c_int;
    /// Multi-GPU inside the library: one process driving n GPUs (devices = null: 0..n-1) ...
    pub fn rbrt_gpu_init_multi(devices: *const c_int, n_devices: c_int, transport: c_int) -> c_int;
    /// ... or one process per GPU: rank 0 makes the id, every rank joins (the id travels over any side channel, e.g. MPI or a file).
    pub fn rbrt_gpu_comm_unique_id(id_out: *mut u8) -> c_int;
    pub fn rbrt_gpu_comm_init_rank(id: *const u8, rank: c_int, world: c_int) -> c_int;
    pub fn rbrt_gpu_comm_info(out: *mut RbrtCommInfo) -> c_int;
    pub fn rbrt_gpu_comm_destroy() -> c_int;
    pub fn rbrt_gpu_set_pool_limit(max_bytes_per_pool: u64) -> c_int;
    pub fn rbrt_gpu_scene_create(spheres: *const RbrtSphereDesc, num_spheres: u32, meshes: *const RbrtMeshDesc, num_meshes: u32,
                                 opts: *const c_void, out: *mut *mut RbrtScene) -> c_int;
    pub fn rbrt_gpu_scene_create_elements(order: *const RbrtElementRef, num_elements: u32, spheres: *const RbrtSphereDesc, num_spheres: u32,
                                          triangles: *const RbrtTriangleDesc, num_triangles: u32, meshes: *const RbrtMeshDesc, num_meshes: u32,
                                          opts: *const c_void, out: *mut *mut RbrtScene) -> c_int;
    pub fn rbrt_gpu_scene_destroy(scene: *mut RbrtScene) -> c_int;
    /// Animation: new vertices for one mesh (same triangle count; the tree is refit, or rebuilt with RBRT_UPDATE_REBUILD), from host
    /// memory or from device memory read in order on `stream`, and new values for Scene.elements (same count and kinds).  Ordered
    /// after every render already enqueued against the scene and before every one enqueued afterwards.
    pub fn rbrt_gpu_scene_update_mesh(scene: *mut RbrtScene, mesh_index: u32, tri_vertices: *const f32, num_triangles: u64,
                                      material: *const RbrtMaterial, flags: u32) -> c_int;
    pub fn rbrt_gpu_scene_update_mesh_device(scene: *mut RbrtScene, mesh_index: u32, d_tri_vertices: *const c_void, num_triangles: u64,
                                             material: *const RbrtMaterial, flags: u32, stream: *mut c_void) -> c_int;
    pub fn rbrt_gpu_scene_update_elements(scene: *mut RbrtScene, order: *const RbrtElementRef, num_elements: u32,
                                          spheres: *const RbrtSphereDesc, num_spheres: u32, triangles: *const RbrtTriangleDesc,
                                          num_triangles: u32) -> c_int;
    pub fn rbrt_gpu_render(scene: *const RbrtScene, cam: *const RbrtCamera, num_samples: u32, opts: *const RbrtRenderOpts,
                           rgb_out: *mut u8, stats: *mut RbrtStats) -> c_int;
    pub fn rbrt_gpu_render_hdr(scene: *const RbrtScene, cam: *const RbrtCamera, num_samples: u32, opts: *const RbrtRenderOpts,
                               rgb_f32_out: *mut f32, stats: *mut RbrtStats) -> c_int;
    /// Multi-GPU / pipelining building blocks: render into a device accumulation buffer on `stream` (stats = null: enqueue only),
    /// then 1/spp, sqrt, x256, saturating u8 on the device.  `opts.flags` bits 3-4 (RBRT_OPT_POOL_*) pick one of four wavefront pools.
    pub fn rbrt_gpu_render_accum_device(scene: *const RbrtScene, cam: *const RbrtCamera, num_samples: u32, opts: *const RbrtRenderOpts,
                                        d_accum: *mut c_void, stream: *mut c_void, stats: *mut RbrtStats) -> c_int;
    /// The same for up to four frames of one scene rendered together in the same wavefront batches (one camera, seed and
    /// accumulation buffer per frame; opts.seed is ignored).
    pub fn rbrt_gpu_render_accum_device_frames(scene: *const RbrtScene, cams: *const RbrtCamera, seeds: *const u64, n_frames: u32,
                                               num_samples: u32, opts: *const RbrtRenderOpts, d_accum: *const *mut c_void,
                                               stream: *mut c_void, stats: *mut RbrtStats) -> c_int;
    /// The collective render with device outputs on rank 0 (shard render -> per-GPU finalise -> gather), enqueue-only when stats = null.
    pub fn rbrt_gpu_render_frames_device(scene: *const RbrtScene, cams: *const RbrtCamera, seeds: *const u64, n_frames: u32, num_samples: u32,
                                         opts: *const RbrtRenderOpts, d_rgb_u8: *const *mut c_void, d_hdr_f32: *const *mut c_void,
                                         stream: *mut c_void, stats: *mut RbrtStats) -> c_int;
    pub fn rbrt_gpu_finalize_device(d_accum: *const c_void, width: u32, height: u32, num_samples: u32, d_rgb: *mut c_void,
                                    d_hdr: *mut c_void, stream: *mut c_void) -> c_int;
    /// First-hit AOVs of the render's camera rays (depth, normal, albedo, coverage, sample 0's ids), host planes; the device variant
    /// takes device planes and enqueues on `stream` (stats = null: no synchronisation).  Not collective: replica 0, whole image.
    pub fn rbrt_gpu_render_aov(scene: *const RbrtScene, cam: *const RbrtCamera, num_samples: u32, seed: u64, out: *const RbrtAovOut,
                               stats: *mut RbrtStats) -> c_int;
    pub fn rbrt_gpu_render_aov_device(scene: *const RbrtScene, cam: *const RbrtCamera, num_samples: u32, seed: u64, d_out: *const RbrtAovOut,
                                      stream: *mut c_void, stats: *mut RbrtStats) -> c_int;
    /// Scene::hit for rays in device memory, each requested plane bit for bit the field rbrt_gpu_trace_rays reports; enqueued on `stream`
    /// (stats = null: no synchronisation).  Not collective: replica 0.
    pub fn rbrt_gpu_query_closest_device(scene: *const RbrtScene, d_rays: *const RbrtRay, n: u64, d_out: *const RbrtQueryOut,
                                         stream: *mut c_void, stats: *mut RbrtStats) -> c_int;
    /// Occlusion for rays in device memory: RBRT_QUERY_OCCLUDED where Scene::hit is a hit with dist < max_dist (null = +inf),
    /// RBRT_QUERY_NAN_RAY for a NaN ray, else RBRT_QUERY_CLEAR.
    pub fn rbrt_gpu_query_occluded_device(scene: *const RbrtScene, d_rays: *const RbrtRay, n: u64, d_max_dist: *const f32,
                                          d_occluded: *mut u8, stream: *mut c_void, stats: *mut RbrtStats) -> c_int;
    /// The nearest surface of the scene to each point (n points, f32 xyz, in device memory): the least (d2, scene order) over every
    /// element and every tested mesh triangle closer than d_max_dist (null = +inf, strict); enqueued on `stream` (stats = null: no
    /// synchronisation).  Not collective: replica 0.
    pub fn rbrt_gpu_query_nearest_device(scene: *const RbrtScene, d_points: *const f32, n: u64, d_max_dist: *const f32,
                                         d_out: *const RbrtNearestOut, stream: *mut c_void, stats: *mut RbrtStats) -> c_int;
    /// The generalized winding number of the scene at each point (n points, f32 xyz, in device memory) over the nearest query's
    /// candidates, and inside = |w| > 0.5; far subtrees by their moments unless opts.beta = +inf (opts may be null: beta 2);
    /// enqueued on `stream` (stats = null: no synchronisation).  Not collective: replica 0.
    pub fn rbrt_gpu_query_winding_device(scene: *const RbrtScene, d_points: *const f32, n: u64, opts: *const RbrtWindingOpts,
                                         d_out: *const RbrtWindingOut, stream: *mut c_void, stats: *mut RbrtStats) -> c_int;
    /// Edge-aware à-trous denoise of a render_hdr image guided by render_aov depth / normal / albedo of the same camera and seed; HOST
    /// pointers, blocks.  hdr_out (W*H*3 f32) and / or rgb_out (W*H*3 u8, k_finalize's tonemap); opts may be null.
    pub fn rbrt_gpu_denoise(width: u32, height: u32, hdr: *const f32, guides: *const RbrtAovOut, opts: *const RbrtDenoiseOpts,
                            hdr_out: *mut f32, rgb_out: *mut u8, stats: *mut RbrtStats) -> c_int;
    /// The same on DEVICE planes of the current render device, enqueued on `stream` (stats = null: no synchronisation).
    pub fn rbrt_gpu_denoise_device(width: u32, height: u32, d_hdr: *const f32, d_guides: *const RbrtAovOut, opts: *const RbrtDenoiseOpts,
                                   d_hdr_out: *mut f32, d_rgb_out: *mut u8, stream: *mut c_void, stats: *mut RbrtStats) -> c_int;
    /// The mean colour of num_samples samples rendered as `splits` (2..16) sample-range shards, and the unbiased variance of that mean
    /// per pixel and channel (W*H*3 f32 each, either may be null); HOST pointers, blocks.
    pub fn rbrt_gpu_render_hdr_variance(scene: *const RbrtScene, cam: *const RbrtCamera, num_samples: u32, splits: u32,
                                        opts: *const RbrtRenderOpts, hdr_out: *mut f32, var_out: *mut f32, stats: *mut RbrtStats) -> c_int;
    /// The same into DEVICE buffers, enqueued on `stream` (stats = null: no synchronisation).
    pub fn rbrt_gpu_render_hdr_variance_device(scene: *const RbrtScene, cam: *const RbrtCamera, num_samples: u32, splits: u32,
                                               opts: *const RbrtRenderOpts, d_hdr_out: *mut f32, d_var_out: *mut f32, stream: *mut c_void,
                                               stats: *mut RbrtStats) -> c_int;
    /// Variance-guided à-trous denoise of a render_hdr_variance frame and its variance, guided by render_aov depth / normal / albedo of
    /// the same camera and seed; HOST pointers, blocks.  opts may be null (5 levels).
    pub fn rbrt_gpu_denoise_variance(width: u32, height: u32, hdr: *const f32, var: *const f32, guides: *const RbrtAovOut,
                                     opts: *const RbrtDenoiseOpts, hdr_out: *mut f32, rgb_out: *mut u8, stats: *mut RbrtStats) -> c_int;
    /// The same on DEVICE planes of the current render device, enqueued on `stream` (stats = null: no synchronisation).
    pub fn rbrt_gpu_denoise_variance_device(width: u32, height: u32, d_hdr: *const f32, d_var: *const f32, d_guides: *const RbrtAovOut,
                                            opts: *const RbrtDenoiseOpts, d_hdr_out: *mut f32, d_rgb_out: *mut u8, stream: *mut c_void,
                                            stats: *mut RbrtStats) -> c_int;
    /// Temporal accumulation: the frame hdr (and its variance var, may be null) at camera `cam`, guided by render_aov depth / normal /
    /// hit_kind / elem_idx of the same camera and seed, blended with the history reprojected from its camera (null: the first frame).
    /// hdr_out, var_out (W*H*3) and len_out (W*H), any may be null, not all, none overlapping an input; HOST pointers, blocks.
    pub fn rbrt_gpu_temporal_accumulate(width: u32, height: u32, cam: *const RbrtCamera, hdr: *const f32, var: *const f32,
                                        guides: *const RbrtAovOut, history: *const RbrtTemporalHistory, opts: *const RbrtTemporalOpts,
                                        hdr_out: *mut f32, var_out: *mut f32, len_out: *mut f32, stats: *mut RbrtStats) -> c_int;
    /// The same on DEVICE planes of the current render device, enqueued on `stream` (stats = null: no synchronisation).
    pub fn rbrt_gpu_temporal_accumulate_device(width: u32, height: u32, cam: *const RbrtCamera, d_hdr: *const f32, d_var: *const f32,
                                               d_guides: *const RbrtAovOut, d_history: *const RbrtTemporalHistory,
                                               opts: *const RbrtTemporalOpts, d_hdr_out: *mut f32, d_var_out: *mut f32,
                                               d_len_out: *mut f32, stream: *mut c_void, stats: *mut RbrtStats) -> c_int;
    /// Records the scene's geometry as "the previous frame" for the motion pass; enqueued on `stream`.
    pub fn rbrt_gpu_scene_snapshot(scene: *mut RbrtScene, stream: *mut c_void) -> c_int;
    /// Per-pixel screen motion from `cam` back to `prev_cam` along the geometry's change since the latest snapshot, and the distance
    /// from prev_cam's position to the previous point; HOST pointers, blocks.
    pub fn rbrt_gpu_render_motion(scene: *const RbrtScene, cam: *const RbrtCamera, prev_cam: *const RbrtCamera, out: *const RbrtMotionOut,
                                  stats: *mut RbrtStats) -> c_int;
    /// The same on DEVICE planes of the scene's first device, enqueued on `stream` (stats = null: no synchronisation).
    pub fn rbrt_gpu_render_motion_device(scene: *const RbrtScene, cam: *const RbrtCamera, prev_cam: *const RbrtCamera,
                                         d_out: *const RbrtMotionOut, stream: *mut c_void, stats: *mut RbrtStats) -> c_int;
    /// rbrt_gpu_temporal_accumulate reprojecting along the frame's motion pass where it is finite; HOST pointers, blocks.
    pub fn rbrt_gpu_temporal_accumulate_motion(width: u32, height: u32, cam: *const RbrtCamera, hdr: *const f32, var: *const f32,
                                               guides: *const RbrtAovOut, history: *const RbrtTemporalHistory, motion: *const RbrtMotionOut,
                                               opts: *const RbrtTemporalOpts, hdr_out: *mut f32, var_out: *mut f32, len_out: *mut f32,
                                               stats: *mut RbrtStats) -> c_int;
    /// The same on DEVICE planes of the current render device, enqueued on `stream` (stats = null: no synchronisation).
    pub fn rbrt_gpu_temporal_accumulate_motion_device(width: u32, height: u32, cam: *const RbrtCamera, d_hdr: *const f32, d_var: *const f32,
                                                      d_guides: *const RbrtAovOut, d_history: *const RbrtTemporalHistory,
                                                      d_motion: *const RbrtMotionOut, opts: *const RbrtTemporalOpts, d_hdr_out: *mut f32,
                                                      d_var_out: *mut f32, d_len_out: *mut f32, stream: *mut c_void,
                                                      stats: *mut RbrtStats) -> c_int;
    pub fn rbrt_gpu_release_cache() -> c_int;
    pub fn rbrt_last_error() -> *const c_char;
    pub fn rbrt_gpu_version() -> *const c_char;
}

/// Keeps the reference's convention: errors are panics (blueprints.rs:80,87, main.rs:86-91).
pub fn check(rc: c_int) {
    if rc != 0 {
        let msg = unsafe { CStr::from_ptr(rbrt_last_error()) }.to_string_lossy().into_owned();
        panic!("rbrt_gpu error {}: {}", rc, msg);
    }
}

/// Owning handle of a GPU scene (flattened SoA buffers + one BVH per mesh).
pub struct GpuScene(*mut RbrtScene);
// Sound since library version 0.2: every entry point takes one process-wide lock (the per-device pools behind the handle are
// shared), so a handle may be created, used and dropped on any thread.  It is NOT Sync-free state: concurrent renders serialise.
unsafe impl Send for GpuScene {}
impl Drop for GpuScene { fn drop(&mut self) { unsafe { rbrt_gpu_scene_destroy(self.0); } } }

impl GpuScene {
    /// `meshes`: world-space triangle soup, 9 f32 per triangle, already scale -> rotate_point -> translate'd (mesh.rs:102-112).
    pub fn new(spheres: &[RbrtSphereDesc], meshes: &[(&[f32], RbrtMaterial)]) -> GpuScene {
        let descs: Vec<RbrtMeshDesc> = meshes.iter()
            .map(|(t, m)| RbrtMeshDesc { tri_vertices: t.as_ptr(), num_triangles: (t.len() / 9) as u64, material: *m }).collect();
        let mut h: *mut RbrtScene = std::ptr::null_mut();
        check(unsafe { rbrt_gpu_scene_create(spheres.as_ptr(), spheres.len() as u32, descs.as_ptr(), descs.len() as u32, std::ptr::null(), &mut h) });
        GpuScene(h)
    }

    /// All GPUs of the box behind the same call: `GpuScene::init_all_gpus(8)` once, BEFORE creating scenes; `render` is then
    /// sharded over them inside the library (the reference spreads render_scene over all cores with rayon, lib.rs:84-86).
    pub fn init_all_gpus(n: i32) { check(unsafe { rbrt_gpu_init_multi(std::ptr::null(), n, RBRT_TRANSPORT_AUTO) }); }

    /// Twin of `render_scene(cam, num_samples, scene)` (lib.rs:75-79): row-major RGB8, W*H*3 bytes =
    /// the buffer of `image::ImageBuffer<Rgb<u8>, Vec<u8>>` (wrap with `ImageBuffer::from_raw(w, h, buf)`).
    pub fn render(&self, cam: &RbrtCamera, num_samples: u32, seed: u64) -> Vec<u8> {
        let mut buf = vec![0u8; (cam.img_width_pix as usize) * (cam.img_height_pix as usize) * 3];
        let opts = RbrtRenderOpts { seed, ..Default::default() };
        check(unsafe { rbrt_gpu_render(self.0, cam, num_samples, &opts, buf.as_mut_ptr(), std::ptr::null_mut()) });
        buf
    }
}
