"""ctypes mirror of include/rbrt_gpu.h (the C-ABI boundary) and the loader of librbrt_gpu.so.

There is no CPU fallback: if the CUDA library was not built, `lib()` raises; if it was built but no
GPU is present, every GPU entry point returns RBRT_E_NODEVICE and `check()` raises RbrtGpuError.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RBRT_GPU_LIB") or os.path.join(_HERE, "librbrt_gpu.so")   # RBRT_GPU_LIB: an experiment build (csrc/Makefile `variant`)


class Vec3C(C.Structure):
    _fields_ = [("x", C.c_float), ("y", C.c_float), ("z", C.c_float)]


class RayC(C.Structure):
    _fields_ = [("origin", Vec3C), ("direction", Vec3C)]


class CameraC(C.Structure):  # cam.rs:4-19, declaration order
    _fields_ = [("hor_fov_rad", C.c_float), ("img_width_pix", C.c_uint32), ("img_height_mm", C.c_float),
                ("vert_fov_rad", C.c_float), ("img_height_pix", C.c_uint32), ("img_width_mm", C.c_float),
                ("position", Vec3C), ("focal_len_mm", C.c_float), ("look_at", Vec3C), ("up", Vec3C),
                ("right", Vec3C), ("img_center_point", Vec3C), ("mm_per_pix_hor", C.c_float),
                ("mm_per_pix_vert", C.c_float)]


class MaterialC(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("albedo", Vec3C), ("param", C.c_float)]


class SphereDescC(C.Structure):
    _fields_ = [("center", Vec3C), ("radius", C.c_float), ("material", MaterialC)]


class TriangleDescC(C.Structure):  # BasicTriangle::new(corners, material) (triangle.rs:9-28)
    _fields_ = [("corners", Vec3C * 3), ("material", MaterialC)]


class ElementRefC(C.Structure):  # one entry of Scene.elements, in order
    _fields_ = [("kind", C.c_uint32), ("index", C.c_uint32)]


class MeshDescC(C.Structure):
    _fields_ = [("tri_vertices", C.POINTER(C.c_float)), ("num_triangles", C.c_uint64), ("material", MaterialC)]


class HitC(C.Structure):
    _fields_ = [("kind", C.c_int32), ("elem_idx", C.c_uint32), ("tri_idx", C.c_uint32), ("t", C.c_float),
                ("dist", C.c_float), ("point", Vec3C), ("normal", Vec3C)]


class SceneOptsC(C.Structure):
    _fields_ = [("simd_lanes", C.c_uint32), ("leaf_size", C.c_uint32), ("box_pad_rel", C.c_float),
                ("flags", C.c_uint32)]


class ScatterInC(C.Structure):  # rbrt_scatter_in
    _fields_ = [("material", MaterialC), ("in_ray", RayC), ("hit_point", Vec3C), ("hit_normal", Vec3C),
                ("pixel", C.c_uint32), ("sample", C.c_uint32), ("bounce", C.c_uint32)]


class ScatterOutC(C.Structure):  # rbrt_scatter_out
    _fields_ = [("scattered", C.c_int32), ("attenuation", Vec3C), ("out_ray", RayC)]


class CommInfoC(C.Structure):  # rbrt_comm_info
    _fields_ = [("active", C.c_int32), ("world", C.c_int32), ("rank", C.c_int32), ("local_devices", C.c_int32),
                ("transport", C.c_int32), ("nccl_version", C.c_int32), ("devices", C.c_int32 * 16)]

    def as_dict(self):
        d = {k: getattr(self, k) for k, _ in self._fields_ if k != "devices"}
        d["devices"] = list(self.devices)[:max(self.local_devices, 0)]
        return d


class RenderOptsC(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("max_depth", C.c_uint32), ("trace_mode", C.c_uint32),
                ("shard_mode", C.c_uint32), ("shard_rank", C.c_uint32), ("shard_count", C.c_uint32),
                ("batch_paths", C.c_uint32), ("integrator", C.c_uint32), ("flags", C.c_uint32)]


class StatsC(C.Structure):
    _fields_ = [("rays", C.c_uint64), ("paths", C.c_uint64), ("nan_rays", C.c_uint64),
                ("node_visits", C.c_uint64), ("tri_tests", C.c_uint64), ("ms_total", C.c_double),
                ("ms_device", C.c_double), ("ms_trace", C.c_double), ("ms_h2d", C.c_double),
                ("ms_d2h", C.c_double), ("launches", C.c_uint32), ("iterations", C.c_uint32),
                ("traversed_rays", C.c_uint64), ("tail_node_visits", C.c_uint64), ("tail_tri_tests", C.c_uint64),
                ("tail_traversed_rays", C.c_uint64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class AovOutC(C.Structure):  # rbrt_aov_out: device or host planes, NULL = pass not produced
    _fields_ = [("depth", C.c_void_p), ("normal", C.c_void_p), ("albedo", C.c_void_p), ("coverage", C.c_void_p),
                ("hit_kind", C.c_void_p), ("elem_idx", C.c_void_p), ("tri_idx", C.c_void_p)]


class QueryOutC(C.Structure):  # rbrt_query_out: device planes, NULL = not produced
    _fields_ = [("t", C.c_void_p), ("dist", C.c_void_p), ("kind", C.c_void_p), ("elem_idx", C.c_void_p), ("tri_idx", C.c_void_p),
                ("point", C.c_void_p), ("normal", C.c_void_p)]


class DenoiseOptsC(C.Structure):  # rbrt_denoise_opts: 0 = default
    _fields_ = [("levels", C.c_uint32), ("sigma_depth", C.c_float), ("sigma_luminance", C.c_float)]


class SceneInfoC(C.Structure):
    _fields_ = [("num_spheres", C.c_uint32), ("num_meshes", C.c_uint32), ("num_triangles", C.c_uint64),
                ("num_triangles_tested", C.c_uint64), ("num_bvh_nodes", C.c_uint64),
                ("device_bytes", C.c_uint64), ("ms_upload", C.c_double), ("ms_build", C.c_double)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


HIT_DTYPE = [("kind", "<i4"), ("elem_idx", "<u4"), ("tri_idx", "<u4"), ("t", "<f4"), ("dist", "<f4"),
             ("point", "<f4", (3,)), ("normal", "<f4", (3,))]

MAT_LAMBERTIAN, MAT_METAL, MAT_DIELECTRIC = 0, 1, 2
SHARD_NONE, SHARD_TILES, SHARD_SAMPLES = 0, 1, 2
TRACE_BVH, TRACE_BRUTE, TRACE_WAVEFRONT = 0, 1, 2
SCENE_LOCAL, SCENE_NO_SAH, SCENE_BROADCAST = 1, 2, 4
TRANSPORT_AUTO, TRANSPORT_NCCL, TRANSPORT_PEER = 0, 1, 2
COMM_ID_BYTES = 128
OPT_COUNT_VISITS, OPT_TIME_KERNELS, OPT_NO_TAIL_KERNEL, OPT_POOL_SHIFT, OPT_SPLIT_BATCHES = 1, 2, 4, 3, 32
MAX_FRAMES = 4          # frames one wavefront batch can hold (rbrt_gpu_render_accum_device_frames)
HIT_NONE, HIT_SPHERE, HIT_MESH, HIT_TRIANGLE = -1, 0, 1, 2
ELEM_SPHERE, ELEM_TRIANGLE = 0, 1
QUERY_CLEAR, QUERY_OCCLUDED, QUERY_NAN_RAY = 0, 1, 2
UPDATE_REFIT, UPDATE_REBUILD = 0, 1
E_INVALID, E_CUDA, E_NODEVICE = 1, 2, 3

P = C.POINTER
# name -> (restype, argtypes) of every function include/rbrt_gpu.h declares
GPU_SIGNATURES = {
    "rbrt_camera_new": (C.c_int, [Vec3C, Vec3C, Vec3C, C.c_uint32, C.c_uint32, C.c_float, P(CameraC)]),
    "rbrt_transform_vertices": (C.c_int, [P(C.c_float), C.c_uint64, C.c_float, Vec3C, Vec3C]),
    "rbrt_mesh_load_obj": (C.c_int, [C.c_char_p, Vec3C, Vec3C, C.c_float, P(P(C.c_float)), P(C.c_uint64)]),
    "rbrt_mesh_free": (None, [P(C.c_float)]),
    "rbrt_gpu_init": (C.c_int, [C.c_int]),
    "rbrt_gpu_init_multi": (C.c_int, [P(C.c_int), C.c_int, C.c_int]),
    "rbrt_gpu_comm_unique_id": (C.c_int, [C.c_void_p]),
    "rbrt_gpu_comm_init_rank": (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    "rbrt_gpu_comm_info": (C.c_int, [P(CommInfoC)]),
    "rbrt_gpu_comm_destroy": (C.c_int, []),
    "rbrt_gpu_set_pool_limit": (C.c_int, [C.c_uint64]),
    "rbrt_gpu_scatter": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p]),
    "rbrt_gpu_render_frames_device": (C.c_int, [C.c_void_p, P(CameraC), P(C.c_uint64), C.c_uint32, C.c_uint32, P(RenderOptsC),
                                                P(C.c_void_p), P(C.c_void_p), C.c_void_p, P(StatsC)]),
    "rbrt_gpu_scene_create": (C.c_int, [P(SphereDescC), C.c_uint32, P(MeshDescC), C.c_uint32, P(SceneOptsC), P(C.c_void_p)]),
    "rbrt_gpu_scene_create_elements": (C.c_int, [P(ElementRefC), C.c_uint32, P(SphereDescC), C.c_uint32, P(TriangleDescC), C.c_uint32,
                                                P(MeshDescC), C.c_uint32, P(SceneOptsC), P(C.c_void_p)]),
    "rbrt_gpu_scene_info": (C.c_int, [C.c_void_p, P(SceneInfoC)]),
    "rbrt_gpu_scene_update_mesh": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint64, P(MaterialC), C.c_uint32]),
    "rbrt_gpu_scene_update_mesh_device": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint64, P(MaterialC), C.c_uint32, C.c_void_p]),
    "rbrt_gpu_scene_update_elements": (C.c_int, [C.c_void_p, P(ElementRefC), C.c_uint32, P(SphereDescC), C.c_uint32, P(TriangleDescC),
                                                C.c_uint32]),
    "rbrt_gpu_scene_destroy": (C.c_int, [C.c_void_p]),
    "rbrt_gpu_render": (C.c_int, [C.c_void_p, P(CameraC), C.c_uint32, P(RenderOptsC), C.c_void_p, P(StatsC)]),
    "rbrt_gpu_render_hdr": (C.c_int, [C.c_void_p, P(CameraC), C.c_uint32, P(RenderOptsC), C.c_void_p, P(StatsC)]),
    "rbrt_gpu_render_accum_device": (C.c_int, [C.c_void_p, P(CameraC), C.c_uint32, P(RenderOptsC), C.c_void_p, C.c_void_p, P(StatsC)]),
    "rbrt_gpu_render_accum_device_frames": (C.c_int, [C.c_void_p, P(CameraC), P(C.c_uint64), C.c_uint32, C.c_uint32, P(RenderOptsC),
                                                      P(C.c_void_p), C.c_void_p, P(StatsC)]),
    "rbrt_gpu_finalize_device": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rbrt_gpu_trace_rays": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, P(StatsC)]),
    "rbrt_gpu_primary_rays": (C.c_int, [P(CameraC), C.c_uint64, C.c_uint32, C.c_void_p]),
    "rbrt_gpu_render_aov": (C.c_int, [C.c_void_p, P(CameraC), C.c_uint32, C.c_uint64, P(AovOutC), P(StatsC)]),
    "rbrt_gpu_render_aov_device": (C.c_int, [C.c_void_p, P(CameraC), C.c_uint32, C.c_uint64, P(AovOutC), C.c_void_p, P(StatsC)]),
    "rbrt_gpu_query_closest_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, P(QueryOutC), C.c_void_p, P(StatsC)]),
    "rbrt_gpu_query_occluded_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, P(StatsC)]),
    "rbrt_gpu_denoise": (C.c_int, [C.c_uint32, C.c_uint32, C.c_void_p, P(AovOutC), P(DenoiseOptsC), C.c_void_p, C.c_void_p, P(StatsC)]),
    "rbrt_gpu_denoise_device": (C.c_int, [C.c_uint32, C.c_uint32, C.c_void_p, P(AovOutC), P(DenoiseOptsC), C.c_void_p, C.c_void_p, C.c_void_p,
                                          P(StatsC)]),
    "rbrt_gpu_render_hdr_variance": (C.c_int, [C.c_void_p, P(CameraC), C.c_uint32, C.c_uint32, P(RenderOptsC), C.c_void_p, C.c_void_p,
                                               P(StatsC)]),
    "rbrt_gpu_render_hdr_variance_device": (C.c_int, [C.c_void_p, P(CameraC), C.c_uint32, C.c_uint32, P(RenderOptsC), C.c_void_p,
                                                      C.c_void_p, C.c_void_p, P(StatsC)]),
    "rbrt_gpu_denoise_variance": (C.c_int, [C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, P(AovOutC), P(DenoiseOptsC), C.c_void_p,
                                            C.c_void_p, P(StatsC)]),
    "rbrt_gpu_denoise_variance_device": (C.c_int, [C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, P(AovOutC), P(DenoiseOptsC),
                                                   C.c_void_p, C.c_void_p, C.c_void_p, P(StatsC)]),
    "rbrt_gpu_release_cache": (C.c_int, []),
    "rbrt_last_error": (C.c_char_p, []),
    "rbrt_gpu_version": (C.c_char_p, []),
}


class RbrtGpuError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"rbrt_gpu error {code}: {msg}")
        self.code = code


_lib = None


def lib():
    """Load rbrt_b200/librbrt_gpu.so (built by __graft_entry__.build() / csrc/Makefile)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RbrtGpuError(E_NODEVICE, f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                                           "(there is no CPU fallback)")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in GPU_SIGNATURES.items():
            f = getattr(l, name)
            f.restype, f.argtypes = res, args
        _lib = l
    return _lib


def check(rc):
    if rc != 0:
        raise RbrtGpuError(rc, lib().rbrt_last_error().decode("utf-8", "replace"))
