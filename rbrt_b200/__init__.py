"""rbrt_b200 — B200-native (sm_100a) path tracer behind rbrt_lib's render/scene API.

Host mirror of the reference's public surface (names and argument order as in rbrt_lib):
    Vec3, Ray, Camera.new, Lambertian, Metal, Dielectric, Sphere, TriangleMesh.new, Scene,
    load_blueprints_from_yaml_file, create_scene_from_scene_blueprint, render_scene
The hot path runs in rbrt_b200/librbrt_gpu.so (hand-written CUDA, csrc/) through the C-ABI of
include/rbrt_gpu.h.  There is no CPU fallback.
"""
from ._abi import (HIT_DTYPE, HIT_MESH, HIT_NONE, HIT_SPHERE, HIT_TRIANGLE, SHARD_NONE, SHARD_SAMPLES, SHARD_TILES, TRACE_BRUTE,
                   TRACE_BVH, RbrtGpuError)
from .blueprints import (CameraBluePrint, SceneBlueprint, SphereBlueprint, TriangleMeshBlueprint,
                         create_material_from_description, create_scene_from_scene_blueprint,
                         load_blueprints_from_yaml_file)
from .cam import Camera
from .materials import Dielectric, Lambertian, Metal
from .mesh import TriangleMesh, load_mesh_vertices_from_file
from .pipeline import FramePipeline
from .render import (AOV_PASSES, ImageBuffer, denoise, denoise_device, denoise_variance, denoise_variance_device, primary_rays, render_aovs,
                     render_aovs_device, render_hdr_variance_device, render_motion, render_motion_device, render_scene, render_scene_hdr,
                     render_scene_hdr_variance, temporal_accumulate, temporal_accumulate_device)
from .scene import Scene
from .temporal import TemporalAccumulator
from .sphere import Sphere
from .triangle import BasicTriangle
from .vec3 import Ray, Vec3


def gpu_init(device=0):
    """Select the CUDA device of this process (one process per GPU)."""
    from . import _abi
    _abi.check(_abi.lib().rbrt_gpu_init(int(device)))
