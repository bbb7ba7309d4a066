"""Meshes of extreme extent on the GPU: the scenes of tests/test_device_source_on_host.py::test_traversal_at_extreme_mesh_extents (the
icosphere plus one small triangle at coordinate `far`) through every path that builds or reads a mesh's node grid — the three
rbrt_gpu_trace_rays modes, a render (every HDR bit), the creation's build, the refit of rbrt_gpu_scene_update_mesh and its
RBRT_UPDATE_REBUILD mode.  Above a grid step of RBRT_QSTEP_MAX (common.cuh) the slab test of an axis would overflow; k_mesh_setup and
the refit then store a NaN step and the traversal does not cull on that axis.  Every comparison is bit-exact against the oracle."""
import numpy as np
import pytest

import rbrt_b200 as R
from rbrt_b200 import _abi
from rbrt_b200.vec3 import Vec3

from . import scenes as S
from .test_gpu_trace import MODES, assert_same
from .test_gpu_update import assert_images_equal, count_stats, fresh

pytestmark = pytest.mark.gpu
SPP, SEED = 2, 13
# far = 3e11: the first of the sweep whose step (~4.6e6) overflowed the slab test before the NaN rule; 2e38 overflows it for every direction
CASES = [(3e11, 0), (1e12, 0), (1e20, 0), (1e30, 0), (2e38, 0), (-3.4e38, 0), (np.inf, 0), (1e12, 1), (1e20, 2), (-np.inf, 1), (1e11, 0)]


def extent_scene(far, axis, leaf_size=0):
    scene = S.spheres_scene(leaf_size=leaf_size)
    scene.triangle_meshes.append(R.TriangleMesh.from_triangles(S.far_triangle_mesh(far, axis), R.Lambertian(Vec3(0.6, 0.5, 0.4))))
    return scene


def check(oracle, scene, rays, what):
    want = oracle.OracleScene.from_scene(scene).hit(rays)
    assert (want["kind"] == _abi.HIT_MESH).sum() > 1000 and ((want["kind"] == _abi.HIT_MESH)[2000:3000]).sum() > 300, what   # axis-parallel rays hit too
    for mode in MODES:
        assert_same(scene.hit(rays, mode), want, f"{what} mode {mode}")
    cam = S.example_camera(48, 36)
    ref = oracle.OracleScene.from_scene(scene).render_hdr(cam.to_c(), SPP, _abi.RenderOptsC(seed=SEED))
    assert_images_equal(R.render_scene_hdr(cam, SPP, scene, seed=SEED), ref, what)


@pytest.mark.parametrize("far,axis", CASES)
@pytest.mark.parametrize("leaf", [1, 4])
def test_creation_at_extreme_extents(gpu, oracle, far, axis, leaf):
    check(oracle, extent_scene(far, axis, leaf), S.extent_rays(1000, 5), f"far {far:g} axis {axis} leaf {leaf}")


@pytest.mark.parametrize("far,axis", CASES)
def test_refit_and_rebuild_into_and_out_of_extreme_extents(gpu, oracle, far, axis):
    """A scene created with the far triangle beside the icosphere, refit with it moved to `far`, refit back, then rebuilt at `far`."""
    rays = S.extent_rays(1000, 9)
    scene = extent_scene(1.0, axis)
    near = scene.triangle_meshes[0].triangles.copy()
    check(oracle, scene, rays, "created")
    moved = S.far_triangle_mesh(far, axis)
    scene.update_mesh(0, moved)
    check(oracle, scene, rays, f"refit to far {far:g} axis {axis}")
    scene.update_mesh(0, near)
    check(oracle, scene, rays, "refit back")
    scene.update_mesh(0, moved, rebuild=True)
    check(oracle, scene, rays, f"rebuilt at far {far:g} axis {axis}")
    (_, st_rb), (_, st_fr) = count_stats(scene), count_stats(fresh(scene))
    assert st_rb == st_fr and st_rb["traversed_rays"] > 500, (st_rb, st_fr)      # the rebuild is the creation's build
