"""Scene updates without a GPU: the refit module is built and exports its launch interface, the new entry points refuse bad
calls and fail loudly without a device, the Python mirror follows an update, and FramePipeline launches a pending group of the
updated scene first (its GPU work replaced by a recorder, as in test_pipeline_logic.py)."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import rbrt_b200 as R
from rbrt_b200 import _abi, pipeline
from rbrt_b200.vec3 import Vec3

from .test_pipeline_logic import RecordingPipeline, _Cam, _Scene

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
UPD = os.path.join(ROOT, "rbrt_b200", "librbrt_gpu_update.so")


def test_refit_module_is_built_for_sm_100a_and_exports_its_interface():
    lib = C.CDLL(UPD)
    lib.rbrt_update_scratch_bytes.restype = C.c_size_t
    lib.rbrt_update_scratch_bytes.argtypes = [C.c_uint64]
    small, big = lib.rbrt_update_scratch_bytes(1), lib.rbrt_update_scratch_bytes(1 << 20)
    assert small % 256 == 0 and big % 256 == 0
    assert big >= (32 + 140) * ((1 << 20) - 1)                             # leaf boxes + per-node links and child boxes
    assert hasattr(lib, "rbrt_update_refit")
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump is not here")
    sass = subprocess.run([cuobjdump, "-sass", UPD], capture_output=True, text=True, check=True).stdout
    names = set(re.findall(r"Function : \S*?(k_upd_\w+?)E", sass))
    assert names == {"k_upd_aabb_init", "k_upd_aabb", "k_upd_setup", "k_upd_tris", "k_upd_links", "k_upd_nodes"}, names
    assert "arch = sm_100a" in sass


def test_update_entry_points_refuse_without_a_scene():
    lib = _abi.lib()
    v = np.zeros((1, 3, 3), np.float32)
    assert lib.rbrt_gpu_scene_update_mesh(None, 0, v.ctypes.data, 1, None, 0) == _abi.E_INVALID
    assert b"null" in lib.rbrt_last_error()
    assert lib.rbrt_gpu_scene_update_mesh_device(None, 0, v.ctypes.data, 1, None, 0, None) == _abi.E_INVALID
    assert lib.rbrt_gpu_scene_update_elements(None, None, 0, None, 0, None, 0) == _abi.E_INVALID


def test_update_needs_a_gpu_once_the_scene_exists():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present; the refusal path is exercised on the CPU-only build box")
    scene = R.Scene(triangle_meshes=[R.TriangleMesh.from_triangles(np.ones((4, 3, 3), np.float32), R.Lambertian(Vec3(0.5, 0.5, 0.5)))])
    with pytest.raises(_abi.RbrtGpuError) as e:
        scene.handle()
    assert e.value.code in (_abi.E_NODEVICE, _abi.E_CUDA)


def test_mirror_follows_updates_before_the_scene_exists():
    """Before the library scene exists an update only changes the host mirror (what the scene will be created from, and what the
    CPU oracle reads through OracleScene.from_scene)."""
    m0 = R.Lambertian(Vec3(0.5, 0.5, 0.5))
    scene = R.Scene(elements=[R.Sphere(Vec3(0, 0, -3), 1.0, m0)],
                    triangle_meshes=[R.TriangleMesh.from_triangles(np.zeros((5, 3, 3), np.float32), m0)])
    new = np.arange(45, dtype=np.float32).reshape(5, 3, 3)
    scene.update_mesh(0, new)
    assert np.array_equal(scene.triangle_meshes[0].triangles, new) and scene.triangle_meshes[0].material is m0
    m1 = R.Metal(Vec3(0.9, 0.9, 0.9), 0.1)
    scene.update_mesh(0, new * 2, material=m1)
    assert np.array_equal(scene.triangle_meshes[0].triangles, new * 2) and scene.triangle_meshes[0].material is m1
    s2 = R.Sphere(Vec3(1, 2, -4), 0.5, m1)
    scene.update_elements([s2])
    assert scene.elements == [s2]
    assert scene._handle is None


def test_an_update_launches_the_pending_group_of_its_scene_first():
    """frames_per_batch = 4: frames of scene a wait in a pending group.  An update of a launches that group (its frames keep the old
    geometry); a pipeline holding frames of another scene keeps its pending group; the frames that left meanwhile come back with the
    next submit."""
    a, b = _Scene(11), _Scene(22)
    p = RecordingPipeline(2, 4)
    q = RecordingPipeline(2, 4)
    pipeline._live.add(p)
    pipeline._live.add(q)
    try:
        p.submit(_Cam(), 4, a, tag=0)
        p.submit(_Cam(), 4, a, tag=1)
        q.submit(_Cam(), 4, b, tag=10)
        assert not p.groups and not q.groups
        pipeline.launch_pending(C.c_void_p(11))
        assert [g[2] for g in p.groups] == [[0, 1]] and not p._pending
        assert not q.groups and len(q._pending) == 1
        out = p.submit(_Cam(), 4, a, tag=2)
        out += p.submit(_Cam(), 4, a, tag=3)
        pipeline.launch_pending(11)
        out += p.drain()
        assert [t for _, t in out] == [0, 1, 2, 3]
        assert [g[2] for g in p.groups] == [[0, 1], [2, 3]]
    finally:
        pipeline._live.discard(p)
        pipeline._live.discard(q)
