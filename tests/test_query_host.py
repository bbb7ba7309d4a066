"""Ray queries on device memory without a GPU: the query module is built for sm_100a and exports its launch interface, rbrt_query_out has the
header's layout, the entry points refuse bad calls without touching a device, the Python wrappers check their arguments, and the occlusion
rule of csrc/query.cuh, compiled for the host, equals Scene::hit composed with the strict max_dist compare on adversarial rays."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import rbrt_b200 as R
from rbrt_b200 import _abi

from . import query_ref as Q
from .test_device_source_on_host import scene_args

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
QRY = os.path.join(ROOT, "rbrt_b200", "librbrt_gpu_query.so")
HEADER = os.path.join(ROOT, "include", "rbrt_gpu.h")
HD = os.path.join(ROOT, "tests", "host_device")
CSRC = os.path.join(ROOT, "rbrt_b200", "csrc")
PLANES = ["t", "dist", "kind", "elem_idx", "tri_idx", "point", "normal"]
P = C.POINTER


@pytest.fixture(scope="module", autouse=True)
def query_module():
    if not os.path.exists(QRY):
        subprocess.run(["make", "-C", CSRC], check=True)
    return QRY


@pytest.fixture(scope="module")
def hq():
    out = os.path.join(HD, "build", "libhost_query.so")
    os.makedirs(os.path.dirname(out), exist_ok=True)
    srcs = [os.path.join(HD, f) for f in ("query_harness.cpp", "harness.cpp", "cuda_runtime.h")] + \
           [os.path.join(CSRC, f) for f in ("common.cuh", "intersect.cuh", "shade.cuh", "cull.cuh", "query.cuh")]
    if not os.path.exists(out) or any(os.path.getmtime(s) > os.path.getmtime(out) for s in srcs):
        # the flags of tests/test_device_source_on_host.py: the stand-in cuda_runtime.h first, no contraction, no FMA
        subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-mno-fma", "-DRBRT_LDG128", "-Wno-unknown-pragmas", "-fPIC", "-shared",
                        "-I", HD, "-I", CSRC, "-o", out, srcs[0]], check=True)
    lib = C.CDLL(out)
    lib.hd_occluded.argtypes = [P(_abi.ElementRefC), C.c_uint32, P(_abi.SphereDescC), P(_abi.TriangleDescC), P(_abi.MeshDescC), C.c_uint32, C.c_uint32,
                                C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_void_p, P(C.c_uint64)]
    lib.hd_trace_rays.argtypes = [P(_abi.ElementRefC), C.c_uint32, P(_abi.SphereDescC), P(_abi.TriangleDescC), P(_abi.MeshDescC), C.c_uint32, C.c_uint32,
                                  C.c_uint32, C.c_void_p, C.c_uint64, C.c_void_p, P(C.c_uint64), P(C.c_uint64)]
    return lib


def host_hits(hq, scene, rays):
    hits = np.zeros(len(rays), dtype=_abi.HIT_DTYPE)
    args, keep = scene_args(scene)
    assert hq.hd_trace_rays(*args, 0, rays.ctypes.data, len(rays), hits.ctypes.data, None, None) == 0
    return hits


def host_occluded(hq, scene, rays, max_dist, leaf_size, ref_bvh):
    occ, ref = np.full(len(rays), 9, np.uint8), np.full(len(rays), 9, np.uint8)
    args, keep = scene_args(scene)
    nodes = C.c_uint64(0)
    assert hq.hd_occluded(*args, leaf_size, rays.ctypes.data, np.ascontiguousarray(max_dist, np.float32).ctypes.data, len(rays), ref_bvh,
                          occ.ctypes.data, ref.ctypes.data, C.byref(nodes)) == 0
    return occ, ref, nodes.value


# ============================================================================== module, layout, refusals
def test_query_module_is_built_for_sm_100a_and_exports_its_interface():
    lib = C.CDLL(QRY)
    assert hasattr(lib, "rbrt_query_launch")
    raw = C.CDLL(_abi.LIB_PATH)
    assert hasattr(raw, "rbrt_gpu_query_closest_device") and hasattr(raw, "rbrt_gpu_query_occluded_device")
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump is not here")
    sass = subprocess.run([cuobjdump, "-sass", QRY], capture_output=True, text=True, check=True).stdout
    names = re.findall(r"Function : (\S+)", sass)
    assert len(names) == 4 and all("k_query" in n for n in names), names
    assert "arch = sm_100a" in sass


def test_query_out_layout_matches_the_header(tmp_path):
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{HEADER}"', "int main(void){",
             'printf("size %zu\\n", sizeof(rbrt_query_out));']
    lines += [f'printf("{f} %zu\\n", offsetof(rbrt_query_out, {f}));' for f in PLANES]
    lines.append("return 0;}")
    src = tmp_path / "query_layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "query_layout"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-o", str(exe), str(src)], check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    assert [f for f, _ in _abi.QueryOutC._fields_] == PLANES
    assert int(got["size"]) == C.sizeof(_abi.QueryOutC)
    for f in PLANES:
        assert int(got[f]) == getattr(_abi.QueryOutC, f).offset, f


def test_refusals_before_any_device_work():
    lib = _abi.lib()
    buf = np.full(8, 7, np.float32)
    occ = np.full(8, 7, np.uint8)
    out = _abi.QueryOutC(t=buf.ctypes.data)
    rays = np.zeros((8, 6), np.float32)
    h = C.c_void_p(1)                                                     # never dereferenced: every call below is refused first
    closest, occluded = lib.rbrt_gpu_query_closest_device, lib.rbrt_gpu_query_occluded_device
    st = _abi.StatsC(rays=5)
    assert closest(None, None, 0, None, None, st) == 0 and st.rays == 0    # n = 0: nothing to do, stats zeroed
    assert occluded(None, None, 0, None, None, None, None) == 0
    assert closest(None, rays.ctypes.data, 8, out, None, None) == _abi.E_INVALID
    assert b"null" in lib.rbrt_last_error()
    assert closest(h, None, 8, out, None, None) == _abi.E_INVALID
    assert closest(h, rays.ctypes.data, 8, None, None, None) == _abi.E_INVALID
    assert closest(h, rays.ctypes.data, 8, _abi.QueryOutC(), None, None) == _abi.E_INVALID
    assert b"every plane" in lib.rbrt_last_error()
    assert closest(h, rays.ctypes.data, 2 ** 32, out, None, None) == _abi.E_INVALID
    assert occluded(None, rays.ctypes.data, 8, None, occ.ctypes.data, None, None) == _abi.E_INVALID
    assert occluded(h, None, 8, None, occ.ctypes.data, None, None) == _abi.E_INVALID
    assert occluded(h, rays.ctypes.data, 8, None, None, None, None) == _abi.E_INVALID
    assert occluded(h, rays.ctypes.data, 2 ** 32, None, occ.ctypes.data, None, None) == _abi.E_INVALID
    assert b"2^32" in lib.rbrt_last_error()
    assert (buf == 7).all() and (occ == 7).all()


def test_queries_need_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present; the refusal path is exercised on the CPU-only build box")
    scene = R.Scene(elements=[R.Sphere((0, 0, -3), 1.0, R.Lambertian((0.5, 0.5, 0.5)))])
    with pytest.raises(_abi.RbrtGpuError) as e:
        scene.handle()
    assert e.value.code in (_abi.E_NODEVICE, _abi.E_CUDA)


def test_python_argument_checks():
    """Anything but a contiguous float32 CUDA tensor [N,6] is refused before the scene is created or a device is touched."""
    import torch
    scene = R.Scene(elements=[R.Sphere((0, 0, -3), 1.0, R.Lambertian((0.5, 0.5, 0.5)))])
    bad = [np.zeros((4, 6), np.float32), torch.zeros(4, 6), torch.zeros(4, 6, dtype=torch.float64), [[0.0] * 6], torch.zeros(4, 5), torch.zeros(24)]
    for rays in bad:
        with pytest.raises(ValueError):
            scene.intersect_device(rays)
        with pytest.raises(ValueError):
            scene.occluded_device(rays)
    assert scene._handle is None
    from rbrt_b200.scene import QUERY_PASSES
    assert QUERY_PASSES == tuple(PLANES)


def test_rust_crate_mirrors_query_out_and_the_new_functions():
    rs = open(os.path.join(ROOT, "integration", "rust", "rbrt_gpu_sys", "src", "lib.rs")).read()
    m = re.search(r"pub struct RbrtQueryOut\s*\{(.*?)\}", rs, re.S)
    assert m and re.findall(r"pub (\w+)\s*:", m.group(1)) == PLANES
    for name, arity in (("rbrt_gpu_query_closest_device", 6), ("rbrt_gpu_query_occluded_device", 7)):
        f = re.search(r"pub fn %s\s*\((.*?)\)\s*->" % name, rs, re.S)
        assert f and len([a for a in f.group(1).split(",") if a.strip()]) == arity, name


# ============================================================================== the occlusion rule (query.cuh) on the host
def test_numpy_nan_mask_equals_scene_hit(hq):
    """tests/query_ref.py's NaN-ray mask (what the GPU tests compose with) against scene_hit's own verdict."""
    scene = Q.adversarial_scene()
    rays = Q.adversarial_rays(3000, 1)
    nan = Q.nan_rays(scene, rays)
    _, ref, _ = host_occluded(hq, scene, rays, np.full(len(rays), np.inf, np.float32), 1, 0)
    assert np.array_equal(ref == 2, nan)
    assert 50 < nan.sum() < 0.75 * len(rays)
    hits = host_hits(hq, scene, rays)
    assert ((hits["kind"] == _abi.HIT_NONE) | ~nan).all()                # a NaN ray is reported as a miss


@pytest.mark.parametrize("leaf_size", [1, 4, 8])
def test_occlusion_rule_equals_the_composition(hq, leaf_size):
    scene = Q.adversarial_scene(leaf_size)
    rays = Q.adversarial_rays(4000, leaf_size)
    hits = host_hits(hq, scene, rays)
    nan = Q.nan_rays(scene, rays)
    seen = {0: 0, 1: 0, 2: 0}
    for k, md in enumerate(Q.max_dist_variants(hits["dist"])):
        for ref_bvh in (0, 1):
            occ, ref, _ = host_occluded(hq, scene, rays, md, leaf_size, ref_bvh)
            assert np.array_equal(ref, Q.occluded(hits, nan, md)), (k, ref_bvh)
            bad = np.flatnonzero(occ != ref)
            assert not len(bad), f"bounds {k}, leaf {leaf_size}: {len(bad)} rays differ; first ray {rays[bad[0]]} md {md[bad[0]]} got {occ[bad[0]]} want {ref[bad[0]]}"
        for v in (0, 1, 2):
            seen[v] += int((occ == v).sum())
    assert min(seen.values()) > 100, seen


def test_short_directions_min_t_triangle_decides(hq):
    """|d| = 1e-4 straight down through both quads: the near one (t = 5, dist 0.0005) is the mesh's minimum-t triangle and too close, so
    Scene::hit reports no mesh hit although the far one (t = 50, dist 0.005) is in the window: not occluded, whatever max_dist."""
    scene = Q.adversarial_scene(1)
    n = 64
    o = np.stack([np.linspace(-0.7, 0.7, n), np.linspace(0.6, -0.6, n), np.zeros(n)], 1).astype(np.float32)
    rays = np.concatenate([o, np.tile(np.float32([[0.0, 0.0, -1e-4]]), (n, 1))], 1).astype(np.float32)
    hits = host_hits(hq, scene, rays)
    assert (hits["kind"] == _abi.HIT_NONE).all()
    occ, ref, _ = host_occluded(hq, scene, rays, np.full(n, np.inf, np.float32), 1, 0)
    assert (occ == 0).all() and (ref == 0).all()
    rays[:, 5] = np.float32(-1.0)                                         # a unit direction: the near quad is hit at dist 0.0005... too close
    hits = host_hits(hq, scene, rays)                                     # ...and it is still the minimum-t triangle
    occ, ref, _ = host_occluded(hq, scene, rays, np.full(n, np.inf, np.float32), 1, 0)
    assert np.array_equal(occ, ref) and np.array_equal(ref, Q.occluded(hits, np.zeros(n, bool), np.full(n, np.inf, np.float32)))


def test_nan_sphere_after_an_earlier_hit(hq):
    """Rays at the first sphere with |d.x| large: hit at once, then the sphere 3e19 away gives a NaN discriminant -> 2, never 1."""
    scene = Q.adversarial_scene(1)
    o = np.tile(np.float32([[0.0, 2.0, 0.0]]), (32, 1))                   # (clear of the quads below the origin)
    d = np.array([-3.0, -2.0, -5.0], np.float32) + np.random.default_rng(3).normal(size=(32, 3)).astype(np.float32) * np.float32(0.1)
    rays = np.concatenate([o, d], 1).astype(np.float32)
    no_far = Q.adversarial_scene(1)
    del no_far.elements[2]
    hits = host_hits(hq, no_far, rays)
    assert (hits["kind"] == _abi.HIT_SPHERE).all()                        # without the far sphere every ray hits sphere 0
    occ, ref, _ = host_occluded(hq, scene, rays, np.full(32, np.inf, np.float32), 1, 0)
    assert (ref == 2).all() and (occ == 2).all()


def test_early_exit_visits_fewer_nodes(hq):
    """With max_dist = +inf the first triangle that proves occlusion ends the traversal: fewer node visits than the closest search."""
    scene = Q.adversarial_scene(1)
    del scene.elements[2]                                                 # (without the sphere that makes these rays NaN rays)
    rng = np.random.default_rng(5)
    o = np.tile(np.float32([[2.5, 1.0, -2.0]]), (500, 1))
    d = (np.float32([2.5, 1.0, -8.0]) + rng.normal(size=(500, 3)).astype(np.float32) * np.float32(0.5)) - o
    rays = np.concatenate([o, d], 1).astype(np.float32)
    inf, _, n_any = host_occluded(hq, scene, rays, np.full(500, np.inf, np.float32), 1, 1)
    args, keep = scene_args(scene)
    hits = np.zeros(500, dtype=_abi.HIT_DTYPE)
    nodes = C.c_uint64(0)
    assert hq.hd_trace_rays(*args, 1 + 16, rays.ctypes.data, 500, hits.ctypes.data, C.byref(nodes), None) == 0
    assert (inf == 1).sum() > 300 and n_any < nodes.value, (n_any, nodes.value)
