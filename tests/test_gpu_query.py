"""Ray queries on device memory (rbrt_gpu_query_closest_device / rbrt_gpu_query_occluded_device; csrc/query.cu, csrc/api.cu) on the GPU.

Both queries are defined by the parity hook (include/rbrt_gpu.h, DESIGN.md section 12): every plane of the closest query is, bit for bit,
the field rbrt_gpu_trace_rays (Scene.hit) reports, and the occlusion answer is that hit composed with the strict max_dist compare
(tests/query_ref.py).  Every comparison is on uint32 views, so NaN and +-inf compare too."""
import ctypes as C
import os
import subprocess
import sys
import time

import numpy as np
import pytest

import rbrt_b200 as R
from rbrt_b200 import _abi

from . import golden_util as G
from . import query_ref as Q
from . import scenes as S
from .test_gpu_aov import meshes_scene, negative_radius_scene
from .test_gpu_trace import mixed_element_scene
from .test_gpu_update import fresh, moved_elements, twist

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
QRY_SO = os.path.join(ROOT, "rbrt_b200", "librbrt_gpu_query.so")
PLANES = ("t", "dist", "kind", "elem_idx", "tri_idx", "point", "normal")


@pytest.fixture(scope="module", autouse=True)
def query_module():
    """The session fixture only builds librbrt_gpu.so when it is missing; the query module is built here when it is."""
    if not os.path.exists(QRY_SO):
        subprocess.run(["make", "-C", os.path.join(ROOT, "rbrt_b200", "csrc")], check=True)
    return QRY_SO


def u32(t):
    """A CUDA tensor of 4-byte values as a numpy uint32 array (bit pattern)."""
    import torch
    return t.contiguous().view(torch.int32).cpu().numpy().view(np.uint32)


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).cuda()


def assert_planes(got, hits, what):
    for k in got:
        want = bits(hits[k].astype({"kind": np.int32, "elem_idx": np.uint32, "tri_idx": np.uint32}.get(k, np.float32)))
        g = u32(got[k]).reshape(want.shape)
        bad = np.flatnonzero((g != want).reshape(len(hits), -1).any(1))
        assert not len(bad), f"{what}: plane {k}: {len(bad)} of {len(hits)} rays differ; first ray {bad[0]}: got {g[bad[0]]} want {want[bad[0]]}"


def check_closest(scene, rays, what, oracle=None):
    hits = scene.hit(rays)
    got = scene.intersect_device(dev(rays))
    assert set(got) == set(PLANES)
    assert_planes(got, hits, f"{what} vs Scene.hit")
    assert S.hits_equal(scene.hit(rays, trace_mode=_abi.TRACE_BRUTE), hits).all(), f"{what}: BVH and BRUTE hooks differ"
    if oracle is not None:
        assert S.hits_equal(oracle.OracleScene.from_scene(scene).hit(rays), hits).all(), f"{what}: the oracle differs"
    return hits


def check_occluded(scene, rays, hits, what):
    nan = Q.nan_rays(scene, rays)
    t = dev(rays)
    seen = set()
    for k, md in enumerate(Q.max_dist_variants(hits["dist"])):
        got = scene.occluded_device(t, dev(md)).cpu().numpy()
        want = Q.occluded(hits, nan, md)
        bad = np.flatnonzero(got != want)
        assert not len(bad), f"{what}, bounds {k}: {len(bad)} rays differ; first {rays[bad[0]]} md {md[bad[0]]} got {got[bad[0]]} want {want[bad[0]]}"
        seen |= set(np.unique(got).tolist())
    assert np.array_equal(scene.occluded_device(t).cpu().numpy(), Q.occluded(hits, nan, np.full(len(rays), np.inf, np.float32))), what
    return seen


# ============================================================================== 1. golden rays (oracle outputs)
@pytest.mark.parametrize("name", G.NAMES)
def test_golden_rays(gpu, name):
    z, scene, cam = G.load(name)
    rays = np.ascontiguousarray(z["rays"], np.float32)
    got = scene.intersect_device(dev(rays))
    assert_planes(got, z["hits"], name)
    check_occluded(scene, rays, z["hits"], name)


# ============================================================================== 2. the scenes of the parity tests
SCENES = {"spheres": S.spheres_scene, "negative_radius": negative_radius_scene, "mixed_elements": mixed_element_scene, "meshes_leaf8": meshes_scene,
          "meshes_leaf1": lambda: meshes_scene(1), "example_leaf1": lambda: S.small_mesh_scene(3, leaf_size=1),
          "adversarial_leaf1": lambda: Q.adversarial_scene(1), "adversarial_leaf8": lambda: Q.adversarial_scene(8), "quirk": S.quirk_scene}


@pytest.mark.parametrize("name", list(SCENES))
def test_scenes(gpu, oracle, name):
    scene = SCENES[name]()
    rays = np.concatenate([R.primary_rays(S.example_camera(64, 48), 3, 0), S.random_rays(6000, (0.0, 1.0, -7.0), 4.0, 2),
                           Q.adversarial_rays(2000, 3)], 0)
    hits = check_closest(scene, rays, name, oracle)
    assert (hits["kind"] != _abi.HIT_NONE).sum() > 300
    seen = check_occluded(scene, rays, hits, name)
    assert {0, 1} <= seen, seen
    if name.startswith("adversarial"):
        assert seen == {0, 1, 2}


# ============================================================================== 3. C3 at full size: camera rays and bounce-like rays
def c3_rays():
    scene, cam = S.big_scene(8)
    cam_rays = R.primary_rays(cam, 3, 0)
    first = scene.hit(cam_rays)
    hit = first["kind"] != _abi.HIT_NONE
    rng = np.random.default_rng(11)
    d = rng.normal(size=(int(hit.sum()), 3)).astype(np.float32)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    bounce = np.concatenate([first["point"][hit], d], 1).astype(np.float32)
    return scene, cam_rays, first, bounce


def test_c3_camera_and_bounce_rays(gpu):
    scene, cam_rays, first, bounce = c3_rays()
    got = scene.intersect_device(dev(cam_rays))
    assert_planes(got, first, "C3 camera rays")
    assert (first["kind"] == _abi.HIT_MESH).sum() > 100000
    bh = scene.hit(bounce)
    assert_planes(scene.intersect_device(dev(bounce)), bh, "C3 bounce rays")
    for rays, hits, what in ((cam_rays, first, "camera"), (bounce, bh, "bounce")):
        nan = Q.nan_rays(scene, rays)
        t = dev(rays)
        for md in (hits["dist"], np.nextafter(hits["dist"], np.float32(np.inf)), np.full(len(rays), np.inf, np.float32),
                   np.random.default_rng(1).uniform(0, 50, len(rays)).astype(np.float32)):
            got = scene.occluded_device(t, dev(md)).cpu().numpy()
            assert np.array_equal(got, Q.occluded(hits, nan, md)), what


# ============================================================================== 4. sizes
@pytest.mark.parametrize("n", [1, 31, 33, 2 ** 24 + 5])
def test_sizes(gpu, n):
    import torch
    scene = S.small_mesh_scene(3)
    g = torch.Generator(device="cuda").manual_seed(n)
    o = torch.randn(n, 3, device="cuda", generator=g) * 4.0 + torch.tensor([3.0, 1.0, -10.0], device="cuda")
    d = torch.randn(n, 3, device="cuda", generator=g)
    rays = torch.cat([o, d], 1).contiguous()
    got = scene.intersect_device(rays, passes=("t", "kind", "tri_idx", "normal"))
    host = rays.cpu().numpy()
    hits = scene.hit(host)
    assert_planes(got, hits, f"n={n}")
    occ = scene.occluded_device(rays).cpu().numpy()
    assert np.array_equal(occ, Q.occluded(hits, Q.nan_rays(scene, host), np.full(n, np.inf, np.float32))), n
    if n > 1000:
        assert (hits["kind"] == _abi.HIT_MESH).sum() > n // 50


# ============================================================================== 5. pass subsets, sentinels, streams, stats
def test_pass_subsets_keep_sentinel_bytes(gpu):
    """All seven planes are carved from ONE block filled with a sentinel; a call gets pointers to some of them only.  The others, and the
    gaps between the planes, keep the sentinel."""
    import torch
    scene = mixed_element_scene()
    rays = np.concatenate([R.primary_rays(S.example_camera(24, 20), 1, 0), S.random_rays(500, (0, 4, -9), 5.0, 3)], 0)
    n = len(rays)
    hits = scene.hit(rays)
    comps = {k: 3 if k in ("point", "normal") else 1 for k in PLANES}
    off, o = {}, 0
    for k in PLANES:
        off[k] = o
        o += comps[k] * n + 16
    SENT = 0x7FA5A5A5
    block = torch.empty(o, dtype=torch.int32, device="cuda")
    s = torch.cuda.Stream()
    t = dev(rays)
    lib = _abi.lib()
    for requested in [[k] for k in PLANES] + [["t", "point"], list(PLANES)]:
        block.fill_(SENT)
        torch.cuda.synchronize()
        out = _abi.QueryOutC(**{k: block.data_ptr() + 4 * off[k] for k in requested})
        _abi.check(lib.rbrt_gpu_query_closest_device(scene.handle(), t.data_ptr(), n, out, s.cuda_stream, None))
        s.synchronize()
        b = block.cpu().numpy().view(np.uint32)
        touched = np.zeros(o, bool)
        for k in requested:
            want = bits(hits[k].astype({"kind": np.int32, "elem_idx": np.uint32, "tri_idx": np.uint32}.get(k, np.float32))).ravel()
            assert np.array_equal(b[off[k]:off[k] + comps[k] * n], want), (requested, k)
            touched[off[k]:off[k] + comps[k] * n] = True
        assert (b[~touched] == SENT).all(), f"{requested}: bytes outside the requested planes were written"
    one = scene.intersect_device(t, passes="dist")
    assert set(one) == {"dist"} and np.array_equal(u32(one["dist"]), bits(hits["dist"]))


def test_side_stream_without_stats_does_not_synchronise(gpu):
    import torch
    scene = S.small_mesh_scene(3)
    rays = S.random_rays(4000, (5.0, 1.4, -12.5), 4.0, 1)
    hits = scene.hit(rays)                                                # the scene is built
    t = dev(rays)
    scene.occluded_device(t)                                              # the module is loaded
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        torch.cuda._sleep(int(2e9))                                       # about a second of work ahead of the calls on their stream
        t0 = time.perf_counter()
        got = scene.intersect_device(t, stream=s)
        occ = scene.occluded_device(t, stream=s)
        dt = time.perf_counter() - t0
        busy = not s.query()
    s.synchronize()
    assert busy and dt < 0.3, (busy, dt)
    assert_planes(got, hits, "side stream")
    assert np.array_equal(occ.cpu().numpy(), Q.occluded(hits, Q.nan_rays(scene, rays), np.full(len(rays), np.inf, np.float32)))


def test_stats(gpu):
    scene = S.small_mesh_scene(3)
    rays = S.random_rays(5000, (5.0, 1.4, -12.5), 4.0, 2)
    t = dev(rays)
    for f in (lambda st: scene.intersect_device(t, stats=st), lambda st: scene.occluded_device(t, stats=st)):
        st = {}
        f(st)
        assert st["rays"] == 5000 and st["launches"] == 1 and st["ms_device"] > 0 and st["ms_total"] >= st["ms_device"]
        assert st["nan_rays"] == 0 and st["node_visits"] > 0 and st["tri_tests"] > 0
    ref = {}
    scene.hit(rays, stats=ref)
    st_c, st_o = {}, {}
    scene.intersect_device(t, stats=st_c)
    scene.occluded_device(t, stats=st_o)
    assert st_o["node_visits"] <= st_c["node_visits"]                    # the first occluding triangle ends a traversal
    # a sphere with a NaN centre makes every ray a NaN ray (the reference panics): misses in the closest query, 2 in the occlusion query
    nan_scene = R.Scene(elements=[R.Sphere(R.Vec3(0.0, 0.0, -3.0), 1.0, R.Lambertian(R.Vec3(0.5, 0.5, 0.5))),
                                  R.Sphere(R.Vec3(float("nan"), 0.0, -3.0), 1.0, R.Lambertian(R.Vec3(0.5, 0.5, 0.5)))])
    st = {}
    got = nan_scene.intersect_device(t, stats=st)
    assert st["nan_rays"] == 5000 and (got["kind"].cpu().numpy() == _abi.HIT_NONE).all() and not u32(got["t"]).any()
    st = {}
    assert (nan_scene.occluded_device(t, stats=st).cpu().numpy() == 2).all() and st["nan_rays"] == 5000


# ============================================================================== 6. ordering against updates
def test_ordering_against_a_device_mesh_update(gpu):
    import torch
    scene = S.small_mesh_scene(3)
    rays = np.concatenate([R.primary_rays(S.example_camera(48, 36), 4, 0), S.random_rays(3000, (5.0, 1.4, -12.5), 4.0, 5)], 0)
    old = fresh(scene).hit(rays)
    new = twist(scene.triangle_meshes[0].triangles, 0.8)
    ref_scene = fresh(scene)
    ref_scene.triangle_meshes[0] = R.TriangleMesh.from_triangles(new, ref_scene.triangle_meshes[0].material)
    want_new = ref_scene.hit(rays)
    assert not S.hits_equal(old, want_new).all(), "the deformation must change the hits"
    scene.hit(rays)                                                       # built and in use before the update
    t = dev(rays)
    t_new = torch.from_numpy(new.copy()).cuda()
    torch.cuda.synchronize()
    nan = np.zeros(len(rays), bool)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        torch.cuda._sleep(int(5e8))                                       # the first query waits in the stream while the update is enqueued
        a, oa = scene.intersect_device(t, stream=s), scene.occluded_device(t, stream=s)
        scene.update_mesh_device(0, t_new, stream=s)
        b, ob = scene.intersect_device(t, stream=s), scene.occluded_device(t, stream=s)
    s.synchronize()
    assert_planes(a, old, "before the update")
    assert_planes(b, want_new, "after the update")
    inf = np.full(len(rays), np.inf, np.float32)
    assert np.array_equal(oa.cpu().numpy(), Q.occluded(old, nan, inf)) and np.array_equal(ob.cpu().numpy(), Q.occluded(want_new, nan, inf))


def test_ordering_against_an_element_update(gpu):
    import torch
    scene = mixed_element_scene()
    rays = np.concatenate([R.primary_rays(S.example_camera(48, 36), 4, 0), S.random_rays(3000, (0, 4, -9), 5.0, 6)], 0)
    old = fresh(scene).hit(rays)
    moved = moved_elements(scene.elements, 3)
    ref_scene = fresh(scene)
    ref_scene.elements = list(moved)
    want_new = ref_scene.hit(rays)
    assert not S.hits_equal(old, want_new).all(), "the update must change the hits"
    scene.hit(rays)
    t = dev(rays)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        torch.cuda._sleep(int(5e8))
        a = scene.intersect_device(t, stream=s)
        scene.update_elements(moved)
        b = scene.intersect_device(t, stream=s)
    s.synchronize()
    assert_planes(a, old, "before the update")
    assert_planes(b, want_new, "after the update")


# ============================================================================== 7. communicator, refusals, missing module
def test_emulated_communicator_gives_the_same_answers(gpu):
    rays = S.random_rays(4000, (5.0, 1.4, -12.5), 4.0, 7)
    ref = S.small_mesh_scene(3).hit(rays)
    lib = _abi.lib()
    devs = (C.c_int * 2)(0, 0)
    _abi.check(lib.rbrt_gpu_init_multi(devs, 2, _abi.TRANSPORT_PEER))
    try:
        scene = S.small_mesh_scene(3)
        t = dev(rays)
        assert_planes(scene.intersect_device(t), ref, "under a one-GPU two-rank communicator")
        inf = np.full(len(rays), np.inf, np.float32)
        assert np.array_equal(scene.occluded_device(t).cpu().numpy(), Q.occluded(ref, np.zeros(len(rays), bool), inf))
        scene.close()
    finally:
        _abi.check(lib.rbrt_gpu_comm_destroy())
    R.gpu_init(0)


def test_refusals(gpu):
    import torch
    lib = _abi.lib()
    scene = S.small_mesh_scene(3)
    h = scene.handle()
    rays = dev(S.random_rays(64, (5.0, 1.4, -12.5), 4.0, 1))
    plane = torch.full((64,), 7.0, device="cuda")
    occ = torch.full((64,), 7, dtype=torch.uint8, device="cuda")
    out = _abi.QueryOutC(t=plane.data_ptr())
    closest, occluded = lib.rbrt_gpu_query_closest_device, lib.rbrt_gpu_query_occluded_device
    assert closest(None, rays.data_ptr(), 64, out, None, None) == _abi.E_INVALID
    assert closest(h, None, 64, out, None, None) == _abi.E_INVALID
    assert closest(h, rays.data_ptr(), 64, None, None, None) == _abi.E_INVALID
    assert closest(h, rays.data_ptr(), 64, _abi.QueryOutC(), None, None) == _abi.E_INVALID
    assert closest(h, rays.data_ptr(), 2 ** 32, out, None, None) == _abi.E_INVALID
    host_rays = S.random_rays(64, (5.0, 1.4, -12.5), 4.0, 1)
    assert closest(h, host_rays.ctypes.data, 64, out, None, None) == _abi.E_INVALID          # unregistered host memory
    assert b"device memory" in lib.rbrt_last_error()
    host_plane = np.zeros(64, np.float32)
    assert closest(h, rays.data_ptr(), 64, _abi.QueryOutC(t=host_plane.ctypes.data), None, None) == _abi.E_INVALID
    assert occluded(None, rays.data_ptr(), 64, None, occ.data_ptr(), None, None) == _abi.E_INVALID
    assert occluded(h, None, 64, None, occ.data_ptr(), None, None) == _abi.E_INVALID
    assert occluded(h, rays.data_ptr(), 64, None, None, None, None) == _abi.E_INVALID
    assert occluded(h, rays.data_ptr(), 64, host_plane.ctypes.data, occ.data_ptr(), None, None) == _abi.E_INVALID
    assert occluded(h, rays.data_ptr(), 2 ** 32, None, occ.data_ptr(), None, None) == _abi.E_INVALID
    st = _abi.StatsC(rays=9)
    assert closest(h, rays.data_ptr(), 0, out, None, st) == 0 and st.rays == 0
    torch.cuda.synchronize()
    assert (plane.cpu().numpy() == 7.0).all() and (occ.cpu().numpy() == 7).all() and not host_plane.any()
    with pytest.raises(ValueError):
        scene.intersect_device(rays.cpu())
    with pytest.raises(ValueError):
        scene.intersect_device(rays[:, :5].contiguous())
    with pytest.raises(ValueError):
        scene.intersect_device(rays.t().contiguous().t())                 # not contiguous
    with pytest.raises(ValueError):
        scene.intersect_device(rays, passes=("t", "velocity"))
    with pytest.raises(ValueError):
        scene.occluded_device(rays, max_dist=torch.zeros(63, device="cuda"))
    with pytest.raises(ValueError):
        scene.occluded_device(rays, max_dist=torch.zeros(64, device="cuda", dtype=torch.float64))
    _abi.check(closest(h, rays.data_ptr(), 64, out, None, None))          # the same call, valid
    torch.cuda.synchronize()
    assert not (plane.cpu().numpy() == 7.0).all()


def test_missing_module_is_refused_with_a_message(gpu):
    """Without librbrt_gpu_query.so the calls fail with a message naming the module, and the rest of the library works."""
    code = ("import sys; sys.path.insert(0, %r)\n"
            "import numpy as np, torch, rbrt_b200 as R\nfrom tests import scenes as S\nfrom rbrt_b200 import _abi\n"
            "R.gpu_init(0); sc = S.small_mesh_scene(3); rays = torch.zeros(8, 6, device='cuda')\n"
            "for f in (sc.intersect_device, sc.occluded_device):\n"
            "    try:\n        f(rays)\n        print('NO ERROR')\n"
            "    except _abi.RbrtGpuError as e:\n        print('CODE', e.code, str(e))\n"
            "print('HIT', sc.hit(np.zeros((4, 6), np.float32)).shape)\n") % ROOT
    env = dict(os.environ, RBRT_GPU_QUERY_LIB=os.path.join(ROOT, "no-such-dir", "librbrt_gpu_query.so"))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr
    assert r.stdout.count(f"CODE {_abi.E_CUDA}") == 2 and "query module is missing" in r.stdout, r.stdout
    assert "HIT (4,)" in r.stdout, r.stdout
