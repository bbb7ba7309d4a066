"""Nearest-surface queries on device memory (rbrt_gpu_query_nearest_device; csrc/point.cu, csrc/api.cu) on the GPU.

Every plane is checked bit for bit (uint32 views, so NaN and +-inf compare too) against the brute force of tests/point_ref.py over the
scene's stored geometry: numpy for the small scenes, the same op sequence in torch on the GPU for C3's 1.31 M triangles and the largest
sizes (test_torch_brute_force_equals_numpy pins the two restatements to each other)."""
import ctypes as C
import os
import subprocess
import sys
import time

import numpy as np
import pytest

import rbrt_b200 as R
from rbrt_b200 import _abi
from rbrt_b200.vec3 import Vec3

from . import golden_util as G
from . import point_ref as P
from . import scenes as S
from .test_gpu_trace import mixed_element_scene
from .test_gpu_update import moved_elements, twist

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PT_SO = os.path.join(ROOT, "rbrt_b200", "librbrt_gpu_point.so")
PLANES = ("dist", "kind", "elem_idx", "tri_idx", "point", "normal", "uv")
F = np.float32


@pytest.fixture(scope="module", autouse=True)
def point_module():
    if not os.path.exists(PT_SO):
        subprocess.run(["make", "-C", os.path.join(ROOT, "rbrt_b200", "csrc")], check=True)
    return PT_SO


def u32(t):
    import torch
    return t.contiguous().view(torch.int32).cpu().numpy().view(np.uint32)


def dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, F)).cuda()


def assert_planes(got, want, what):
    n = len(want["dist"])
    for k in got:
        w = np.ascontiguousarray(want[k]).view(np.uint32).reshape(n, -1)
        g = u32(got[k]).reshape(n, -1)
        bad = np.flatnonzero((g != w).any(1))
        assert not len(bad), (f"{what}: plane {k}: {len(bad)} of {n} points differ; first {bad[0]}: got {g[bad[0]]} want {w[bad[0]]} "
                              f"(dist got {u32(got['dist'])[bad[0]].view(F) if 'dist' in got else '-'} want {want['dist'][bad[0]]})")


def check(scene, points, what, max_dist=None, X=P.NP, stats=None):
    cand = P.candidates(scene)
    want = P.nearest(cand, points, max_dist, X=X)
    got = scene.nearest_device(dev(points), max_dist=None if max_dist is None else dev(max_dist), stats=stats)
    assert set(got) == set(PLANES)
    assert_planes(got, want, what)
    return want


def scene_points(scene, n, seed, far=True):
    """Points of four kinds: uniform in the scene box inflated by half its size, on surfaces (candidate points of random triangles and
    spheres), offset from surfaces along their normals by 1e-3 ... 10, and far away (1e3 ... 1e6)."""
    rng = np.random.default_rng(seed)
    cand = P.candidates(scene)
    rec = cand["rec"]
    tri = cand["is_tri"]
    # surface samples
    k = rng.integers(0, len(rec), n)
    a, b = rng.random(n), rng.random(n)
    flip = a + b > 1
    a[flip], b[flip] = 1 - a[flip], 1 - b[flip]
    r = rec[k].astype(np.float64)
    on_tri = r[:, 0, :3] + a[:, None] * r[:, 1, :3] + b[:, None] * r[:, 2, :3]
    dirs = rng.normal(size=(n, 3))
    dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    on_sph = r[:, 0, :3] + np.abs(r[:, 0, 3:4]) * dirs
    on = np.where(tri[k][:, None], on_tri, on_sph)
    nrm = np.where(tri[k][:, None], cand["normal"][k].astype(np.float64), dirs)
    off = on + nrm * (10.0 ** rng.uniform(-3, 1, n))[:, None] * rng.choice([-1, 1], n)[:, None]
    pts = np.concatenate([on, off], 0)
    lo, hi = np.nanmin(pts, 0), np.nanmax(pts, 0)
    lo = np.maximum(lo, -1e4)
    hi = np.minimum(hi, 1e4)
    c, h = (lo + hi) / 2, (hi - lo) * 0.75 + 1e-3
    uni = c + rng.uniform(-1, 1, (n, 3)) * h
    out = [uni, on, off]
    if far:
        fd = rng.normal(size=(n, 3))
        fd /= np.linalg.norm(fd, axis=1, keepdims=True)
        out.append(c + fd * (10.0 ** rng.uniform(3, 6, n))[:, None])
    return np.concatenate(out, 0).astype(F)


# ============================================================================== 1. scenes (golden, C1, C2, C4, elements of both kinds)
SCENES = {"spheres_C1": S.spheres_scene, "small_mesh_C2": S.small_mesh_scene, "stress_C4": S.stress_scene, "mixed_elements": mixed_element_scene,
          "quirk": S.quirk_scene}


@pytest.mark.parametrize("name", G.NAMES)
def test_golden_scenes(gpu, name):
    _, scene, _ = G.load(name)
    want = check(scene, scene_points(scene, 1500, 1), name)
    assert (want["kind"] != P.HIT_NONE).all()


@pytest.mark.parametrize("name", list(SCENES))
def test_scenes(gpu, name):
    scene = SCENES[name]()
    X = P.TORCH if name == "stress_C4" else P.NP
    want = check(scene, scene_points(scene, 2000, 2), name, X=X)
    kinds = set(np.unique(want["kind"]).tolist())
    assert P.HIT_NONE not in kinds and (P.HIT_MESH in kinds or not scene.triangle_meshes)
    if name == "mixed_elements":
        assert kinds == {P.HIT_SPHERE, P.HIT_MESH, P.HIT_TRIANGLE}


def test_torch_brute_force_equals_numpy(gpu):
    scene = mixed_element_scene()
    pts = scene_points(scene, 500, 3)
    cand = P.candidates(scene)
    a, b = P.nearest(cand, pts), P.nearest(cand, pts, X=P.TORCH)
    for k in PLANES:
        assert np.array_equal(np.ascontiguousarray(a[k]).view(np.uint32), np.ascontiguousarray(b[k]).view(np.uint32)), k


# ============================================================================== 2. exact ties
def test_exact_ties(gpu):
    """Equal d2 from two spheres, from two coincident triangles in one mesh and from one triangle in two meshes: the first in scene order
    wins (the lower element index, the lower original index, the earlier mesh)."""
    mat = R.Lambertian(Vec3(0.5, 0.5, 0.5))
    tri = np.array([[(0, 0, 10), (1, 0, 10), (0, 1, 10)]], F)
    other = np.array([[(5, 5, 5), (6, 5, 5), (5, 6, 5)]], F)
    scene = R.Scene(elements=[R.Sphere(Vec3(-4.0, 0.0, 0.0), 1.0, mat), R.Sphere(Vec3(4.0, 0.0, 0.0), 1.0, mat)],
                    triangle_meshes=[R.TriangleMesh.from_triangles(np.concatenate([other, tri, other, tri] + [other] * 4), mat),
                                     R.TriangleMesh.from_triangles(np.concatenate([tri] + [other] * 7), mat)], leaf_size=1)
    pts = np.array([(0.0, 0.0, 0.0), (0.0, 3.0, 0.0), (0.0, -3.0, 0.0), (0.25, 0.25, 12.0), (0.2, 0.3, 9.0), (0.0, 0.0, 11.0)], F)
    want = check(scene, pts, "ties")
    got = {k: want[k] for k in ("kind", "elem_idx", "tri_idx")}
    for i in (0, 1, 2):                                                        # on the plane x = 0 both spheres are equally near
        assert got["kind"][i] == P.HIT_SPHERE and got["elem_idx"][i] == 0, (i, got)
    for i in (3, 4, 5):                                                        # the coincident triangles 1 and 3 of mesh 0, and mesh 1's copy
        assert got["kind"][i] == P.HIT_MESH and got["elem_idx"][i] == 0 and got["tri_idx"][i] == 1, (i, got)


def test_ties_across_slots(gpu):
    """Two mirror images of one triangle about the plane z = 0 are exactly equidistant from every point on that plane.  The Morton order
    puts the z = -1 copy (original index 1) in the lower slot; the winner is original index 0 whatever the slots."""
    mat = R.Lambertian(Vec3(0.5, 0.5, 0.5))
    t = np.array([(0.0, 0.0, 1.0), (1.0, 0.0, 1.0), (0.0, 1.0, 1.0)], F)
    m = t * np.array([1, 1, -1], F)
    far = [t + np.array([40.0 + 3 * k, 0, 0], F) for k in range(6)]
    for leaf in (1, 8):
        scene = R.Scene(triangle_meshes=[R.TriangleMesh.from_triangles(np.stack([t, m] + far), mat)], leaf_size=leaf)
        pts = np.array([(0.0, 0.0, 0.0), (0.2, 0.3, 0.0), (-1.0, 0.5, 0.0), (2.0, 2.0, 0.0), (0.5, -3.0, 0.0)], F)
        want = check(scene, pts, f"mirror tie leaf {leaf}")
        assert (want["kind"] == P.HIT_MESH).all() and (want["tri_idx"] == 0).all(), want["tri_idx"]


def test_prune_slack_covers_the_rounding_of_a_vertex(gpu):
    """The computed vertex v0 + e1 of a triangle can lie an ulp outside the mesh's exact box (e1 = b - a is rounded).  A point just beyond
    it is then nearer to the triangle than to the box (d2 < box bound).  A point element placed so that its d2 lies between the two makes
    the mesh's pre-test decide: without the prune slack of point.cuh the mesh would be skipped and the element reported."""
    ax, bx = F(0.15260756), F(-3.3237813)
    assert F(ax + F(bx - ax)) < bx
    a, b, c = np.array([ax, 0, 0], F), np.array([bx, 0.5, 0], F), np.array([ax, 1, 0], F)
    tri = np.stack([a, b, c])
    tris = np.stack([tri] + [tri + np.array([0, 10.0 + k, 0], F) for k in range(7)]).astype(F)
    p = np.array([F(bx - F(1e-6)), 0.5, 0.0], F)
    elem = (float(p[0]), 0.5, 8.5e-7)
    scene = R.Scene(elements=[R.Sphere(Vec3(*elem), 0.0, R.Lambertian(Vec3(0.5, 0.5, 0.5)))],
                    triangle_meshes=[R.TriangleMesh.from_triangles(tris, R.Lambertian(Vec3(0.5, 0.5, 0.5)))])
    cand = P.candidates(scene)
    d2 = P._pair_d2(P.NP, p[None], cand["rec"], cand["is_tri"])[0]
    box = np.float32(max(F(tris[:, :, 0].min() - p[0]), F(0))) ** 2
    assert d2[1] < d2[0] < box, (d2[:2], box)                                 # triangle < element < the mesh box's bound
    want = check(scene, p[None], "vertex outside the box")
    assert want["kind"][0] == P.HIT_MESH and want["tri_idx"][0] == 0


# ============================================================================== 3. C3 at full size
def test_c3_full_size(gpu):
    scene, _ = S.big_scene(8)
    pts = scene_points(scene, 1024, 4)                                         # 4 096 points: uniform, on, off the surface, far
    want = check(scene, pts, "C3", X=P.TORCH)
    assert len(pts) >= 4096 and (want["kind"] == P.HIT_MESH).sum() > 2000
    # on the surface a point tests a handful of triangles, four orders of magnitude below the brute force's 1.31 M (points deep inside
    # the sphere, nearly equidistant from all of it, and points 1e3 ... 1e6 away, whose prune slack grows with |p|, test far more)
    n_tris = scene.info()["num_triangles_tested"]
    st = {}
    scene.nearest_device(dev(pts[1024:2048]), stats=st)
    assert st["rays"] == 1024 and st["tri_tests"] / 1024 < n_tris * 1e-4, st
    sub = pts[::128]                                                           # the numpy restatement itself on a subset
    assert_planes(scene.nearest_device(dev(sub)), P.nearest(P.candidates(scene), sub), "C3 numpy subset")


# ============================================================================== 4. the tree does not matter
@pytest.mark.parametrize("leaf", [1, 2, 4, 8])
@pytest.mark.parametrize("sah", [True, False])
def test_tree_independence_refit_and_rebuild(gpu, leaf, sah):
    scene = S.small_mesh_scene(3, leaf_size=leaf, sah=sah)
    pts = scene_points(scene, 800, 5)
    base = check(scene, pts, f"leaf {leaf} sah {sah}")
    ref = S.small_mesh_scene(3)
    assert_planes(ref.nearest_device(dev(pts)), base, "another tree, the same answers")
    new = twist(scene.triangle_meshes[0].triangles, 0.7)
    scene.update_mesh_device(0, dev(new))
    check(scene, pts, "after a refit")
    scene.update_mesh(0, twist(new, -0.3), rebuild=True)
    check(scene, pts, "after a rebuild")


# ============================================================================== 5. extreme extents
EXTENTS = [(3e11, 0), (1e12, 0), (1e20, 0), (2e38, 0), (np.inf, 0), (1e12, 1), (-np.inf, 1), (1e11, 2)]


@pytest.mark.parametrize("far,axis", EXTENTS)
def test_extreme_extents(gpu, far, axis):
    scene = S.spheres_scene(leaf_size=2)
    scene.triangle_meshes.append(R.TriangleMesh.from_triangles(S.far_triangle_mesh(far, axis), R.Lambertian(Vec3(0.6, 0.5, 0.4))))
    pts = scene_points(S.small_mesh_scene(3), 600, 6)
    want = check(scene, pts, f"far {far:g} axis {axis}")
    assert (want["kind"] == P.HIT_MESH).sum() > 300


def test_qstep_nan_axis_contributes_nothing(gpu):
    """A mesh whose x extent (1e12) gives a grid step above RBRT_QSTEP_MAX: the step is NaN, the x axis adds 0 to every box bound, and the
    query still finds the icosphere's triangles exactly (a NaN bound that rejected boxes would lose them).  (The far triangle also sets the
    mesh's coordinate scale, and with it a prune slack of ~1e7: here every point tests every triangle, DESIGN.md section 17.)"""
    tris = S.far_triangle_mesh(1e12, 0)
    ext = tris.reshape(-1, 3).max(0) - tris.reshape(-1, 3).min(0)
    assert ext[0] / 65500 > 2e6
    scene = R.Scene(triangle_meshes=[R.TriangleMesh.from_triangles(tris, R.Lambertian(Vec3(0.5, 0.5, 0.5)))], leaf_size=1)
    pts = scene_points(S.small_mesh_scene(3), 800, 7, far=False)
    want = check(scene, pts, "qstep NaN")
    assert (want["kind"] == P.HIT_MESH).all()


def test_tiny_mesh_and_mesh_far_from_the_origin(gpu):
    base = S.far_triangle_mesh(1.0, 0)
    c = base.reshape(-1, 3).mean(0)
    tiny = ((base - c) * F(1e-4) + c).astype(F)
    far_mesh = (base + F(3e5)).astype(F)
    rng = np.random.default_rng(8)
    near_tiny = np.concatenate([c + rng.normal(0, 50, (500, 3)), c + rng.normal(0, 1e-4, (500, 3))]).astype(F)
    near_far = (far_mesh.reshape(-1, 3)[::4] + rng.normal(0, 0.5, (len(far_mesh.reshape(-1, 3)[::4]), 3))).astype(F)
    for tris, pts, what in ((tiny, near_tiny, "points far from and near a tiny mesh"), (far_mesh, near_far, "near a mesh at 3e5")):
        for leaf in (1, 8):
            scene = R.Scene(triangle_meshes=[R.TriangleMesh.from_triangles(tris, R.Lambertian(Vec3(0.5, 0.5, 0.5)))], leaf_size=leaf)
            want = check(scene, pts, f"{what} leaf {leaf}")
            assert (want["kind"] == P.HIT_MESH).all()


# ============================================================================== 6. max_dist
def test_max_dist(gpu):
    scene = mixed_element_scene()
    pts = scene_points(scene, 1000, 11)
    cand = P.candidates(scene)
    free = P.nearest(cand, pts)
    n = len(pts)
    rng = np.random.default_rng(12)
    exact = free["dist"].copy()
    variants = {"equal to the distance (strict: rejected)": exact,
                "just above": np.nextafter(exact, F(np.inf)).astype(F),
                "random": rng.uniform(0, 5, n).astype(F),
                "specials": np.array([0.0, -0.0, -1.0, np.nan, np.inf, 1e-30], F)[rng.integers(0, 6, n)]}
    for what, md in variants.items():
        want = check(scene, pts, what, max_dist=md)
        if what.startswith("equal"):
            # the winner within a strict bound equal to the free winner's distance has a smaller distance, or there is none
            assert (want["dist"] < exact)[want["kind"] != P.HIT_NONE].all()
        if what == "just above":
            assert np.array_equal(want["which"], free["which"])
        if what == "specials":
            none = ~(variants[what] > 0)
            assert (want["kind"][none] == P.HIT_NONE).all() and np.isinf(want["dist"][none]).all()


# ============================================================================== 7. sizes, special points, pass subsets
@pytest.mark.parametrize("n", [1, 31, 33, 2 ** 24 + 5])
def test_sizes(gpu, n):
    import torch
    scene = S.small_mesh_scene(3, n_keep=60)                                    # 60 triangles, all tested, + 4 spheres
    g = torch.Generator(device="cuda").manual_seed(n)
    pts = (torch.randn(n, 3, device="cuda", generator=g) * 5.0 + torch.tensor([3.0, 1.0, -10.0], device="cuda")).contiguous()
    got = scene.nearest_device(pts, passes=("dist", "kind", "tri_idx", "uv"))
    want = P.nearest(P.candidates(scene), pts.cpu().numpy(), X=P.TORCH)
    assert_planes(got, want, f"n={n}")


def test_nan_and_inf_points(gpu):
    scene = S.small_mesh_scene(3)
    pts = scene_points(scene, 200, 13)
    pts[::7, 0] = np.nan
    pts[1::7, 1] = np.inf
    pts[2::7, 2] = -np.inf
    st = {}
    want = check(scene, pts, "NaN and inf points", stats=st)
    assert st["nan_rays"] == np.isnan(pts).any(1).sum()
    assert (want["kind"][~np.isfinite(pts).all(1)] == P.HIT_NONE).all()
    assert st["rays"] == len(pts) and st["launches"] == 1 and st["ms_device"] > 0 and st["ms_total"] >= st["ms_device"]


def test_pass_subsets_keep_sentinel_bytes(gpu):
    import torch
    scene = mixed_element_scene()
    pts = scene_points(scene, 300, 14)
    n = len(pts)
    want = P.nearest(P.candidates(scene), pts)
    comps = {"point": 3, "normal": 3, "uv": 2}
    off, o = {}, 0
    for k in PLANES:
        off[k] = o
        o += comps.get(k, 1) * n + 16
    SENT = 0x7FA5A5A5
    block = torch.empty(o, dtype=torch.int32, device="cuda")
    s = torch.cuda.Stream()
    t = dev(pts)
    lib = _abi.lib()
    for requested in [[k] for k in PLANES] + [["dist", "uv"], list(PLANES)]:
        block.fill_(SENT)
        torch.cuda.synchronize()
        out = _abi.NearestOutC(**{k: block.data_ptr() + 4 * off[k] for k in requested})
        _abi.check(lib.rbrt_gpu_query_nearest_device(scene.handle(), t.data_ptr(), n, None, out, s.cuda_stream, None))
        s.synchronize()
        b = block.cpu().numpy().view(np.uint32)
        touched = np.zeros(o, bool)
        for k in requested:
            w = np.ascontiguousarray(want[k]).view(np.uint32).ravel()
            assert np.array_equal(b[off[k]:off[k] + comps.get(k, 1) * n], w), (requested, k)
            touched[off[k]:off[k] + comps.get(k, 1) * n] = True
        assert (b[~touched] == SENT).all(), f"{requested}: bytes outside the requested planes were written"


# ============================================================================== 8. ordering against updates, streams, the cache
def test_ordering_against_a_device_mesh_update(gpu):
    import torch
    scene = S.small_mesh_scene(3)
    pts = scene_points(scene, 500, 15)
    old = P.nearest(P.candidates(scene), pts)
    new = twist(scene.triangle_meshes[0].triangles, 0.8)
    t, t_new = dev(pts), torch.from_numpy(new.copy()).cuda()
    scene.nearest_device(t)
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        torch.cuda._sleep(int(5e8))
        a = scene.nearest_device(t, stream=s)
        scene.update_mesh_device(0, t_new, stream=s)
        b = scene.nearest_device(t, stream=s)
    s.synchronize()
    assert_planes(a, old, "before the update")
    want_new = P.nearest(P.candidates(scene), pts)
    assert not np.array_equal(want_new["dist"], old["dist"])
    assert_planes(b, want_new, "after the update")


def test_ordering_against_an_element_update_and_release_cache(gpu):
    import torch
    scene = mixed_element_scene()
    pts = scene_points(scene, 500, 16)
    old = P.nearest(P.candidates(scene), pts)
    moved = moved_elements(scene.elements, 3)
    t = dev(pts)
    scene.nearest_device(t)
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        torch.cuda._sleep(int(5e8))
        a = scene.nearest_device(t, stream=s)
        scene.update_elements(moved)
        b = scene.nearest_device(t, stream=s)
    s.synchronize()
    assert_planes(a, old, "before the element update")
    want_new = P.nearest(P.candidates(scene), pts)
    assert_planes(b, want_new, "after the element update")
    _abi.check(_abi.lib().rbrt_gpu_release_cache())
    assert_planes(scene.nearest_device(t), want_new, "after rbrt_gpu_release_cache")


def test_side_stream_without_stats_does_not_synchronise(gpu):
    import torch
    scene = S.small_mesh_scene(3)
    pts = scene_points(scene, 1000, 17)
    t = dev(pts)
    want = P.nearest(P.candidates(scene), pts)
    scene.nearest_device(t)
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        torch.cuda._sleep(int(2e9))
        t0 = time.perf_counter()
        got = scene.nearest_device(t, stream=s)
        dt = time.perf_counter() - t0
        busy = not s.query()
    s.synchronize()
    assert busy and dt < 0.3, (busy, dt)
    assert_planes(got, want, "side stream")


# ============================================================================== 9. communicator, refusals, missing module
def test_emulated_communicator_gives_the_same_answers(gpu):
    pts = scene_points(S.small_mesh_scene(3), 500, 18)
    want = P.nearest(P.candidates(S.small_mesh_scene(3)), pts)
    lib = _abi.lib()
    devs = (C.c_int * 2)(0, 0)
    _abi.check(lib.rbrt_gpu_init_multi(devs, 2, _abi.TRANSPORT_PEER))
    try:
        scene = S.small_mesh_scene(3)
        assert_planes(scene.nearest_device(dev(pts)), want, "under a one-GPU two-rank communicator")
        scene.close()
    finally:
        _abi.check(lib.rbrt_gpu_comm_destroy())
    R.gpu_init(0)


def test_refusals(gpu):
    import torch
    lib = _abi.lib()
    scene = S.small_mesh_scene(3)
    h = scene.handle()
    pts = dev(scene_points(scene, 16, 19))                                      # 64 points
    n = pts.shape[0]
    plane = torch.full((n,), 7.0, device="cuda")
    out = _abi.NearestOutC(dist=plane.data_ptr())
    f = lib.rbrt_gpu_query_nearest_device
    assert f(None, pts.data_ptr(), n, None, out, None, None) == _abi.E_INVALID
    assert f(h, None, n, None, out, None, None) == _abi.E_INVALID
    assert f(h, pts.data_ptr(), n, None, None, None, None) == _abi.E_INVALID
    assert f(h, pts.data_ptr(), n, None, _abi.NearestOutC(), None, None) == _abi.E_INVALID
    assert f(h, pts.data_ptr(), 2 ** 32, None, out, None, None) == _abi.E_INVALID
    host_pts = pts.cpu().numpy()
    assert f(h, host_pts.ctypes.data, n, None, out, None, None) == _abi.E_INVALID
    assert b"device memory" in lib.rbrt_last_error()
    host_plane = np.zeros(n, F)
    assert f(h, pts.data_ptr(), n, host_plane.ctypes.data, out, None, None) == _abi.E_INVALID
    assert f(h, pts.data_ptr(), n, None, _abi.NearestOutC(uv=host_plane.ctypes.data), None, None) == _abi.E_INVALID
    st = _abi.StatsC(rays=9)
    assert f(h, pts.data_ptr(), 0, None, out, None, st) == 0 and st.rays == 0
    torch.cuda.synchronize()
    assert (plane.cpu().numpy() == 7.0).all() and not host_plane.any()
    for bad in (pts.cpu(), pts[:, :2].contiguous(), pts.t().contiguous().t(), pts.double()):
        with pytest.raises(ValueError):
            scene.nearest_device(bad)
    with pytest.raises(ValueError):
        scene.nearest_device(pts, passes=("dist", "velocity"))
    with pytest.raises(ValueError):
        scene.nearest_device(pts, max_dist=torch.zeros(n - 1, device="cuda"))
    with pytest.raises(ValueError):
        scene.nearest_device(pts, max_dist=torch.zeros(n, device="cuda", dtype=torch.float64))
    _abi.check(f(h, pts.data_ptr(), n, None, out, None, None))
    torch.cuda.synchronize()
    assert not (plane.cpu().numpy() == 7.0).all()


def test_missing_module_is_refused_with_a_message(gpu):
    code = ("import sys; sys.path.insert(0, %r)\n"
            "import numpy as np, torch, rbrt_b200 as R\nfrom tests import scenes as S\nfrom rbrt_b200 import _abi\n"
            "R.gpu_init(0); sc = S.small_mesh_scene(3); pts = torch.zeros(8, 3, device='cuda')\n"
            "try:\n    sc.nearest_device(pts)\n    print('NO ERROR')\n"
            "except _abi.RbrtGpuError as e:\n    print('CODE', e.code, str(e))\n"
            "print('HIT', sc.hit(np.zeros((4, 6), np.float32)).shape)\n") % ROOT
    env = dict(os.environ, RBRT_GPU_POINT_LIB=os.path.join(ROOT, "no-such-dir", "librbrt_gpu_point.so"))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr
    assert f"CODE {_abi.E_CUDA}" in r.stdout and "nearest-surface module is missing" in r.stdout, r.stdout
    assert "HIT (4,)" in r.stdout, r.stdout
