"""Winding numbers on device memory (rbrt_gpu_query_winding_device, Scene.winding_device, Scene.signed_distance_device; csrc/wind.cu,
csrc/api.cu) on the GPU.

The reference is the exact float64 sum of tests/winding_ref.py over the scene's stored candidates: numpy for the small scenes, the same
code on CUDA float64 tensors for C4 and C3's 1.31 M triangles.  beta = +inf (the exact sum in the kernel: f32 terms, f64 sum) and the
default beta = 2 (the far-field expansion) each have a pinned bound on |w - w64|, measured on an NVIDIA B200 and kept with a margin.
Points on a surface are ill-conditioned (rounding decides which side of a triangle's plane they lie on, a jump of up to 1 in w): there
only |w - w64| <= 1 + the pin is required."""
import ctypes as C
import os
import subprocess
import sys
import time

import numpy as np
import pytest

import rbrt_b200 as R
from rbrt_b200 import _abi, synth
from rbrt_b200.vec3 import Vec3

from . import golden_util as G
from . import point_ref as P
from . import scenes as S
from . import winding_ref as W
from .motion_ref import tri_records
from .test_gpu_extents import CASES as EXTENT_CASES
from .test_gpu_point import dev, scene_points
from .test_gpu_trace import mixed_element_scene
from .test_gpu_update import moved_elements, twist

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WD_SO = os.path.join(ROOT, "rbrt_b200", "librbrt_gpu_wind.so")
F = np.float32
INF = float("inf")
# Largest |w - w64| off the surfaces, beta = +inf and beta = 2 (measured: 4.8e-4, on the quirk scene, and 0.063).
EXACT_PIN = 1e-3
BETA2_PIN = 0.1
# test_error_falls_with_beta: the largest |w - w64| off the surfaces by scene and beta (measured: C2 0.058, 0.0126, 0.0031; the soup
# 0.0113, 0.00138, 9.9e-5; without the parallel-axis shift of the merge the soup gives 0.027, 0.0037, 5.1e-4).
BETA_PINS = {"C2": {2.0: BETA2_PIN, 4.0: 0.02, 8.0: 0.005}, "soup": {2.0: 0.017, 4.0: 0.002, 8.0: 1.5e-4}}
# Classification is checked where ||w64| - 0.5| exceeds this.
CLASS_MARGIN = BETA2_PIN


@pytest.fixture(scope="module", autouse=True)
def wind_module():
    if not os.path.exists(WD_SO):
        subprocess.run(["make", "-C", os.path.join(ROOT, "rbrt_b200", "csrc")], check=True)
    return WD_SO


def wind(scene, pts, beta=None, stats=None, stream=None):
    got = scene.winding_device(dev(pts) if isinstance(pts, np.ndarray) else pts, beta=beta, stats=stats, stream=stream)
    return got["winding"].cpu().numpy(), got["inside"].cpu().numpy()


def off_surface(n_pts):
    """scene_points' kinds (uniform, on, offset, far), n each: a mask of the points not on a surface."""
    m = np.ones(n_pts, bool)
    n = n_pts // 4
    m[n:2 * n] = False
    return m


def check(scene, pts, what, beta=None, X=W.NP, on=None, pin=None):
    """w and inside against the float64 reference; returns (w, inside, w64)."""
    w64 = W.winding(P.candidates(scene), pts, X=X)
    w, ins = wind(scene, pts, beta)
    pin = pin or (EXACT_PIN if beta == INF else BETA2_PIN)
    nan = np.isnan(pts).any(1)
    assert np.isnan(w[nan]).all() and not ins[nan].any()
    ok = ~nan
    err = np.abs(w[ok].astype(np.float64) - w64[ok])
    off = np.ones(len(pts), bool) if on is None else ~on
    e_off = np.abs(w.astype(np.float64) - w64)[off & ok]
    print(f"{what} beta {beta}: max |w - w64| {e_off.max() if len(e_off) else 0:.3g} off the surface, {err.max():.3g} overall")
    assert (e_off <= pin).all(), f"{what}: max |w - w64| {e_off.max():g} > {pin:g} at {pts[off & ok][e_off.argmax()]}"
    assert (err <= 1.0 + pin).all(), f"{what}: on-surface |w - w64| {err.max():g}"
    assert np.array_equal(ins.astype(bool), np.abs(w) > 0.5)
    sure = ok & off & (np.abs(np.abs(w64) - 0.5) > max(pin, CLASS_MARGIN if beta != INF else pin))
    assert np.array_equal(ins[sure].astype(bool), np.abs(w64[sure]) > 0.5), what
    return w, ins, w64


def pts_of(scene, n, seed, far=True):
    pts = scene_points(scene, n, seed, far=far)
    return pts, ~off_surface(len(pts)) if far else np.r_[np.zeros(n, bool), np.ones(n, bool), np.zeros(n, bool)]


# ============================================================================== 1. scenes, beta = +inf and beta = 2
SCENES = {"spheres_C1": S.spheres_scene, "small_mesh_C2": S.small_mesh_scene, "stress_C4": S.stress_scene, "mixed_elements": mixed_element_scene,
          "quirk": S.quirk_scene}


@pytest.mark.parametrize("beta", [INF, None])
@pytest.mark.parametrize("name", G.NAMES)
def test_golden_scenes(gpu, name, beta):
    _, scene, _ = G.load(name)
    pts, on = pts_of(scene, 800, 1)
    check(scene, pts, name, beta, on=on)


@pytest.mark.parametrize("beta", [INF, None])
@pytest.mark.parametrize("name", list(SCENES))
def test_scenes(gpu, name, beta):
    scene = SCENES[name]()
    pts, on = pts_of(scene, 1500, 2)
    check(scene, pts, name, beta, X=W.TORCH if name == "stress_C4" else W.NP, on=on)


def test_c3_full_size(gpu):
    """C3 (1.31 M triangles, radius 40) on 4 096 points against the float64 brute force, both betas; points offset by >= 1e-3 of the
    radius along the normals classify as intended."""
    scene, _ = S.big_scene(8)
    pts, on = pts_of(scene, 1024, 4)
    for beta in (INF, None):
        w, ins, w64 = check(scene, pts, "C3", beta, X=W.TORCH, on=on)
    st = {}
    scene.winding_device(dev(pts[1024:2048]), stats=st)
    n_tris = scene.info()["num_triangles_tested"]
    print("C3 beta 2 near the surface, per point:", st["node_visits"] / 1024, "node visits,", st["tri_tests"] / 1024, "triangle terms")
    assert st["rays"] == 1024 and st["tri_tests"] / 1024 < n_tris * 1e-2, st
    # offsets along the normals of random surface points, by 1e-3 ... 1 times the radius, in and out
    rng = np.random.default_rng(40)
    cand = P.candidates(scene)
    k = rng.integers(len(scene.elements), len(cand["rec"]), 2048)
    r = cand["rec"][k].astype(np.float64)
    q = r[:, 0, :3] + (r[:, 1, :3] + r[:, 2, :3]) / 3
    h = 40.0 * 10.0 ** rng.uniform(-3, -1, len(k))
    sign = rng.choice([-1.0, 1.0], len(k))
    p = (q + cand["normal"][k] * (sign * h)[:, None]).astype(F)
    w, ins, w64 = check(scene, p, "C3 offsets", None, X=W.TORCH)
    intended = (sign < 0)
    in_spheres = W.winding({"rec": cand["rec"][:len(scene.elements)], "is_tri": cand["is_tri"][:len(scene.elements)]}, p) != 0
    sel = ~in_spheres
    agree = (np.abs(w64) > 0.5) == intended
    assert agree[sel].mean() > 0.999                                       # (a few offsets near a concave edge cross a neighbour)
    assert np.array_equal(ins[sel & agree].astype(bool), intended[sel & agree])


def test_error_falls_with_beta(gpu):
    """The expansion's error off the surfaces at beta = 2, 4, 8 on C2 and on a soup of randomly oriented triangles, each below its pin.
    The soup is what the T term of a merged subtree matters for: on a smooth surface the children's normals are nearly parallel and the
    parallel-axis shift N_k (x) (c_k - c) nearly cancels, in a soup it does not."""
    rng = np.random.default_rng(42)
    soup = (rng.uniform(-3, 3, (3000, 1, 3)) + rng.normal(0, 0.4, (3000, 3, 3))).astype(F)
    scenes = {"C2": S.small_mesh_scene(3), "soup": R.Scene(triangle_meshes=[R.TriangleMesh.from_triangles(soup, MAT)])}
    for name, scene in scenes.items():
        pts, on = pts_of(scene, 1000, 41)
        w64 = W.winding(P.candidates(scene), pts)
        errs = {}
        for beta in (2.0, 4.0, 8.0):
            w, _ = wind(scene, pts, beta)
            errs[beta] = float(np.abs(w.astype(np.float64) - w64)[~on].max())
        print(f"{name}: max |w - w64| off the surface by beta:", errs)
        for beta, pin in BETA_PINS[name].items():
            assert errs[beta] <= pin, (name, errs)


# ============================================================================== 2. structure
MAT = R.Lambertian(Vec3(0.5, 0.5, 0.5))


def ico(subdiv=3, r=3.0, c=(0.0, 0.0, 0.0)):
    return synth.displaced_icosphere(subdiv, r, c, amplitude=0.0)


def test_nesting_open_surface_and_inward_faces(gpu):
    """A point inside a sphere inside a mesh: w = 2.  An open hemisphere: fractional w, against float64.  An inward-facing copy of a
    mesh: w = -1 inside, and inside = 1 all the same."""
    tris = ico()
    nested = R.Scene(elements=[R.Sphere(Vec3(0.0, 0.0, 0.0), 1.0, MAT)], triangle_meshes=[R.TriangleMesh.from_triangles(tris, MAT)])
    w, ins, _ = check(nested, np.array([(0.1, 0.2, -0.1), (2.0, 0.0, 0.0), (9.0, 0.0, 0.0)], F), "nested", INF)
    assert np.allclose(w, [2.0, 1.0, 0.0], atol=1e-4) and ins.tolist() == [1, 1, 0]
    top = tris[tris[:, :, 2].mean(1) > 0]
    hemi = R.Scene(triangle_meshes=[R.TriangleMesh.from_triangles(top, MAT)])
    pts = np.random.default_rng(9).uniform(-4, 4, (2000, 3)).astype(F)
    for beta in (INF, None):
        w, _, w64 = check(hemi, pts, "hemisphere", beta)
    assert ((np.abs(w64) > 0.05) & (np.abs(w64) < 0.95)).mean() > 0.1
    inward = R.Scene(triangle_meshes=[R.TriangleMesh.from_triangles(tris[:, ::-1].copy(), MAT)])
    for beta in (INF, None):
        w, ins, _ = check(inward, np.array([(0.0, 0.5, 0.0), (5.0, 0.0, 0.0)], F), "inward", beta)
        assert np.allclose(w, [-1.0, 0.0], atol=EXACT_PIN if beta == INF else BETA2_PIN) and ins.tolist() == [1, 0]


def test_tail_dropped_triangles_are_not_candidates(gpu):
    """simd_lanes = 4 with a mesh of 4k + 1 triangles: the last one is not tested, and w follows the tested ones only."""
    tris = ico()[:-3]                                                      # 1277 = 4 * 319 + 1: one dropped
    assert P.n_tested(len(tris), 4) == len(tris) - 1
    scene = R.Scene(triangle_meshes=[R.TriangleMesh.from_triangles(tris, MAT)], simd_lanes=4)
    assert scene.info()["num_triangles_tested"] == len(tris) - 1
    dropped = tris[-1].astype(np.float64)
    c = dropped.mean(0)
    pts = (c + np.random.default_rng(10).normal(0, 0.2, (500, 3))).astype(F)
    w, _, w64 = check(scene, pts, "lanes 4", INF)
    full = W.winding({"rec": tri_records(tris), "is_tri": np.ones(len(tris), bool)}, pts)
    assert np.abs(full - w64).max() > 0.1                                  # the dropped triangle matters to these points


# ============================================================================== 3. trees, refit, rebuild, extents
@pytest.mark.parametrize("leaf", [1, 2, 4, 8])
@pytest.mark.parametrize("sah", [True, False])
def test_trees_refit_and_rebuild(gpu, leaf, sah):
    scene = S.small_mesh_scene(3, leaf_size=leaf, sah=sah)
    pts, on = pts_of(scene, 600, 5)
    check(scene, pts, f"leaf {leaf} sah {sah}", None, on=on)
    new = twist(scene.triangle_meshes[0].triangles, 0.7)
    scene.update_mesh_device(0, dev(new))
    check(scene, pts, "after a refit", None, on=on)
    scene.update_mesh(0, twist(new, -0.3), rebuild=True)
    check(scene, pts, "after a rebuild", None, on=on)


@pytest.mark.parametrize("rebuild", [False, True])
def test_translated_mesh_inside_set_follows(gpu, rebuild):
    """After an update that moves a closed mesh by 10, the points inside it are those of the moved mesh: the moments were recomputed."""
    tris = ico(3, 3.0, (0.0, 0.0, 0.0))
    scene = R.Scene(triangle_meshes=[R.TriangleMesh.from_triangles(tris, MAT)])
    pts = np.random.default_rng(11).uniform(-5, 15, (4000, 3)).astype(F)
    _, ins0 = wind(scene, pts)
    moved = (tris + F(10.0)).astype(F)
    if rebuild:
        scene.update_mesh(0, moved, rebuild=True)
    else:
        scene.update_mesh_device(0, dev(moved))
    _, ins1 = wind(scene, pts)
    c0 = np.linalg.norm(pts, axis=1) < 2.9
    c1 = np.linalg.norm(pts - 10.0, axis=1) < 2.9
    assert ins0[c0].all() and not ins0[c1].any() and ins1[c1].all() and not ins1[c0].any()
    check(scene, pts, "moved", None)


@pytest.mark.parametrize("far,axis", EXTENT_CASES)
def test_extreme_extents(gpu, far, axis):
    """The meshes of tests/test_gpu_extents.py: the icosphere plus one small triangle at coordinate `far` (1e12 on x gives a NaN grid
    step: the moments never read the node boxes)."""
    scene = R.Scene(triangle_meshes=[R.TriangleMesh.from_triangles(S.far_triangle_mesh(far, axis), MAT)], leaf_size=2)
    pts, on = pts_of(S.small_mesh_scene(3), 400, 6, far=False)
    for beta in (INF, None):
        check(scene, pts, f"far {far:g} axis {axis}", beta, on=on)


# ============================================================================== 4. sizes and inputs
@pytest.mark.parametrize("n", [1, 31, 33, 2 ** 24 + 5])
def test_sizes(gpu, n):
    import torch
    scene = S.small_mesh_scene(3, n_keep=60)
    g = torch.Generator(device="cuda").manual_seed(n)
    pts = (torch.randn(n, 3, device="cuda", generator=g) * 5.0 + torch.tensor([5.0, 1.4, -12.5], device="cuda")).contiguous()
    w, ins = wind(scene, pts, INF)
    idx = np.unique(np.r_[np.arange(min(n, 4096)), np.random.default_rng(n).integers(0, n, 4096), n - 1])
    w64 = W.winding(P.candidates(scene), pts.cpu().numpy()[idx])
    assert np.abs(w[idx] - w64).max() <= EXACT_PIN
    assert np.array_equal(ins.astype(bool), np.abs(w) > 0.5)


def test_nan_and_inf_points_and_stats(gpu):
    scene = S.small_mesh_scene(3)
    pts, on = pts_of(scene, 200, 13)
    pts[::7, 0] = np.nan
    pts[1::7, 1] = np.inf
    pts[2::7, 2] = -np.inf
    st = {}
    w, ins = wind(scene, pts, stats=st)
    nan = np.isnan(pts).any(1)
    assert np.isnan(w[nan]).all() and not ins[nan].any() and np.isfinite(w[~nan]).all()
    assert st["nan_rays"] == nan.sum() and st["rays"] == len(pts) and st["launches"] == 1
    assert st["ms_device"] > 0 and st["ms_total"] >= st["ms_device"] and st["node_visits"] > 0 and st["tri_tests"] > 0
    check(scene, pts, "NaN and inf", INF, on=on)


def test_one_plane_keeps_sentinels(gpu):
    import torch
    scene = S.small_mesh_scene(3)
    pts, _ = pts_of(scene, 200, 14)
    n = len(pts)
    t = dev(pts)
    w_all, ins_all = wind(scene, pts)
    lib = _abi.lib()
    for which in ("winding", "inside"):
        wbuf = torch.full((n + 8,), 7.5, device="cuda")
        ibuf = torch.full((n + 8,), 0xA5, dtype=torch.uint8, device="cuda")
        out = _abi.WindingOutC(**({"winding": wbuf.data_ptr()} if which == "winding" else {"inside": ibuf.data_ptr()}))
        _abi.check(lib.rbrt_gpu_query_winding_device(scene.handle(), t.data_ptr(), n, None, out, None, None))
        torch.cuda.synchronize()
        wb, ib = wbuf.cpu().numpy(), ibuf.cpu().numpy()
        if which == "winding":
            assert np.array_equal(wb[:n].view(np.uint32), w_all.view(np.uint32)) and (wb[n:] == 7.5).all() and (ib == 0xA5).all()
        else:
            assert np.array_equal(ib[:n], ins_all) and (ib[n:] == 0xA5).all() and (wb == 7.5).all()


# ============================================================================== 5. ordering
def test_ordering_against_a_mesh_update_on_another_stream(gpu):
    import torch
    scene = S.small_mesh_scene(3)
    pts, _ = pts_of(scene, 500, 15)
    old = wind(scene, pts)[0]
    new = twist(scene.triangle_meshes[0].triangles, 0.8)
    t, t_new = dev(pts), torch.from_numpy(new.copy()).cuda()
    torch.cuda.synchronize()
    s, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    with torch.cuda.stream(s):
        torch.cuda._sleep(int(5e8))
        a = scene.winding_device(t, stream=s)["winding"]
    scene.update_mesh_device(0, t_new, stream=s2)
    with torch.cuda.stream(s):
        b = scene.winding_device(t, stream=s)["winding"]
    s.synchronize(); s2.synchronize()
    assert np.array_equal(a.cpu().numpy(), old)
    want = wind(scene, pts)[0]
    assert not np.array_equal(want, old)
    assert np.array_equal(b.cpu().numpy(), want)
    check(scene, pts, "after the update", None)


def test_two_streams_right_after_an_update(gpu):
    """Two winding calls on two streams right after an update (the first recomputes the moments, the second waits for them): both equal
    the sequential result."""
    import torch
    scene = S.small_mesh_scene(3)
    pts, _ = pts_of(scene, 500, 16)
    t = dev(pts)
    wind(scene, pts)
    new = twist(scene.triangle_meshes[0].triangles, 0.5)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    scene.update_mesh_device(0, torch.from_numpy(new.copy()).cuda())
    with torch.cuda.stream(s1):
        torch.cuda._sleep(int(3e8))
        a = scene.winding_device(t, stream=s1)["winding"]
    with torch.cuda.stream(s2):
        b = scene.winding_device(t, stream=s2)["winding"]
    s1.synchronize(); s2.synchronize()
    want = wind(scene, pts)[0]
    assert np.array_equal(a.cpu().numpy(), want) and np.array_equal(b.cpu().numpy(), want)


def test_element_update_release_cache_and_destroy_in_flight(gpu):
    import torch
    scene = mixed_element_scene()
    pts, on = pts_of(scene, 500, 17)
    t = dev(pts)
    wind(scene, pts)
    scene.update_elements(moved_elements(scene.elements, 3))
    check(scene, pts, "after an element update", INF, on=on)
    _abi.check(_abi.lib().rbrt_gpu_release_cache())
    check(scene, pts, "after rbrt_gpu_release_cache", INF, on=on)
    s = torch.cuda.Stream()
    want = wind(scene, pts)[0]
    with torch.cuda.stream(s):
        torch.cuda._sleep(int(5e8))
        got = scene.winding_device(t, stream=s)["winding"]
    scene.close()                                                           # the block is freed behind the call in flight
    s.synchronize()
    assert np.array_equal(got.cpu().numpy(), want)


def test_side_stream_without_stats_does_not_synchronise(gpu):
    import torch
    scene = S.small_mesh_scene(3)
    pts, _ = pts_of(scene, 1000, 18)
    t = dev(pts)
    want = wind(scene, pts)[0]
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        torch.cuda._sleep(int(2e9))
        t0 = time.perf_counter()
        got = scene.winding_device(t, stream=s)["winding"]
        dt = time.perf_counter() - t0
        busy = not s.query()
    s.synchronize()
    assert busy and dt < 0.3, (busy, dt)
    assert np.array_equal(got.cpu().numpy(), want)


# ============================================================================== 6. communicator, refusals, missing module
def test_emulated_communicator_gives_the_same_answers(gpu):
    pts, _ = pts_of(S.small_mesh_scene(3), 300, 19)
    want = wind(S.small_mesh_scene(3), pts)[0]
    lib = _abi.lib()
    devs = (C.c_int * 2)(0, 0)
    _abi.check(lib.rbrt_gpu_init_multi(devs, 2, _abi.TRANSPORT_PEER))
    try:
        scene = S.small_mesh_scene(3)
        assert np.array_equal(wind(scene, pts)[0], want)
        scene.close()
    finally:
        _abi.check(lib.rbrt_gpu_comm_destroy())
    R.gpu_init(0)


def test_refusals(gpu):
    import torch
    lib = _abi.lib()
    scene = S.small_mesh_scene(3)
    h = scene.handle()
    pts = dev(scene_points(scene, 16, 20))
    n = pts.shape[0]
    plane = torch.full((n,), 7.0, device="cuda")
    out = _abi.WindingOutC(winding=plane.data_ptr())
    f = lib.rbrt_gpu_query_winding_device
    assert f(None, pts.data_ptr(), n, None, out, None, None) == _abi.E_INVALID
    assert f(h, None, n, None, out, None, None) == _abi.E_INVALID
    assert f(h, pts.data_ptr(), n, None, None, None, None) == _abi.E_INVALID
    assert f(h, pts.data_ptr(), n, None, _abi.WindingOutC(), None, None) == _abi.E_INVALID
    assert f(h, pts.data_ptr(), 2 ** 32, None, out, None, None) == _abi.E_INVALID
    host_pts = pts.cpu().numpy()
    assert f(h, host_pts.ctypes.data, n, None, out, None, None) == _abi.E_INVALID
    assert b"device memory" in lib.rbrt_last_error()
    host_plane = np.zeros(n, np.uint8)
    assert f(h, pts.data_ptr(), n, None, _abi.WindingOutC(inside=host_plane.ctypes.data), None, None) == _abi.E_INVALID
    for beta in (1.0, 0.5, -2.0, float("nan"), -INF):
        assert f(h, pts.data_ptr(), n, _abi.WindingOptsC(beta), out, None, None) == _abi.E_INVALID, beta
        assert b"beta" in lib.rbrt_last_error()
    st = _abi.StatsC(rays=9)
    assert f(h, pts.data_ptr(), 0, None, out, None, st) == 0 and st.rays == 0
    torch.cuda.synchronize()
    assert (plane.cpu().numpy() == 7.0).all() and not host_plane.any()
    for bad in (pts.cpu(), pts[:, :2].contiguous(), pts.double()):
        with pytest.raises(ValueError):
            scene.winding_device(bad)
    with pytest.raises(ValueError):
        scene.winding_device(pts, passes=("winding", "depth"))
    with pytest.raises(ValueError):
        scene.winding_device(pts, beta=1.0)
    for beta in (1.0001, 2.0, 100.0, INF):
        _abi.check(f(h, pts.data_ptr(), n, _abi.WindingOptsC(beta), out, None, None))
    torch.cuda.synchronize()
    assert not (plane.cpu().numpy() == 7.0).all()


def test_missing_module_is_refused_with_a_message(gpu):
    code = ("import sys; sys.path.insert(0, %r)\n"
            "import numpy as np, torch, rbrt_b200 as R\nfrom tests import scenes as S\nfrom rbrt_b200 import _abi\n"
            "R.gpu_init(0); sc = S.small_mesh_scene(3); pts = torch.zeros(8, 3, device='cuda')\n"
            "try:\n    sc.winding_device(pts)\n    print('NO ERROR')\n"
            "except _abi.RbrtGpuError as e:\n    print('CODE', e.code, str(e))\n"
            "print('NEAR', sc.nearest_device(pts)['dist'].shape)\n") % ROOT
    env = dict(os.environ, RBRT_GPU_WIND_LIB=os.path.join(ROOT, "no-such-dir", "librbrt_gpu_wind.so"))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr
    assert f"CODE {_abi.E_CUDA}" in r.stdout and "winding-number module is missing" in r.stdout, r.stdout
    assert "NEAR torch.Size([8])" in r.stdout, r.stdout


# ============================================================================== 7. signed distance
def test_signed_distance(gpu):
    import torch
    tris = ico(4, 3.0, (1.0, 2.0, 3.0))
    scene = R.Scene(triangle_meshes=[R.TriangleMesh.from_triangles(tris, MAT)])
    pts = np.random.default_rng(21).uniform(-4, 6, (3000, 3)).astype(F)
    t = dev(pts)
    sd = scene.signed_distance_device(t).cpu().numpy()
    dist = scene.nearest_device(t, passes="dist")["dist"].cpu().numpy()
    ins = scene.winding_device(t, passes="inside")["inside"].cpu().numpy()
    assert np.array_equal(sd.view(np.uint32), np.where(ins.astype(bool), -dist, dist).view(np.uint32))
    r = np.linalg.norm(pts - np.array([1.0, 2.0, 3.0]), axis=1)
    clear = np.abs(r - 3.0) > 0.1
    assert (np.sign(sd[clear]) == np.sign(r[clear] - 3.0)).all()
    band = scene.signed_distance_device(t, max_dist=0.5).cpu().numpy()
    deep, out = r < 2.0, r > 4.0
    assert (band[deep] == -np.inf).all() and (band[out] == np.inf).all()
    near = np.isfinite(band)
    assert np.array_equal(band[near], sd[near])
    tb = torch.full((len(pts),), 0.5, device="cuda")
    assert np.array_equal(scene.signed_distance_device(t, max_dist=tb).cpu().numpy().view(np.uint32), band.view(np.uint32))
