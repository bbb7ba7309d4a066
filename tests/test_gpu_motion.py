"""Per-object motion vectors (rbrt_gpu_scene_snapshot, rbrt_gpu_render_motion*, rbrt_gpu_temporal_accumulate_motion*; csrc/motion.cu,
csrc/temporal.cu, csrc/api.cu) on the GPU.

The reference of every case: the pixel-centre rays built in numpy (tests/motion_ref.py), Scene.hit (rbrt_gpu_trace_rays), then
motion_ref with the geometry the test itself fed to the scene before and after its update.  Results are compared bit for bit (NaN equal
to NaN whatever its payload).  The quality test measures temporal accumulation along the motion against camera reprojection alone on a
moving sphere and a deforming mesh under a static camera."""
import ctypes as C
import dataclasses
import os
import subprocess
import sys
import time

import numpy as np
import pytest

import rbrt_b200 as R
from rbrt_b200 import _abi

from . import motion_ref as M
from . import scenes as S
from . import temporal_ref as T
from .test_gpu_denoise import rmse
from .test_gpu_temporal import render_frame, same_all, workload

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "rbrt_b200", "librbrt_gpu_motion.so")
F = np.float32


@pytest.fixture(scope="module", autouse=True)
def motion_module():
    """The session fixture only builds librbrt_gpu.so when it is missing; the module is built here when it is."""
    if not os.path.exists(LIB):
        subprocess.run(["make", "-C", os.path.join(ROOT, "rbrt_b200", "csrc")], check=True)
    return LIB


# ============================================================================== geometry the tests feed and remember
def geometry(scene):
    """The scene's geometry as motion_ref.motion_from_hits reads it."""
    els = []
    for e in scene.elements:
        if isinstance(e, R.Sphere):
            els.append(("sphere", (e.center.x, e.center.y, e.center.z), e.radius))
        else:
            els.append(("triangle", np.array([[c.x, c.y, c.z] for c in e.corners], F)))
    return {"elements": els, "meshes": [np.array(m.triangles, F) for m in scene.triangle_meshes]}


def expected(scene, cam, prev, now, snap):
    hits = scene.hit(M.camera_rays(cam))
    return M.motion_from_hits(cam, prev, hits, now, snap)


def same_planes(got, want):
    return T.same_bits(got[0], want[0]) and T.same_bits(got[1], want[1])


def to_np(t):
    return t.cpu().numpy()


def check(scene, cam, prev, snap, what):
    got = R.render_motion(cam, prev, scene)
    want = expected(scene, cam, prev, geometry(scene), snap)
    assert same_planes(got, want), what
    return got


def moved_sphere(els, k, d):
    e = els[k]
    return R.Sphere(R.Vec3(e.center.x + d[0], e.center.y + d[1], e.center.z + d[2]), e.radius * d[3], e.material)


def mixed_scene():
    """Spheres (one with a negative radius), BasicTriangles and two meshes."""
    scene = S.small_mesh_scene(3)
    mat = R.Lambertian(R.Vec3(0.5, 0.6, 0.7))
    scene.elements.append(R.Sphere(R.Vec3(-1.2, 0.6, -0.4), -0.35, mat))
    scene.elements.append(R.BasicTriangle.new([R.Vec3(-2.0, 0.0, -1.5), R.Vec3(-0.5, 0.1, -1.6), R.Vec3(-1.2, 1.4, -1.4)], mat))
    scene.elements.append(R.BasicTriangle.new([R.Vec3(0.8, 0.0, -1.2), R.Vec3(2.0, 0.2, -1.0), R.Vec3(1.4, 1.1, -1.3)], mat))
    second = np.array(scene.triangle_meshes[0].triangles, F) * F(0.5) + np.array([1.3, 0.1, 0.4], F)
    scene.triangle_meshes.append(R.TriangleMesh.from_triangles(second, mat))
    return scene


def wave(tris, k):
    """scripts/update_time.py's travelling wave, step k, in float32."""
    base = np.asarray(tris, F)
    return (base + F(0.6) * np.sin(F(0.15) * np.roll(base, 1, axis=-1) + F(0.05 * k))).astype(F)


def small_wave(tris, k):
    base = np.asarray(tris, F)
    return (base + F(0.02) * np.sin(F(3.0) * np.roll(base, 1, axis=-1) + F(0.7 * k))).astype(F)


# ============================================================================== 1. a snapshot of a static scene
@pytest.mark.parametrize("name,W,H", [("c1", 256, 192), ("c2", 256, 192), ("c4", 256, 192), ("c3", 1920, 1080)])
def test_static_scene_gives_zero_motion(gpu, name, W, H):
    scene, cam = workload(name, W, H)
    scene.snapshot()
    m, pd = R.render_motion(cam, cam, scene)
    hits = scene.hit(M.camera_rays(cam))
    hit = (hits["kind"] >= 0).reshape(H, W)
    assert hit.mean() > 0.3
    assert (m[hit].view(np.uint32) == 0).all()                            # (+0, +0) exactly
    assert np.isnan(m[~hit]).all() and np.isposinf(pd[~hit]).all()
    pos = T.cam_values(cam)[0]
    D = [hits["point"][:, k] - pos[k] for k in range(3)]
    assert T.same_bits(pd[hit], np.sqrt(T.dot(D, D)).astype(F).reshape(H, W)[hit])
    assert same_planes((m, pd), expected(scene, cam, cam, geometry(scene), geometry(scene)))


def test_snapshot_of_an_unchanged_scene_twice_is_the_same(gpu):
    scene = mixed_scene()
    cam = S.example_camera(64, 48)
    prev = dataclasses.replace(cam, position=R.Vec3(cam.position.x + 0.2, cam.position.y, cam.position.z))
    scene.snapshot()
    a = R.render_motion(cam, prev, scene)
    scene.snapshot()
    scene.snapshot()
    assert same_planes(R.render_motion(cam, prev, scene), a)


# ============================================================================== 2. geometry changes
def test_sphere_translated_and_rescaled(gpu):
    scene = mixed_scene()
    cam = S.example_camera(96, 72)
    scene.snapshot()
    snap = geometry(scene)
    els = list(scene.elements)
    els[0] = moved_sphere(els, 0, (0.1, 0.05, -0.02, 1.1))
    els[1] = moved_sphere(els, 1, (-0.05, 0.0, 0.03, 0.9))
    els[4] = moved_sphere(els, 4, (0.04, -0.02, 0.0, 1.3))                # the negative radius
    scene.update_elements(els)
    for prev in (cam, S.example_camera(96, 72), dataclasses.replace(cam, position=R.Vec3(cam.position.x - 0.3, cam.position.y, cam.position.z))):
        m, _ = check(scene, cam, prev, snap, "spheres moved")
    assert (np.isfinite(m).all(-1) & (m != 0).any(-1)).sum() > 50


def test_basic_triangle_corners_moved(gpu):
    mat = R.Lambertian(R.Vec3(0.5, 0.6, 0.7))
    scene = R.Scene(elements=[R.Sphere(R.Vec3(0.0, 0.0, -6.0), 1.0, mat),
                              R.BasicTriangle.new([R.Vec3(-2.0, -1.0, -3.0), R.Vec3(-0.2, -1.1, -3.2), R.Vec3(-1.1, 1.0, -2.9)], mat),
                              R.BasicTriangle.new([R.Vec3(0.3, -1.0, -3.5), R.Vec3(2.0, -0.8, -3.3), R.Vec3(1.2, 1.2, -3.6)], mat)])
    cam = R.Camera.new(R.Vec3(0.0, 0.0, 0.0), R.Vec3(0.0, 0.0, -1.0), R.Vec3(0.0, 1.0, 0.0), 72, 96, 35.0)
    scene.snapshot()
    snap = geometry(scene)
    els = list(scene.elements)
    for k in (1, 2):
        t = els[k]
        els[k] = R.BasicTriangle.new([R.Vec3(c.x + 0.05 * i, c.y - 0.03, c.z + 0.02 * i) for i, c in enumerate(t.corners)], t.material)
    scene.update_elements(els)
    hits = scene.hit(M.camera_rays(cam))
    assert (hits["kind"] == _abi.HIT_TRIANGLE).sum() > 500 and (hits["kind"] == _abi.HIT_SPHERE).sum() > 50
    m, _ = check(scene, cam, cam, snap, "BasicTriangles moved")
    tri = (hits["kind"] == _abi.HIT_TRIANGLE).reshape(72, 96)
    assert (m[tri] != 0).any(-1).mean() > 0.9 and (m[(hits["kind"] == _abi.HIT_SPHERE).reshape(72, 96)].view(np.uint32) == 0).all()


@pytest.mark.parametrize("rebuild", [False, True])
def test_deforming_mesh(gpu, rebuild):
    """RBRT_UPDATE_REFIT keeps the record slots; RBRT_UPDATE_REBUILD permutes them: the snapshot is keyed by the original index."""
    scene = mixed_scene()
    cam = S.example_camera(96, 72)
    scene.snapshot()
    snap = geometry(scene)
    for k in (1, 2):
        scene.update_mesh(0, small_wave(snap["meshes"][0], k), rebuild=rebuild)
        m, _ = check(scene, cam, cam, snap, f"mesh step {k}")
    hits = scene.hit(M.camera_rays(cam))
    mesh0 = ((hits["kind"] == _abi.HIT_MESH) & (hits["elem_idx"] == 0)).reshape(m.shape[:2])
    assert mesh0.sum() > 100 and (m[mesh0] != 0).any(-1).mean() > 0.5


def test_only_one_of_several_meshes_moves(gpu):
    scene = mixed_scene()
    cam = S.example_camera(96, 72)
    scene.snapshot()
    snap = geometry(scene)
    scene.update_mesh(1, small_wave(snap["meshes"][1], 3))
    m, _ = check(scene, cam, cam, snap, "mesh 1 moved")
    hits = scene.hit(M.camera_rays(cam))
    kind, el = hits["kind"].reshape(m.shape[:2]), hits["elem_idx"].reshape(m.shape[:2])
    still = (kind >= 0) & ~((kind == _abi.HIT_MESH) & (el == 1))
    assert (m[still].view(np.uint32) == 0).all()
    assert (m[(kind == _abi.HIT_MESH) & (el == 1)] != 0).any()


@pytest.mark.parametrize("W,H", [(1, 1), (1, 40), (40, 1), (33, 17)])
def test_odd_image_shapes(gpu, W, H):
    scene = mixed_scene()
    cam = S.example_camera(W, H)
    prev = dataclasses.replace(cam, position=R.Vec3(cam.position.x + 0.1, cam.position.y + 0.05, cam.position.z))
    scene.snapshot()
    snap = geometry(scene)
    els = list(scene.elements)
    els[0] = moved_sphere(els, 0, (0.05, 0.0, 0.0, 1.0))
    scene.update_elements(els)
    scene.update_mesh(0, small_wave(snap["meshes"][0], 1), rebuild=True)
    check(scene, cam, prev, snap, f"{W}x{H}")


def test_analytic_sphere_translation(gpu):
    """A sphere translated by Δ under a static camera: inside its silhouette the motion is the float64 projection of P + Δ minus that of
    P, within 1e-3 px."""
    scene, cam = workload("c1", 256, 192)
    scene.snapshot()
    els = list(scene.elements)
    k = max(range(len(els)), key=lambda i: els[i].radius if els[i].radius < 50 else -1)
    delta = np.array([0.08, 0.03, -0.05])
    els[k] = moved_sphere(els, k, (*delta, 1.0))
    scene.update_elements(els)
    m, _ = R.render_motion(cam, cam, scene)
    hits = scene.hit(M.camera_rays(cam))
    kind, el = hits["kind"].reshape(192, 256), hits["elem_idx"].reshape(192, 256)
    on = (kind == _abi.HIT_SPHERE) & (el == k)
    inner = on & np.roll(on, 1, 0) & np.roll(on, -1, 0) & np.roll(on, 1, 1) & np.roll(on, -1, 1)
    assert inner.sum() > 100

    def proj(P):
        pos, right, up, center, mmh, mmv, W, H = (np.asarray(v, np.float64) if isinstance(v, np.ndarray) else v for v in T.cam_values(cam))
        Dv, Cv = P - pos, center - pos
        ru = np.cross(right, up)
        det = Dv @ ru
        a = (Dv @ np.cross(up, Cv)) / det
        b = (Dv @ np.cross(right, Cv)) / det
        return np.stack([a / 0.001 / float(mmh) + W // 2, b / 0.001 / float(mmv) + H // 2], -1)

    P = hits["point"].reshape(192, 256, 3)[inner].astype(np.float64)
    want = proj(P - delta) - proj(P)                                      # P was at P - Δ at the snapshot
    err = np.abs(m[inner] - want).max()
    print(f"analytic: {int(inner.sum())} pixels, |motion| up to {np.abs(want).max():.3f} px, max error {err:.2e} px")
    assert err < 1e-3


# ============================================================================== 3. ordering
def test_update_on_another_stream_after_a_snapshot_does_not_leak_into_it(gpu):
    import torch
    scene = mixed_scene()
    cam = S.example_camera(64, 48)
    scene.snapshot()                                                      # the module is loaded and the block allocated
    snap = geometry(scene)
    new = small_wave(snap["meshes"][0], 2)
    t = torch.from_numpy(new).cuda()
    torch.cuda.synchronize()
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    with torch.cuda.stream(s1):
        torch.cuda._sleep(int(1e9))                                       # the snapshot waits in its stream
        scene.snapshot(stream=s1)
    with torch.cuda.stream(s2):
        scene.update_mesh_device(0, t, stream=s2)                         # enqueued while the snapshot is still waiting
    torch.cuda.synchronize()
    got = R.render_motion(cam, cam, scene)
    now = {"elements": snap["elements"], "meshes": [new] + snap["meshes"][1:]}
    assert same_planes(got, expected(scene, cam, cam, now, snap))
    assert (np.isfinite(got[0]) & (got[0] != 0)).any()


def test_motion_after_a_second_snapshot_sees_it(gpu):
    """The second snapshot waits behind a second of work on its stream; the motion call on another stream, enqueued meanwhile, must see
    it and not the first one.  The planes are allocated and the kernel loaded beforehand, so nothing synchronises the device in between."""
    import torch
    scene = mixed_scene()
    cam = S.example_camera(64, 48)
    scene.snapshot()
    snap0 = geometry(scene)
    scene.update_mesh(0, small_wave(snap0["meshes"][0], 2))
    stale = R.render_motion(cam, cam, scene)                              # against the first snapshot: moving
    assert (np.isfinite(stale[0]) & (stale[0] != 0)).any()
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    m = torch.full((48, 64, 2), 7.0, device="cuda")
    pd = torch.full((48, 64), 7.0, device="cuda")
    out = _abi.MotionOutC(m.data_ptr(), pd.data_ptr())
    lib = _abi.lib()
    _abi.check(lib.rbrt_gpu_render_motion_device(scene.handle(), cam.to_c(), cam.to_c(), out, s2.cuda_stream, None))   # the kernel is loaded
    torch.cuda.synchronize()                                              # (a first launch may wait for the device)
    m.fill_(7.0)
    pd.fill_(7.0)
    torch.cuda.synchronize()
    with torch.cuda.stream(s1):
        torch.cuda._sleep(int(2e9))
        scene.snapshot(stream=s1)                                         # of the updated scene
    _abi.check(lib.rbrt_gpu_render_motion_device(scene.handle(), cam.to_c(), cam.to_c(), out, s2.cuda_stream, None))
    busy = not s1.query()
    torch.cuda.synchronize()
    assert busy
    now = geometry(scene)
    assert same_planes((to_np(m), to_np(pd)), expected(scene, cam, cam, now, now))


def test_two_motion_calls_in_flight_on_two_streams(gpu):
    import torch
    scene = mixed_scene()
    cam = S.example_camera(64, 48)
    scene.snapshot()
    snap = geometry(scene)
    els = list(scene.elements)
    els[0] = moved_sphere(els, 0, (0.1, 0.0, 0.0, 1.0))
    scene.update_elements(els)
    prevs = [cam, dataclasses.replace(cam, position=R.Vec3(cam.position.x + 0.3, cam.position.y, cam.position.z))]
    want = [expected(scene, cam, p, geometry(scene), snap) for p in prevs]
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    outs = []
    for s, p in zip(streams, prevs):
        with torch.cuda.stream(s):
            torch.cuda._sleep(int(3e8))
            outs.append(R.render_motion_device(cam, p, scene, stream=s))
    torch.cuda.synchronize()
    for (m, pd), w in zip(outs, want):
        assert same_planes((to_np(m), to_np(pd)), w)


def test_scene_destroyed_with_a_snapshot_pending(gpu):
    import torch
    scene = mixed_scene()
    cam = S.example_camera(64, 48)
    scene.snapshot()
    snap = geometry(scene)
    els = list(scene.elements)
    els[1] = moved_sphere(els, 1, (0.0, 0.1, 0.0, 1.0))
    scene.update_elements(els)
    want = expected(scene, cam, cam, geometry(scene), snap)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        m, pd = R.render_motion_device(cam, cam, scene, stream=s)
        torch.cuda._sleep(int(1e9))
        scene.snapshot(stream=s)
    scene.close()
    torch.cuda.synchronize()
    assert same_planes((to_np(m), to_np(pd)), want)
    again = mixed_scene()                                                 # the library still works
    again.snapshot()
    assert same_planes(R.render_motion(cam, cam, again), expected(again, cam, cam, geometry(again), geometry(again)))


def test_release_cache_between_motion_calls(gpu):
    scene = mixed_scene()
    cam = S.example_camera(64, 48)
    scene.snapshot()
    snap = geometry(scene)
    scene.update_mesh(0, small_wave(snap["meshes"][0], 1))
    a = check(scene, cam, cam, snap, "before")
    _abi.check(_abi.lib().rbrt_gpu_release_cache())
    assert same_planes(R.render_motion(cam, cam, scene), a)


# ============================================================================== 4. host and device, stats
def test_device_variant_on_a_side_stream_equals_the_host_variant(gpu):
    import torch
    scene = mixed_scene()
    cam = S.example_camera(50, 30)
    prev = dataclasses.replace(cam, position=R.Vec3(cam.position.x + 0.2, cam.position.y, cam.position.z))
    scene.snapshot()
    els = list(scene.elements)
    els[0] = moved_sphere(els, 0, (0.05, 0.05, 0.0, 1.1))
    scene.update_elements(els)
    st = {}
    host = R.render_motion(cam, prev, scene, stats=st)
    assert st["rays"] == 50 * 30 and st["nan_rays"] == 0 and st["launches"] == 1 and st["ms_device"] > 0 and st["node_visits"] > 0
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        dev = R.render_motion_device(cam, prev, scene, stream=s)
    s.synchronize()
    assert same_planes((to_np(dev[0]), to_np(dev[1])), host)


def test_nan_rays_are_counted(gpu):
    mat = R.Lambertian(R.Vec3(0.5, 0.5, 0.5))
    scene = R.Scene(elements=[R.Sphere(R.Vec3(0.0, 0.0, -3.0), float("nan"), mat)])
    cam = S.example_camera(16, 12)
    scene.snapshot()
    st = {}
    m, pd = R.render_motion(cam, cam, scene, stats=st)
    assert st["rays"] == 16 * 12 and st["nan_rays"] == 16 * 12
    assert np.isnan(m).all() and np.isposinf(pd).all()


def test_device_variant_without_stats_does_not_synchronise(gpu):
    import torch
    scene = mixed_scene()
    cam = S.example_camera(32, 24)
    scene.snapshot()
    ref = R.render_motion(cam, cam, scene)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        torch.cuda._sleep(int(2e9))
        t0 = time.perf_counter()
        m, pd = R.render_motion_device(cam, cam, scene, stream=s)
        dt = time.perf_counter() - t0
        busy = not s.query()
    s.synchronize()
    assert busy and dt < 0.3, (busy, dt)
    assert same_planes((to_np(m), to_np(pd)), ref)


# ============================================================================== 5. communicator
def test_emulated_communicator_gives_the_same_planes(gpu):
    cam = S.example_camera(40, 30)

    def run():
        scene = mixed_scene()
        scene.snapshot()
        snap = geometry(scene)
        scene.update_mesh(0, small_wave(snap["meshes"][0], 1))
        els = list(scene.elements)
        els[0] = moved_sphere(els, 0, (0.05, 0.0, 0.0, 1.0))
        scene.update_elements(els)
        out = R.render_motion(cam, cam, scene)
        scene.close()
        return out

    ref = run()
    lib = _abi.lib()
    devs = (C.c_int * 2)(0, 0)
    _abi.check(lib.rbrt_gpu_init_multi(devs, 2, _abi.TRANSPORT_PEER))
    try:
        got = run()
    finally:
        _abi.check(lib.rbrt_gpu_comm_destroy())
    R.gpu_init(0)
    assert same_planes(got, ref)


# ============================================================================== 6. refusals and the missing module
def test_refusals_write_nothing(gpu):
    import torch
    from .test_gpu_bvh_build import REFUSED, deep_scene
    lib = _abi.lib()
    scene = mixed_scene()
    cam = S.example_camera(16, 12)
    h = scene.handle()
    m = np.full((12, 16, 2), 7.0, F)
    pd = np.full((12, 16), 7.0, F)
    out = _abi.MotionOutC(m.ctypes.data, pd.ctypes.data)
    c = cam.to_c()
    assert lib.rbrt_gpu_render_motion(h, c, c, out, None) == _abi.E_INVALID and b"snapshot" in lib.rbrt_last_error()
    scene.snapshot()
    cases = [((None, c, c, out), b"null"), ((h, None, c, out), b"null"), ((h, c, None, out), b"null"), ((h, c, c, None), b"null"),
             ((h, c, c, _abi.MotionOutC(None, None)), b"no output"),
             ((h, c, S.example_camera(16, 13).to_c(), out), b"prev_cam"),
             ((h, dataclasses.replace(cam, img_width_pix=0).to_c(), c, out), b"empty"),
             ((h, dataclasses.replace(cam, img_width_pix=65536, img_height_pix=65536).to_c(),
               dataclasses.replace(cam, img_width_pix=65536, img_height_pix=65536).to_c(), out), b"too large"),
             ((h, c, c, _abi.MotionOutC(m.ctypes.data, m.ctypes.data + 8)), b"overlap")]
    for args, msg in cases:
        assert lib.rbrt_gpu_render_motion(*args, None) == _abi.E_INVALID, msg
        assert msg in lib.rbrt_last_error(), (msg, lib.rbrt_last_error())
    dm = torch.full((12, 16, 2), 7.0, device="cuda")
    dpd = torch.full((12, 16), 7.0, device="cuda")
    for o, msg in [(_abi.MotionOutC(m.ctypes.data, dpd.data_ptr()), b"device memory"),
                   (_abi.MotionOutC(dm.data_ptr(), dm.data_ptr() + 4), b"overlap")]:
        assert lib.rbrt_gpu_render_motion_device(h, c, c, o, None, None) == _abi.E_INVALID, msg
        assert msg in lib.rbrt_last_error()
    deep = deep_scene(REFUSED)
    with pytest.raises(_abi.RbrtGpuError, match="BVH deeper than the traversal stack allows"):
        deep.snapshot()
    assert lib.rbrt_gpu_render_motion(deep.handle(), c, c, out, None) == _abi.E_INVALID
    torch.cuda.synchronize()
    assert (m == 7.0).all() and (pd == 7.0).all() and (dm == 7.0).all() and (dpd == 7.0).all()
    assert lib.rbrt_gpu_render_motion(h, c, c, out, None) == 0 and not (pd == 7.0).all()   # the same call, valid


def test_missing_module_is_refused_with_a_message(gpu):
    code = ("import sys; sys.path.insert(0, %r)\n"
            "import numpy as np, rbrt_b200 as R\nfrom tests import scenes as S\nfrom rbrt_b200 import _abi\n"
            "R.gpu_init(0); sc = S.small_mesh_scene(3); cam = S.example_camera(16, 12)\n"
            "for what, f in (('SNAPSHOT', lambda: sc.snapshot()), ('MOTION', lambda: R.render_motion(cam, cam, sc))):\n"
            "    try:\n        f(); print(what, 'NO ERROR')\n"
            "    except _abi.RbrtGpuError as e:\n        print(what, 'CODE', e.code, str(e))\n"
            "print('RENDER', R.render_scene_hdr(cam, 1, sc).shape)\n") % ROOT
    env = dict(os.environ, RBRT_GPU_MOTION_LIB=os.path.join(ROOT, "no-such-dir", "librbrt_gpu_motion.so"))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr
    for what in ("SNAPSHOT", "MOTION"):
        assert f"{what} CODE {_abi.E_CUDA}" in r.stdout and "motion module is missing" in r.stdout, r.stdout
    assert "RENDER (12, 16, 3)" in r.stdout, r.stdout


# ============================================================================== 7. temporal accumulation along the motion
def moving_sphere_frames(n, W=96, H=72, seed=20):
    """C1 under a static camera, its largest small sphere moving sideways; per frame (hdr, var, aovs, motion planes or None)."""
    scene, cam = workload("c1", W, H)
    els = list(scene.elements)
    k = max(range(len(els)), key=lambda i: els[i].radius if els[i].radius < 50 else -1)
    frames = []
    for f in range(n):
        if f:
            scene.snapshot()
            els[k] = moved_sphere(els, k, (0.06, 0.0, 0.0, 1.0))
            scene.update_elements(els)
        hdr, var, aovs = render_frame(scene, cam, seed + f)
        frames.append((hdr, var, aovs, R.render_motion(cam, cam, scene) if f else None))
    return scene, cam, frames


def test_temporal_with_motion_equals_the_reference_on_real_renders(gpu):
    import torch
    scene, cam, frames = moving_sphere_frames(4)
    hist = None
    moved = 0
    for hdr, var, aovs, mo in frames:
        for v in (var, None):
            h = None if hist is None else {**hist, "var": hist["var"] if v is not None else None}
            want = M.accumulate_motion(cam, hdr, v, aovs, h, *mo) if mo is not None else T.accumulate(cam, hdr, v, aovs, h)
            got = R.temporal_accumulate(cam, hdr, aovs, var=v, history=h, motion=mo)
            assert same_all(got, want)
        if mo is not None:
            tens = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
            dh = {"cam": cam, "hdr": tens(hist["hdr"]), "var": tens(hist["var"]), "length": tens(hist["length"]),
                  "aovs": {k: tens(hist["aovs"][k]) for k in ("depth", "normal", "hit_kind", "elem_idx")}}
            dev = R.temporal_accumulate_device(cam, tens(hdr), {k: tens(aovs[k]) for k in dev_keys()}, var=tens(var), history=dh,
                                               motion=(tens(mo[0]), tens(mo[1])))
            torch.cuda.synchronize()
            assert same_all([to_np(x) for x in dev], R.temporal_accumulate(cam, hdr, aovs, var=var, history=hist, motion=mo))
            moved += int((np.isfinite(mo[0]).all(-1) & (mo[0] != 0).any(-1)).sum())
        out = R.temporal_accumulate(cam, hdr, aovs, var=var, history=hist, motion=mo)
        hist = {"cam": cam, "hdr": out[0], "var": out[1], "length": out[2], "aovs": aovs}
    assert moved > 100


def dev_keys():
    return ("depth", "normal", "hit_kind", "elem_idx")


def test_accumulator_without_motion_keeps_the_existing_bits_and_zero_motion_maps_each_pixel_to_itself(gpu):
    """TemporalAccumulator with motion=None gives the existing call's bits.  With a static scene the motion is exactly 0 on every hit,
    so each pixel maps to itself as under the bitwise-equal camera; the two paths differ only in r (the centre ray's prev_dist against
    the camera path's depth AOV, a mean over the jittered samples), which only the depth tolerance reads."""
    import torch
    scene, cam = workload("c2", 64, 48)
    scene.snapshot()
    acc_none, acc_zero = R.TemporalAccumulator(64, 48), R.TemporalAccumulator(64, 48)
    hist = hz = None
    for f in range(3):
        hdr, var, aovs = render_frame(scene, cam, 40 + f)
        tens = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
        dh, dv, da = tens(hdr), tens(var), {k: tens(aovs[k]) for k in dev_keys()}
        ref = R.temporal_accumulate(cam, hdr, aovs, var=var, history=hist)
        hist = {"cam": cam, "hdr": ref[0], "var": ref[1], "length": ref[2], "aovs": aovs}
        a = [to_np(x) for x in acc_none.step(cam, dh, dv, da, motion=None)]
        mo = R.render_motion_device(cam, acc_zero.camera or cam, scene)
        z = [to_np(x) for x in acc_zero.step(cam, dh, dv, da, motion=mo)]
        torch.cuda.synchronize()
        mo = (to_np(mo[0]), to_np(mo[1]))
        assert same_all(a, ref), f
        assert same_all(z, M.accumulate_motion(cam, hdr, var, aovs, hz, *mo)), f
        hz = {"cam": cam, "hdr": z[0], "var": z[1], "length": z[2], "aovs": aovs}
        centre_hit = (scene.hit(M.camera_rays(cam))["kind"] >= 0).reshape(48, 64)
        assert (mo[0][centre_hit].view(np.uint32) == 0).all() and np.isnan(mo[0][~centre_hit]).all()
        same = (z[0].view(np.uint32) == ref[0].view(np.uint32)).all(-1)
        print(f"frame {f}: {same.mean():.4f} of the pixels equal the bitwise-equal camera's result")
        assert same.mean() > 0.9


# ============================================================================== 8. quality: a moving sphere and a deforming mesh
# RMSE / noisy RMSE on the moving object's pixels (current AOV elem_idx) and on the whole frame, the largest over frames 3..7, pinned
# with a margin of 0.02 (DESIGN.md section 16).
BOUNDS = {("c1", "spatial_obj"): 0.98, ("c1", "camera_obj"): 1.88, ("c1", "motion_obj"): 1.10,
          ("c1", "spatial_all"): 0.58, ("c1", "camera_all"): 0.71, ("c1", "motion_all"): 0.63,
          ("c2", "spatial_obj"): 0.70, ("c2", "camera_obj"): 0.69, ("c2", "motion_obj"): 0.65,
          ("c2", "spatial_all"): 0.60, ("c2", "camera_all"): 0.51, ("c2", "motion_all"): 0.50}


def quality_sequence(name):
    W, H = 256, 192
    scene, cam = workload(name, W, H)
    if name == "c1":
        els = list(scene.elements)
        k = max(range(len(els)), key=lambda i: els[i].radius if els[i].radius < 50 else -1)
        # a few pixels per frame: 3 px at the sphere's centre
        pos, right = T.cam_values(cam)[0], T.cam_values(cam)[1]
        c = np.array([els[k].center.x, els[k].center.y, els[k].center.z], np.float64)
        px0 = T.project(cam, [F(c[i] - pos[i]) for i in range(3)])[0]
        px1 = T.project(cam, [F(c[i] + right[i] - pos[i]) for i in range(3)])[0]
        step = 3.0 / float(px1 - px0) * np.asarray(right, np.float64)

        def advance(f):
            els[k] = R.Sphere(R.Vec3(c[0] + f * step[0], c[1] + f * step[1], c[2] + f * step[2]), els[k].radius, els[k].material)
            scene.update_elements(els)

        def moving(aovs):
            return (aovs["hit_kind"] == _abi.HIT_SPHERE) & (aovs["elem_idx"] == k)
    else:
        base = np.array(scene.triangle_meshes[0].triangles, F)

        def advance(f):
            scene.update_mesh(0, wave(base, f))

        def moving(aovs):
            return aovs["hit_kind"] == _abi.HIT_MESH
    return scene, cam, advance, moving


@pytest.mark.parametrize("name", ["c1", "c2"])
def test_quality_of_motion_reprojection(gpu, name):
    """8 frames under a static camera, 4 spp with K = 4 and seeds 11 + f, guides at 4 spp of the same seed, 4096-spp references with
    seed 12345 per frame: the variance-guided filter alone, temporal with camera reprojection then the filter, temporal along the motion
    then the filter."""
    scene, cam, advance, moving = quality_sequence(name)
    hc = hm = None
    rows = []
    for f in range(8):
        if f:
            scene.snapshot()                                              # the previous frame's geometry
        advance(f)
        hdr, var, aovs = render_frame(scene, cam, 11 + f)
        mo = R.render_motion(cam, cam, scene) if f else None
        tc = R.temporal_accumulate(cam, hdr, aovs, var=var, history=hc)
        tm = R.temporal_accumulate(cam, hdr, aovs, var=var, history=hm, motion=mo)
        hc = {"cam": cam, "hdr": tc[0], "var": tc[1], "length": tc[2], "aovs": aovs}
        hm = {"cam": cam, "hdr": tm[0], "var": tm[1], "length": tm[2], "aovs": aovs}
        if f < 3:
            continue
        ref = R.render_scene_hdr(cam, 4096, scene, seed=12345)
        mv = moving(aovs)
        assert mv.sum() > 200
        outs = {"spatial": R.denoise_variance(hdr, var, aovs)[0], "camera": R.denoise_variance(tc[0], tc[1], aovs)[0],
                "motion": R.denoise_variance(tm[0], tm[1], aovs)[0]}
        r = {"frame": f}
        for k, o in outs.items():
            r[k + "_obj"] = rmse(o[mv], ref[mv]) / rmse(hdr[mv], ref[mv])
            r[k + "_all"] = rmse(o, ref) / rmse(hdr, ref)
        r["len_camera_obj"] = float(tc[2][mv].mean())
        r["len_motion_obj"] = float(tm[2][mv].mean())
        rows.append(r)
        print(f"{name} frame {f}: " + " ".join(f"{k} {v:.4f}" for k, v in r.items() if k != "frame"))
    for r in rows:
        assert r["motion_obj"] < r["camera_obj"], (name, r)
        assert r["motion_all"] <= r["camera_all"], (name, r)
    for k in ("spatial_obj", "camera_obj", "motion_obj", "spatial_all", "camera_all", "motion_all"):
        assert max(r[k] for r in rows) <= BOUNDS[name, k], (name, k)
