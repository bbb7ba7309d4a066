"""Parity with the oracle at the far ends of the ranges include/rbrt_gpu.h accepts, where packed fields and fixed-size tables live:

* max_depth up to 1024 (history rows and iteration counters sized by the depth, the pool's `depth_cap` growing and shrinking, the
  tail kernel running paths to their end);
* 65 535 scene elements (sphere and pending-hit element ids in 16 bits with 0xFFFF = none, the u16 scatter history, the element id
  of a mesh = n_spheres + mesh index), and thousands of meshes of which many lose every triangle to the SIMD tail rule;
* the camera-ray cone table (CULL_MAX = 256 entries of elements x frames: culling on at 256, off above);
* image shapes of one row or one column and odd widths, very long sample runs of one pixel, tile and sample shards.

Every comparison is bit-exact, like the rest of the suite, and every test asserts that it reaches the regime it is about."""
import ctypes as C

import numpy as np
import pytest

import rbrt_b200 as R
from rbrt_b200 import _abi, synth
from rbrt_b200.vec3 import Vec3

from . import scenes as S
from .test_gpu_trace import MODES, assert_same

pytestmark = pytest.mark.gpu
P = C.POINTER


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def assert_images_equal(got, ref, what):
    ne = (bits(got) != bits(ref)).any(axis=-1)
    assert not ne.any(), f"{what}: {int(ne.sum())} of {ne.size} pixels differ, first at {np.argwhere(ne)[0]}: {got[ne][0]} vs {ref[ne][0]}"


def accum(scene, cam, spp, **kw):
    """rbrt_gpu_render_accum_device: the per-pixel sums (W x H x 4 f32) and the stats."""
    import torch
    W, H = cam.img_width_pix, cam.img_height_pix
    buf = torch.empty(H * W * 4, dtype=torch.float32, device="cuda")
    st = _abi.StatsC()
    _abi.check(_abi.lib().rbrt_gpu_render_accum_device(scene.handle(), cam.to_c(), spp, R.render.make_opts(**kw), buf.data_ptr(),
                                                       torch.cuda.current_stream().cuda_stream, st))
    torch.cuda.synchronize()
    return buf.cpu().numpy(), st.as_dict()


# ============================================================================== a. depth budgets

DEPTH_WAYS = [{}, {"no_tail_kernel": True}, {"trace_mode": _abi.TRACE_BRUTE}, {"batch_paths": 700}]


@pytest.mark.parametrize("depth", [51, 64, 65, 200, 1024])
def test_deep_paths(gpu, oracle, depth):
    """Paths that scatter far more than 64 times, at depth budgets past 50 up to the limit: the tail kernel, pure wavefront iterations,
    the brute-force integrator and many small batches all give the oracle's image and ray count."""
    scene, cam = S.deep_path_scene(), S.deep_path_camera(32, 24)
    ost = {}
    ref = oracle.OracleScene.from_scene(scene).render_hdr(cam.to_c(), 2, _abi.RenderOptsC(seed=19, max_depth=depth), ost)
    if depth >= 200:
        assert ost["rays"] > 65 * ost["paths"], ost
    assert (ref > 0).any(axis=2).sum() > 32 * 24 // 8                     # not a black image
    for kw in DEPTH_WAYS:
        st = {}
        assert_images_equal(R.render_scene_hdr(cam, 2, scene, stats=st, seed=19, max_depth=depth, **kw), ref, f"depth {depth} {kw}")
        assert st["rays"] == ost["rays"] and st["paths"] == ost["paths"] == 32 * 24 * 2, (kw, st)
    assert np.array_equal(R.render_scene(cam, 2, scene, seed=19, max_depth=depth).pixels,
                          oracle.OracleScene.from_scene(scene).render(cam.to_c(), 2, _abi.RenderOptsC(seed=19, max_depth=depth)))


def test_two_mirrors_use_the_whole_budget(gpu):
    scene, cam = S.two_mirror_scene(), S.two_mirror_camera(8, 4)
    for kw in DEPTH_WAYS[:2]:
        st = {}
        img = R.render_scene_hdr(cam, 3, scene, stats=st, seed=3, max_depth=1024, **kw)
        assert st["rays"] == 1025 * st["paths"] and st["paths"] == 8 * 4 * 3 and not img.any(), (kw, st)
    with pytest.raises(_abi.RbrtGpuError):
        R.render_scene_hdr(cam, 1, scene, max_depth=1025)


def test_wave_pool_lifecycle_across_depths(gpu, oracle):
    """One process, wavefront pool 0 of the device: depth 50, then 1024 (the pool's depth_cap must grow), then rbrt_gpu_trace_rays in
    WAVEFRONT mode with more rays than the pool holds (it re-allocates with room for depth 50 only), then 1024 again (must grow again),
    then 50.  Every result equals its reference."""
    scene, cam = S.deep_path_scene(), S.deep_path_camera(24, 16)
    osc = oracle.OracleScene.from_scene(scene)
    refs = {d: osc.render_hdr(cam.to_c(), 2, _abi.RenderOptsC(seed=23, max_depth=d)) for d in (50, 1024)}
    rays = S.random_rays(300000, (0.0, 0.0, -6.0), 0.6, 9)                # more rays than the renders' pools hold (24 x 16 x 2 paths)
    want = osc.hit(rays)
    assert (want["kind"] == 1).sum() > 100000
    for step, d in enumerate((50, 1024, None, 1024, 50)):
        if d is None:
            assert_same(scene.hit(rays, _abi.TRACE_WAVEFRONT), want, "wavefront trace between renders")
        else:
            assert_images_equal(R.render_scene_hdr(cam, 2, scene, seed=23, max_depth=d), refs[d], f"step {step}: depth {d}")


def test_frame_accumulators_across_image_sizes(gpu):
    """The accumulators rbrt_gpu_render / rbrt_gpu_render_frames_device keep per pool are reused across calls: a large lone frame, then
    four small frames per batch, then four frames of a size in between, all on pool 0.  Each frame equals its lone render.  (The frames
    added to a pool once got the size of the image at hand instead of the pool's, and the last call was refused with a CUDA error.)"""
    scene = S.small_mesh_scene(2)
    R.render_scene_hdr(S.example_camera(128, 96), 1, scene, seed=1)
    cb = synth.example_camera_blueprint()
    for w, h in ((16, 8), (64, 48)):
        cams = [R.Camera.new(Vec3(cb.camera_position.x + 0.4 * k, cb.camera_position.y, cb.camera_position.z), cb.camera_look_at, cb.camera_up,
                             h, w, cb.camera_focal_length_mm) for k in range(4)]
        want = [R.render_scene_hdr(c, 2, scene, seed=30 + k) for k, c in enumerate(cams)]
        pipe = R.FramePipeline(w, h, depth=1, hdr=True, frames_per_batch=4)
        got = []
        for k, c in enumerate(cams):
            got += pipe.submit(c, 2, scene, tag=k, seed=30 + k)
        got += pipe.drain()
        assert [t for _, t in got] == [0, 1, 2, 3]
        for img, t in got:
            assert np.array_equal(bits(img), bits(want[t])), f"{w}x{h} frame {t} differs"


def test_frame_pipeline_deep_paths(gpu):
    """FramePipeline, two frames per batch, depth 300: the same images as lone renders."""
    scene = S.deep_path_scene()
    cams = [R.Camera.new(Vec3(0.1 * k - 0.2, 0.05 * k, -0.2), Vec3(0.05 - 0.03 * k, 0.02, -1.0), Vec3(0, 1, 0), 16, 24, 24.0) for k in range(5)]
    want = [R.render_scene_hdr(c, 2, scene, seed=50 + k, max_depth=300) for k, c in enumerate(cams)]
    pipe = R.FramePipeline(24, 16, depth=2, hdr=True, frames_per_batch=2)
    got = []
    for k, c in enumerate(cams):
        got += pipe.submit(c, 2, scene, tag=k, seed=50 + k, max_depth=300)
    got += pipe.drain()
    assert [t for _, t in got] == list(range(len(cams)))
    for img, t in got:
        assert np.array_equal(bits(img), bits(want[t])), f"frame {t} differs"


# ============================================================================== b. element counts

LIMIT = 65535


def sphere_descs(n, rng):
    """n rbrt_sphere_desc (9 x 32 bit each) built in numpy: small Lambertian spheres (material kind 0)."""
    a = np.zeros((n, 9), np.float32)
    a[:, :3] = rng.uniform(-50, 50, (n, 3))
    a[:, 3] = 0.1
    a[:, 5:8] = 0.5
    return a, C.cast(a.ctypes.data, P(_abi.SphereDescC))


def create(entry, ns, nt=0, nm=0, seed=0):
    """Scene of ns spheres, nt BasicTriangle elements and nm one-triangle meshes through `entry` ("plain": rbrt_gpu_scene_create,
    "elements": rbrt_gpu_scene_create_elements).  Returns (rc, handle, message)."""
    lib = _abi.lib()
    rng = np.random.default_rng(seed)
    sph, sph_p = sphere_descs(ns, rng)
    tri = np.zeros((max(nt, 1), 14), np.float32)
    tri[:, :9] = rng.uniform(-50, 50, (max(nt, 1), 9))
    tri[:, 10:13] = 0.5
    verts = np.array([[0, 0, -60, 1, 0, -60, 0, 1, -60]], np.float32)
    meshes = (_abi.MeshDescC * max(nm, 1))(*[_abi.MeshDescC(verts.ctypes.data_as(P(C.c_float)), 1, _abi.MaterialC(1, _abi.Vec3C(0.9, 0.9, 0.9), 0.1))
                                               for _ in range(nm)])
    opts = _abi.SceneOptsC(8, 0, 0.0, 0)
    h = C.c_void_p()
    if entry == "plain":
        assert nt == 0
        rc = lib.rbrt_gpu_scene_create(sph_p, ns, meshes, nm, opts, C.byref(h))
    else:
        order = np.zeros((ns + nt, 2), np.uint32)
        order[ns:, 0] = _abi.ELEM_TRIANGLE
        order[:ns, 1] = np.arange(ns)
        order[ns:, 1] = np.arange(nt)
        rc = lib.rbrt_gpu_scene_create_elements(C.cast(order.ctypes.data, P(_abi.ElementRefC)), ns + nt, sph_p, ns,
                                                C.cast(tri.ctypes.data, P(_abi.TriangleDescC)), nt, meshes, nm, opts, C.byref(h))
    return rc, h, lib.rbrt_last_error().decode()


@pytest.mark.parametrize("entry,mix", [("plain", (1, 0, 0)), ("elements", (1, 0, 0)), ("elements", (0.9, 0.1, 0)),
                                       ("plain", (0, 0, 3)), ("elements", (0, 0, 3)), ("elements", (0.8, 0.2, 3))])
def test_element_limit(gpu, entry, mix):
    """65 535 elements (spheres + BasicTriangles + meshes) are accepted, 65 536 refused on the host with the reason."""
    lib = _abi.lib()
    for n, ok in ((LIMIT, True), (LIMIT + 1, False)):
        nm = mix[2]
        nt = int((n - nm) * mix[1])
        ns = n - nm - nt
        rc, h, msg = create(entry, ns, nt, nm)
        if ok:
            assert rc == 0, msg
            info = _abi.SceneInfoC()
            _abi.check(lib.rbrt_gpu_scene_info(h, info))
            assert (info.num_spheres, info.num_meshes) == (ns + nt, nm)
            _abi.check(lib.rbrt_gpu_scene_destroy(h))
        else:
            assert rc == _abi.E_INVALID and "65535" in msg and not h.value, (rc, msg)


def high_index_scene():
    """65 534 spheres + 1 mesh (element id 65 534).  Everything the camera sees sits at indices above 32 767: sixteen spheres at
    40 000.., their exact duplicates with other materials at 50 000.. (the lower index must win the tie) and the ground sphere at
    65 533.  The other spheres are small ones behind the camera, each with its own material, so a truncated element id would pick
    a wrong material."""
    rng = np.random.default_rng(65534)
    mats = [R.Lambertian(Vec3(0.7, 0.3, 0.2)), R.Metal(Vec3(0.9, 0.9, 0.9), 0.05), R.Dielectric(1.6), R.Lambertian(Vec3(0.2, 0.6, 0.8))]
    pos = rng.uniform((-60, -60, 150), (60, 60, 400), (65534, 3)).astype(np.float32)
    alb = rng.uniform(0.05, 0.95, (65534, 3)).astype(np.float32)
    els = [R.Sphere(Vec3(*map(float, p)), 0.5, R.Lambertian(Vec3(*map(float, a))) if i % 3 else R.Metal(Vec3(*map(float, a)), 0.2))
           for i, (p, a) in enumerate(zip(pos, alb))]
    for k in range(16):
        c = Vec3(-1.5 + 1.0 * (k % 4), 0.4 + 0.8 * (k // 4), -6.0 - 0.3 * (k % 3))
        els[40000 + k] = R.Sphere(c, 0.4, mats[k % 4])
        els[50000 + k] = R.Sphere(c, 0.4, mats[(k + 1) % 4])
    els[65533] = R.Sphere(Vec3(0.0, -1000.0, -6.0), 1000.0, R.Lambertian(Vec3(0.5, 0.5, 0.3)))
    sc = R.Scene()
    sc.elements = els
    sc.triangle_meshes.append(R.TriangleMesh.from_triangles(synth.displaced_icosphere(2, 0.8, (2.5, 1.0, -7.0)), mats[1]))
    return sc


def test_high_element_indices(gpu, oracle):
    scene = high_index_scene()
    cam = R.Camera.new(Vec3(0.0, 1.0, 0.0), Vec3(0.0, -0.08, -1.0), Vec3(0, 1, 0), 24, 32, 18.0)
    osc = oracle.OracleScene.from_scene(scene)
    rays = np.concatenate([R.primary_rays(cam, 5, 0), S.random_rays(3000, (0.0, 0.5, -6.0), 1.5, 3)], 0)
    want = osc.hit(rays)
    hit_spheres = set(want["elem_idx"][want["kind"] == 0].tolist())
    assert {40000, 40007, 40015, 65533} <= hit_spheres and not hit_spheres & set(range(50000, 50016)), sorted(hit_spheres)[:20]
    assert (want["elem_idx"][want["kind"] == 0] > 32767).sum() > 1000 and (want["kind"] == 1).sum() > 50
    for mode in MODES:
        assert_same(scene.hit(rays, mode), want, f"65534 spheres + 1 mesh, trace mode {mode}")
    ost = {}
    ref = osc.render_hdr(cam.to_c(), 2, _abi.RenderOptsC(seed=13), ost)
    for kw in [{}, {"no_tail_kernel": True}]:
        st = {}
        assert_images_equal(R.render_scene_hdr(cam, 2, scene, stats=st, seed=13, **kw), ref, f"high indices {kw}")
        assert st["rays"] == ost["rays"] > 3 * st["paths"] // 2


def n_tested(n, lanes):
    r = n % lanes
    return n if (r == 0 or 2 * r >= lanes) else n - r


@pytest.mark.parametrize("lanes", [8, 4])
def test_thousands_of_meshes(gpu, oracle, lanes):
    """4 096 meshes of 1..9 triangles in a 64 x 64 grid (with AVX lanes the meshes of 1, 2 and 3 triangles lose them all to the tail
    rule, interleaved with live meshes) + a ground sphere: scene info, the three trace modes and a render against the oracle."""
    rng = np.random.default_rng(4096)
    mats = [R.Lambertian(Vec3(0.6, 0.3, 0.2)), R.Metal(Vec3(0.9, 0.9, 0.9), 0.05), R.Dielectric(1.6)]
    sc = R.Scene(simd_lanes=lanes)
    sc.elements.append(R.Sphere(Vec3(0.0, -1000.0, -20.0), 1000.0, R.Lambertian(Vec3(0.3, 0.5, 0.3))))
    sizes = []
    for k in range(4096):
        n = 1 + (k * 7 + k // 64) % 9
        centre = np.array((-16.0 + 0.5 * (k % 64), 0.3 + 0.5 * (k // 64), -20.0), np.float32)
        tris = (centre + rng.uniform(-0.3, 0.3, (n, 3, 3))).astype(np.float32)
        sc.triangle_meshes.append(R.TriangleMesh.from_triangles(tris, mats[k % 3]))
        sizes.append(n)
    assert sc.info()["num_triangles_tested"] == sum(n_tested(n, lanes) for n in sizes)
    if lanes == 8:
        assert sum(n <= 3 for n in sizes) > 1000
    cam = R.Camera.new(Vec3(0.0, 16.0, 10.0), Vec3(0.0, -0.02, -1.0), Vec3(0, 1, 0), 48, 64, 14.0)
    osc = oracle.OracleScene.from_scene(sc)
    rays = np.concatenate([R.primary_rays(cam, 2, 0), S.random_rays(4000, (0.0, 16.0, -20.0), 8.0, 5)], 0)
    want = osc.hit(rays)
    hit_meshes = want["elem_idx"][want["kind"] == 1]
    assert len(np.unique(hit_meshes)) > 500
    assert all(n_tested(sizes[m], lanes) > 0 for m in np.unique(hit_meshes))
    for mode in MODES:
        assert_same(sc.hit(rays, mode), want, f"4096 meshes lanes {lanes} mode {mode}")
    ref = osc.render_hdr(cam.to_c(), 2, _abi.RenderOptsC(seed=8))
    for kw in [{}, {"no_tail_kernel": True}]:
        assert_images_equal(R.render_scene_hdr(cam, 2, sc, seed=8, **kw), ref, f"4096 meshes lanes {lanes} {kw}")


# ============================================================================== c. the camera-ray cone table

def cone_scene(n_tab):
    """n_tab - 1 spheres (some pixel-sized) + 1 mesh: n_tab entries of the cone table per frame."""
    rng = np.random.default_rng(n_tab)
    mats = [R.Lambertian(Vec3(0.6, 0.3, 0.2)), R.Metal(Vec3(0.9, 0.9, 0.9), 0.05), R.Dielectric(1.6)]
    sc = R.Scene()
    sc.elements.append(R.Sphere(Vec3(0.0, -1000.0, -10.0), 1000.0, mats[0]))
    for k in range(n_tab - 2):
        c = rng.uniform((-6, 0, -14), (6, 5, -6))
        sc.elements.append(R.Sphere(Vec3(*map(float, c)), float(rng.choice([0.02, 0.3, 0.6])), mats[k % 3]))
    sc.triangle_meshes.append(R.TriangleMesh.from_triangles(synth.displaced_icosphere(2, 0.8, (1.0, 1.0, -8.0)), mats[2]))
    return sc


def cone_cams(n):
    return [R.Camera.new(Vec3(0.3 * k, 2.0, 2.0), Vec3(-0.03 * k, -0.1, -1.0), Vec3(0, 1, 0), 24, 40, 20.0) for k in range(n)]


@pytest.mark.parametrize("n_tab", [256, 257])
def test_cone_table_lone_frames(gpu, oracle, n_tab):
    sc = cone_scene(n_tab)
    assert len(sc.elements) + len(sc.triangle_meshes) == n_tab
    cam = cone_cams(1)[0]
    ref = oracle.OracleScene.from_scene(sc).render_hdr(cam.to_c(), 2, _abi.RenderOptsC(seed=61, max_depth=4))
    assert_images_equal(R.render_scene_hdr(cam, 2, sc, seed=61, max_depth=4), ref, f"{n_tab} cone-table entries")


@pytest.mark.parametrize("n_tab,fpb", [(64, 4), (65, 4), (128, 2), (129, 2)])
def test_cone_table_frames_per_batch(gpu, oracle, n_tab, fpb):
    """elements x frames of one batch = 256 (culling on) and 258 / 260 (off): every frame equals its lone render and the oracle."""
    sc = cone_scene(n_tab)
    cams = cone_cams(fpb)
    osc = oracle.OracleScene.from_scene(sc)
    pipe = R.FramePipeline(40, 24, depth=1, hdr=True, frames_per_batch=fpb)
    got = []
    for k, c in enumerate(cams):
        got += pipe.submit(c, 2, sc, tag=k, seed=70 + k, max_depth=4)
    got += pipe.drain()
    assert [t for _, t in got] == list(range(fpb))
    for img, t in got:
        lone = R.render_scene_hdr(cams[t], 2, sc, seed=70 + t, max_depth=4)
        assert np.array_equal(bits(img), bits(lone)), f"frame {t} vs its lone render"
        assert_images_equal(lone, osc.render_hdr(cams[t].to_c(), 2, _abi.RenderOptsC(seed=70 + t, max_depth=4)), f"frame {t} vs the oracle")


# ============================================================================== d. image shapes and long sample runs

def test_one_pixel_long_sample_run(gpu, oracle):
    """One pixel, 65 537 samples: the per-pixel sum runs in sample order across batches (default, small batches, a small pool limit)."""
    scene, cam = S.small_mesh_scene(2), S.example_camera(1, 1)
    ost = {}
    ref = oracle.OracleScene.from_scene(scene).render_hdr(cam.to_c(), 65537, _abi.RenderOptsC(seed=99), ost)
    lib = _abi.lib()
    for kw, limit in [({}, 0), ({"batch_paths": 32 * 4099}, 0), ({}, 176 * 32 * 1000)]:
        _abi.check(lib.rbrt_gpu_set_pool_limit(limit))
        try:
            st = {}
            assert_images_equal(R.render_scene_hdr(cam, 65537, scene, stats=st, seed=99, **kw), ref, f"1x1 {kw} pool limit {limit}")
        finally:
            _abi.check(lib.rbrt_gpu_set_pool_limit(0))
        assert st["rays"] == ost["rays"] and st["paths"] == 65537
        if kw or limit:
            assert st["iterations"] >= 16, st                             # several batches


@pytest.mark.parametrize("w,h", [(1, 4099), (4099, 1), (8193, 3)])
def test_extreme_image_shapes_and_shards(gpu, oracle, w, h):
    """One column, one row and an odd 8193 x 3 strip (ragged 8 x 4 tiles): the image, tile shards of 3 and 8 (disjoint, their sum is the
    unsharded accumulator bit for bit, each equals the oracle's shard) and sample shards with more shards than samples (some empty)."""
    scene, cam = S.small_mesh_scene(2), S.example_camera(w, h)
    osc = oracle.OracleScene.from_scene(scene)
    ref = osc.render_hdr(cam.to_c(), 2, _abi.RenderOptsC(seed=6))
    assert_images_equal(R.render_scene_hdr(cam, 2, scene, seed=6), ref, f"{w}x{h}")
    full, st_full = accum(scene, cam, 2, seed=6)
    assert np.array_equal(bits(full), bits(osc.render_accum(cam.to_c(), 2, _abi.RenderOptsC(seed=6))))
    for n in (3, 8):
        parts = [accum(scene, cam, 2, seed=6, shard_mode=_abi.SHARD_TILES, shard_rank=r, shard_count=n) for r in range(n)]
        assert np.array_equal(bits(np.sum([p for p, _ in parts], 0, dtype=np.float32)), bits(full)), f"tiles x{n}"
        assert sum(s["paths"] for _, s in parts) == st_full["paths"] and sum(s["rays"] for _, s in parts) == st_full["rays"]
        for r, (p, _) in enumerate(parts):
            want = osc.render_accum(cam.to_c(), 2, _abi.RenderOptsC(seed=6, shard_mode=_abi.SHARD_TILES, shard_rank=r, shard_count=n))
            assert np.array_equal(bits(p), bits(want)), f"tile shard {r}/{n}"
    spp, n = 3, 8
    empty = 0
    for r in range(n):
        p, s = accum(scene, cam, spp, seed=6, shard_mode=_abi.SHARD_SAMPLES, shard_rank=r, shard_count=n)
        want = osc.render_accum(cam.to_c(), spp, _abi.RenderOptsC(seed=6, shard_mode=_abi.SHARD_SAMPLES, shard_rank=r, shard_count=n))
        assert np.array_equal(bits(p), bits(want)), f"sample shard {r}/{n}"
        if spp * r // n == spp * (r + 1) // n:
            empty += 1
            assert not p.any() and s["paths"] == s["rays"] == 0
    assert empty == n - spp
