"""Scenes updated in place (rbrt_gpu_scene_update_mesh / _mesh_device / _update_elements; csrc/update.cu, csrc/api.cu).

The traversal's result does not depend on the tree's shape (DESIGN.md section 2), so a refit tree — the creation's topology with new
boxes — must give the oracle's images and hits for the new geometry bit for bit, like a freshly created scene.  And because min / max
are exact, a refit with the unchanged vertices must reproduce the creation's tree: the node-visit counters are equal.  Every
comparison below is bit-exact, and every test asserts that it reaches the regime it is about."""
import ctypes as C

import numpy as np
import pytest

import rbrt_b200 as R
from rbrt_b200 import _abi, synth
from rbrt_b200.vec3 import Vec3

from . import scenes as S
from .test_gpu_trace import MODES, assert_same

pytestmark = pytest.mark.gpu
MESH_AT = np.float32([5.0, 1.4, -12.5])
W, H, SPP, SEED = 48, 36, 2, 11


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def assert_images_equal(got, ref, what):
    ne = (bits(got) != bits(ref)).reshape(got.shape[0], got.shape[1], -1).any(axis=-1)
    assert not ne.any(), f"{what}: {int(ne.sum())} of {ne.size} pixels differ, first at {np.argwhere(ne)[0]}"


def fresh(scene):
    """A newly created scene with the same contents and options (the reference an updated scene must equal)."""
    return R.Scene(list(scene.elements), [R.TriangleMesh(m.triangles, m.material) for m in scene.triangle_meshes],
                   simd_lanes=scene.simd_lanes, leaf_size=scene.leaf_size, box_pad_rel=scene.box_pad_rel, sah=scene.sah)


def cam(w=W, h=H):
    return S.example_camera(w, h)


def hdr(scene, c=None, **kw):
    return R.render_scene_hdr(c or cam(), SPP, scene, seed=SEED, **kw)


def oracle_hdr(oracle, scene, c=None):
    return oracle.OracleScene.from_scene(scene).render_hdr((c or cam()).to_c(), SPP, _abi.RenderOptsC(seed=SEED))


def mesh_scene(subdiv=3, **kw):
    return S.small_mesh_scene(subdiv=subdiv, **kw)


# ---------------------------------------------------------------- deformations (seeded, same triangle count)
def noise(t, s=0.05, seed=1):
    return (t + np.random.default_rng(seed).normal(size=t.shape).astype(np.float32) * np.float32(s)).astype(np.float32)


def twist(t, turns=0.6):
    c = t - MESH_AT
    a = (c[..., 1] * np.float32(turns)).astype(np.float32)
    x = c[..., 0] * np.cos(a) - c[..., 2] * np.sin(a)
    z = c[..., 0] * np.sin(a) + c[..., 2] * np.cos(a)
    return (np.stack([x, c[..., 1], z], -1) + MESH_AT).astype(np.float32)


def translate(t, d=(500.0, 0.0, 0.0)):
    return (t + np.float32(d)).astype(np.float32)


def scale(t, f):
    return ((t - MESH_AT) * np.float32(f) + MESH_AT).astype(np.float32)


def scramble(t, seed=3):
    """Every triangle moved to another one's place: the topology the tree was built for no longer fits the geometry at all."""
    p = np.random.default_rng(seed).permutation(len(t))
    return (t - t.mean(1, keepdims=True) + t[p].mean(1, keepdims=True)).astype(np.float32)


DEFORMS = {"noise": noise, "twist": twist, "translate500": translate, "scale100": lambda t: scale(t, 100.0),
           "scale0.1": lambda t: scale(t, 0.1), "scale0.01": lambda t: scale(t, 0.01)}


def count_stats(scene, **kw):
    st = {}
    img = hdr(scene, stats=st, count_visits=True, **kw)
    return img, {k: st[k] for k in ("rays", "node_visits", "tri_tests", "traversed_rays", "tail_node_visits", "tail_tri_tests",
                                    "tail_traversed_rays")}


# ============================================================================== 1. identity refit
@pytest.mark.parametrize("leaf", [1, 2, 4, 8])
@pytest.mark.parametrize("sah", [True, False])
def test_identity_refit_reproduces_the_creation(gpu, leaf, sah):
    scene = mesh_scene(subdiv=6, leaf_size=leaf, sah=sah)                 # C2's 81 920-triangle displaced icosphere + C1's spheres
    c = cam(64, 48)
    img0, st0 = count_stats(scene, c=c)
    u8 = R.render_scene(c, SPP, scene, seed=SEED).pixels
    assert st0["traversed_rays"] > 500 and st0["node_visits"] > st0["traversed_rays"], st0
    scene.update_mesh(0, scene.triangle_meshes[0].triangles)
    img1, st1 = count_stats(scene, c=c)
    assert_images_equal(img1, img0, "identity refit")
    assert st1 == st0, (st0, st1)
    assert np.array_equal(R.render_scene(c, SPP, scene, seed=SEED).pixels, u8)


# ============================================================================== 2. deformed meshes
@pytest.mark.parametrize("name", list(DEFORMS))
def test_deformed_mesh_equals_oracle_and_fresh_scene(gpu, oracle, name):
    scene = mesh_scene()
    hdr(scene)                                                            # the old tree is built and used
    new = DEFORMS[name](scene.triangle_meshes[0].triangles)
    scene.update_mesh(0, new)
    ref = oracle_hdr(oracle, scene)
    assert_images_equal(hdr(scene), ref, f"{name}: refit vs oracle")
    assert_images_equal(hdr(fresh(scene)), ref, f"{name}: fresh vs oracle")
    centre = new.reshape(-1, 3).mean(0)
    spread = float(np.abs(new.reshape(-1, 3) - centre).max())
    rays = S.random_rays(20000, centre, spread, seed=5)
    want = oracle.OracleScene.from_scene(scene).hit(rays)
    # x0.01: edges of ~0.006 give |det| < 1e-3, which the reference culls (triangle.rs): the mesh is invisible, and the refit's tiny
    # boxes on a grid of ~1e-7 steps must not make it visible either
    assert (want["kind"] == _abi.HIT_MESH).sum() > 500 if name != "scale0.01" else (want["kind"] == _abi.HIT_MESH).sum() == 0
    for mode in MODES:
        assert_same(scene.hit(rays, mode), want, f"{name} mode {mode}")


def test_small_mesh_near_the_origin_far_rays_after_refit(gpu, oracle):
    """The padding floor 2^-21 * (mx + 1000) is re-derived by the refit: a small mesh near the world origin, deformed, hit by
    edge-aimed rays from 990 units away (the regime of test_gpu_trace.py::test_small_mesh_near_the_world_origin_far_ray_origins)."""
    tris = synth.displaced_icosphere(2, 0.3, (0.05, 0.02, -0.03))
    scene = R.Scene()
    scene.triangle_meshes.append(R.TriangleMesh.from_triangles(synth.displaced_icosphere(2, 5.0, (40.0, 0.0, 0.0)), R.Lambertian(Vec3(0.5, 0.5, 0.5))))
    scene.hit(S.random_rays(100, (40, 0, 0), 5.0))                         # built for a large mesh far away: a coarse grid
    new = noise(tris, 0.002, seed=9)
    scene.update_mesh(0, new)
    rays = S.edge_aimed_rays(new, 60000, 990.0, seed=2)
    want = oracle.OracleScene.from_scene(scene).hit(rays)
    assert (want["kind"] == 1).sum() > 30000
    for mode in MODES:
        assert_same(scene.hit(rays, mode), want, f"mode {mode}")


# ============================================================================== 3. degenerate updates
def _check_hits_and_image(oracle, scene, rays, what):
    want = oracle.OracleScene.from_scene(scene).hit(rays)
    for mode in MODES:
        assert_same(scene.hit(rays, mode), want, f"{what} mode {mode}")
    assert_images_equal(hdr(scene), oracle_hdr(oracle, scene), what)
    return want


def test_collapsed_and_nan_vertices(gpu, oracle):
    scene = mesh_scene()
    tris = scene.triangle_meshes[0].triangles
    rays = S.random_rays(8000, MESH_AT, 4.0, seed=1)
    hdr(scene)
    scene.update_mesh(0, np.broadcast_to(MESH_AT, tris.shape).copy())      # every vertex on one point
    want = _check_hits_and_image(oracle, scene, rays, "collapsed")
    assert (want["kind"] == _abi.HIT_MESH).sum() == 0
    bad = noise(tris, 0.05, seed=4)
    bad[::7, 1, 0] = np.nan
    bad[::11, :, 2] = np.nan
    scene.update_mesh(0, bad)
    want = _check_hits_and_image(oracle, scene, rays, "nan")
    assert (want["kind"] == _abi.HIT_MESH).sum() > 500


@pytest.mark.parametrize("lanes,n", [(8, 8 * 40 + 1), (8, 8 * 40 + 2), (8, 8 * 40 + 3), (4, 4 * 80 + 1), (8, 1), (8, 3), (8, 5)])
def test_tail_dropped_triangle_moved_far_outside(gpu, oracle, lanes, n):
    """The AABB covers the triangles the SIMD tail rule drops; moving one far outside grows the box (and the slab pre-test changes).
    n = 1 and 3 under AVX leave N_eff = 0; n = 5 keeps all five in one leaf (leaf_size 8: no nodes).  (N_eff = 1 is not reachable
    under either tail rule.)"""
    tris = synth.displaced_icosphere(3, 3.0, tuple(MESH_AT))[:n].copy()
    scene = R.Scene(simd_lanes=lanes, leaf_size=8 if n == 5 else 0)
    scene.elements += [R.Sphere(Vec3(0.0, -1000.0, -5.0), 1000.0, R.Lambertian(Vec3(0.2, 0.3, 0.1)))]
    scene.triangle_meshes.append(R.TriangleMesh.from_triangles(tris, R.Metal(Vec3(0.8, 0.7, 0.6), 0.1)))
    rays = S.random_rays(6000, MESH_AT, 3.0, seed=n)
    before = _check_hits_and_image(oracle, scene, rays, "before")
    moved = tris.copy()
    moved[-1] += np.float32([300.0, 200.0, -400.0])                        # the last triangle: dropped by the tail rule unless N_eff = n
    scene.update_mesh(0, moved)
    after = _check_hits_and_image(oracle, scene, rays, "after")
    n_eff = scene.info()["num_triangles_tested"]
    assert n_eff < n or n == 5
    if n_eff >= 8:
        assert (after["kind"] == _abi.HIT_MESH).sum() > 100 and (before["kind"] == _abi.HIT_MESH).sum() > 100


# ============================================================================== 4. rebuild mode
def test_rebuild_equals_a_fresh_build_and_refit_costs_visits(gpu, oracle):
    scene = mesh_scene(subdiv=4)
    hdr(scene)
    new = scramble(scene.triangle_meshes[0].triangles)
    scene.update_mesh(0, new, rebuild=True)
    img_rb, st_rb = count_stats(scene)
    assert_images_equal(img_rb, oracle_hdr(oracle, scene), "rebuild vs oracle")
    img_fr, st_fr = count_stats(fresh(scene))
    assert st_rb == st_fr and st_rb["traversed_rays"] > 500, (st_rb, st_fr)
    scene.update_mesh(0, scene.triangle_meshes[0].triangles * np.float32(1.0))    # unchanged values, the creation's topology is gone:
    _, st_id = count_stats(scene)                                                  # a refit of the rebuilt tree is that tree
    assert st_id == st_rb
    ref_scene = mesh_scene(subdiv=4)
    hdr(ref_scene)
    ref_scene.update_mesh(0, new)                                         # refit of the original topology to the scrambled mesh
    img_rf, st_rf = count_stats(ref_scene)
    assert_images_equal(img_rf, img_rb, "refit vs rebuild")
    assert st_rf["node_visits"] > st_rb["node_visits"], (st_rf, st_rb)


# ============================================================================== 5. several meshes
def test_update_one_of_several_meshes_and_its_material(gpu, oracle):
    scene = S.quirk_scene()
    scene.triangle_meshes.append(R.TriangleMesh.from_triangles(synth.displaced_icosphere(3, 1.0, (0.0, 1.5, -4.5)), R.Lambertian(Vec3(0.3, 0.6, 0.2))))
    c = S.quirk_camera(W, H)
    before = [m.triangles.copy() for m in scene.triangle_meshes]
    hdr(scene, c)
    scene.update_mesh(3, twist(before[3], 2.0), material=R.Metal(Vec3(0.9, 0.8, 0.7), 0.02))
    ref = oracle_hdr(oracle, scene, c)
    assert_images_equal(hdr(scene, c), ref, "mesh 3 twisted, lambertian -> metal")
    assert_images_equal(hdr(fresh(scene), c), ref, "fresh")
    scene.update_mesh(0, before[0], material=R.Dielectric(1.3))           # vertices unchanged, material kind changed
    assert_images_equal(hdr(scene, c), oracle_hdr(oracle, scene, c), "mesh 0 lambertian -> glass")
    for i in (1, 2):
        assert np.array_equal(scene.triangle_meshes[i].triangles, before[i])


# ============================================================================== 6. elements
def element_scene(n_spheres):
    rng = np.random.default_rng(n_spheres)
    scene = mesh_scene()
    for k in range(n_spheres):
        c = Vec3(*[float(x) for x in rng.uniform([-6, 0.2, -16], [8, 4, -6])])
        scene.elements.append(R.Sphere(c, float(rng.uniform(0.1, 0.4)), R.Lambertian(Vec3(0.5, 0.4, 0.3))))
    scene.elements.insert(2, R.BasicTriangle.new([(-2, 0, -8), (0, 0, -8), (-1, 2, -8)], R.Metal(Vec3(0.7, 0.7, 0.7), 0.0)))
    scene.elements.append(R.BasicTriangle.new([(1, 0, -6), (3, 0, -6), (2, 1.5, -6)], R.Lambertian(Vec3(0.9, 0.2, 0.2))))
    return scene


def moved_elements(elements, seed):
    rng = np.random.default_rng(seed)
    out = []
    for k, e in enumerate(elements):
        if isinstance(e, R.BasicTriangle):
            d = rng.uniform(-0.5, 0.5, 3)
            out.append(R.BasicTriangle.new([tuple(np.float32([c.x, c.y, c.z]) + np.float32(d)) for c in e.corners], R.Dielectric(1.5)))
        else:
            c = e.center
            mat = [R.Lambertian(Vec3(0.2, 0.8, 0.3)), R.Metal(Vec3(0.8, 0.8, 0.9), 0.2), R.Dielectric(1.6)][k % 3]
            out.append(R.Sphere(Vec3(c.x + float(rng.uniform(-0.4, 0.4)), c.y, c.z + float(rng.uniform(-0.4, 0.4))),
                                float(e.radius) * float(rng.uniform(0.7, 1.3)), mat))
    return out


@pytest.mark.parametrize("n_spheres,frames", [(20, 1), (20, 4), (300, 1)])
def test_elements_move_and_change_material(gpu, oracle, n_spheres, frames):
    """Spheres moved and resized, material kinds changed, BasicTriangles moved.  The camera-ray cone table (CULL_MAX = 256 entries of
    elements x frames, render.cu) is on below that and off above; it is built per frame from the block, so it follows the update."""
    scene = element_scene(n_spheres)
    assert (len(scene.elements) * frames <= 256) == (n_spheres == 20)
    c = cam()
    ref0 = oracle_hdr(oracle, scene, c)
    assert_images_equal(hdr(scene, c), ref0, "elements before")
    scene.update_elements(moved_elements(scene.elements, 1))
    ref1 = oracle_hdr(oracle, scene, c)
    assert (bits(ref0) != bits(ref1)).any(axis=2).sum() > W * H // 20
    if frames == 1:
        assert_images_equal(hdr(scene, c), ref1, "elements moved")
    else:
        import torch
        cams = (_abi.CameraC * frames)(*[c.to_c()] * frames)
        seeds = (C.c_uint64 * frames)(*[SEED] * frames)
        outs = [torch.empty(H * W * 3, dtype=torch.float32, device="cuda") for _ in range(frames)]
        ptrs = (C.c_void_p * frames)(*[o.data_ptr() for o in outs])
        s = torch.cuda.current_stream()
        _abi.check(_abi.lib().rbrt_gpu_render_frames_device(scene.handle(), cams, seeds, frames, SPP, R.render.make_opts(), None, ptrs,
                                                            s.cuda_stream, None))
        s.synchronize()
        for o in outs:
            assert_images_equal(o.cpu().numpy().reshape(H, W, 3), ref1, "elements moved, 4 frames per batch")


def test_element_refusals_leave_the_scene_unchanged(gpu):
    scene = element_scene(4)
    img = hdr(scene)
    els = moved_elements(scene.elements, 2)
    swapped = list(els)
    swapped[1], swapped[2] = swapped[2], swapped[1]                       # a sphere where a BasicTriangle was
    for bad, what in ((els[:-1], "elements"), (swapped, "kind")):
        with pytest.raises(_abi.RbrtGpuError) as e:
            scene.update_elements(bad)
        assert e.value.code == _abi.E_INVALID and what in str(e.value)
    lib = _abi.lib()
    order, sph, tris, ne, ns, nt = R.scene.element_arrays(els)
    sph[0].material.kind = 7
    assert lib.rbrt_gpu_scene_update_elements(scene.handle(), order, ne, sph, ns, tris, nt) == _abi.E_INVALID
    assert b"material" in lib.rbrt_last_error()
    assert lib.rbrt_gpu_scene_update_elements(scene.handle(), None, ne, sph, ns, tris, nt) == _abi.E_INVALID
    assert_images_equal(hdr(scene), img, "after refused updates")


# ============================================================================== 7. ordering
@pytest.mark.parametrize("depth,fpb", [(2, 1), (2, 4), (4, 1), (4, 4)])
def test_pipeline_frames_see_the_geometry_of_their_submission(gpu, oracle, depth, fpb):
    scene = mesh_scene()
    geo = {"A": scene.triangle_meshes[0].triangles.copy()}
    geo["B"] = twist(noise(geo["A"], 0.1), 1.0)
    c = cam()
    want = {}

    def expect(g, seed):
        if (g, seed) not in want:
            ref = R.Scene(list(scene.elements), [R.TriangleMesh(geo[g], scene.triangle_meshes[0].material)])
            want[(g, seed)] = oracle.OracleScene.from_scene(ref).render_hdr(c.to_c(), SPP, _abi.RenderOptsC(seed=seed))
        return want[(g, seed)]

    pipe = R.FramePipeline(W, H, depth=depth, hdr=True, frames_per_batch=fpb)
    got, k = [], 0
    for g, n in (("A", 3), ("B", 6), ("A", 2)):
        if k:
            scene.update_mesh(0, geo[g])
        for _ in range(n):
            got += pipe.submit(c, SPP, scene, tag=(g, k % 3), seed=k % 3)
            k += 1
    got += pipe.drain()
    assert [t for _, t in got] == [(g, j % 3) for j, g in enumerate("AAABBBBBBAA")]
    for img, (g, seed) in got:
        assert_images_equal(img, expect(g, seed), f"frame on {g}, seed {seed}")
    assert (bits(expect("A", 0)) != bits(expect("B", 0))).any(axis=2).sum() > 50


def test_enqueue_only_renders_on_two_streams_around_an_update_and_destroy(gpu, oracle):
    import torch
    scene = mesh_scene()
    a = scene.triangle_meshes[0].triangles.copy()
    b = scale(twist(a, 1.5), 1.3)
    c = cam()
    ref = {g: oracle.OracleScene.from_scene(R.Scene(list(scene.elements), [R.TriangleMesh(t, scene.triangle_meshes[0].material)]))
           .render_accum(c.to_c(), SPP, _abi.RenderOptsC(seed=SEED)) for g, t in (("A", a), ("B", b))}
    lib = _abi.lib()
    streams = [torch.cuda.Stream() for _ in range(3)]
    bufs = [torch.empty(H * W * 4, dtype=torch.float32, device="cuda") for _ in range(3)]

    def enqueue(k):
        _abi.check(lib.rbrt_gpu_render_accum_device(scene.handle(), c.to_c(), SPP, R.render.make_opts(seed=SEED, pool=k),
                                                    bufs[k].data_ptr(), streams[k].cuda_stream, None))
    enqueue(0)
    scene.update_mesh(0, b)
    enqueue(1)
    scene.update_mesh(0, a)
    enqueue(2)
    scene.update_mesh(0, b)
    scene.close()                                                         # destroyed with three frames and an update in flight
    torch.cuda.synchronize()
    for k, g in enumerate("ABA"):
        assert np.array_equal(bits(bufs[k].cpu().numpy()), bits(ref[g])), f"frame {k} on {g}"


# ============================================================================== 8. device pointers
@pytest.mark.parametrize("rebuild", [False, True])
def test_device_pointer_update_on_a_side_stream(gpu, oracle, rebuild):
    import torch
    scene = mesh_scene()
    hdr(scene)
    new = twist(scene.triangle_meshes[0].triangles, 1.2)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        t = torch.from_numpy(new.copy()).pin_memory().to("cuda", non_blocking=True)   # produced on the side stream
        scene.update_mesh_device(0, t, rebuild=rebuild, stream=s)
        t.fill_(float("nan"))                                             # overwritten in stream order right after the update
    s.synchronize()
    assert torch.isnan(t).all()
    assert np.array_equal(scene.triangle_meshes[0].triangles, new)        # the host mirror holds the values handed in
    assert_images_equal(hdr(scene), oracle_hdr(oracle, scene), "device-pointer update")


# ============================================================================== 9. communicator
@pytest.mark.parametrize("world", [2, 3])
def test_collective_render_after_update(gpu, oracle, world):
    lib = _abi.lib()
    devs = (C.c_int * world)(*([0] * world))
    _abi.check(lib.rbrt_gpu_init_multi(devs, world, _abi.TRANSPORT_PEER))
    try:
        scene = mesh_scene()
        hdr(scene)
        scene.update_mesh(0, twist(scene.triangle_meshes[0].triangles, 0.8), material=R.Metal(Vec3(0.8, 0.6, 0.4), 0.1))
        scene.update_elements(moved_elements(scene.elements, 3))
        assert_images_equal(hdr(scene), oracle_hdr(oracle, scene), f"{world} ranks after the update")
        scene.close()
    finally:
        _abi.check(lib.rbrt_gpu_comm_destroy())
    R.gpu_init(0)


# ============================================================================== 10. refusals
def test_mesh_update_refusals_leave_the_scene_unchanged(gpu):
    scene = mesh_scene()
    img = hdr(scene)
    tris = scene.triangle_meshes[0].triangles
    lib = _abi.lib()
    h = scene.handle()
    other = noise(tris, 0.3)
    cases = [
        (lambda: lib.rbrt_gpu_scene_update_mesh(h, 0, other.ctypes.data, len(tris) - 1, None, 0), "triangles"),
        (lambda: lib.rbrt_gpu_scene_update_mesh(h, 1, other.ctypes.data, len(tris), None, 0), "out of range"),
        (lambda: lib.rbrt_gpu_scene_update_mesh(h, 0, None, len(tris), None, 0), "null"),
        (lambda: lib.rbrt_gpu_scene_update_mesh(h, 0, other.ctypes.data, len(tris), C.byref(_abi.MaterialC(3, _abi.Vec3C(1, 1, 1), 0.0)), 0), "material"),
        (lambda: lib.rbrt_gpu_scene_update_mesh(h, 0, other.ctypes.data, len(tris), None, 2), "flags"),
        (lambda: lib.rbrt_gpu_scene_update_mesh_device(h, 0, None, len(tris), None, 0, None), "null"),
        (lambda: lib.rbrt_gpu_scene_update_mesh(None, 0, other.ctypes.data, len(tris), None, 0), "null"),
    ]
    for call, what in cases:
        assert call() == _abi.E_INVALID
        assert what in lib.rbrt_last_error().decode(), (what, lib.rbrt_last_error())
    assert_images_equal(hdr(scene), img, "after refused updates")
