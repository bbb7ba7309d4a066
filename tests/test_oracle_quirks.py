"""The oracle's restatement of the reference's unpinned behaviour (SURVEY.md parity-quirk checklist
Q1-Q15).  The reference has no test for these; each case below is derived by hand from the cited lines,
so that the oracle (the only pin for these rows) is itself pinned to a reading of the source."""
import numpy as np
import pytest

import rbrt_b200 as R
from rbrt_b200 import _abi
from rbrt_b200.vec3 import Vec3

from . import scenes as S


def one_tri_scene(tri, n_copies=8, **kw):
    sc = R.Scene(**kw)
    sc.triangle_meshes.append(R.TriangleMesh.from_triangles(np.array([tri] * n_copies, np.float32), R.Lambertian(Vec3(1, 1, 1))))
    return sc


def trace(oracle, scene, rays):
    return oracle.OracleScene.from_scene(scene).hit(np.array(rays, np.float32))


TRI = ((-1, -1, -5), (1, -1, -5), (0, 1, -5))


def test_q1_two_sided_and_absolute_determinant_cull(oracle):  # triangle.rs:198-200
    sc = one_tri_scene(TRI)
    h = trace(oracle, sc, [[0, 0, 0, 0, 0, -1], [0, 0, -10, 0, 0, 1]])
    assert list(h["kind"]) == [1, 1] and np.allclose(h["t"], 5.0)          # front and back face both hit
    assert np.array_equal(h["normal"], np.float32([[0, 0, 1], [0, 0, 1]]))    # geometric normal, never flipped (Q10)
    tiny = tuple(tuple(np.float32(c) * np.float32(0.01) + (0, 0, -5)[i] * np.float32(0.99) for i, c in enumerate(v)) for v in TRI)
    # 2*area = 0.0004 < 1e-3 -> |a| < eps even head-on: invisible
    assert trace(oracle, one_tri_scene(tiny), [[0, 0, 0, 0, 0, -1]])["kind"][0] == -1


def test_q2_t_window(oracle):  # triangle.rs:146,239-241: eps < t < 999.99994
    far = tuple((x * 400, y * 400, -999.0) for x, y, _ in TRI)
    assert trace(oracle, one_tri_scene(far), [[0, 0, 0, 0, 0, -1]])["kind"][0] == 1
    far = tuple((x * 400, y * 400, -1000.0) for x, y, _ in TRI)
    assert trace(oracle, one_tri_scene(far), [[0, 0, 0, 0, 0, -1]])["kind"][0] == -1   # t = 1000 > 999.99994
    near = tuple((x, y, -0.0009) for x, y, _ in TRI)
    assert trace(oracle, one_tri_scene(near), [[0, 0, 0, 0, 0, -1]])["kind"][0] == -1  # t < eps


def test_q3_first_index_wins_ties(oracle):  # triangle.rs:400
    h = trace(oracle, one_tri_scene(TRI, 16), [[0, 0, 0, 0, 0, -1]])
    assert h["tri_idx"][0] == 0


def test_q4_avx_tail_drop(oracle):  # mesh.rs:136-144 + triangle.rs:167
    for n, tested in [(8, 8), (9, 8), (10, 8), (11, 8), (12, 12), (13, 13), (15, 15), (1, 0), (3, 0), (4, 4)]:
        tris = [((-1, -1, -50 + i), (1, -1, -50 + i), (0, 1, -50 + i)) for i in range(n)]   # triangle i at z=-50+i: the LAST is nearest
        sc = R.Scene()
        sc.triangle_meshes.append(R.TriangleMesh.from_triangles(np.array(tris, np.float32), R.Lambertian(Vec3(1, 1, 1))))
        h = trace(oracle, sc, [[0, 0, 0, 0, 0, -1]])
        if tested == 0:
            assert h["kind"][0] == -1, n
        else:
            assert h["kind"][0] == 1 and h["tri_idx"][0] == tested - 1, (n, h["tri_idx"][0])
    # SSE lanes: N % 4 == 1 drops the last triangle (triangle.rs:296)
    for n, tested in [(5, 4), (6, 6), (7, 7), (8, 8), (9, 8)]:
        tris = [((-1, -1, -50 + i), (1, -1, -50 + i), (0, 1, -50 + i)) for i in range(n)]
        sc = R.Scene(simd_lanes=4)
        sc.triangle_meshes.append(R.TriangleMesh.from_triangles(np.array(tris, np.float32), R.Lambertian(Vec3(1, 1, 1))))
        assert trace(oracle, sc, [[0, 0, 0, 0, 0, -1]])["tri_idx"][0] == tested - 1, n


def test_q6_q8_dist_key_and_element_order(oracle):  # mesh.rs:247-249, scene.rs:23-41
    # direction of length 2: t = 2.5 but dist = 5; a sphere surface at dist 4.9 must win over the mesh at dist 5
    sc = one_tri_scene(TRI)
    sc.elements.append(R.Sphere(Vec3(0, 0, -5.9), 1.0, R.Lambertian(Vec3(1, 1, 1))))
    h = trace(oracle, sc, [[0, 0, 0, 0, 0, -2]])
    assert h["kind"][0] == 0 and abs(h["dist"][0] - 4.9) < 1e-5 and abs(h["t"][0] - 2.45) < 1e-5
    # exact tie in dist: the sphere (earlier in Scene::hit) wins, strict <
    sc = one_tri_scene(TRI)
    sc.elements.append(R.Sphere(Vec3(0, 0, -6.0), 1.0, R.Lambertian(Vec3(1, 1, 1))))
    h = trace(oracle, sc, [[0, 0, 0, 0, 0, -1]])
    assert h["kind"][0] == 0 and h["dist"][0] == 5.0


def test_q7_mesh_aabb_pretest(oracle):  # aabbox.rs:28-58
    L = oracle.lib()
    V, Ray = _abi.Vec3C, _abi.RayC
    assert L.rbrt_ref_kat_bbox_hit(V(-1, -1, -6), V(1, 1, -5), Ray(V(0, 0, 0), V(0, 0, -1))) == 1   # 0/0 lanes are NaN and ignored
    assert L.rbrt_ref_kat_bbox_hit(V(-1, -1, -6), V(1, 1, -5), Ray(V(0, 0, 0), V(0, 0, 1))) == 0    # t_max < 0
    assert L.rbrt_ref_kat_bbox_hit(V(-1, -1, -6), V(1, 1, -5), Ray(V(3, 0, 0), V(0, 0, -1))) == 0   # t_min > t_max
    # a flat mesh (zero-extent box) is still hit
    assert trace(oracle, one_tri_scene(TRI), [[0, 0, 0, 0.01, 0.01, -1]])["kind"][0] == 1


def test_q9_sphere_near_root_quirk(oracle):  # sphere.rs:42-55
    L = oracle.lib()
    V, Ray = _abi.Vec3C, _abi.RayC
    h = _abi.HitC()
    # origin just inside the surface heading out: near root < 0 -> far root used
    assert L.rbrt_ref_kat_sphere(V(0, 0, 0), 1.0, Ray(V(0, 0, 0.5), V(0, 0, 1)), 0.001, 2000.0, h) == 1 and h.t == 0.5
    # origin 0.0005 OUTSIDE the surface heading in: near root in [0, 0.001) -> rejected by dist, far root never tried
    assert L.rbrt_ref_kat_sphere(V(0, 0, 0), 1.0, Ray(V(0, 0, 1.0005), V(0, 0, -1)), 0.001, 2000.0, h) == 0
    # sphere behind the ray: both roots negative
    assert L.rbrt_ref_kat_sphere(V(0, 0, 5), 1.0, Ray(V(0, 0, 0), V(0, 0, -1)), 0.001, 2000.0, h) == 0
    # Q16 (found by the round-2 GPU parity runs): a sphere BEHIND the ray whose line is exactly tangent — discriminant == 0.0 — IS hit:
    # num_hits == 1, so the negative root is kept (the far root is only tried when there are two, sphere.rs:34-44) and only the
    # distance window is checked: l = (-1,0,-5), b = 10, c = 25, sol = 100 - 100 = 0, t = -5, point (0,0,5), normal (-1,0,0)
    assert L.rbrt_ref_kat_sphere(V(1, 0, 5), 1.0, Ray(V(0, 0, 0), V(0, 0, -1)), 0.001, 2000.0, h) == 1
    assert h.t == -5.0 and h.dist == 5.0 and (h.point.x, h.point.y, h.point.z) == (0.0, 0.0, 5.0) and (h.normal.x, h.normal.y, h.normal.z) == (-1.0, 0.0, 0.0)
    # ... while a line that cuts the same sphere (two roots, both negative) is a miss
    assert L.rbrt_ref_kat_sphere(V(0.5, 0, 5), 1.0, Ray(V(0, 0, 0), V(0, 0, -1)), 0.001, 2000.0, h) == 0
    # max_dist is inclusive for spheres (sphere.rs:52)
    assert L.rbrt_ref_kat_sphere(V(0, 0, -2001), 1.0, Ray(V(0, 0, 0), V(0, 0, -1)), 0.001, 2000.0, h) == 1
    # NaN discriminant: the reference panics (sphere.rs:33)
    assert L.rbrt_ref_kat_sphere(V(0, 0, 0), 1.0, Ray(V(0, 0, 0), V(float("nan"), 0, 1)), 0.001, 2000.0, h) == -1


def test_q10_sphere_normal_not_normalised(oracle):  # sphere.rs:56
    sc = R.Scene()
    sc.elements.append(R.Sphere(Vec3(0, 0, -10), 3.0, R.Lambertian(Vec3(1, 1, 1))))
    h = trace(oracle, sc, [[0, 0, 0, 0, 0, -1]])
    assert np.array_equal(h["normal"][0], np.float32([0, 0, 3]))


def scatter(oracle, mat, d, n, seed=1, pixel=0, sample=0, bounce=1, point=(0, 0, 0)):
    V, Ray = _abi.Vec3C, _abi.RayC
    att, out = V(), Ray()
    ok = oracle.lib().rbrt_ref_kat_scatter(mat.to_c(), Ray(V(9, 9, 9), V(*d)), V(*point), V(*n), seed, pixel, sample, bounce, att, out)
    return ok, (att.x, att.y, att.z), (out.origin.x, out.origin.y, out.origin.z), np.float32([out.direction.x, out.direction.y, out.direction.z])


def test_q12_metal(oracle):  # metal.rs:12-25
    m = R.Metal(Vec3(0.8, 0.7, 0.6), 0.0)
    ok, att, org, d = scatter(oracle, m, (1, -1, 0), (0, 2, 0), point=(1, 2, 3))
    assert ok == 1 and att == tuple(float(np.float32(x)) for x in (0.8, 0.7, 0.6)) and org == (1, 2, 3)
    assert np.allclose(d, [0.70710678, 0.70710678, 0], atol=1e-6)
    # reflected direction points into the surface w.r.t. the RAW normal -> absorbed
    ok, *_ = scatter(oracle, m, (1, 1, 0), (0, 2, 0))
    assert ok == 0


def test_q13_dielectric(oracle):  # dielectric.rs:11-85
    m = R.Dielectric(1.5)
    seen = set()
    for px in range(64):
        ok, att, _, d = scatter(oracle, m, (0, -1, 0), (0, 1, 0), pixel=px)
        assert ok == 1 and att == (1.0, 1.0, 1.0)
        seen.add(tuple(np.round(d, 5)))
    assert seen == {(0.0, 1.0, 0.0), (0.0, -1.0, 0.0)}            # head-on: reflect (4 %) or pass straight through
    # total internal reflection: discr <= 0 -> reflect_prob = 1
    for px in range(16):
        _, _, _, d = scatter(oracle, m, (1, 0.2, 0), (0, 1, 0), pixel=px)
        assert d[1] < 0
    # refracted direction is NOT re-normalised (dielectric.rs:81)
    L = oracle.lib()
    V = _abi.Vec3C
    out = V()
    assert L.rbrt_ref_kat_refract(V(1, -1, 0), V(0, 1, 0), 1.0 / 1.5, out) == 1
    assert abs(np.sqrt(out.x ** 2 + out.y ** 2) - 1.0) < 1e-6    # unit only because v^, n^ are unit and Snell holds
    assert abs(L.rbrt_ref_kat_schlick(1.0, 1.5) - 0.04) < 1e-7 and L.rbrt_ref_kat_schlick(1.5, 1.8) < L.rbrt_ref_kat_schlick(1.0, 1.8)


def test_lambertian_not_faced_forward(oracle):  # lambertian.rs:11-24
    m = R.Lambertian(Vec3(0.3, 0.4, 0.5))
    for px in range(32):
        ok, att, _, d = scatter(oracle, m, (0, 1, 0), (0, 5, 0), pixel=px)      # ray arrives from BELOW the surface
        assert ok == 1 and abs(np.linalg.norm(d) - 1) < 1e-6 and d[1] >= -1e-6  # still scatters around +n


def test_q14_camera(oracle):  # cam.rs:22-82
    cam = S.example_camera(256, 192)
    assert cam.up.as_tuple() == Vec3(0.0, 1.0, -0.4).as_tuple()        # stored raw
    assert cam.mm_per_pix_hor == float(np.float32(35.0) / np.float32(256))
    rays = oracle.primary_rays(cam.to_c(), 11, 0)
    assert np.array_equal(rays[:, :3], np.tile(np.float32([0, 5, 4]), (256 * 192, 1)))
    assert np.allclose(np.linalg.norm(rays[:, 3:], axis=1), 1.0, atol=1e-6)
    c = rays.reshape(192, 256, 6)[96, 128, 3:]                            # centre pixel looks along look_at (within the jitter)
    la = np.float32([0, -0.1, -1]) / np.linalg.norm([0, -0.1, -1])
    assert np.abs(c - la).max() < 2e-3
    assert not np.array_equal(rays, oracle.primary_rays(cam.to_c(), 11, 1))   # jitter depends on the sample index


def test_q11_q15_depth_and_output(oracle):  # lib.rs:54-66,99,101,118-120
    # two facing perfect mirrors: every path bounces until the depth budget is gone -> black
    sc = R.Scene()
    tris = np.array([((-50, -50, -5), (50, -50, -5), (0, 50, -5))] * 8 + [((-50, -50, 5), (0, 50, 5), (50, -50, 5))] * 8, np.float32)   # second mirror wound so its normal faces -z (metal absorbs on raw-normal back faces, Q12)
    sc.triangle_meshes.append(R.TriangleMesh.from_triangles(tris, R.Metal(Vec3(1, 1, 1), 0.0)))
    cam = R.Camera.new(Vec3(0, 0, 0), Vec3(0, 0, -1), Vec3(0, 1, 0), 2, 2, 2800.0)   # long lens: rays stay between the mirrors
    st = {}
    img = oracle.OracleScene.from_scene(sc).render_hdr(cam.to_c(), 1, _abi.RenderOptsC(seed=3), st)
    assert st["rays"] == 4 * 51 and not img.any()                        # 1 primary + 50 scattered rays per path
    st = {}
    oracle.OracleScene.from_scene(sc).render_hdr(cam.to_c(), 1, _abi.RenderOptsC(seed=3, max_depth=7), st)
    assert st["rays"] == 4 * 8
    # empty scene: pure sky; (sqrt(c) * 256) as u8 saturates at c = 1
    cam = R.Camera.new(Vec3(0, 0, 0), Vec3(0, 1, 0), Vec3(0, 0, 1), 1, 1, 28000.0)     # looking straight up: t = 1 -> white
    osc = oracle.OracleScene.from_scene(R.Scene())
    hdr = osc.render_hdr(cam.to_c(), 4, _abi.RenderOptsC(seed=0))
    assert np.allclose(hdr, 1.0, atol=1e-5), hdr
    rgb = osc.render(cam.to_c(), 4, _abi.RenderOptsC(seed=0))
    assert (rgb >= 254).all()


def test_depth_budget_up_to_the_limit(oracle):  # lib.rs:54-66; the product accepts max_depth <= 1024
    """Past 64 bounces (the size of a fixed attenuation store the oracle once had) up to the product's limit, and the limit itself."""
    osc = oracle.OracleScene.from_scene(S.two_mirror_scene())
    cam = S.two_mirror_camera()
    for depth in (64, 65, 1024):
        st = {}
        img = osc.render_hdr(cam.to_c(), 1, _abi.RenderOptsC(seed=3, max_depth=depth), st)
        assert st["rays"] == 4 * (depth + 1) and st["paths"] == 4 and not img.any()
    for depth in (1025, 2 ** 32 - 1):
        with pytest.raises(RuntimeError, match="max_depth"):
            osc.render_hdr(cam.to_c(), 1, _abi.RenderOptsC(seed=3, max_depth=depth))
        with pytest.raises(RuntimeError, match="max_depth"):
            osc.render(cam.to_c(), 1, _abi.RenderOptsC(seed=3, max_depth=depth))


def test_basic_triangle_element(oracle):  # triangle.rs:9-28, 92-130, 412-441
    """BasicTriangle as an element of Scene.elements: CCW unit normal, same Moeller-Trumbore arithmetic as the mesh sweep
    but no upper cap on t (a mesh triangle at t = 1500 is invisible, a BasicTriangle is hit), dist window inclusive, element
    order decides exact ties, and it shares `elements` with the spheres."""
    big = ((-900, -900, -1500), (900, -900, -1500), (0, 900, -1500))
    sc = R.Scene()
    sc.elements.append(R.BasicTriangle.new(big, R.Lambertian(Vec3(1, 1, 1))))
    h = trace(oracle, sc, [[0, 0, 0, 0, 0, -1]])
    assert h["kind"][0] == 2 and abs(h["t"][0] - 1500.0) < 1e-2 and np.array_equal(h["normal"][0], np.float32([0, 0, 1]))
    assert trace(oracle, one_tri_scene(big), [[0, 0, 0, 0, 0, -1]])["kind"][0] == -1          # the mesh sweep caps t at 999.99994
    far = tuple((x, y, -2001.0) for x, y, _ in big)
    sc = R.Scene(); sc.elements.append(R.BasicTriangle.new(far, R.Lambertian(Vec3(1, 1, 1))))
    assert trace(oracle, sc, [[0, 0, 0, 0, 0, -1]])["kind"][0] == -1                             # dist > max_dist
    # exact tie between a sphere surface and a triangle at dist 5: whichever comes first in `elements` wins (strict <)
    tri = R.BasicTriangle.new(TRI, R.Metal(Vec3(1, 1, 1), 0.0))
    sph = R.Sphere(Vec3(0, 0, -6.0), 1.0, R.Lambertian(Vec3(1, 1, 1)))
    for els, want in (([tri, sph], 2), ([sph, tri], 0)):
        sc = R.Scene(elements=els)
        h = trace(oracle, sc, [[0, 0, 0, 0, 0, -1]])
        assert h["kind"][0] == want and h["elem_idx"][0] == 0 and h["dist"][0] == 5.0
    # back face is hit too, the normal is never flipped
    h = trace(oracle, R.Scene(elements=[tri]), [[0, 0, -10, 0, 0, 1]])
    assert h["kind"][0] == 2 and np.array_equal(h["normal"][0], np.float32([0, 0, 1]))
