"""The SOURCE of the product's per-ray arithmetic, checked without a GPU.

rbrt_b200/csrc/common.cuh, intersect.cuh and shade.cuh (Scene::hit with its sphere / BasicTriangle / bounding-box / Moeller-Trumbore
tests, camera rays, Lambertian / Metal / Dielectric scatter, Philox, sky, `as u8`) are compiled for the host by g++ behind a stand-in
cuda_runtime.h (tests/host_device/) and driven by a plain one-ray-at-a-time brute-force loop.  The results must equal the oracle's and the
golden fixtures' bit for bit; the BVH traversal source runs over 4-wide trees built on the host in the product's node format.  This is test infrastructure, not a CPU path of the product (nothing under rbrt_b200/ can reach it): it makes
the CPU-only test run of every round notice a slip in those headers.  The device compiler, the GPU's LBVH build, the warp-voted traversal and
the wavefront kernels are what the `-m gpu` tests cover."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import rbrt_b200 as R
from rbrt_b200 import _abi
from rbrt_b200.scene import element_arrays
from rbrt_b200.vec3 import Vec3

from . import golden_util as G
from . import scenes as S

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HD = os.path.join(ROOT, "tests", "host_device")
CSRC = os.path.join(ROOT, "rbrt_b200", "csrc")
P = C.POINTER


@pytest.fixture(scope="module")
def hd():
    out = os.path.join(HD, "build", "libhost_device.so")
    os.makedirs(os.path.dirname(out), exist_ok=True)
    srcs = [os.path.join(HD, "harness.cpp"), os.path.join(HD, "cuda_runtime.h")] + [os.path.join(CSRC, f) for f in ("common.cuh", "intersect.cuh", "shade.cuh", "cull.cuh")]
    if not os.path.exists(out) or any(os.path.getmtime(s) > os.path.getmtime(out) for s in srcs):
        # -I tests/host_device FIRST: `#include <cuda_runtime.h>` in common.cuh finds the stand-in.  No contraction, no FMA, as the oracle.
        subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-mno-fma", "-DRBRT_LDG128", "-Wno-unknown-pragmas", "-fPIC", "-shared",
                        "-I", HD, "-I", CSRC, "-o", out, srcs[0]], check=True)
    lib = C.CDLL(out)
    scene_args = [P(_abi.ElementRefC), C.c_uint32, P(_abi.SphereDescC), P(_abi.TriangleDescC), P(_abi.MeshDescC), C.c_uint32, C.c_uint32]
    lib.hd_trace_rays.argtypes = scene_args + [C.c_uint32, C.c_void_p, C.c_uint64, C.c_void_p, P(C.c_uint64), P(C.c_uint64)]
    lib.hd_render.argtypes = scene_args + [C.c_uint32, P(_abi.CameraC), C.c_uint32, C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p, P(C.c_uint64), P(C.c_uint64)]
    lib.hd_scatter.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p]
    lib.hd_fastdiv_mismatches.argtypes, lib.hd_fastdiv_mismatches.restype = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32], C.c_uint64
    lib.hd_shard_visits.argtypes = [C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, P(C.c_uint32)]
    lib.hd_set_rcp_error.argtypes = [C.c_float]
    for f in (lib.hd_cull_spheres, lib.hd_cull_boxes):
        f.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_float, C.c_float, C.c_void_p]
    return lib


def scene_args(scene):
    order, spheres, tris, ne, ns, nt = element_arrays(scene.elements)
    nm = len(scene.triangle_meshes)
    meshes = (_abi.MeshDescC * max(nm, 1))(*[m.to_c() for m in scene.triangle_meshes])
    return (order, ne, spheres, tris, meshes, nm, scene.simd_lanes), (order, spheres, tris, meshes)     # (arguments, keep-alive)


def hd_hit(hd, scene, rays, leaf_size=0, counters=None):
    """leaf_size 0: the brute-force loop (scene_hit<true>); 1..8: the BVH traversal (scene_hit<false>) over a host-built 4-wide tree."""
    rays = np.ascontiguousarray(rays, dtype=np.float32).reshape(-1, 6)
    hits = np.zeros(len(rays), dtype=_abi.HIT_DTYPE)
    args, keep = scene_args(scene)
    nodes, tris = C.c_uint64(0), C.c_uint64(0)
    assert hd.hd_trace_rays(*args, leaf_size, rays.ctypes.data, len(rays), hits.ctypes.data, C.byref(nodes), C.byref(tris)) == 0
    if counters is not None:
        counters.update(nodes=nodes.value, tris=tris.value)
    return hits


def hd_render(hd, scene, cam, spp, seed=0, max_depth=0, leaf_size=0):
    h, w = cam.img_height_pix, cam.img_width_pix
    hdr, rgb = np.empty((h, w, 3), np.float32), np.empty((h, w, 3), np.uint8)
    rays, nans = C.c_uint64(0), C.c_uint64(0)
    args, keep = scene_args(scene)
    assert hd.hd_render(*args, leaf_size, cam.to_c(), spp, seed & (2 ** 64 - 1), max_depth, hdr.ctypes.data, rgb.ctypes.data, C.byref(rays), C.byref(nans)) == 0
    return hdr, rgb, rays.value, nans.value


def assert_hits(a, b, what):
    eq = S.hits_equal(a, b)
    assert eq.all(), f"{what}: {int((~eq).sum())} of {len(a)} hits differ; first: got {a[np.argmin(eq)]} want {b[np.argmin(eq)]}"


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


@pytest.mark.parametrize("name", G.NAMES)
def test_golden_fixtures(hd, name):
    """The committed fixtures (oracle outputs; what the GPU tests compare with): hits of the stored rays, the complete render."""
    z, scene, cam = G.load(name)
    assert_hits(hd_hit(hd, scene, z["rays"]), z["hits"], name)
    for leaf in (0, 1, 17):                                                             # brute force, BVH, voted BVH
        hdr, rgb, rays, _ = hd_render(hd, scene, cam, int(z["spp"]), int(z["seed"]), 0, leaf)
        assert np.array_equal(bits(hdr), bits(z["hdr"])), f"{name} leaf {leaf}: {int((bits(hdr) != bits(z['hdr'])).any(axis=2).sum())} pixels differ"
        assert np.array_equal(rgb, z["rgb"]) and rays == int(z["n_rays_rendered"])


def test_scene_hit_against_the_oracle(hd, oracle):
    """Live oracle: the lane rule (N % 8, N % 4 tails), quirk scene, BasicTriangle elements mixed with spheres, ties between equal elements."""
    for lanes in (8, 4):
        for n_keep in (1275, 1277, 1280, 5, 3, 1):
            scene = S.small_mesh_scene(3, n_keep, simd_lanes=lanes)
            rays = np.concatenate([oracle.primary_rays(S.example_camera(48, 36).to_c(), 3, 0), S.random_rays(2048, (5.0, 1.4, -12.5), 4.0, 1)], 0)
            assert_hits(hd_hit(hd, scene, rays), oracle.OracleScene.from_scene(scene).hit(rays), f"n={n_keep} lanes={lanes}")
    scene = S.quirk_scene()
    rays = np.concatenate([oracle.primary_rays(S.quirk_camera(64, 48).to_c(), 9, s) for s in range(3)], 0)
    assert_hits(hd_hit(hd, scene, rays), oracle.OracleScene.from_scene(scene).hit(rays), "quirk scene")
    # BasicTriangle elements between spheres (triangle.rs:9-28,92-130), two coincident elements (the earlier one wins, scene.rs:27)
    mixed = R.Scene()
    mixed.elements += [R.Sphere(Vec3(0, 0, -6), 1.0, R.Lambertian(Vec3(0.5, 0.5, 0.5))),
                       R.BasicTriangle([Vec3(-3, -1, -5), Vec3(3, -1, -5), Vec3(0, 2.5, -5)], R.Metal(Vec3(0.9, 0.9, 0.9), 0.1)),
                       R.Sphere(Vec3(0, 0, -6), 1.0, R.Dielectric(1.5)),
                       R.BasicTriangle([Vec3(-3, -1, -5), Vec3(3, -1, -5), Vec3(0, 2.5, -5)], R.Lambertian(Vec3(0.1, 0.2, 0.3))),
                       R.Sphere(Vec3(0, -101, -6), 100.0, R.Lambertian(Vec3(0.2, 0.8, 0.2)))]
    rays = S.random_rays(4096, (0.0, 0.0, -5.5), 3.0, 4)
    got, want = hd_hit(hd, mixed, rays), oracle.OracleScene.from_scene(mixed).hit(rays)
    assert_hits(got, want, "mixed elements")
    assert {0, 2} <= set(np.unique(got["kind"]).tolist())                   # spheres and BasicTriangle elements were both hit


def test_bvh_traversal_source_against_the_oracle(hd, oracle):
    """The TRAVERSAL the trace kernels share (ray_slabs, the 16-bit node decode, bvh4_step's ordering and stack, leaf_step, the prune bounds,
    scene_hit<false>'s limit from the spheres) over 4-wide trees built on the host in the product's node format: same hits as the oracle's
    O(N) sweep, for every leaf size, with rays that are axis-parallel, start inside the mesh, graze it, or carry zero components."""
    from rbrt_b200 import synth
    rng = np.random.default_rng(8)
    centre = np.array((5.0, 1.4, -12.5), np.float32)
    for lanes, n_keep in ((8, 1280), (8, 1277), (4, 1277), (8, 9), (8, 3), (8, 1)):
        scene = S.small_mesh_scene(3, n_keep, simd_lanes=lanes)
        rays = [oracle.primary_rays(S.example_camera(48, 36).to_c(), 3, 0), S.random_rays(3000, tuple(centre), 4.0, 1)]
        inside = np.concatenate([np.tile(centre, (600, 1)) + rng.normal(0, 0.5, (600, 3)).astype(np.float32), rng.normal(size=(600, 3)).astype(np.float32)], 1)
        axis = np.zeros((600, 6), np.float32)
        axis[:, :3] = centre + rng.uniform(-4, 4, (600, 3)).astype(np.float32)
        axis[np.arange(600), 3 + rng.integers(0, 3, 600)] = rng.choice([-1.0, 1.0], 600)                 # two zero direction components
        planar = inside.copy(); planar[:, 3 + 1] = 0.0                                                    # one zero component
        rays = np.concatenate(rays + [inside, axis, planar], 0).astype(np.float32)
        want = oracle.OracleScene.from_scene(scene).hit(rays)
        brute = {}
        assert_hits(hd_hit(hd, scene, rays, 0, brute), want, f"brute n={n_keep}")
        for leaf in (1, 2, 4, 8):
            cnt, vcnt = {}, {}
            assert_hits(hd_hit(hd, scene, rays, leaf, cnt), want, f"bvh n={n_keep} lanes={lanes} leaf={leaf}")
            # + 16: traverse_voted (one node visit or ONE triangle test per step: leaf_step_one, tri_intersect_masks), what k_trace / k_tail run
            assert_hits(hd_hit(hd, scene, rays, leaf + 16, vcnt), want, f"voted n={n_keep} lanes={lanes} leaf={leaf}")
            assert vcnt == cnt                                                                            # the same visits and tests, in another schedule
            if n_keep >= 1277:
                assert 0 < cnt["nodes"] and cnt["tris"] < brute["tris"] / 20                              # the tree did prune
    # ties and near-ties: every triangle three times (exact copies and a copy shifted by a few ulp), shuffled — "the first index with the smallest t"
    # (triangle.rs:392-410) must survive the prune bound that follows the best hit so far
    base = synth.displaced_icosphere(2, 3.0, (5.0, 1.4, -12.5))
    shifted = base + np.float32(3e-6) * rng.normal(size=(len(base), 1, 3)).astype(np.float32)
    stack = np.concatenate([base, base, shifted], 0)[rng.permutation(3 * len(base))]
    scene = R.Scene()
    scene.triangle_meshes.append(R.TriangleMesh.from_triangles(stack, R.Lambertian(Vec3(0.5, 0.5, 0.5))))
    rays = np.concatenate([oracle.primary_rays(S.example_camera(64, 48).to_c(), 11, 0), S.random_rays(3000, (5.0, 1.4, -12.5), 4.0, 6)], 0)
    want = oracle.OracleScene.from_scene(scene).hit(rays)
    assert (want["kind"] == 1).sum() > 500
    for leaf in (1, 2, 8, 17, 24):
        assert_hits(hd_hit(hd, scene, rays, leaf), want, f"stacked copies leaf={leaf}")
    # a larger mesh (20 480 triangles) + the fixture's spheres in front of and behind it: the limit handed to the traversal comes from the spheres
    scene = S.spheres_scene()
    scene.triangle_meshes.append(R.TriangleMesh.from_triangles(synth.displaced_icosphere(5, 3.0, (5.0, 1.4, -12.5)), R.Dielectric(0.2)))
    rays = np.concatenate([oracle.primary_rays(S.example_camera(96, 72).to_c(), 5, 0), S.random_rays(4000, (5.0, 1.4, -12.5), 5.0, 2)], 0)
    want = oracle.OracleScene.from_scene(scene).hit(rays)
    assert (want["kind"] == 1).sum() > 500 and (want["kind"] == 0).sum() > 500
    for leaf in (1, 4, 17, 20):
        assert_hits(hd_hit(hd, scene, rays, leaf), want, f"icosphere 5 leaf={leaf}")


def test_renders_against_the_oracle(hd, oracle):
    """Complete renders, all three materials, depth budgets 0 / 3 / 50 (lib.rs:54-55), three seeds; every bit of the HDR image, the u8 image
    and the ray count."""
    cases = [(S.spheres_scene(), S.example_camera(40, 30), 3), (S.quirk_scene(), S.quirk_camera(32, 24), 4),
             (S.small_mesh_scene(2, None, material=R.Dielectric(0.2)), S.example_camera(32, 24), 2)]
    for k, (scene, cam, spp) in enumerate(cases):
        osc = oracle.OracleScene.from_scene(scene)
        for seed, depth in ((0, 0), (0x5EED, 3), (2 ** 63 + 5, 0), (7, 1)):
            st = {}
            want = osc.render_hdr(cam.to_c(), spp, _abi.RenderOptsC(seed=seed, max_depth=depth), st)
            hdr, rgb, rays, nans = hd_render(hd, scene, cam, spp, seed, depth)
            assert np.array_equal(bits(hdr), bits(want)), (k, seed, depth, int((bits(hdr) != bits(want)).any(axis=2).sum()))
            assert rays == st["rays"] and nans == st.get("nan_rays", 0)
            assert np.array_equal(rgb, osc.render(cam.to_c(), spp, _abi.RenderOptsC(seed=seed, max_depth=depth)))
            if scene.triangle_meshes and depth != 1:                                     # the same frame with every closest hit through the BVH traversals
                for leaf in (1, 20):
                    hdr_b, rgb_b, rays_b, _ = hd_render(hd, scene, cam, spp, seed, depth, leaf)
                    assert np.array_equal(bits(hdr_b), bits(want)) and rays_b == rays, (k, seed, depth, leaf)


def test_deep_paths_against_the_oracle(hd, oracle):
    """Depth budgets past 64 up to the product's limit of 1024 on a scene whose paths scatter far more than 64 times: every bit of the HDR
    image, the u8 image and the ray count; depth 200 also with every closest hit through the voted BVH traversal."""
    scene, cam = S.deep_path_scene(), S.deep_path_camera(12, 8)
    osc = oracle.OracleScene.from_scene(scene)
    for depth in (64, 65, 200, 1024):
        st = {}
        want = osc.render_hdr(cam.to_c(), 2, _abi.RenderOptsC(seed=41, max_depth=depth), st)
        hdr, rgb, rays, nans = hd_render(hd, scene, cam, 2, 41, depth)
        assert np.array_equal(bits(hdr), bits(want)), (depth, int((bits(hdr) != bits(want)).any(axis=2).sum()))
        assert rays == st["rays"] and nans == st["nan_rays"] == 0
        assert np.array_equal(rgb, osc.render(cam.to_c(), 2, _abi.RenderOptsC(seed=41, max_depth=depth)))
        assert (want > 0).any(axis=2).sum() >= want.shape[0] * want.shape[1] // 4           # not a black image
        if depth >= 200:
            assert st["rays"] > 65 * st["paths"], st                                          # the regime this is about
        if depth == 200:
            hdr_b, _, rays_b, _ = hd_render(hd, scene, cam, 2, 41, depth, 17)
            assert np.array_equal(bits(hdr_b), bits(want)) and rays_b == rays


def test_scatter_against_the_oracle(hd, oracle):
    """scatter() alone on the inputs of tests/test_gpu_scatter.py (random + grazing + normal incidence, ref_idx 0.2 ... 3.5)."""
    from .test_gpu_scatter import oracle_scatter
    rng = np.random.default_rng(17)
    mats = [R.Lambertian(Vec3(0.7, 0.3, 0.2)), R.Metal(Vec3(0.8, 0.8, 0.8), 0.005), R.Metal(Vec3(0.9, 0.9, 0.5), 0.0),
            R.Metal(Vec3(0.5, 0.6, 0.7), 0.9), R.Dielectric(1.8), R.Dielectric(1.5), R.Dielectric(0.2), R.Dielectric(1.0), R.Dielectric(3.5)]
    items = []
    for k in range(3000):
        d, n = rng.normal(size=3).astype(np.float32), rng.normal(size=3).astype(np.float32)
        if k % 4 == 0:
            n *= np.float32(rng.uniform(0.01, 1000.0))
        if k % 7 == 0:
            t = np.cross(n, rng.normal(size=3)).astype(np.float32)
            d = (t / np.float32(np.linalg.norm(t)) + np.float32(0.02) * n / np.float32(np.linalg.norm(n)) * np.float32(rng.choice([-1, 1]))).astype(np.float32)
        if k % 11 == 0:
            d = (-n).astype(np.float32)
        items.append((mats[k % len(mats)], d, (rng.normal(size=3) * 20).astype(np.float32), n, int(rng.integers(0, 2 ** 21)), int(rng.integers(0, 1024)),
                      int(rng.integers(1, 51))))
    arr = (_abi.ScatterInC * len(items))()
    for k, (mat, d, p, nrm, pixel, sample, bounce) in enumerate(items):
        a = arr[k]
        a.material = mat.to_c()
        a.in_ray.direction = _abi.Vec3C(*[float(x) for x in d]); a.hit_point = _abi.Vec3C(*[float(x) for x in p]); a.hit_normal = _abi.Vec3C(*[float(x) for x in nrm])
        a.pixel, a.sample, a.bounce = pixel, sample, bounce
    out = (_abi.ScatterOutC * len(items))()
    seed = 0x5EED0123456789
    assert hd.hd_scatter(C.cast(arr, C.c_void_p), len(items), seed, C.cast(out, C.c_void_p)) == 0
    o_sc, o_att, o_od = oracle_scatter(oracle, items, seed)
    g_sc = np.array([o.scattered for o in out], np.int32)
    g_att = np.array([[o.attenuation.x, o.attenuation.y, o.attenuation.z] for o in out], np.float32)
    g_od = np.array([[o.out_ray.direction.x, o.out_ray.direction.y, o.out_ray.direction.z] for o in out], np.float32)
    assert np.array_equal(g_sc, o_sc) and np.array_equal(bits(g_att), bits(o_att)) and np.array_equal(bits(g_od), bits(o_od))
    assert 0 < g_sc.sum() < len(items)


def directions_around(axis, half_angle, m, rng):
    """m directions per axis [n,3] (f64): most within a relative 1e-8 .. 1e-1 of the cone of `half_angle` [n] on either side, some anywhere,
    some exactly along / against the axis; returned as f32 with lengths that are not exactly 1."""
    n = len(axis)
    a = axis / np.linalg.norm(axis, axis=1, keepdims=True)
    helper = np.where(np.abs(a[:, :1]) < 0.9, np.array([[1.0, 0.0, 0.0]]), np.array([[0.0, 1.0, 0.0]]))
    u = np.cross(a, helper); u /= np.linalg.norm(u, axis=1, keepdims=True)
    v = np.cross(a, u)
    delta = 10.0 ** rng.uniform(-8, -1, (n, m)) * rng.choice([-1.0, 1.0], (n, m))
    # ... of the TRUE cone (where the exact test changes its answer) for one half of them, of the cull's own cone (cos^2 lowered by the 1e-4 margin:
    # where the cull changes ITS answer) for the other
    cull_angle = np.arccos(np.sqrt(np.clip(np.cos(half_angle) ** 2 - 1e-4, 0.0, 1.0)))
    theta = np.where(rng.random((n, m)) < 0.5, half_angle[:, None], cull_angle[:, None]) * (1.0 + delta)
    anywhere = rng.random((n, m)) < 0.15
    theta = np.where(anywhere, rng.uniform(0, np.pi, (n, m)), theta)
    theta[:, 0] = 0.0; theta[:, 1] = np.pi                                  # along and against the axis
    theta[:, 2] = np.pi - half_angle; theta[:, 3] = np.pi - half_angle * (1 + 1e-6)     # the cone BEHIND the origin (quirk Q16: not a provable miss for spheres)
    phi = rng.uniform(0, 2 * np.pi, (n, m))
    d = (np.cos(theta)[..., None] * a[:, None, :] + np.sin(theta)[..., None] * (np.cos(phi)[..., None] * u[:, None, :] + np.sin(phi)[..., None] * v[:, None, :]))
    d *= 1.0 + rng.uniform(-2e-7, 2e-7, (n, m, 1))
    return np.ascontiguousarray(d, dtype=np.float32)


def test_camera_ray_culling_only_skips_provable_misses(hd):
    """cull.cuh: the cone tests k_generate puts in front of the exact sphere test and the mesh-box test for camera rays.  A skipped test must be one
    the exact arithmetic answers with "no hit" — for spheres and boxes of every size and distance, origins far from the world origin, directions
    hugging the cone from both sides (and the mirrored cone behind the camera), with the cone record perturbed the way the device's approximate
    rsqrtf may perturb it.  ~25 M (element, direction) pairs; both outcomes of both tests occur in quantity."""
    rng = np.random.default_rng(23)
    totals = np.zeros(4, np.uint64)
    origins = [(0.0, 5.0, 4.0), (0.0, 0.0, 0.0), (-37.5, 12.25, 80.0), (1.0e4, -2.0e3, 5.0e3), (3.0e5, 3.0e5, -3.0e5)]
    for oi, origin in enumerate(origins):
        o = np.array(origin, np.float64)
        n, m = 600, 1400
        r = 10.0 ** rng.uniform(-3, 3, n)
        dist = r * (1.0 + 10.0 ** rng.uniform(-2.2, 3.5, n))                # from 0.6 % outside the surface (never culled: within 1 %) to 3000 radii away
        axis = rng.normal(size=(n, 3))
        axis /= np.linalg.norm(axis, axis=1, keepdims=True)
        centre = o + axis * dist[:, None]
        spheres = np.ascontiguousarray(np.concatenate([centre, r[:, None]], 1), dtype=np.float32)
        # the angles are taken from the f32 values the kernel sees
        c32, r32, o32 = spheres[:, :3].astype(np.float64), spheres[:, 3].astype(np.float64), np.array(origin, np.float32).astype(np.float64)
        l = c32 - o32
        D = np.linalg.norm(l, axis=1)
        ok = D > r32 * 1.0001
        half = np.arcsin(np.clip(r32 / np.maximum(D, 1e-300), 0, 1))
        dirs = directions_around(np.where(ok[:, None], l, axis), np.where(ok, half, 0.3), m, rng)
        o_f32 = np.array(origin, np.float32)
        for scale, shift in ((1.0, 0.0), (1.0 + 3e-7, 2e-7), (1.0 - 3e-7, 2e-7)):
            out = np.zeros(4, np.uint64)
            assert hd.hd_cull_spheres(o_f32.ctypes.data, spheres.ctypes.data, n, dirs.ctypes.data, m, scale, shift, out.ctypes.data) == 0
            assert out[2] == 0, f"origin {origin}: {int(out[2])} sphere tests were skipped although the exact test reports a hit (scale {scale}, shift {shift})"
            totals += out
        # boxes: random extents (flat ones too) around the same centres
        ext = r[:, None] * 10.0 ** rng.uniform(-2, 0, (n, 3))
        boxes = np.ascontiguousarray(np.concatenate([centre - ext, centre + ext], 1), dtype=np.float32)
        b_lo, b_hi = boxes[:, :3].astype(np.float64), boxes[:, 3:].astype(np.float64)
        bc, br = 0.5 * (b_lo + b_hi), 0.5 * np.linalg.norm(b_hi - b_lo, axis=1)
        lb = bc - o32
        Db = np.linalg.norm(lb, axis=1)
        okb = Db > br * 1.0001
        halfb = np.arcsin(np.clip(br / np.maximum(Db, 1e-300), 0, 1))
        dirs = directions_around(np.where(okb[:, None], lb, axis), np.where(okb, halfb, 0.3), m, rng)
        dirs[:, 4:40, rng.integers(0, 3)] = 0.0                              # axis-parallel components: the slab test divides by them (aabbox.rs:30-47)
        for scale, shift in ((1.0, 0.0), (1.0 + 3e-7, 2e-7)):
            out = np.zeros(4, np.uint64)
            assert hd.hd_cull_boxes(o_f32.ctypes.data, boxes.ctypes.data, n, dirs.ctypes.data, m, scale, shift, out.ctypes.data) == 0
            assert out[2] == 0, f"origin {origin}: {int(out[2])} box tests were skipped although the slab test reports a hit (scale {scale}, shift {shift})"
            totals += out
    pairs, skipped, wrong, hits = (int(x) for x in totals)
    assert pairs > 2e7 and wrong == 0
    assert skipped > 0.15 * pairs and hits > 0.15 * pairs                    # the cull is active and the exact tests do hit: neither side is vacuous


def test_pixel_mapping_of_tile_shards(hd):
    """common.cuh: fast_div equals `/` for every divisor the mapping can see, and shard_pixel over all ranks of a tile-sharded image visits every
    pixel exactly once — for image sizes that are not multiples of the 8 x 4 tile, 1 .. 8 and odd rank counts, more ranks than tiles."""
    rng = np.random.default_rng(3)
    divisors = np.unique(np.concatenate([np.arange(1, 600), 2 ** np.arange(0, 32), 2 ** np.arange(1, 32) - 1, 2 ** np.arange(1, 31) + 1,
                                         rng.integers(1, 2 ** 32, 300), [240, 480, 1920 // 8, 3840 // 8, 0xFFFFFFFF, 0xFFFFFFFE, 0x80000000]])).astype(np.uint32)
    dividends = np.unique(np.concatenate([np.arange(0, 5000), 2 ** 32 - 1 - np.arange(0, 5000), rng.integers(0, 2 ** 32, 20000),
                                          (divisors.astype(np.uint64)[:, None] * rng.integers(1, 2 ** 16, (len(divisors), 8)).astype(np.uint64) + np.array([-1, 0, 1, 0, -1, 1, 0, -1])).ravel() % 2 ** 32])).astype(np.uint32)
    assert hd.hd_fastdiv_mismatches(divisors.ctypes.data, len(divisors), dividends.ctypes.data, len(dividends)) == 0
    for W, H in ((1920, 1080), (64, 48), (13, 10), (8, 4), (7, 3), (1, 1), (257, 129), (3840, 2160)):
        for count in (1, 2, 3, 4, 7, 8, 64):
            if W * H > 3e6 and count not in (1, 8):
                continue
            visits = np.zeros(W * H, np.uint32)
            most = C.c_uint32(0)
            assert hd.hd_shard_visits(W, H, count, visits.ctypes.data, C.byref(most)) == 0
            assert (visits == 1).all(), (W, H, count, int((visits != 1).sum()))
            tiles = ((W + 7) // 8) * ((H + 3) // 4)
            assert most.value == 32 * ((tiles + count - 1) // count)             # interleaved tiles: no rank has more than one tile above its share


def test_small_mesh_near_the_world_origin_far_ray_origins(hd, oracle, monkeypatch):
    """Found with this host build: a box padding that is only RELATIVE to the mesh's coordinates is too small for a small mesh near the world
    origin when rays start hundreds of units away (they may: t < 1000, triangle.rs:146) — the exact test's `o - v0` then carries ~ulp(|o|) and accepts
    rays that miss the padded boxes.  k_mesh_setup (bvh_build.cu) therefore keeps the padding above 2^-21 * (mx + 1000); the harness' builder follows
    the same rule.  With the floor the traversal returns the oracle's hits; without it (HD_NO_PAD_FLOOR) the same rays show the mismatches."""
    from rbrt_b200 import synth
    total_without = 0
    for subdiv, size, centre, dist in ((1, 0.2, (0, 0, 0), 990.0), (0, 0.05, (0, 0, 0), 100.0), (0, 0.05, (0, 0, 0), 990.0), (2, 0.3, (0.05, 0.02, -0.03), 990.0),
                                       (1, 0.2, (0, 0, 0), 10.0), (2, 1.0, (0, 0, 0), 990.0)):
        tris = synth.displaced_icosphere(subdiv, size, centre)
        scene = R.Scene()
        scene.triangle_meshes.append(R.TriangleMesh.from_triangles(tris, R.Lambertian(Vec3(0.5, 0.5, 0.5))))
        rays = S.edge_aimed_rays(tris, 60000, dist, seed=subdiv + int(dist))
        want = oracle.OracleScene.from_scene(scene).hit(rays)
        assert (want["kind"] == 1).sum() > 30000
        for leaf in (1, 4, 17):
            assert_hits(hd_hit(hd, scene, rays, leaf), want, f"size {size} dist {dist} leaf {leaf}")
        for err in (2.4e-7, -2.4e-7):                                        # the device's reciprocal in ray_slabs is not the exact quotient: twice its ~1 ulp, both ways
            hd.hd_set_rcp_error(err)
            try:
                assert_hits(hd_hit(hd, scene, rays, 1), want, f"size {size} dist {dist} reciprocal error {err}")
            finally:
                hd.hd_set_rcp_error(0.0)
        monkeypatch.setenv("HD_NO_PAD_FLOOR", "1")
        total_without += int((~S.hits_equal(hd_hit(hd, scene, rays, 1), want)).sum())
        monkeypatch.delenv("HD_NO_PAD_FLOOR")
    assert total_without > 100                                               # the floor is what closes the gap


def test_traversal_in_awkward_regimes(hd, oracle):
    """Regimes the GPU suite's scenes do not reach, swept once with scripts/host_model/explore.py at 200 000 rays each and kept here at a smaller size:
    bounce rays that start ON the surface (also nearly tangent, also inward), direction components down to 1e-38, a flat mesh with in-plane rays,
    coordinates of 1e5, un-normalised directions from 1e-2 to 1e6, a sphere coinciding with the mesh (sphere / mesh near-ties: the limit handed to the
    traversal) seen from 10 to 900 units away."""
    from rbrt_b200 import synth
    rng = np.random.default_rng(42)
    n = 40000
    tris = synth.displaced_icosphere(4, 3.0, (5.0, 1.4, -12.5))

    def mesh_scene(t):
        sc = R.Scene()
        sc.triangle_meshes.append(R.TriangleMesh.from_triangles(np.asarray(t, np.float32), R.Lambertian(Vec3(0.5, 0.5, 0.5))))
        return sc

    def check(name, scene, rays, min_hits):
        rays = np.ascontiguousarray(rays, dtype=np.float32)
        want = oracle.OracleScene.from_scene(scene).hit(rays)
        assert (want["kind"] == 1).sum() >= min_hits, (name, int((want["kind"] == 1).sum()))
        for leaf in (1, 17, 4):
            assert_hits(hd_hit(hd, scene, rays, leaf), want, f"{name} leaf {leaf}")

    ti = rng.integers(0, len(tris), n)
    b = rng.random((n, 3)); b /= b.sum(1, keepdims=True)
    p = (tris[ti].astype(np.float64) * b[:, :, None]).sum(1)
    nrm = np.cross(tris[ti, 1] - tris[ti, 0], tris[ti, 2] - tris[ti, 0]).astype(np.float64); nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    d = rng.normal(size=(n, 3)); d /= np.linalg.norm(d, axis=1, keepdims=True)
    tangent = d - (d * nrm).sum(1, keepdims=True) * nrm * (1 - 10.0 ** rng.uniform(-6, -1, (n, 1)))
    d = np.where(rng.random((n, 1)) < 0.5, d, tangent); d /= np.linalg.norm(d, axis=1, keepdims=True)
    scene = mesh_scene(tris)
    check("bounce rays from the surface", scene, np.concatenate([p, d], 1), 10000)
    check("inward rays from the surface", scene, np.concatenate([p, -np.abs((d * nrm).sum(1, keepdims=True)) * nrm + 0.3 * d], 1), 10000)
    d2 = d.copy(); d2[np.arange(n), rng.integers(0, 3, n)] *= 10.0 ** rng.uniform(-38, -5, n)
    check("tiny direction components", scene, np.concatenate([np.array((5.0, 1.4, -12.5)) + rng.normal(0, 4, (n, 3)), d2], 1), 3000)
    base = np.concatenate([S.random_rays(n // 2, (5.0, 1.4, -12.5), 4.0, 1), S.edge_aimed_rays(tris, n // 2, 30.0, 2)], 0)
    for scale, min_hits in ((1e-2, 50), (0.1, 10000), (10.0, 10000), (1e3, 10000), (1e6, 50)):
        r = base.copy(); r[:, 3:] *= np.float32(scale)
        check(f"|d| = {scale:g}", scene, r, min_hits)
    g = np.linspace(-2, 2, 21)
    X, Y = np.meshgrid(g, g)
    Pz = np.stack([X, Y, np.full_like(X, -5.0)], -1)
    flat = np.array([t for i in range(20) for j in range(20) for t in ([Pz[i, j], Pz[i + 1, j], Pz[i, j + 1]], [Pz[i + 1, j], Pz[i + 1, j + 1], Pz[i, j + 1]])])
    inplane = np.concatenate([np.stack([rng.uniform(-3, 3, n // 4), rng.uniform(-3, 3, n // 4), np.full(n // 4, -5.0)], 1),
                              np.stack([rng.normal(size=n // 4), rng.normal(size=n // 4), np.zeros(n // 4)], 1)], 1)
    check("flat mesh", mesh_scene(flat), np.concatenate([S.random_rays(n // 2, (0, 0, -5), 3.0, 3), inplane, S.edge_aimed_rays(flat, n // 4, 50.0, 1)], 0), 5000)
    c = (1e5, 0.5e5, -1e5)
    far = synth.displaced_icosphere(3, 300.0, c)
    check("coordinates of 1e5", mesh_scene(far), np.concatenate([S.edge_aimed_rays(far, n // 2, 900.0, 3), S.random_rays(n // 2, c, 400.0, 4)], 0), 10000)
    both = R.Scene()
    both.elements.append(R.Sphere(Vec3(5.0, 1.4, -12.5), 3.0, R.Dielectric(1.5)))
    both.triangle_meshes.append(R.TriangleMesh.from_triangles(tris, R.Lambertian(Vec3(0.5, 0.5, 0.5))))
    for dist in (10.0, 300.0, 900.0):
        check(f"sphere inside the mesh from {dist:g}", both, S.edge_aimed_rays(tris, n, dist, 3 + int(dist)), 10000)
    # three meshes in YAML order — two interpenetrating, one of them the SAME mesh twice (exact ties between meshes: the earlier one wins, scene.rs:36) —
    # and an empty one: the best hit so far bounds the traversal of the next mesh
    several = R.Scene()
    other = synth.displaced_icosphere(3, 2.5, (6.0, 1.0, -11.5), seed=99)
    for t, m in ((other, R.Metal(Vec3(0.9, 0.9, 0.9), 0.1)), (tris, R.Lambertian(Vec3(0.5, 0.5, 0.5))), (np.zeros((0, 3, 3), np.float32), R.Dielectric(1.5)),
                 (tris, R.Dielectric(0.2))):
        several.triangle_meshes.append(R.TriangleMesh.from_triangles(t, m))
    several.elements.append(R.Sphere(Vec3(4.0, 1.4, -9.0), 1.0, R.Dielectric(1.8)))
    rays = np.concatenate([S.edge_aimed_rays(tris, n // 2, 40.0, 12), S.edge_aimed_rays(other, n // 2, 700.0, 13), S.random_rays(n // 2, (5.5, 1.2, -12.0), 3.0, 14)], 0)
    want = oracle.OracleScene.from_scene(several).hit(rays)
    assert set(np.unique(want["elem_idx"][want["kind"] == 1]).tolist()) == {0, 1} and (want["kind"] == 0).sum() > 100     # mesh 3 never beats its twin, mesh 1
    for leaf in (1, 17, 4):
        assert_hits(hd_hit(hd, several, rays, leaf), want, f"several meshes leaf {leaf}")


EXTENT_FAR = (1e6, 1e9, 1e11, 1.4e11, 2.6e11, 3e11, 1e12, 1e15, 1e20, 1e25, 1e30, 1e35, 2e38, 3.4e38, np.inf)


def test_traversal_at_extreme_mesh_extents(hd, oracle):
    """Meshes whose box is huge on one axis: the icosphere of tests/scenes.py with ONE small triangle at coordinate `far` (1e6 ... 3.4e38, inf,
    and negative) on each axis, and the icosphere scaled to extents 1e8 ... 1e36; rays of scenes.extent_rays (random, edge-aimed, exactly
    axis-parallel, direction components down to 1e-30).  The BVH traversals must return the oracle's hits.

    What went wrong first: ray_slabs (intersect.cuh) forms B' = (qorg - o) / d - 2^23 * qstep / d, with 1/d clamped to 1e25 for a direction
    component of 0 or |d| <= 1e-25.  Once the grid step of an axis exceeds ~4.05e6 (a padded extent of ~2.65e11: far = 3e11 here) that product
    overflows to inf, every slab t of the axis becomes -inf and rays with such a component reject the boxes they are in: before the fix, far =
    2.6e11 (step 3.97e6) still passed and far = 3e11 lost 384 of these 4000 hits.  For other directions the same happens when
    qstep / |d| > 4e31 (far = 2e38: every hit lost).  Up to step 2e6 (far = 1.3e11) the arithmetic stays finite and the one-step margin of the
    quantisation covers B's rounding.  Beyond it k_mesh_setup stores qstep = NaN for the axis: its slab t is NaN, fminf / fmaxf drop it, and the
    traversal culls on the remaining axes (common.cuh, RBRT_QSTEP_MAX).  The harness' builder applies the same rule."""
    rays = S.extent_rays(1000, 5)
    cases = [(far, 0) for far in EXTENT_FAR] + [(-far, 0) for far in (1e12, 1e20, 3.4e38, np.inf)]
    cases += [(far, ax) for ax in (1, 2) for far in (1e11, 1e12, 1e20, 1e30, 2e38, -np.inf)]
    for far, ax in cases:
        scene = R.Scene()
        scene.triangle_meshes.append(R.TriangleMesh.from_triangles(S.far_triangle_mesh(far, ax), R.Lambertian(Vec3(0.5, 0.5, 0.5))))
        want = oracle.OracleScene.from_scene(scene).hit(rays)
        assert (want["kind"] == 1).sum() > 1500, (far, ax)                  # the icosphere is hit
        assert ((want["kind"] == 1)[2000:3000]).sum() > 300                  # ... also by the axis-parallel rays
        for leaf in (1, 4, 17):
            assert_hits(hd_hit(hd, scene, rays, leaf), want, f"far {far:g} on axis {ax} leaf {leaf}")
    rng = np.random.default_rng(6)
    for extent in (1e8, 1e12, 1e16, 1e20, 1e24, 1e28, 1e32, 1e36):
        tris, _ = S.scaled_mesh(extent)
        scene = R.Scene()
        scene.triangle_meshes.append(R.TriangleMesh.from_triangles(tris, R.Lambertian(Vec3(0.5, 0.5, 0.5))))
        # a hit counts up to dist 2000 (lib.rs:45): edge-aimed rays from 500 away, and axis-parallel ones at triangle centres from 500 away
        target = tris[rng.integers(0, len(tris), 1500)].astype(np.float64).mean(1)
        k = rng.integers(0, 3, 1500)
        d = np.zeros((1500, 3)); d[np.arange(1500), k] = rng.choice([-1.0, 1.0], 1500)
        r = np.concatenate([S.edge_aimed_rays(tris, 2500, 500.0, 7), np.concatenate([target - 500.0 * d, d], 1).astype(np.float32)], 0)
        want = oracle.OracleScene.from_scene(scene).hit(r)
        if extent <= 1e8:
            assert (want["kind"] == 1).sum() > 1500, extent                  # (from ~1e10 on, ulp(|o|) > 500 and the origins snap onto the surface)
        for leaf in (1, 4, 17):
            assert_hits(hd_hit(hd, scene, r, leaf), want, f"mesh scaled to {extent:g} leaf {leaf}")
