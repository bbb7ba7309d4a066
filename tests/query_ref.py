"""The occlusion query's definition in numpy, and the adversarial scene and rays its tests use (tests/test_query_host.py on the CPU,
tests/test_gpu_query.py on the GPU).

occluded[i] = 2 when ray i is a NaN ray (a NaN sphere discriminant, sphere.rs:33, on ANY sphere of Scene.elements), else 1 when Scene::hit
reports a hit with dist < max_dist[i] (strict), else 0.  `nan_rays` restates the discriminant in float32 with the reference's op order
(sphere.rs:20-33); numpy does not contract, so the bits are the device's."""
import numpy as np

import rbrt_b200 as R
from rbrt_b200 import _abi, synth
from rbrt_b200.vec3 import Vec3

f32 = np.float32


def nan_rays(scene, rays):
    """Boolean mask of the NaN rays of `rays` [N,6] in `scene` (only spheres can give a NaN discriminant)."""
    o, d = rays[:, :3].astype(f32), rays[:, 3:].astype(f32)
    out = np.zeros(len(rays), bool)
    with np.errstate(all="ignore"):
        for e in scene.elements:
            if isinstance(e, R.BasicTriangle):
                continue
            cv = Vec3.from_any(e.center)
            c = np.array([cv.x, cv.y, cv.z], f32)
            r = f32(e.radius)

            def dot(a, b):
                return (a[:, 0] * b[:, 0] + a[:, 1] * b[:, 1]) + a[:, 2] * b[:, 2]
            a = dot(d, d)
            l = o - c
            b = dot(d * f32(2.0), l)
            cc = dot(l, l) - r * r
            sol = b * b - (f32(4.0) * a) * cc
            out |= np.isnan(sol)
    return out


def occluded(hits, nan, max_dist):
    """The composition: Scene::hit's records (HIT_DTYPE), the NaN mask, the bounds."""
    with np.errstate(invalid="ignore"):
        hit = (hits["kind"] != _abi.HIT_NONE) & (hits["dist"] < np.asarray(max_dist, f32))
    return np.where(nan, 2, hit.astype(np.uint8)).astype(np.uint8)


def adversarial_scene(leaf_size=1):
    """Elements: a sphere, a BasicTriangle, a sphere 3e19 away whose discriminant is NaN for every ray with |d.x| above about 0.3 of |d|
    (b*b and 4*a*cc both overflow: inf - inf; so rays that hit the first sphere are NaN rays too), a negative-radius sphere.  Meshes: two
    parallel quads 0.0005 and 0.005 below the origin plane (a ray with |d| = 1e-4 straight down meets the near one at t = 5, dist 0.0005,
    too close, and the far one at t = 50, dist 0.005: Scene::hit reports no mesh hit), an icosphere, an empty mesh."""
    mat = R.Lambertian(Vec3(0.5, 0.5, 0.5))
    els = [R.Sphere(Vec3(-3.0, 0.0, -5.0), 1.5, mat),
           R.BasicTriangle.new([(1.0, -1.0, -4.0), (3.0, -1.0, -4.0), (2.0, 1.5, -4.0)], mat),
           R.Sphere(Vec3(3e19, 0.0, 0.0), 1.0, mat),
           R.Sphere(Vec3(0.0, 3.0, -6.0), -1.0, R.Dielectric(1.5))]
    quads = []
    for z in (-0.0005, -0.005):
        a, b, c, d = (-1.0, -1.0, z), (1.0, -1.0, z), (1.0, 1.0, z), (-1.0, 1.0, z)
        quads += [[a, b, c], [a, c, d]]
    scene = R.Scene(elements=els, leaf_size=leaf_size)
    scene.triangle_meshes.append(R.TriangleMesh.from_triangles(np.array(quads, f32), mat))
    scene.triangle_meshes.append(R.TriangleMesh.from_triangles(synth.displaced_icosphere(2, 1.5, (2.5, 1.0, -8.0)), mat))
    scene.triangle_meshes.append(R.TriangleMesh.from_triangles(np.zeros((0, 3, 3), f32), mat))
    return scene


def adversarial_rays(n=4000, seed=0):
    """|d| from 1e-4 to 1e4, origins up to 1e5 away, short straight-down rays at the quads, rays at the first sphere (NaN through the far
    sphere), exact zeros, and +-inf / NaN components."""
    rng = np.random.default_rng(seed)
    aim = np.array([0.0, 0.5, -6.0], f32)
    o = (rng.normal(size=(n, 3)) * 3.0).astype(f32) + aim
    d = rng.normal(size=(n, 3)).astype(f32)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    d *= (10.0 ** rng.uniform(-4, 4, size=(n, 1))).astype(f32)
    far = rng.normal(size=(n // 4, 3)).astype(f32)
    far *= (10.0 ** rng.uniform(2, 5, size=(n // 4, 1)) / np.linalg.norm(far, axis=1, keepdims=True)).astype(f32)
    fo = aim + far
    fd = (aim + rng.normal(size=far.shape).astype(f32) - fo) * (10.0 ** rng.uniform(-4, 1, size=(n // 4, 1))).astype(f32)
    k = n // 4                                                            # short directions at the two quads
    so = np.stack([rng.uniform(-0.8, 0.8, k), rng.uniform(-0.8, 0.8, k), np.zeros(k)], 1).astype(f32)
    sd = np.stack([rng.uniform(-0.1, 0.1, k), rng.uniform(-0.1, 0.1, k), -np.ones(k)], 1).astype(f32)
    sd *= rng.choice(f32([1e-4, 1.5e-4, 3e-4, 5e-4, 1e-3, 2e-3, 1e-2, 1.0]), k)[:, None]
    so[::7, 2] = f32(0.3)                                                 # some from above the plane z = 0
    to = np.tile(np.float32([[0.0, 0.0, 0.0]]), (k, 1)) + rng.normal(size=(k, 3)).astype(f32) * f32(0.2)
    td = (np.array([-3.0, 0.0, -5.0], f32) + rng.normal(size=(k, 3)).astype(f32) * f32(0.8)) - to
    special = []
    for v in (np.inf, -np.inf, np.nan, 0.0):
        for comp in range(6):
            r = np.array([0.1, 0.2, 0.0, -0.3, 0.1, -1.0], f32)
            r[comp] = v
            special.append(r)
    rays = np.concatenate([np.concatenate([o, d], 1), np.concatenate([fo, fd], 1), np.concatenate([so, sd], 1), np.concatenate([to, td], 1),
                           np.array(special, f32)], 0)
    return np.ascontiguousarray(rays, dtype=f32)


def max_dist_variants(dist):
    """Bounds for rays whose closest hit has distance `dist` (0 for a miss): exactly the hit dist, one ulp above and below, 0, negative,
    NaN, +-inf, 2000, 0.001, and random values."""
    dist = np.asarray(dist, f32)
    rng = np.random.default_rng(len(dist))
    n = len(dist)
    return [dist, np.nextafter(dist, f32(np.inf)), np.nextafter(dist, f32(-np.inf)), np.zeros(n, f32), np.full(n, -1.0, f32),
            np.full(n, np.nan, f32), np.full(n, np.inf, f32), np.full(n, -np.inf, f32), np.full(n, 2000.0, f32), np.full(n, 1e-3, f32),
            rng.uniform(0, 20, n).astype(f32)]
