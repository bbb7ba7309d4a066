"""Scene builders shared by the parity tests, the golden-vector generator and smoke()."""
import numpy as np

import rbrt_b200 as R
from rbrt_b200 import synth
from rbrt_b200.vec3 import Vec3


def example_camera(width, height):
    cb = synth.example_camera_blueprint()
    return R.Camera.new(cb.camera_position, cb.camera_look_at, cb.camera_up, height, width, cb.camera_focal_length_mm)


def spheres_scene(**kw):
    """Config C1: the four spheres of scenes/example_scene.yaml:33-75, no mesh."""
    return R.create_scene_from_scene_blueprint(synth.spheres_only_blueprint(), **kw)


def small_mesh_scene(subdiv=3, n_keep=None, material=None, **kw):
    """C1's spheres + a displaced icosphere where the fixture's bunny stands (example_scene.yaml:18-23)."""
    scene = spheres_scene(**kw)
    tris = synth.displaced_icosphere(subdiv, 3.0, (5.0, 1.4, -12.5))
    if n_keep is not None:
        tris = tris[:n_keep]
    scene.triangle_meshes.append(R.TriangleMesh.from_triangles(tris, material or R.Dielectric(0.2)))
    return scene


def quirk_scene(**kw):
    """Hand-built geometry that exercises the reference's quirks (SURVEY.md Q1-Q10):
    mesh 0: 11 triangles (N % 8 == 3 -> the last three are never tested), including two coplanar duplicates
            (equal t -> lowest index wins), a sliver with |det| < 1e-3 (culled) and a back-facing triangle;
    mesh 1: 12 triangles (N % 8 == 4 -> all tested) placed behind mesh 0;
    mesh 2: 0 triangles;  spheres: a lambertian, a metal, a glass sphere and a huge ground sphere."""
    t = []
    def quad(z, x0, x1, y0, y1, flip=False):
        a, b, c, d = (x0, y0, z), (x1, y0, z), (x1, y1, z), (x0, y1, z)
        return [(a, c, b), (a, d, c)] if flip else [(a, b, c), (a, c, d)]
    m0 = quad(-6.0, -2, 2, 0, 3) + quad(-6.0, -2, 2, 0, 3)            # 0-3: duplicates of the same two triangles
    m0 += quad(-5.0, -0.5, 0.5, 1, 2, flip=True)                       # 4-5: back-facing, in front
    m0 += [((3.0, 0.0, -6.0), (3.0001, 0.0, -6.0), (3.0, 3.0, -6.0))]  # 6: sliver, |det| < 1e-3 for most rays
    m0 += [((-4, 0, -7), (-3, 0, -7), (-3.5, 2, -7))]                  # 7
    m0 += quad(-4.0, -1, 1, 0.5, 2.5)[:2] + [((2, 0, -4), (3, 0, -4), (2.5, 2, -4))]   # 8-10: dropped by the AVX tail rule
    m1 = quad(-9.0, -6, 6, 0, 6) * 6                                   # 12 triangles, all tested
    scene = R.Scene(**kw)
    scene.elements += [
        R.Sphere(Vec3(0.0, -1000.0, -5.0), 1000.0, R.Lambertian(Vec3(0.02, 0.2, 0.1))),
        R.Sphere(Vec3(-3.0, 1.0, -3.5), 1.0, R.Lambertian(Vec3(0.1, 0.1, 0.9))),
        R.Sphere(Vec3(3.0, 1.0, -3.0), 1.0, R.Metal(Vec3(0.8, 0.8, 0.8), 0.05)),
        R.Sphere(Vec3(0.0, 0.8, -2.0), 0.8, R.Dielectric(1.8)),
    ]
    scene.triangle_meshes += [
        R.TriangleMesh.from_triangles(np.array(m0, np.float32), R.Lambertian(Vec3(0.7, 0.3, 0.2))),
        R.TriangleMesh.from_triangles(np.array(m1, np.float32), R.Metal(Vec3(0.9, 0.9, 0.5), 0.3)),
        R.TriangleMesh.from_triangles(np.zeros((0, 3, 3), np.float32), R.Dielectric(1.5)),
    ]
    return scene


def quirk_camera(width, height):
    return R.Camera.new(Vec3(0.0, 1.5, 3.0), Vec3(0.0, -0.05, -1.0), Vec3(0.0, 1.0, 0.0), height, width, 24.0)


def _quads(quads, inward):
    """Two triangles per quad (corners in order around it), wound so that the normal (triangle.rs:30-34) points along `inward`."""
    tris = []
    for q, n in zip(np.asarray(quads, np.float32), np.asarray(inward, np.float32)):
        a, b, c, d = q
        tris += [(a, b, c), (a, c, d)] if np.dot(np.cross(b - a, c - a), n) > 0 else [(a, c, b), (a, d, c)]
    return np.array(tris, np.float32)


def deep_path_scene(length=12.0, hole=0.3, **kw):
    """A long 2 x 2 box along -z, its walls facing inwards, open only through a `2 hole` x `2 hole` window in the front wall at z = 0:
    Lambertian floor, ceiling, left wall, far end and front wall (albedo 0.95), a metal right wall (fuzz 0.05) in four segments and a glass sphere
    in the middle.  A path has to diffuse back to the window to reach the sky, so most paths scatter well over 64 times and still
    end with radiance > 0.  Both meshes have N % 8 == 0 triangles (every triangle is tested)."""
    L, h = -float(length), float(hole)
    lam = _quads([[(-1, -1, 0), (1, -1, 0), (1, -1, L), (-1, -1, L)],          # floor
                  [(-1, 1, 0), (1, 1, 0), (1, 1, L), (-1, 1, L)],              # ceiling
                  [(-1, -1, 0), (-1, 1, 0), (-1, 1, L), (-1, -1, L)],          # left wall
                  [(-1, -1, L), (1, -1, L), (1, 1, L), (-1, 1, L)],            # far end
                  [(-1, -1, 0), (1, -1, 0), (1, -h, 0), (-1, -h, 0)],          # front wall: four frames around the window
                  [(-1, h, 0), (1, h, 0), (1, 1, 0), (-1, 1, 0)],
                  [(-1, -h, 0), (-h, -h, 0), (-h, h, 0), (-1, h, 0)],
                  [(h, -h, 0), (1, -h, 0), (1, h, 0), (h, h, 0)]],
                 [(0, 1, 0), (0, -1, 0), (1, 0, 0), (0, 0, 1)] + [(0, 0, -1)] * 4)
    seg = [L * k / 4 for k in range(5)]
    metal = _quads([[(1, -1, z0), (1, 1, z0), (1, 1, z1), (1, -1, z1)] for z0, z1 in zip(seg, seg[1:])], [(-1, 0, 0)] * 4)
    scene = R.Scene(**kw)
    scene.elements.append(R.Sphere(Vec3(0.2, -0.3, L / 2), 0.5, R.Dielectric(1.5)))
    scene.triangle_meshes += [R.TriangleMesh.from_triangles(lam, R.Lambertian(Vec3(0.95, 0.95, 0.95))),
                              R.TriangleMesh.from_triangles(metal, R.Metal(Vec3(0.95, 0.9, 0.95), 0.05))]
    return scene


def deep_path_camera(width, height):
    """Just inside the opening of deep_path_scene, looking down the box."""
    return R.Camera.new(Vec3(0.0, 0.0, -0.2), Vec3(0.05, 0.02, -1.0), Vec3(0.0, 1.0, 0.0), height, width, 24.0)


def two_mirror_scene():
    """Two facing perfect mirrors, 10 apart, eight copies of each triangle: every path of two_mirror_camera bounces until its depth
    budget is gone, so a render gives exactly (max_depth + 1) rays per path and a black image (lib.rs:54-66)."""
    sc = R.Scene()
    tris = np.array([((-50, -50, -5), (50, -50, -5), (0, 50, -5))] * 8 + [((-50, -50, 5), (0, 50, 5), (50, -50, 5))] * 8, np.float32)
    sc.triangle_meshes.append(R.TriangleMesh.from_triangles(tris, R.Metal(Vec3(1, 1, 1), 0.0)))
    return sc


def two_mirror_camera(width=2, height=2):
    """A long lens on the axis between the mirrors of two_mirror_scene: the rays stay between them."""
    return R.Camera.new(Vec3(0, 0, 0), Vec3(0, 0, -1), Vec3(0, 1, 0), height, width, 28000.0)


def random_rays(n, center, spread, seed=0):
    """Secondary-like rays: origins scattered around `center`, random unit directions, plus degenerate
    ones (axis-aligned directions with exact zeros, un-normalised and tiny directions)."""
    rng = np.random.default_rng(seed)
    o = rng.normal(size=(n, 3)).astype(np.float32) * np.float32(spread) + np.asarray(center, np.float32)
    d = rng.normal(size=(n, 3)).astype(np.float32)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    k = n // 16
    d[:k] = np.eye(3, dtype=np.float32)[rng.integers(0, 3, k)] * rng.choice(np.float32([-1, 1]), k)[:, None]
    d[k:2 * k, rng.integers(0, 3)] = 0.0
    d[2 * k:3 * k] *= np.float32(7.5)
    d[3 * k:4 * k] *= np.float32(1e-3)
    return np.concatenate([o, d], 1).astype(np.float32)


def hits_equal(a, b):
    """Bit-exact comparison of two HIT_DTYPE arrays; returns the boolean mask of equal records."""
    u = np.uint32
    return ((a["kind"] == b["kind"]) & (a["elem_idx"] == b["elem_idx"]) & (a["tri_idx"] == b["tri_idx"])
            & (a["t"].view(u) == b["t"].view(u)) & (a["dist"].view(u) == b["dist"].view(u))
            & (a["point"].view(u) == b["point"].view(u)).all(1) & (a["normal"].view(u) == b["normal"].view(u)).all(1))


_BIG = {}


def big_scene(subdiv, sah=True):
    """Configs C3 (subdiv 8: 1 310 720 triangles, radius 40) / C5 (subdiv 9: 5 242 880 triangles, radius 100) exactly as
    bench.py builds them (synth.big_mesh_config); the triangle soup is cached per process.  Returns (scene, camera at the
    config's full size)."""
    radius, (W, H) = {8: (40.0, (1920, 1080)), 9: (100.0, (3840, 2160))}[subdiv]
    if subdiv not in _BIG:
        _BIG[subdiv] = synth.big_mesh_config(subdiv, radius)
    camkw, spheres, tris, mat = _BIG[subdiv]
    scene = R.Scene(sah=sah)
    scene.elements += [R.Sphere(c, r, m) for c, r, m in spheres]
    scene.triangle_meshes.append(R.TriangleMesh.from_triangles(tris, mat))
    cam = R.Camera.new(camkw["position"], camkw["look_at"], camkw["up"], H, W, camkw["focal_len_mm"])
    return scene, cam


def stress_scene():
    """Config C4 exactly as bench.py builds it (synth.stress_config): 33 glass / metal spheres + a 20 480-triangle glass mesh."""
    spheres, tris, mat = synth.stress_config()
    scene = R.Scene()
    scene.elements += [R.Sphere(c, r, m) for c, r, m in spheres]
    scene.triangle_meshes.append(R.TriangleMesh.from_triangles(tris, mat))
    return scene


def edge_aimed_rays(tris, n, dist, seed=0):
    """n rays that start `dist` away and aim at points on the edges and corners of the triangles [N,3,3]: where a closest-hit answer hangs on the
    last bits of the arithmetic (used for far origins: `o - v0` and the direction then carry ~ulp(|o|) of noise)."""
    rng = np.random.default_rng(seed)
    ti = rng.integers(0, len(tris), n)
    b = rng.random((n, 3))
    kind = rng.integers(0, 3, n)
    b[kind == 0, 0] = 0.0
    b[kind == 1, :2] = 0.0
    b /= b.sum(1, keepdims=True)
    target = (np.asarray(tris, np.float64)[ti] * b[:, :, None]).sum(1)
    back = rng.normal(size=(n, 3))
    back /= np.linalg.norm(back, axis=1, keepdims=True)
    o = (target - back * dist).astype(np.float32)
    d = target - o.astype(np.float64)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    return np.concatenate([o, d.astype(np.float32)], 1).astype(np.float32)


EXTENT_CENTRE = (5.0, 1.4, -12.5)


def far_triangle_mesh(far, axis=0):
    """The 1280-triangle icosphere of small_mesh_scene, one small triangle whose corners lie at coordinate `far` on `axis` (inf and -inf
    too), and seven copies of the first triangles: 1288 = 161 x 8, so the 8-lane tail rule drops nothing and every triangle is in the tree.
    The far triangle stretches the mesh box, its padding and the node grid on that axis; the icosphere, where the rays hit, stays put."""
    base = synth.displaced_icosphere(3, 3.0, EXTENT_CENTRE)
    tri = np.zeros((1, 3, 3), np.float32)
    tri[0, :, axis] = np.float32(far)
    tri[0, 1, (axis + 1) % 3] = 1.0
    tri[0, 2, (axis + 2) % 3] = 1.0
    return np.concatenate([base, tri, base[:7]], 0).astype(np.float32)


def scaled_mesh(extent):
    """The icosphere of far_triangle_mesh scaled about the world origin until its box is `extent` wide; returns (triangles, scale)."""
    base = synth.displaced_icosphere(3, 3.0, EXTENT_CENTRE).astype(np.float64)
    s = extent / float(np.ptp(base.reshape(-1, 3), axis=0).max())
    return (base * s).astype(np.float32), s


def extent_rays(n, seed=0, tris=None):
    """Four kinds of rays at the icosphere of far_triangle_mesh, n of each: random (random_rays: also axis-aligned, zero components,
    un-normalised), edge-aimed from 30 units away, exactly axis-parallel (two zero components, either sign) and directions with one or two
    components scaled down to 1e-30 ... 1e-5."""
    rng = np.random.default_rng(seed)
    c = np.asarray(EXTENT_CENTRE, np.float32)
    tris = synth.displaced_icosphere(3, 3.0, EXTENT_CENTRE) if tris is None else tris
    axis = np.zeros((n, 6), np.float32)
    axis[:, :3] = c + rng.uniform(-3.5, 3.5, (n, 3)).astype(np.float32)
    k = rng.integers(0, 3, n)
    axis[np.arange(n), k] = c[k] - np.float32(20.0) * np.sign(rng.uniform(-1, 1, n)).astype(np.float32)
    axis[np.arange(n), 3 + k] = np.sign(c[k] - axis[np.arange(n), k])
    tiny = random_rays(n, EXTENT_CENTRE, 4.0, seed + 1)
    tiny[:, 3:] = rng.normal(size=(n, 3)).astype(np.float32)
    scale = (10.0 ** rng.uniform(-30, -5, (n, 2))).astype(np.float32)
    tiny[np.arange(n), 3 + k] *= scale[:, 0]
    two = rng.random(n) < 0.3
    tiny[np.arange(n)[two], 3 + (k[two] + 1) % 3] *= scale[two, 1]
    return np.concatenate([random_rays(n, EXTENT_CENTRE, 4.0, seed + 2), edge_aimed_rays(tris, n, 30.0, seed + 3), axis, tiny], 0).astype(np.float32)
