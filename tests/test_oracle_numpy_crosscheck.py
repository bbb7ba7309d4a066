"""A SECOND, independent restatement of Scene::hit — written from the reference's lines in numpy float32, one IEEE
operation per numpy call — checked bit for bit against the C++/AVX oracle on random rays.

The reference has no test for ray-triangle `t` / index, `BoundingBox::hit` or `Scene::hit` ordering (SURVEY.md
section 8c), so the oracle is the only pin for those rows; two restatements that share no code (scalar/vectorised
numpy here, `_mm256_*` intrinsics there) agreeing on every bit is the strongest check available without rustc.

Lines followed: sphere.rs:20-66, aabbox.rs:28-58, mesh.rs:57-60,136-144,225-268, triangle.rs:30-34,134-262,392-410,
vec3.rs:111-134, vec3_avx.rs:10-45, scene.rs:19-43, ray.rs:10-12.
"""
import numpy as np
import pytest


from rbrt_b200 import _abi

from . import scenes as S

F = np.float32
EPS, MAX_DIST = F(0.001), F(2000.0)
T_CAP = F(1.0) / F(0.001)                                   # 999.99994 (triangle.rs:146)


def dot(a, b):                                              # (x*x' + y*y') + z*z'  (vec3.rs:115-117, vec3_avx.rs:18-21)
    return (a[..., 0] * b[..., 0] + a[..., 1] * b[..., 1]) + a[..., 2] * b[..., 2]


def cross(a, b):                                            # mul, mul, sub per component (vec3.rs:128-134, vec3_avx.rs:40-42)
    return np.stack([a[..., 1] * b[..., 2] - a[..., 2] * b[..., 1],
                     a[..., 2] * b[..., 0] - a[..., 0] * b[..., 2],
                     a[..., 0] * b[..., 1] - a[..., 1] * b[..., 0]], axis=-1).astype(F)


def length(a):                                              # sqrt((x*x + y*y) + z*z)  (vec3.rs:111-113)
    return np.sqrt((a[..., 0] * a[..., 0] + a[..., 1] * a[..., 1]) + a[..., 2] * a[..., 2]).astype(F)


def sphere_hit(o, d, c, r):                                 # sphere.rs:20-66 -> (t, dist) or None
    a = dot(d, d)
    l = (o - c).astype(F)
    b = dot((d * F(2.0)).astype(F), l)
    cc = F(dot(l, l) - r * r)
    sol = F(b * b - F(F(4.0) * a) * cc)
    if not sol >= 0:                                        # sol < 0 -> miss (NaN would panic: not generated here)
        return None
    sq = np.sqrt(sol).astype(F)
    t = F(F(-b - sq) / F(F(2.0) * a))
    if sol > 0 and t < 0:
        t = F(F(-b + sq) / F(F(2.0) * a))
        if t < 0:
            return None
    p = (o + t * d).astype(F)
    dist = length((o - p).astype(F))
    if dist < EPS or dist > MAX_DIST:
        return None
    return t, dist


def bbox_hit(o, d, lo, hi):                                 # aabbox.rs:28-58 (f32::min / max ignore NaN = fmin / fmax)
    with np.errstate(divide="ignore", invalid="ignore"):
        tl = ((lo - o).astype(F) / d).astype(F)
        tu = ((hi - o).astype(F) / d).astype(F)
    mn, mx = np.fmin(tl, tu), np.fmax(tl, tu)
    t_min = np.fmax(np.fmax(mn[0], mn[1]), mn[2])
    t_max = np.fmin(np.fmin(mx[0], mx[1]), mx[2])
    return not (t_max < 0 or t_min > t_max)


class NpMesh:
    def __init__(self, tris, lanes=8):
        v = np.asarray(tris, dtype=F).reshape(-1, 3, 3)
        self.lo, self.hi = v.reshape(-1, 3).min(axis=0), v.reshape(-1, 3).max(axis=0)    # aabbox.rs:62-88: ALL vertices
        n, r = len(v), len(v) % lanes
        self.n_eff = n if (r == 0 or 2 * r >= lanes) else n - r                          # mesh.rs:136-144 + chunks_exact
        self.v0 = v[:, 0]
        self.e1 = (v[:, 1] - v[:, 0]).astype(F)                                           # mesh.rs:57-60
        self.e2 = (v[:, 2] - v[:, 0]).astype(F)
        n_ = cross(self.e1, self.e2)                                                      # triangle.rs:30-34
        self.normals = (n_ / length(n_)[:, None]).astype(F)

    def hit(self, o, d):                                    # mesh.rs:225-268 -> (t, dist, idx) or None
        if self.n_eff == 0 or not bbox_hit(o, d, self.lo, self.hi):
            return None
        v0, e1, e2 = self.v0[:self.n_eff], self.e1[:self.n_eff], self.e2[:self.n_eff]
        with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
            h = cross(np.broadcast_to(d, e2.shape), e2)                                   # triangle.rs:189-247
            a = dot(e1, h)
            c1 = (-EPS < a) & (a < EPS)
            f = (F(1.0) / a).astype(F)
            s = (o - v0).astype(F)
            u = (f * dot(s, h)).astype(F)
            c2 = (u < 0) | (u > 1)
            q = cross(s, e1)
            v = (f * dot(np.broadcast_to(d, q.shape), q)).astype(F)
            c3 = (v < 0) | ((u + v).astype(F) > 1)
            t = (f * dot(e2, q)).astype(F)
            c4 = (t > EPS) & (t < T_CAP)
        ok = ~(c1 | c2 | c3) & c4
        if not ok.any():
            return None
        tt = np.where(ok, t, F(np.inf))
        idx = int(np.argmin(tt))                            # first index with the smallest t (triangle.rs:392-410)
        if not tt[idx] < F(100000.0):
            return None
        tb = tt[idx]
        p = (o + tb * d).astype(F)                          # ray.point_at (ray.rs:10-12)
        dist = length((o - p).astype(F))
        if not (dist > EPS and dist < MAX_DIST):            # mesh.rs:249
            return None
        return tb, dist, idx


def scene_hit(spheres, meshes, o, d):                       # scene.rs:19-43: spheres in order, then meshes, strict <
    closest, best = F(np.finfo(np.float32).max), (-1, 0, 0, F(0), F(0))
    for i, (c, r) in enumerate(spheres):
        h = sphere_hit(o, d, c, r)
        if h is not None and h[1] < closest:
            closest, best = h[1], (0, i, 0, h[0], h[1])
    for mi, m in enumerate(meshes):
        h = m.hit(o, d)
        if h is not None and h[1] < closest:
            closest, best = h[1], (1, mi, h[2], h[0], h[1])
    return best


def bits(x):
    return np.asarray(x, dtype=F).view(np.uint32)


@pytest.mark.parametrize("n_keep,lanes", [(None, 8), (1275, 8), (1277, 8), (1279, 4), (1277, 4)])
def test_numpy_restatement_agrees_with_the_oracle(oracle, n_keep, lanes):
    """1280-ish triangle mesh (N % 8 in {0, 3, 5}, N % 4 in {3, 1}: both SIMD tail rules) + the four fixture spheres,
    camera rays and rays leaving the surfaces in random directions."""
    rng = np.random.default_rng(20241018)
    scene = S.small_mesh_scene(3, n_keep=n_keep, simd_lanes=lanes)
    tris = np.asarray(scene.triangle_meshes[0].triangles, dtype=F).reshape(-1, 3, 3)
    mesh = NpMesh(tris, lanes)
    spheres = [(np.array([e.center.x, e.center.y, e.center.z], F), F(e.radius)) for e in scene.elements]
    cam = S.example_camera(40, 30)
    rays = [np.asarray(oracle.primary_rays(cam.to_c(), 3, 0), dtype=F).reshape(-1, 6)]      # inputs only: any rays would do
    centres = tris.mean(axis=1)[rng.integers(0, len(tris), 300)]
    dirs = rng.normal(size=(300, 3)).astype(F)
    rays.append(np.concatenate([centres, dirs], axis=1).astype(F))                       # rays starting ON the mesh
    on_sphere = np.array([spheres[k % 4][0] + spheres[k % 4][1] * (v / np.linalg.norm(v)).astype(F)
                          for k, v in enumerate(rng.normal(size=(100, 3)).astype(F))], F)
    rays.append(np.concatenate([on_sphere, rng.normal(size=(100, 3)).astype(F)], axis=1).astype(F))
    rays = np.concatenate(rays).astype(F)
    want = oracle.OracleScene.from_scene(scene).hit(rays)
    kinds = {0: 0, 1: 0, -1: 0}
    for k, ray in enumerate(rays):
        o, d = ray[:3].copy(), ray[3:].copy()
        kind, elem, tri, t, dist = scene_hit(spheres, [mesh], o, d)
        w = want[k]
        kinds[kind] += 1
        assert (kind if kind >= 0 else _abi.HIT_NONE) == w["kind"], (k, kind, w)
        if kind < 0:
            continue
        assert elem == w["elem_idx"] and tri == w["tri_idx"], (k, elem, tri, w)
        assert bits(t) == bits(w["t"]) and bits(dist) == bits(w["dist"]), (k, t, dist, w)
        p = (o + t * d).astype(F)
        n = mesh.normals[tri] if kind == 1 else (p - spheres[elem][0]).astype(F)          # mesh.rs:253-257 / sphere.rs:56
        assert (bits(p) == bits(w["point"])).all() and (bits(n) == bits(w["normal"])).all(), (k, p, n, w)
    assert kinds[0] > 50 and kinds[1] > 100 and kinds[-1] > 50, kinds                    # every arm was exercised


# ====================================================================== the rest of the path: camera, colorize, scatter
# (cam.rs:22-82, lib.rs:43-73,96-101, materials.rs:14-37, lambertian.rs:11-24, metal.rs:12-25, dielectric.rs:11-85),
# driven by the same counter-based RNG streams as the oracle and the GPU (Philox4x32-10, key = seed,
# counter = (pixel, sample, bounce, round): csrc/shade.cuh).

def philox4x32_10(c, k):
    c, k = [int(x) for x in c], [int(x) for x in k]
    for _ in range(10):
        p0, p1 = 0xD2511F53 * c[0], 0xCD9E8D57 * c[2]
        c = [(p1 >> 32) ^ c[1] ^ k[0], p1 & 0xFFFFFFFF, (p0 >> 32) ^ c[3] ^ k[1], p0 & 0xFFFFFFFF]
        k = [(k[0] + 0x9E3779B9) & 0xFFFFFFFF, (k[1] + 0xBB67AE85) & 0xFFFFFFFF]
    return c


def unit(u):                                                # rand 0.8 Standard f32: 24 bits, [0,1)
    return F(F(u >> 8) * F(1.0 / 16777216.0))


def normalize(a):                                           # three true divisions by the length (vec3.rs:119-126)
    return (a / length(a)).astype(F)


def vec(v):
    return np.array([v.x, v.y, v.z], F)


def camera_ray(cam, row, col, key, sample):                 # cam.rs:64-82
    W, H = cam.img_width_pix, cam.img_height_pix
    r = philox4x32_10([row * W + col, sample, 0, 0], key)
    u1, u2 = unit(r[0]), unit(r[1])
    cx, cy = F(F(col) - F(W // 2)), F(F(row) - F(H // 2))
    x_mm = F(F(F(cx + u1) - F(0.5)) * F(cam.mm_per_pix_hor))
    y_mm = F(F(F(cy + u2) - F(0.5)) * F(cam.mm_per_pix_vert))
    pos = vec(cam.position)
    target = ((vec(cam.img_center_point) + F(F(0.001) * x_mm) * vec(cam.right)).astype(F) - F(F(0.001) * y_mm) * vec(cam.up)).astype(F)
    return pos, normalize((target - pos).astype(F))


def random_point_in_unit_sphere(key, pixel, sample, bounce):   # materials.rs:14-30
    rnd = 0
    while True:
        r = philox4x32_10([pixel, sample, bounce, rnd], key)
        rnd += 1
        p = (F(2.0) * np.array([unit(r[0]), unit(r[1]), unit(r[2])], F) - np.ones(3, F)).astype(F)
        if not length(p) > 1.0:
            return p


def reflect(d, n):                                          # materials.rs:32-37
    du, nu = normalize(d), normalize(n)
    return normalize((du - (F(2.0) * nu).astype(F) * dot(du, nu)).astype(F))


def refract(d, n, ni):                                      # dielectric.rs:68-85
    vu, nu = normalize(d), normalize(n)
    c = dot(vu, nu)
    discr = F(F(1.0) - F(F(ni * ni) * F(F(1.0) - F(c * c))))
    if discr > 0:
        return ((ni * (vu - (nu * c).astype(F)).astype(F)).astype(F) - (np.sqrt(discr).astype(F) * nu).astype(F)).astype(F)
    return None


def schlick(cosine, ref_idx):                               # dielectric.rs:63-66 (powi(2), powi(5))
    r0 = F(F(F(1.0) - ref_idx) / F(F(1.0) + ref_idx))
    r0 = F(r0 * r0)
    x = F(F(1.0) - cosine)
    x2 = F(x * x)
    return F(r0 + F(F(F(1.0) - r0) * F(x * F(x2 * x2))))


COVER = {}


def scatter(mat, d, point, normal, key, pixel, sample, bounce):   # -> (attenuation, new direction) or None
    from rbrt_b200 import Dielectric, Lambertian, Metal
    COVER[type(mat).__name__] = COVER.get(type(mat).__name__, 0) + 1
    COVER["max_bounce"] = max(COVER.get("max_bounce", 0), bounce)
    if isinstance(mat, Lambertian):                         # lambertian.rs:11-24
        target = ((point + normalize(normal)).astype(F) + random_point_in_unit_sphere(key, pixel, sample, bounce)).astype(F)
        return vec(mat.albedo), normalize((target - point).astype(F))
    if isinstance(mat, Metal):                              # metal.rs:12-25
        out = normalize((reflect(d, normal) + (F(mat.roughness) * random_point_in_unit_sphere(key, pixel, sample, bounce)).astype(F)).astype(F))
        return (vec(mat.albedo), out) if dot(out, normal) > 0 else None
    assert isinstance(mat, Dielectric)                      # dielectric.rs:11-60
    ref_idx = F(mat.ref_idx)
    refl = reflect(d, normal)
    a = dot(normalize(d), normalize(normal))
    if a > 0:
        outward, ni, cosine = (F(-1.0) * normal).astype(F), ref_idx, F(ref_idx * a)
    else:
        outward, ni, cosine = normal, F(F(1.0) / ref_idx), F(-a)
    refr = refract(d, outward, ni)
    prob = schlick(cosine, ref_idx) if refr is not None else F(1.0)
    COVER["refracted" if refr is not None else "total_reflection"] = COVER.get("refracted" if refr is not None else "total_reflection", 0) + 1
    u = unit(philox4x32_10([pixel, sample, bounce, 0], key)[0])
    return np.ones(3, F), (refl if u < prob else (refr if refr is not None else np.zeros(3, F)))


def colorize(o, d, max_depth, world, key, pixel, sample):   # lib.rs:43-73: the recursion unrolled into a loop
    spheres, meshes, mats = world
    atts = []                                               # the attenuations in path order: the recursion's pending factors
    depth = max_depth
    while True:
        kind, elem, tri, t, dist = scene_hit(spheres, meshes, o, d)
        if kind < 0:
            tt = F(F(0.5) * F(d[1] + F(1.0)))               # lib.rs:68-71
            leaf = ((tt * np.ones(3, F)).astype(F) + (F(F(1.0) - tt) * np.array([0.05, 0.05, 0.8], F)).astype(F)).astype(F)
            break
        point = (o + t * d).astype(F)
        normal = meshes[elem].normals[tri] if kind == 1 else (point - spheres[elem][0]).astype(F)
        mat = mats[elem if kind == 0 else len(spheres) + elem]
        sc = scatter(mat, d, point, normal, key, pixel, sample, max_depth - depth + 1) if depth > 0 else None
        if sc is None:
            leaf = np.zeros(3, F)
            break
        atts.append(sc[0])
        o, d, depth = point, sc[1], depth - 1
    for a in reversed(atts):                                # att_1 * (att_2 * (... * leaf)): innermost first, as the recursion returns
        leaf = (a * leaf).astype(F)
    return leaf


def numpy_render(scene, cam, spp, seed, max_depth=50):
    """render_scene (lib.rs:75-124) by the numpy restatement: the HDR image (pre-gamma mean colour)."""
    W, H = cam.img_width_pix, cam.img_height_pix
    meshes = [NpMesh(np.asarray(m.triangles, dtype=F).reshape(-1, 3, 3), scene.simd_lanes) for m in scene.triangle_meshes]
    spheres = [(vec(e.center), F(e.radius)) for e in scene.elements]
    mats = [e.material for e in scene.elements] + [m.material for m in scene.triangle_meshes]
    key = [seed & 0xFFFFFFFF, seed >> 32]
    got = np.zeros((H, W, 3), F)
    inv = F(F(1.0) / F(spp))                                # lib.rs:101
    for row in range(H):
        for col in range(W):
            color = np.zeros(3, F)
            for s in range(spp):                            # lib.rs:96-100
                o, d = camera_ray(cam, row, col, key, s)
                color = (color + colorize(o, d, max_depth, (spheres, meshes, mats), key, row * W + col, s)).astype(F)
            got[row, col] = (color * inv).astype(F)
    return got


def test_numpy_render_agrees_with_the_oracle(oracle):
    """A whole (tiny) render — 20x15, 3 spp, spheres of all three materials + a 320-triangle glass mesh — by the numpy
    restatement of render_scene, bit for bit against the oracle's HDR image."""
    seed = 0x1234_5678_9ABC
    COVER.clear()
    scene = S.small_mesh_scene(2)
    cam = S.example_camera(20, 15)
    W, H, spp = 20, 15, 3
    want = oracle.OracleScene.from_scene(scene).render_hdr(cam.to_c(), spp, _abi.RenderOptsC(seed=seed))
    got = numpy_render(scene, cam, spp, seed)
    bad = (got.view(np.uint32) != want.view(np.uint32)).any(axis=2)
    assert not bad.any(), f"{int(bad.sum())} of {W * H} pixels differ, first at {np.argwhere(bad)[:3].tolist()}"
    # every arm of the path was exercised
    assert COVER.get("Lambertian", 0) > 50 and COVER.get("Metal", 0) > 10 and COVER.get("Dielectric", 0) > 20, COVER
    assert COVER.get("refracted", 0) > 5 and COVER.get("total_reflection", 0) > 0 and COVER["max_bounce"] >= 5, COVER


def test_numpy_render_of_deep_paths_agrees_with_the_oracle(oracle):
    """Paths that scatter far more than 64 times (tests/scenes.py deep_path_scene) at max_depth 300: the bounce index of the Philox
    stream runs to max_depth - depth + 1 past 64, and the oracle's attenuation store holds every factor of such a path."""
    COVER.clear()
    scene, cam = S.deep_path_scene(), S.deep_path_camera(6, 4)
    st = {}
    want = oracle.OracleScene.from_scene(scene).render_hdr(cam.to_c(), 2, _abi.RenderOptsC(seed=77, max_depth=300), st)
    got = numpy_render(scene, cam, 2, 77, max_depth=300)
    bad = (got.view(np.uint32) != want.view(np.uint32)).any(axis=2)
    assert not bad.any(), f"{int(bad.sum())} of 24 pixels differ, first at {np.argwhere(bad)[:3].tolist()}"
    assert st["rays"] > 65 * st["paths"] and COVER["max_bounce"] > 100 and (want > 0).any(axis=2).sum() >= 8, (st, COVER)
