"""Procedural scenes for BASELINE.json's configs (the Stanford bunny.obj the reference renders is not
shipped, .gitignore:5 of the reference, and there is no network): displaced icospheres written as real
.obj files or handed over as triangle soup, plus the spheres of scenes/example_scene.yaml:33-75."""
import atexit
import os
import shutil
import tempfile

import numpy as np

from .blueprints import CameraBluePrint, SceneBlueprint, SphereBlueprint, TriangleMeshBlueprint
from .materials import Dielectric, Lambertian, Metal
from .vec3 import Vec3

_T = (1.0 + 5.0 ** 0.5) / 2.0
_ICO_V = np.array([[-1, _T, 0], [1, _T, 0], [-1, -_T, 0], [1, -_T, 0], [0, -1, _T], [0, 1, _T], [0, -1, -_T], [0, 1, -_T],
                   [_T, 0, -1], [_T, 0, 1], [-_T, 0, -1], [-_T, 0, 1]], dtype=np.float64)
_ICO_F = np.array([[0, 11, 5], [0, 5, 1], [0, 1, 7], [0, 7, 10], [0, 10, 11], [1, 5, 9], [5, 11, 4], [11, 10, 2], [10, 7, 6],
                   [7, 1, 8], [3, 9, 4], [3, 4, 2], [3, 2, 6], [3, 6, 8], [3, 8, 9], [4, 9, 5], [2, 4, 11], [6, 2, 10],
                   [8, 6, 7], [9, 8, 1]], dtype=np.int64)


def icosphere(subdiv):
    """Unit icosphere: 20 * 4**subdiv CCW triangles. Returns (verts [V,3] f64, faces [F,3] i64)."""
    v = _ICO_V / np.linalg.norm(_ICO_V, axis=1, keepdims=True)
    f = _ICO_F
    for _ in range(subdiv):
        e = np.concatenate([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]], axis=0)
        e.sort(axis=1)
        key = e[:, 0] * (len(v) + 1) + e[:, 1]
        uniq, inv = np.unique(key, return_inverse=True)
        a, b = uniq // (len(v) + 1), uniq % (len(v) + 1)
        mid = v[a] + v[b]
        mid /= np.linalg.norm(mid, axis=1, keepdims=True)
        base = len(v)
        v = np.concatenate([v, mid], axis=0)
        n = len(f)
        m01, m12, m20 = base + inv[:n], base + inv[n:2 * n], base + inv[2 * n:]
        f = np.concatenate([np.stack([f[:, 0], m01, m20], 1), np.stack([f[:, 1], m12, m01], 1),
                            np.stack([f[:, 2], m20, m12], 1), np.stack([m01, m12, m20], 1)], axis=0)
    return v, f


def displace(verts, amplitude=0.05, seed=1234, octaves=6):
    """Smooth radial displacement r = 1 + amplitude * noise(p), |noise| <= 1 (sum of random sinusoids)."""
    rng = np.random.default_rng(seed)
    k = rng.normal(size=(octaves, 3)) * np.linspace(2.0, 9.0, octaves)[:, None]
    phase = rng.uniform(0, 2 * np.pi, size=octaves)
    w = 1.0 / np.arange(1, octaves + 1)
    noise = (np.sin(verts @ k.T + phase) * w).sum(axis=1) / w.sum()
    return verts * (1.0 + amplitude * noise)[:, None]


def displaced_icosphere(subdiv, radius=1.0, center=(0.0, 0.0, 0.0), amplitude=0.05, seed=1234):
    """Triangle soup [F,3,3] f32 of a displaced icosphere."""
    v, f = icosphere(subdiv)
    v = displace(v, amplitude, seed) * radius + np.asarray(center, dtype=np.float64)
    return v.astype(np.float32)[f]


def write_obj(path, verts, faces):
    with open(path, "w") as fh:
        fh.write("# rbrt_b200 procedural mesh\no mesh\n")
        np.savetxt(fh, verts, fmt="v %.9g %.9g %.9g")
        np.savetxt(fh, faces + 1, fmt="f %d %d %d")


# ---- the fixture of scenes/example_scene.yaml --------------------------------------------------
EXAMPLE_CAMERA = dict(camera_up=(0.0, 1.0, -0.4), camera_look_at=(0.0, -0.1, -1.0), camera_position=(0.0, 5.0, 4.0),
                      camera_focal_length_mm=28.0)  # example_scene.yaml:2-15


def example_camera_blueprint():
    c = EXAMPLE_CAMERA
    return CameraBluePrint(Vec3(*c["camera_up"]), Vec3(*c["camera_look_at"]), Vec3(*c["camera_position"]),
                           c["camera_focal_length_mm"])


def example_sphere_blueprints():  # example_scene.yaml:33-75
    return [
        SphereBlueprint(1000.0, Vec3(0.0, -1000.0, -5.0), "lambertian", Vec3(0.02, 0.2, 0.1), None),
        SphereBlueprint(1.5, Vec3(-5.0, 1.5, -9.0), "lambertian", Vec3(0.1, 0.1, 0.9), None),
        SphereBlueprint(3.0, Vec3(-2.5, 2.9, -15.0), "metal", Vec3(0.8, 0.8, 0.8), 0.005),
        SphereBlueprint(1.5, Vec3(1.5, 1.25, -9.0), "dielectric", None, 1.8),
    ]


def write_bunny_standin(path, subdiv=6, seed=1234):
    """A closed displaced icosphere in bunny-like object coordinates: with the fixture's scale 45 and
    translation (5,-1.8,-12.5) (example_scene.yaml:18-23) it is ~6.3 units across and rests on the ground."""
    v, f = icosphere(subdiv)
    v = displace(v, 0.05, seed) * 0.07 + np.array([0.0, 0.11, 0.0])
    write_obj(path, v.astype(np.float32), f)
    return len(f)


def example_scene_blueprint(obj_path):
    """= scenes/example_scene.yaml with `obj_path` substituted for bunny.obj (config C2)."""
    mesh = TriangleMeshBlueprint(obj_path, 45.0, Vec3(5.0, -1.8, -12.5), Vec3(0.0, 0.0, 0.0), "dielectric",
                                 Vec3(0.8, 0.8, 0.8), 0.2)
    return SceneBlueprint(example_camera_blueprint(), [mesh], example_sphere_blueprints())


def header_card_blueprint(obj_path):
    """= scenes/header_card.yaml of the reference (the scene of its README banner: 7 spheres + a red lambertian bunny at scale 45,
    translation (3.5, -1.8, -14)) with `obj_path` substituted for bunny.obj.  tests/test_host.py compares it field by field
    with the reference's file when the reference tree is mounted."""
    mesh = TriangleMeshBlueprint(obj_path, 45.0, Vec3(3.5, -1.8, -14.0), Vec3(0.0, 0.0, 0.0), "lambertian", Vec3(1.0, 0.0, 0.0), None)
    spheres = [
        SphereBlueprint(1000.0, Vec3(0.0, -1000.0, -12.0), "lambertian", Vec3(0.02, 0.2, 0.1), None),
        SphereBlueprint(1.5, Vec3(-7.5, 1.5, -10.5), "lambertian", Vec3(0.1, 0.1, 0.9), None),
        SphereBlueprint(0.7, Vec3(3.0, 0.7, -9.5), "lambertian", Vec3(0.5, 0.5, 0.1), None),
        SphereBlueprint(2.5, Vec3(-4.5, 2.5, -16.0), "metal", Vec3(0.9, 0.9, 0.9), 0.005),
        SphereBlueprint(4.0, Vec3(9.5, 4.0, -20.0), "metal", Vec3(0.9, 0.9, 0.9), 0.001),
        SphereBlueprint(1.0, Vec3(-1.5, 1.0, -8.0), "dielectric", None, 1.8),
        SphereBlueprint(1.5, Vec3(7.0, 1.5, -10.0), "dielectric", None, 1.8),
    ]
    return SceneBlueprint(example_camera_blueprint(), [mesh], spheres)


def blueprint_to_yaml(bp):
    """A SceneBlueprint as the YAML text load_blueprints_from_yaml_file reads (blueprints.rs:15-48 field names)."""
    import yaml
    v = lambda a: None if a is None else {"x": float(a.x), "y": float(a.y), "z": float(a.z)}
    opt = lambda d: {k: x for k, x in d.items() if x is not None}
    c = bp.camera_blueprint
    return yaml.safe_dump({
        "camera_blueprint": {"camera_up": v(c.camera_up), "camera_look_at": v(c.camera_look_at), "camera_position": v(c.camera_position),
                             "camera_focal_length_mm": float(c.camera_focal_length_mm)},
        "mesh_blueprints": [opt({"obj_filepath": m.obj_filepath, "scale": float(m.scale), "translation": v(m.translation),
                                 "rotation_rad": v(m.rotation_rad), "material_type": m.material_type, "albedo": v(m.albedo),
                                 "material_param": m.material_param}) for m in bp.mesh_blueprints],
        "sphere_blueprints": [opt({"radius": float(sp.radius), "center": v(sp.center), "material_type": sp.material_type, "albedo": v(sp.albedo),
                                   "material_param": sp.material_param}) for sp in bp.sphere_blueprints]}, sort_keys=False)


def spheres_only_blueprint():
    """Config C1: example_scene.yaml with the mesh removed."""
    return SceneBlueprint(example_camera_blueprint(), [], example_sphere_blueprints())


def big_mesh_config(subdiv, radius, seed=1234):
    """Configs C3 / C5: one displaced icosphere of `radius` resting on a ground sphere, three feature
    spheres in front, camera pulled back so everything is within t < 1000 (the reference's triangle
    window, triangle.rs:146).  Triangle size keeps 2*area well above the 1e-3 determinant cull.
    Returns (camera kwargs for Camera.new, spheres, triangles, mesh material)."""
    tris = displaced_icosphere(subdiv, radius, (0.0, radius * 1.02, -3.2 * radius), 0.05, seed)
    r = radius
    spheres = [
        (Vec3(0.0, -1000.0, -3.2 * r), 1000.0, Lambertian(Vec3(0.02, 0.2, 0.1))),
        (Vec3(-1.6 * r, 0.45 * r, -1.7 * r), 0.45 * r, Lambertian(Vec3(0.1, 0.1, 0.9))),
        (Vec3(1.7 * r, 0.5 * r, -2.0 * r), 0.5 * r, Metal(Vec3(0.8, 0.8, 0.8), 0.005)),
        (Vec3(0.3 * r, 0.3 * r, -1.2 * r), 0.3 * r, Dielectric(1.8)),
    ]
    cam = dict(position=Vec3(0.0, 1.6 * r, 1.2 * r), look_at=Vec3(0.0, -0.12, -1.0), up=Vec3(0.0, 1.0, -0.12),
               focal_len_mm=28.0)
    return cam, spheres, tris, Lambertian(Vec3(0.7, 0.35, 0.2))


def stress_config(seed=4321):
    """Config C4: divergence stress — a 6x6 field of glass (ref_idx 1.5-1.8) and low-roughness metal spheres around
    a glass displaced icosphere (20 480 triangles), on the fixture's ground sphere, seen by the fixture camera.
    More than half of the frame is covered by specular material, so paths use the 50-bounce budget.
    Returns (spheres, triangles, mesh material)."""
    rng = np.random.default_rng(seed)
    spheres = [(Vec3(0.0, -1000.0, -5.0), 1000.0, Lambertian(Vec3(0.02, 0.2, 0.1)))]
    for i in range(6):
        for j in range(6):
            if (i, j) in ((2, 2), (3, 2), (2, 3), (3, 3)):
                continue                                  # the mesh stands here
            r = float(rng.uniform(0.9, 1.3))
            x, z = -9.0 + 3.6 * i + float(rng.uniform(-0.3, 0.3)), -5.0 - 3.4 * j + float(rng.uniform(-0.3, 0.3))
            if (i + j) % 2 == 0:
                mat = Dielectric(float(rng.uniform(1.5, 1.8)))
            else:
                mat = Metal(Vec3(*rng.uniform(0.6, 0.95, size=3)), float(rng.uniform(0.0, 0.02)))
            spheres.append((Vec3(x, r, z), r, mat))
    tris = displaced_icosphere(5, 3.0, (0.0, 3.0, -13.5), 0.05, seed)
    return spheres, tris, Dielectric(1.5)


_TMP_CACHE = []


def cache_dir():
    """Where generated scene files go: RBRT_B200_CACHE, else a temporary directory of this process, removed when it exits (the
    source tree may be read-only, and a directory of its own keeps processes from reading each other's half-written files)."""
    d = os.environ.get("RBRT_B200_CACHE")
    if not d:
        if not _TMP_CACHE:
            _TMP_CACHE.append(tempfile.mkdtemp(prefix="rbrt_b200_synth_"))
            atexit.register(shutil.rmtree, _TMP_CACHE[0], True)
        d = _TMP_CACHE[0]
    os.makedirs(d, exist_ok=True)
    return d
