"""First-hit AOVs (rbrt_gpu_render_aov / rbrt_gpu_render_aov_device; csrc/aov.cu, csrc/api.cu) on the GPU.

Every pass is defined by the parity hooks (include/rbrt_gpu.h, DESIGN.md section 11): the renderer's primary rays of each sample, their
closest hits as rbrt_gpu_trace_rays reports them, and f32 sums in sample order.  tests/aov_ref.py restates those rules in numpy, so
every comparison below is bit-exact, on uint32 views (NaN and +-inf compare too)."""
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

from . import aov_ref as A
from . import golden_util as G
from . import scenes as S
from .test_cli_cpp import write_scene
from .test_gpu_trace import mixed_element_scene
from .test_gpu_update import fresh, moved_elements, twist

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
AOV_SO = os.path.join(ROOT, "rbrt_b200", "librbrt_gpu_aov.so")
PLANES = {"depth": 1, "normal": 3, "albedo": 3, "coverage": 1, "hit_kind": 1, "elem_idx": 1, "tri_idx": 1}
PASS_PLANES = {"depth": ["depth"], "normal": ["normal"], "albedo": ["albedo"], "coverage": ["coverage"],
               "ids": ["hit_kind", "elem_idx", "tri_idx"]}


@pytest.fixture(scope="module", autouse=True)
def aov_module():
    """The session fixture only builds librbrt_gpu.so when it is missing; the AOV module is built here when it is."""
    if not os.path.exists(AOV_SO):
        subprocess.run(["make", "-C", os.path.join(ROOT, "rbrt_b200", "csrc")], check=True)
    return AOV_SO


def assert_passes(got, want, what):
    bad = A.mismatches(got, want)
    assert not bad, f"{what}: differing values per pass {bad}"


def to_np(t):
    """A CUDA tensor of 4-byte values as a numpy uint32 array (bit pattern)."""
    import torch
    return t.contiguous().view(torch.int32).cpu().numpy().view(np.uint32)


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def negative_radius_scene():
    """C1's spheres plus a hollow glass ball: a sphere inside a negative-radius sphere of the same centre (normals point inward)."""
    scene = S.spheres_scene()
    scene.elements += [R.Sphere(Vec3(1.0, 1.2, -4.0), 0.9, R.Dielectric(1.5)), R.Sphere(Vec3(1.0, 1.2, -4.0), -0.8, R.Dielectric(1.5)),
                       R.Sphere(Vec3(-1.5, 0.8, -3.5), -0.7, R.Metal(Vec3(0.7, 0.6, 0.5), 0.1))]
    return scene


def meshes_scene(leaf_size=8):
    """Three meshes of the three material kinds, among C1's spheres."""
    scene = S.small_mesh_scene(3, leaf_size=leaf_size)
    scene.triangle_meshes.append(R.TriangleMesh.from_triangles(synth.displaced_icosphere(2, 1.2, (-3.0, 1.5, -8.0)), R.Lambertian(Vec3(0.3, 0.6, 0.9))))
    scene.triangle_meshes.append(R.TriangleMesh.from_triangles(synth.displaced_icosphere(3, 2.0, (1.0, 3.5, -10.0)), R.Metal(Vec3(0.9, 0.8, 0.2), 0.05)))
    return scene


SCENES = {"example_leaf1": lambda: S.small_mesh_scene(3, leaf_size=1), "example_leaf8": lambda: S.small_mesh_scene(3, leaf_size=8),
          "mixed_elements": mixed_element_scene, "negative_radius": negative_radius_scene, "meshes": meshes_scene}


# ============================================================================== 1. golden vectors, S = 1
@pytest.mark.parametrize("name", G.NAMES)
def test_golden_scenes_one_sample(gpu, name):
    z, scene, cam = G.load(name)
    W, H = cam.img_width_pix, cam.img_height_pix
    want = A.compose([z["hits"][:W * H]], *A.albedo_tables(scene), shape=(H, W))
    assert (want["hit_kind"] != _abi.HIT_NONE).sum() > 100
    assert_passes(R.render_aovs(cam, 1, scene, seed=int(z["seed"])), want, name)


# ============================================================================== 2. composition from the parity hooks (and the oracle)
@pytest.mark.parametrize("spp", [1, 3, 16])
@pytest.mark.parametrize("name", list(SCENES))
def test_composition_of_primary_rays_and_hits(gpu, oracle, name, spp):
    scene = SCENES[name]()
    cam = S.example_camera(64, 48)
    want = A.expected(cam, spp, scene, seed=9)
    got = R.render_aovs(cam, spp, scene, seed=9)
    assert_passes(got, want, f"{name} S={spp}")
    assert_passes(A.expected(cam, spp, scene, seed=9, oracle=oracle), want, f"{name} S={spp}: oracle composition")
    kinds = set(np.unique(want["hit_kind"]).tolist())
    assert _abi.HIT_SPHERE in kinds
    if name != "negative_radius":
        assert (_abi.HIT_MESH in kinds or _abi.HIT_TRIANGLE in kinds), kinds
    if name == "mixed_elements":
        assert {_abi.HIT_MESH, _abi.HIT_TRIANGLE} <= kinds
        alb = want["albedo"][want["coverage"] == 1].reshape(-1, 3)
        assert (alb == 1).all(1).any() and (alb != 1).any(1).any()       # Dielectric (1,1,1) and coloured Lambertian / Metal
    if spp > 1:
        cov = want["coverage"]
        assert ((cov > 0) & (cov < 1)).any()                              # edges: some samples hit, some do not


# ============================================================================== 3. C3 (1.31 M triangles)
def test_c3_reduced_composition_and_full_size_ids(gpu):
    scene, cam_full = S.big_scene(8)
    camkw = S._BIG[8][0]
    small = R.Camera.new(camkw["position"], camkw["look_at"], camkw["up"], 270, 480, camkw["focal_len_mm"])
    st = {}
    got = R.render_aovs(small, 4, scene, seed=3, stats=st)
    want = A.expected(small, 4, scene, seed=3)
    assert (want["hit_kind"] == _abi.HIT_MESH).sum() > 10000
    assert_passes(got, want, "C3 480x270 S=4")
    assert st["rays"] == 480 * 270 * 4 and st["node_visits"] > 0 and st["launches"] == 1
    hits = scene.hit(R.primary_rays(cam_full, 3, 0))
    ids = R.render_aovs(cam_full, 1, scene, seed=3, passes="ids")
    assert set(ids) == {"hit_kind", "elem_idx", "tri_idx"}
    H, W = 1080, 1920
    assert np.array_equal(ids["hit_kind"], hits["kind"].reshape(H, W))
    assert np.array_equal(ids["elem_idx"], hits["elem_idx"].reshape(H, W))
    assert np.array_equal(ids["tri_idx"], hits["tri_idx"].reshape(H, W))


# ============================================================================== 4. image shapes
@pytest.mark.parametrize("wh", [(1, 1), (1, 37), (29, 1), (13, 7), (50, 3), (9, 5)])
def test_image_shapes(gpu, wh):
    w, h = wh
    scene = S.small_mesh_scene(3)
    cam = S.example_camera(w, h)
    got = R.render_aovs(cam, 2, scene, seed=1)
    assert got["depth"].shape == (h, w) and got["normal"].shape == (h, w, 3)
    assert_passes(got, A.expected(cam, 2, scene, seed=1), f"{w}x{h}")


# ============================================================================== 5. pass subsets and refusals
def test_pass_subsets_equal_the_full_set(gpu):
    scene = S.small_mesh_scene(3)
    cam = S.example_camera(40, 30)
    full = R.render_aovs(cam, 3, scene, seed=2)
    assert set(full) == set(PLANES)
    for p, planes in PASS_PLANES.items():
        one = R.render_aovs(cam, 3, scene, seed=2, passes=(p,))
        assert set(one) == set(planes), p
        assert_passes(one, {k: full[k] for k in planes}, f"pass {p} alone")


def test_unrequested_planes_keep_their_sentinel_bytes(gpu):
    """All seven planes are carved from ONE device block filled with a sentinel; a call gets pointers to some of them only.  The
    others, and the gaps between the planes, must keep the sentinel."""
    import torch
    scene = S.small_mesh_scene(3)
    cam = S.example_camera(24, 20)
    n = 24 * 20
    full = R.render_aovs(cam, 3, scene, seed=2)
    off, o = {}, 0
    for k, c in PLANES.items():
        off[k] = o
        o += c * n + 16                                                   # a 64-byte gap after every plane
    SENT = 0x7FA5A5A5
    block = torch.empty(o, dtype=torch.int32, device="cuda")
    s = torch.cuda.Stream()
    lib = _abi.lib()
    for requested in [[p] for p in PASS_PLANES] + [list(PASS_PLANES)]:
        planes = [k for p in requested for k in PASS_PLANES[p]]
        block.fill_(SENT)
        torch.cuda.synchronize()
        out = _abi.AovOutC(**{k: block.data_ptr() + 4 * off[k] for k in planes})
        _abi.check(lib.rbrt_gpu_render_aov_device(scene.handle(), cam.to_c(), 3, 2, out, s.cuda_stream, None))
        s.synchronize()
        b = block.cpu().numpy().view(np.uint32)
        touched = np.zeros(o, bool)
        for k in planes:
            seg = b[off[k]:off[k] + PLANES[k] * n]
            assert np.array_equal(seg, bits(full[k]).ravel()), (requested, k)
            touched[off[k]:off[k] + PLANES[k] * n] = True
        assert (b[~touched] == SENT).all(), f"{requested}: bytes outside the requested planes were written"


def test_refusals(gpu):
    lib = _abi.lib()
    scene = S.small_mesh_scene(3)
    cam = S.example_camera(16, 12)
    depth = np.full(16 * 12, 7.0, np.float32)
    out = _abi.AovOutC(depth=depth.ctypes.data)
    h, c = scene.handle(), cam.to_c()
    assert lib.rbrt_gpu_render_aov(h, c, 1, 0, _abi.AovOutC(), None) == _abi.E_INVALID       # every pass NULL
    assert lib.rbrt_gpu_render_aov(h, c, 0, 0, out, None) == _abi.E_INVALID                  # zero samples
    assert lib.rbrt_gpu_render_aov(h, S.example_camera(0, 12).to_c(), 1, 0, out, None) == _abi.E_INVALID   # empty image
    assert lib.rbrt_gpu_render_aov(None, c, 1, 0, out, None) == _abi.E_INVALID              # NULL scene
    assert lib.rbrt_gpu_render_aov(h, None, 1, 0, out, None) == _abi.E_INVALID              # NULL camera
    assert lib.rbrt_gpu_render_aov(h, c, 1, 0, None, None) == _abi.E_INVALID                # NULL out
    assert lib.rbrt_gpu_render_aov_device(h, c, 0, 0, out, None, None) == _abi.E_INVALID
    assert (depth == 7.0).all()
    assert _abi.lib().rbrt_gpu_render_aov(h, c, 1, 0, out, None) == 0 and not (depth == 7.0).all()   # the same call, valid


def test_missing_module_is_refused_with_a_message(gpu):
    """Without librbrt_gpu_aov.so the call fails with a message naming the module, and the rest of the library works."""
    code = ("import sys; sys.path.insert(0, %r)\n"
            "import numpy as np, rbrt_b200 as R\nfrom tests import scenes as S\nfrom rbrt_b200 import _abi\n"
            "R.gpu_init(0); sc = S.small_mesh_scene(3); cam = S.example_camera(16, 12)\n"
            "try:\n    R.render_aovs(cam, 1, sc)\n    print('NO ERROR')\n"
            "except _abi.RbrtGpuError as e:\n    print('CODE', e.code, str(e))\n"
            "print('RENDER', R.render_scene_hdr(cam, 1, sc).shape)\n") % ROOT
    env = dict(os.environ, RBRT_GPU_AOV_LIB=os.path.join(ROOT, "no-such-dir", "librbrt_gpu_aov.so"))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr
    assert f"CODE {_abi.E_CUDA}" in r.stdout and "AOV module is missing" in r.stdout, r.stdout
    assert "RENDER (12, 16, 3)" in r.stdout, r.stdout


# ============================================================================== 6. device variant
def test_device_variant_on_a_side_stream_equals_the_host_variant(gpu):
    import torch
    scene = mixed_element_scene()
    cam = S.example_camera(50, 30)
    host = R.render_aovs(cam, 4, scene, seed=5)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        dev = R.render_aovs_device(cam, 4, scene, seed=5, stream=s)
    s.synchronize()
    assert set(dev) == set(host)
    for k, t in dev.items():
        assert t.device.type == "cuda" and tuple(t.shape) == host[k].shape, k
        assert np.array_equal(to_np(t), bits(host[k])), k


def test_device_variant_without_stats_does_not_synchronise(gpu):
    import torch
    scene = S.small_mesh_scene(3)
    cam = S.example_camera(32, 24)
    ref = R.render_aovs(cam, 2, scene, seed=8)                            # the scene is built and the module loaded
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        torch.cuda._sleep(int(2e9))                                       # about a second of work ahead of the call on its stream
        t0 = time.perf_counter()
        dev = R.render_aovs_device(cam, 2, scene, seed=8, stream=s)
        dt = time.perf_counter() - t0
        busy = not s.query()
    s.synchronize()
    assert busy and dt < 0.3, (busy, dt)
    for k, t in dev.items():
        assert np.array_equal(to_np(t), bits(ref[k])), k


def test_stats(gpu):
    import torch
    lib = _abi.lib()
    scene = S.small_mesh_scene(3)
    cam = S.example_camera(40, 30)
    st = {}
    R.render_aovs(cam, 5, scene, seed=1, stats=st)
    assert st["rays"] == 40 * 30 * 5 and st["launches"] == 1 and st["ms_device"] > 0 and st["ms_total"] >= st["ms_device"]
    assert st["nan_rays"] == 0 and st["node_visits"] > 0
    t = torch.empty(40 * 30, dtype=torch.float32, device="cuda")
    dst = _abi.StatsC()
    _abi.check(lib.rbrt_gpu_render_aov_device(scene.handle(), cam.to_c(), 5, 1, _abi.AovOutC(coverage=t.data_ptr()), None, dst))
    assert dst.rays == 40 * 30 * 5 and dst.launches == 1 and dst.ms_device > 0
    # a sphere with a NaN centre makes every ray a NaN ray (the reference panics): misses, counted
    nan_scene = R.Scene(elements=[R.Sphere(Vec3(float("nan"), 0.0, -3.0), 1.0, R.Lambertian(Vec3(0.5, 0.5, 0.5)))])
    st = {}
    got = R.render_aovs(cam, 3, nan_scene, seed=1, stats=st)
    assert st["nan_rays"] == 40 * 30 * 3
    assert (got["coverage"] == 0).all() and np.isinf(got["depth"]).all() and (got["hit_kind"] == _abi.HIT_NONE).all()
    assert_passes(got, A.expected(cam, 3, nan_scene, seed=1), "NaN rays")


# ============================================================================== 7. ordering against updates
def test_ordering_against_a_device_mesh_update(gpu):
    import torch
    scene = S.small_mesh_scene(3)
    cam = S.example_camera(48, 36)
    old = R.render_aovs(cam, 2, fresh(scene), seed=4)
    new = twist(scene.triangle_meshes[0].triangles, 0.8)
    ref_scene = fresh(scene)
    ref_scene.triangle_meshes[0] = R.TriangleMesh.from_triangles(new, ref_scene.triangle_meshes[0].material)
    want_new = R.render_aovs(cam, 2, ref_scene, seed=4)
    assert A.mismatches(old, want_new), "the deformation must change the passes"
    R.render_aovs(cam, 1, scene)                                          # built and in use before the update
    t_new = torch.from_numpy(new.copy()).cuda()
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        torch.cuda._sleep(int(5e8))                                       # the first AOV waits in the stream while the update is enqueued
        a = R.render_aovs_device(cam, 2, scene, seed=4, stream=s)
        scene.update_mesh_device(0, t_new, stream=s)
        b = R.render_aovs_device(cam, 2, scene, seed=4, stream=s)
    s.synchronize()
    for k in PLANES:
        assert np.array_equal(to_np(a[k]), bits(old[k])), f"before the update: {k}"
        assert np.array_equal(to_np(b[k]), bits(want_new[k])), f"after the update: {k}"


def test_ordering_against_an_element_update(gpu):
    import torch
    scene = mixed_element_scene()
    cam = S.example_camera(48, 36)
    old = R.render_aovs(cam, 2, fresh(scene), seed=4)
    moved = moved_elements(scene.elements, 3)
    ref_scene = fresh(scene)
    ref_scene.elements = list(moved)
    want_new = R.render_aovs(cam, 2, ref_scene, seed=4)
    assert A.mismatches(old, want_new), "the update must change the passes"
    R.render_aovs(cam, 1, scene)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        torch.cuda._sleep(int(5e8))
        a = R.render_aovs_device(cam, 2, scene, seed=4, stream=s)
        scene.update_elements(moved)
        b = R.render_aovs_device(cam, 2, scene, seed=4, stream=s)
    s.synchronize()
    for k in PLANES:
        assert np.array_equal(to_np(a[k]), bits(old[k])), f"before the update: {k}"
        assert np.array_equal(to_np(b[k]), bits(want_new[k])), f"after the update: {k}"


# ============================================================================== 8. seeds
@pytest.mark.parametrize("seed", [0, 2**64 - 1])
def test_seeds(gpu, seed):
    scene = S.small_mesh_scene(3)
    cam = S.example_camera(40, 30)
    assert_passes(R.render_aovs(cam, 3, scene, seed=seed), A.expected(cam, 3, scene, seed=seed), f"seed {seed}")


# ============================================================================== 9. communicator
def test_emulated_communicator_gives_the_same_passes(gpu):
    cam = S.example_camera(40, 30)
    ref = R.render_aovs(cam, 3, S.small_mesh_scene(3), seed=6)
    lib = _abi.lib()
    devs = (C.c_int * 2)(0, 0)
    _abi.check(lib.rbrt_gpu_init_multi(devs, 2, _abi.TRANSPORT_PEER))
    try:
        scene = S.small_mesh_scene(3)
        assert_passes(R.render_aovs(cam, 3, scene, seed=6), ref, "under a one-GPU two-rank communicator")
        scene.close()
    finally:
        _abi.check(lib.rbrt_gpu_comm_destroy())
    R.gpu_init(0)


# ============================================================================== 10. CLI
def read_pfm(path):
    data = open(path, "rb").read()
    parts = data.split(b"\n", 3)
    kind, (w, h), scale = parts[0], map(int, parts[1].split()), float(parts[2])
    ch = {b"PF": 3, b"Pf": 1}[kind]
    assert scale < 0                                                      # little-endian
    v = np.frombuffer(parts[3], dtype="<f4")
    assert v.size == w * h * ch
    img = v.reshape(h, w, ch)[::-1]                                       # rows are stored bottom to top
    return img[..., 0] if ch == 1 else img


def test_cli_writes_pfm_aovs(gpu, tmp_path):
    cli = os.path.join(ROOT, "rbrt_b200", "rbrt")
    y, _ = write_scene(tmp_path)
    bp = R.load_blueprints_from_yaml_file(y)
    cb = bp.camera_blueprint
    cam = R.Camera.new(cb.camera_position, cb.camera_look_at, cb.camera_up, 30, 44, cb.camera_focal_length_mm)
    scene = R.create_scene_from_scene_blueprint(bp)
    for extra, spp in [([], 2), (["--aov-samples", "5"], 5)]:
        prefix = str(tmp_path / f"out{spp}")
        r = subprocess.run([cli, "-c", y, "--height", "30", "-w", "44", "-s", "2", "--seed", "5", "-t", prefix + ".png", "--aov", prefix] + extra,
                           capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        assert os.path.exists(prefix + ".png")
        want = R.render_aovs(cam, spp, scene, seed=5, passes=("depth", "normal", "albedo", "coverage"))
        for k in ("depth", "normal", "albedo", "coverage"):
            got = read_pfm(f"{prefix}.{k}.pfm")
            assert np.array_equal(bits(got), bits(want[k])), (spp, k)
