"""Per-object motion vectors without a GPU: the module is built for sm_100a with its two kernels, the struct matches the header, the entry
points refuse bad calls without touching a device, and tests/motion_ref.py equals the host build of csrc/motion.cuh (the motion pass) and
of csrc/temporal.cuh (the motion variant of the temporal step) bit for bit: every hit kind, changed and unchanged elements, negative
radii, cameras equal but not bitwise, points behind either camera, and ±0, ±inf and NaN inputs."""
import ctypes as C
import dataclasses
import os
import shutil
import subprocess

import numpy as np
import pytest

import rbrt_b200 as R
from rbrt_b200 import _abi

from . import motion_ref as M
from . import temporal_ref as T
from .test_temporal_host import CASE_NAMES, camera, cases, frame, history, same_all

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "rbrt_b200", "librbrt_gpu_motion.so")
HD = os.path.join(ROOT, "tests", "host_device")
CSRC = os.path.join(ROOT, "rbrt_b200", "csrc")
F = np.float32
SPECIALS = np.array([0.0, -0.0, np.inf, -np.inf, np.nan], F)


@pytest.fixture(scope="module", autouse=True)
def motion_module():
    if not os.path.exists(LIB):
        subprocess.run(["make", "-C", CSRC], check=True)
    return LIB


@pytest.fixture(scope="module")
def hd():
    out = os.path.join(HD, "build", "libhost_motion.so")
    os.makedirs(os.path.dirname(out), exist_ok=True)
    srcs = [os.path.join(HD, f) for f in ("motion_harness.cpp", "cuda_runtime.h")] + \
           [os.path.join(CSRC, f) for f in ("common.cuh", "denoise.cuh", "temporal.cuh", "motion.cuh")]
    if not os.path.exists(out) or any(os.path.getmtime(s) > os.path.getmtime(out) for s in srcs):
        # the flags of tests/test_device_source_on_host.py: the stand-in cuda_runtime.h first, no contraction, no FMA
        subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-mno-fma", "-Wno-unknown-pragmas", "-fPIC", "-shared",
                        "-I", HD, "-I", CSRC, "-o", out, srcs[0]], check=True)
    lib = C.CDLL(out)
    P = C.POINTER(_abi.CameraC)
    lib.hd_motion.argtypes = [C.c_uint32, P, P] + [C.c_void_p] * 6
    lib.hd_pixel_dirs.argtypes = [P, C.c_void_p]
    lib.hd_temporal_motion.argtypes = [C.c_uint32, C.c_uint32, P, P] + [C.c_void_p] * 7
    return lib


def host_motion(hd, cam, prev, tri, o, d, t, cur, old):
    n = len(t)
    odt = np.ascontiguousarray(np.concatenate([o, d, np.asarray(t, F)[:, None]], 1), F)
    tri = np.ascontiguousarray(tri, np.int32)
    cur, old = np.ascontiguousarray(cur, F), np.ascontiguousarray(old, F)
    m, pd = np.zeros((n, 2), F), np.zeros(n, F)
    assert hd.hd_motion(n, cam.to_c(), prev.to_c(), tri.ctypes.data, odt.ctypes.data, cur.ctypes.data, old.ctypes.data, m.ctypes.data,
                        pd.ctypes.data) == 0
    return m, pd


# ============================================================================== synthetic hits
def hits(cam, n, seed, specials=False):
    """n hits seen from cam: (tri, o, d, t, cur, old).  Triangles and spheres in front of the camera, each unchanged, translated, scaled
    or deformed since the snapshot; spheres with negative radii too; with specials, ±0, ±inf and NaN in records, rays and t."""
    rng = np.random.default_rng(seed)
    pos = T.cam_values(cam)[0].astype(np.float64)
    tri = rng.random(n) < 0.6
    cur = np.zeros((n, 3, 4), F)
    centre = pos + np.array([0.0, 0.0, -6.0]) + rng.normal(0, 1.5, (n, 3))
    cur[:, 0, :3] = centre
    cur[:, 1, :3] = rng.normal(0, 1.0, (n, 3))
    cur[:, 2, :3] = rng.normal(0, 1.0, (n, 3))
    radius = rng.uniform(0.2, 1.5, n) * np.where(rng.random(n) < 0.2, -1, 1)
    cur[~tri, 0, 3] = radius[~tri]
    cur[~tri, 1:] = 0
    a, b = rng.random(n) * 0.5, rng.random(n) * 0.5
    target = np.where(tri[:, None], cur[:, 0, :3] + a[:, None] * cur[:, 1, :3] + b[:, None] * cur[:, 2, :3],
                      centre + np.abs(radius)[:, None] * rng.normal(0, 0.3, (n, 3)))
    dv = target - pos
    t = np.linalg.norm(dv, axis=1)
    d = (dv / t[:, None]).astype(F)
    o = np.broadcast_to(pos, (n, 3)).astype(F)
    old = cur.copy()
    how = rng.integers(0, 4, n)                                           # 0 unchanged, 1 translated, 2 scaled, 3 deformed
    old[how == 1, 0, :3] += rng.normal(0, 0.3, ((how == 1).sum(), 3)).astype(F)
    old[how == 2, 0, 3] *= F(1.25)
    old[(how == 2) & tri, 1:, :3] *= F(1.25)
    old[how == 3, 1:, :3] += rng.normal(0, 0.1, ((how == 3).sum(), 2, 3)).astype(F)
    old[(how == 3) & ~tri, 0, 3] = -old[(how == 3) & ~tri, 0, 3]
    old[~tri, 1:] = 0
    if specials:
        for arr, k in ((cur, 8), (old, 8), (d, 4), (t := t.astype(F), 4)):
            flat = arr.reshape(-1)
            flat[rng.integers(0, flat.size, k)] = rng.choice(SPECIALS, k)
        cur[rng.integers(0, n, 2), 0, 3] = 0.0                            # r = 0: r' / r is ±inf or NaN
    return tri, o, d, np.asarray(t, F), cur, old


def motion_cases(W, H):
    cam = camera(W, H)
    return [
        ("same", cam, cam),
        ("equal_but_not_bitwise", cam, dataclasses.replace(cam, hor_fov_rad=cam.hor_fov_rad * 2)),
        ("translation", cam, camera(W, H, position=(0.3, -0.2, 0.5))),
        ("rotation", cam, camera(W, H, look_at=(0.2, 0.05, -1.0))),
        ("non_orthogonal_up", cam, dataclasses.replace(cam, up=R.Vec3(0.15, 1.3, -0.2))),
        ("prev_among_the_points", cam, camera(W, H, position=(0.0, 0.0, -6.0))),
        ("cam_behind", camera(W, H, position=(0.0, 0.0, -12.0)), cam),
    ]


MOTION_CASES = [c[0] for c in motion_cases(8, 6)]


# ============================================================================== the motion pass
@pytest.mark.parametrize("name", MOTION_CASES)
@pytest.mark.parametrize("specials", [False, True])
def test_host_build_of_the_motion_pass_equals_numpy(hd, name, specials):
    (case,) = [c for c in motion_cases(64, 48) if c[0] == name]
    _, cam, prev = case
    h = hits(cam, 4000, 7 + specials, specials)
    got = host_motion(hd, cam, prev, *h)
    want = M.motion(cam, prev, *h)
    assert T.same_bits(got[0], want[0]) and T.same_bits(got[1], want[1]), name


def test_the_hits_reach_every_rule(hd):
    """Changed and unchanged elements of both kinds, negative radii, finite and NaN motion, points behind a camera."""
    W, H = 64, 48
    cam = camera(W, H)
    tri, o, d, t, cur, old = hits(cam, 4000, 7)
    m, pd = M.motion(cam, camera(W, H, position=(0.3, -0.2, 0.5)), tri, o, d, t, cur, old)
    same = (cur.view(np.uint32) == old.view(np.uint32)).all((1, 2))
    assert (tri & same).any() and (tri & ~same).any() and (~tri & same).any() and (~tri & ~same).any()
    assert (cur[~tri, 0, 3] < 0).any() and np.isfinite(m).all(1).mean() > 0.9
    m2, _ = M.motion(cam, camera(W, H, position=(0.0, 0.0, -6.0)), tri, o, d, t, cur, old)   # inside the cloud of hits
    assert np.isnan(m2).all(1).any() and np.isfinite(m2).all(1).any()


def test_unchanged_geometry_and_the_same_camera_give_zero_motion(hd):
    W, H = 64, 48
    cam = camera(W, H)
    tri, o, d, t, cur, _ = hits(cam, 2000, 9)
    for prev in (cam, dataclasses.replace(cam, hor_fov_rad=cam.hor_fov_rad * 2)):
        m, pd = host_motion(hd, cam, prev, tri, o, d, t, cur, cur)
        assert (m.view(np.uint32) == 0).all()                             # +0 exactly
        P = [o[:, k] + t * d[:, k] for k in range(3)]
        D = [P[k] - o[:, k] for k in range(3)]
        assert T.same_bits(pd, np.sqrt(T.dot(D, D)).astype(F))


def test_pixel_dirs_equal_the_host_build_and_the_temporal_world_point(hd):
    for W, H in ((33, 17), (1, 1), (1, 40), (40, 1)):
        cam = dataclasses.replace(camera(W, H), up=R.Vec3(0.15, 1.3, -0.2))
        got = np.zeros((H, W, 3), F)
        assert hd.hd_pixel_dirs(cam.to_c(), got.ctypes.data) == 0
        d = M.pixel_dirs(cam)
        assert T.same_bits(got, d)
        y, x = np.mgrid[0:H, 0:W]
        z = np.full((H, W), 3.5, F)
        X = T.world_point(cam, x, y, z)
        pos = T.cam_values(cam)[0]
        assert T.same_bits(np.stack(X, -1), np.stack([pos[k] + z * d[..., k] for k in range(3)], -1))


# ============================================================================== temporal accumulation along the motion
def host_temporal_motion(hd, cam, hdr, var, aovs, hist, mplane, pdist, alpha_min=0.1, sigma_depth=0.02, normal_min=0.9):
    H, W = hdr.shape[:2]
    keep = []

    def arr(*xs):
        a = (C.c_void_p * len(xs))(*[None if x is None else np.ascontiguousarray(x).ctypes.data for x in xs])
        keep.append(xs)
        return a

    g = aovs
    ins = arr(hdr, var, g["depth"], g["normal"], g["hit_kind"], g["elem_idx"])
    hs = None
    if hist is not None:
        ha = hist["aovs"]
        hs = arr(hist["hdr"], hist["var"] if var is not None else None, hist["length"], ha["depth"], ha["normal"], ha["hit_kind"], ha["elem_idx"])
    mv = arr(mplane, pdist)
    opt = np.array([alpha_min, sigma_depth, normal_min], F)
    out, vout, lout = np.zeros((H, W, 3), F), (None if var is None else np.zeros((H, W, 3), F)), np.zeros((H, W), F)
    prev = hist["cam"].to_c() if hist is not None else None
    assert hd.hd_temporal_motion(W, H, cam.to_c(), prev, ins, hs, mv, opt.ctypes.data, out.ctypes.data,
                                 None if vout is None else vout.ctypes.data, lout.ctypes.data) == 0
    return out, vout, lout


def motion_planes(cam, hist_cam, aovs, seed, kind):
    """(motion, prev_dist) on synthetic frames.  kind: "nan" (every pixel falls back to the cameras), "zero" (each pixel to itself,
    prev_dist = the camera path's r), "random" (small motions, some NaN, prev_dist near the camera path's r), "specials"."""
    H, W = aovs["depth"].shape
    y, x = np.mgrid[0:H, 0:W]
    X = T.world_point(cam, x, y, aovs["depth"])
    pp = T.cam_values(hist_cam)[0]
    with np.errstate(all="ignore"):
        r = np.sqrt(T.dot(*([[X[k] - pp[k] for k in range(3)]] * 2))).astype(F)
    rng = np.random.default_rng(seed)
    if kind == "nan":
        return np.full((H, W, 2), np.nan, F), r
    if kind == "zero":
        return np.zeros((H, W, 2), F), r
    m = rng.normal(0, 1.5, (H, W, 2)).astype(F)
    m[rng.random((H, W)) < 0.15] = np.nan
    pd = (r * (1 + rng.normal(0, 0.01, r.shape))).astype(F)
    if kind == "specials":
        for arr, k in ((m, 8), (pd, 6)):
            flat = arr.reshape(-1)
            flat[rng.integers(0, flat.size, k)] = rng.choice(SPECIALS, k)
        m[0, 0] = (np.inf, 0.0)
        m[-1, -1] = (F(W), F(H))                                          # out of the image
    return m, pd


@pytest.mark.parametrize("name", CASE_NAMES)
@pytest.mark.parametrize("kind", ["nan", "zero", "random", "specials"])
def test_host_build_of_the_temporal_motion_step_equals_numpy(hd, name, kind):
    (case,) = [c for c in cases(29, 21) if c[0] == name]
    _, cam, prev, opts = case
    for specials in (False, True):
        hdr, var, aovs = frame(cam, 3, specials)
        hist = history(prev, 4, specials) if prev is not None else None
        mp, pd = motion_planes(cam, prev or cam, aovs, 5, kind)
        for v in (var, None):
            want = M.accumulate_motion(cam, hdr, v, aovs, hist, mp, pd, **opts)
            got = host_temporal_motion(hd, cam, hdr, v, aovs, hist, mp, pd, **{**dict(alpha_min=0.1, sigma_depth=0.02, normal_min=0.9), **opts})
            assert same_all(got, want), (name, kind, specials, v is None)


@pytest.mark.parametrize("name", CASE_NAMES)
def test_nan_motion_falls_back_to_the_camera_reprojection(name):
    (case,) = [c for c in cases(29, 21) if c[0] == name]
    _, cam, prev, opts = case
    hdr, var, aovs = frame(cam, 3, True)
    hist = history(prev, 4, True) if prev is not None else None
    mp, pd = motion_planes(cam, prev or cam, aovs, 5, "nan")
    assert same_all(M.accumulate_motion(cam, hdr, var, aovs, hist, mp, pd, **opts), T.accumulate(cam, hdr, var, aovs, hist, **opts))


def test_zero_motion_maps_each_pixel_to_itself():
    """Zero motion with prev_dist = the camera path's r is the bitwise-equal camera's shortcut, whatever the history's camera."""
    W, H = 29, 21
    cam = camera(W, H)
    hdr, var, aovs = frame(cam, 3)
    hist = history(cam, 4)
    want = T.accumulate(cam, hdr, var, aovs, hist)
    for other in (cam, dataclasses.replace(cam, hor_fov_rad=cam.hor_fov_rad * 2)):
        mp, pd = motion_planes(cam, cam, aovs, 5, "zero")
        assert same_all(M.accumulate_motion(cam, hdr, var, aovs, {**hist, "cam": other}, mp, pd), want)
    assert (want[2] > 1).any()


# ============================================================================== module and entry points, no device needed
def test_module_is_built_for_sm_100a_with_its_two_kernels():
    raw = C.CDLL(LIB)
    assert hasattr(raw, "rbrt_snapshot_launch") and hasattr(raw, "rbrt_motion_launch")
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump is not here")
    sass = subprocess.run([cuobjdump, "-sass", LIB], capture_output=True, text=True, check=True).stdout
    fns = sorted(ln.split(":")[1].strip() for ln in sass.splitlines() if "Function :" in ln)
    assert len(fns) == 3 and sum("k_motion" in f for f in fns) == 2 and sum("k_snapshot" in f for f in fns) == 1
    assert "sm_100a" in subprocess.run([cuobjdump, "-lelf", LIB], capture_output=True, text=True, check=True).stdout


def test_motion_out_layout_matches_the_header(tmp_path):
    src = tmp_path / "m.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "%s"\nint main(void){printf("%%zu %%zu %%zu\\n", sizeof(rbrt_motion_out), '
                   'offsetof(rbrt_motion_out, motion), offsetof(rbrt_motion_out, prev_dist));return 0;}\n'
                   % os.path.join(ROOT, "include", "rbrt_gpu.h"))
    exe = tmp_path / "m"
    subprocess.run(["gcc", "-std=c99", "-o", str(exe), str(src)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert got == [C.sizeof(_abi.MotionOutC), _abi.MotionOutC.motion.offset, _abi.MotionOutC.prev_dist.offset]


def test_refusals_before_any_device_work():
    lib = _abi.lib()
    cam = camera(8, 6)
    m = np.zeros((6, 8, 2), F)
    pd = np.zeros((6, 8), F)
    out = _abi.MotionOutC(m.ctypes.data, pd.ctypes.data)
    assert lib.rbrt_gpu_scene_snapshot(None, None) == _abi.E_INVALID
    assert lib.rbrt_gpu_render_motion(None, cam.to_c(), cam.to_c(), out, None) == _abi.E_INVALID
    assert lib.rbrt_gpu_render_motion_device(None, cam.to_c(), cam.to_c(), out, None, None) == _abi.E_INVALID
    hdr = np.zeros((6, 8, 3), F)
    g = _abi.AovOutC(depth=pd.ctypes.data, normal=hdr.ctypes.data, hit_kind=pd.ctypes.data, elem_idx=pd.ctypes.data)
    o3 = np.zeros((6, 8, 3), F)
    for bad in (None, _abi.MotionOutC(m.ctypes.data, None), _abi.MotionOutC(None, pd.ctypes.data)):
        rc = lib.rbrt_gpu_temporal_accumulate_motion(8, 6, cam.to_c(), hdr.ctypes.data, None, g, None, bad, None, o3.ctypes.data, None,
                                                     None, None)
        assert rc == _abi.E_INVALID and b"motion" in lib.rbrt_last_error()
    assert (m == 0).all() and (pd == 0).all()
