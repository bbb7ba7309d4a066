"""Temporal accumulation without a GPU: the module is built for sm_100a with its one kernel, the structs match the header, the entry points
refuse bad calls without touching a device, and tests/temporal_ref.py equals a plain loop restatement and the host build of
csrc/temporal.cuh bit for bit on planes with every special value and cameras of every kind of motion."""
import ctypes as C
import dataclasses
import os
import shutil
import subprocess

import numpy as np
import pytest

import rbrt_b200 as R
from rbrt_b200 import _abi

from . import temporal_ref as T

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TMP = os.path.join(ROOT, "rbrt_b200", "librbrt_gpu_temporal.so")
HD = os.path.join(ROOT, "tests", "host_device")
CSRC = os.path.join(ROOT, "rbrt_b200", "csrc")
F = np.float32
SPECIALS = np.array([0.0, -0.0, 1e-45, -1e-45, 1e-40, np.inf, -np.inf, np.nan, 3e38, -2.5], F)


@pytest.fixture(scope="module", autouse=True)
def temporal_module():
    if not os.path.exists(TMP):
        subprocess.run(["make", "-C", CSRC], check=True)
    return TMP


@pytest.fixture(scope="module")
def hd():
    out = os.path.join(HD, "build", "libhost_temporal.so")
    os.makedirs(os.path.dirname(out), exist_ok=True)
    srcs = [os.path.join(HD, f) for f in ("temporal_harness.cpp", "cuda_runtime.h")] + \
           [os.path.join(CSRC, f) for f in ("common.cuh", "denoise.cuh", "temporal.cuh")]
    if not os.path.exists(out) or any(os.path.getmtime(s) > os.path.getmtime(out) for s in srcs):
        # the flags of tests/test_device_source_on_host.py: the stand-in cuda_runtime.h first, no contraction, no FMA
        subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-mno-fma", "-Wno-unknown-pragmas", "-fPIC", "-shared",
                        "-I", HD, "-I", CSRC, "-o", out, srcs[0]], check=True)
    lib = C.CDLL(out)
    lib.hd_temporal.argtypes = [C.c_uint32, C.c_uint32, C.POINTER(_abi.CameraC), C.POINTER(_abi.CameraC), C.c_void_p, C.c_void_p,
                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    return lib


# ============================================================================== synthetic frames
def camera(W, H, position=(0.0, 0.0, 0.0), look_at=(0.0, 0.0, -1.0), up=(0.0, 1.0, 0.0), focal=35.0):
    return R.Camera.new(R.Vec3(*position), R.Vec3(*look_at), R.Vec3(*up), H, W, focal)


def _ray_dirs(cam):
    """Pixel-centre ray directions of cam in float64, [H,W,3]."""
    pos, right, up, center, mmh, mmv, W, H = (np.asarray(v, np.float64) if isinstance(v, np.ndarray) else v for v in T.cam_values(cam))
    y, x = np.mgrid[0:H, 0:W].astype(np.float64)
    t = center + (0.001 * (x - W // 2) * float(mmh))[..., None] * right - (0.001 * (y - H // 2) * float(mmv))[..., None] * up
    d = t - pos
    return d / np.linalg.norm(d, axis=-1, keepdims=True)


def frame(cam, seed, specials=False):
    """hdr, var and guides of a world of two planes seen from cam: a tilted wall (elem 0) and, where it is nearer, a floor (elem 1);
    rays that hit neither are misses.  With specials: ±0, subnormals, ±inf, NaN in colour, variance and depth, negative variance and
    mismatched ids."""
    rng = np.random.default_rng(seed)
    W, H = cam.img_width_pix, cam.img_height_pix
    pos = np.array([cam.position.x, cam.position.y, cam.position.z])
    d = _ray_dirs(cam)
    planes = [(np.array([0.1, 0.2, 1.0]) / np.linalg.norm([0.1, 0.2, 1.0]), -6.0), (np.array([0.0, 1.0, 0.0]), -1.5)]
    z = np.full((H, W), np.inf)
    n = np.zeros((H, W, 3))
    elem = np.zeros((H, W), np.uint32)
    for i, (pn, off) in enumerate(planes):
        with np.errstate(all="ignore"):
            t = (off - pos @ pn) / (d @ pn)
        hit = (t > 0) & (t < z)
        z[hit], n[hit], elem[hit] = t[hit], pn, i
    kind = np.where(np.isfinite(z), 1, -1).astype(np.int32)
    n = (n + rng.normal(0, 0.01, n.shape) * np.isfinite(z)[..., None]).astype(F)
    z = (z * (1 + rng.normal(0, 0.002, z.shape))).astype(F)
    hdr = rng.gamma(2.0, 0.3, (H, W, 3)).astype(F)
    var = rng.gamma(0.8, 0.02, (H, W, 3)).astype(F)
    var[rng.random((H, W)) < 0.1] = 0.0
    if specials:
        for arr, k in ((hdr, 6), (var, 6), (z, 4)):
            flat = arr.reshape(-1)
            flat[rng.integers(0, flat.size, k)] = rng.choice(SPECIALS, k)
        var.reshape(-1)[rng.integers(0, var.size, 2)] = -1e-3
        elem.reshape(-1)[rng.integers(0, elem.size, max(1, elem.size // 20))] = 7
    return hdr, var, {"depth": z, "normal": n, "hit_kind": kind, "elem_idx": elem}


def history(prev, seed, specials=False):
    hdr, var, aovs = frame(prev, seed, specials)
    rng = np.random.default_rng(seed + 1000)
    length = rng.choice(np.array([0, 1, 2, 3, 7.5, 40], F), (prev.img_height_pix, prev.img_width_pix)).astype(F)
    return {"cam": prev, "hdr": hdr, "var": var, "length": length, "aovs": aovs}


def cases(W, H):
    """(name, cam, prev or None, opts) of every kind of camera motion the definition distinguishes."""
    cam = camera(W, H)
    odd = dataclasses.replace(cam, up=R.Vec3(0.15, 1.3, -0.2))                 # a raw up, neither unit nor orthogonal to right
    return [
        ("first", cam, None, {}),
        ("identity", cam, cam, {}),
        ("identity_alpha0", cam, cam, {"alpha_min": 0.0}),
        ("identity_alpha1", cam, cam, {"alpha_min": 1.0}),
        ("equal_but_not_bitwise", cam, dataclasses.replace(cam, hor_fov_rad=cam.hor_fov_rad * 2), {}),   # pixel centres and borders
        ("translation", cam, camera(W, H, position=(0.04, -0.03, 0.1)), {}),
        ("rotation", cam, camera(W, H, look_at=(0.06, 0.02, -1.0)), {}),
        ("rotation_up", cam, camera(W, H, up=(0.05, 1.0, 0.0)), {"alpha_min": 0.0}),
        ("non_orthogonal_up", odd, dataclasses.replace(odd, position=R.Vec3(0.02, 0.01, 0.0)), {}),
        ("behind", cam, camera(W, H, position=(0.0, 0.0, -12.0)), {}),
        ("sigmas", cam, camera(W, H, position=(0.03, 0.0, 0.0)), {"sigma_depth": 0.2, "normal_min": 0.0, "alpha_min": 0.5}),
        ("strict", cam, camera(W, H, position=(0.03, 0.0, 0.0)), {"sigma_depth": 0.0, "normal_min": 1.0}),
    ]


CASE_NAMES = [c[0] for c in cases(8, 6)]


def host_temporal(hd, cam, hdr, var, aovs, hist, alpha_min=0.1, sigma_depth=0.02, normal_min=0.9):
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
    opt = np.array([alpha_min, sigma_depth, normal_min], F)
    out, vout, lout = np.zeros((H, W, 3), F), (None if var is None else np.zeros((H, W, 3), F)), np.zeros((H, W), F)
    prev = hist["cam"].to_c() if hist is not None else None
    assert hd.hd_temporal(W, H, cam.to_c(), prev, ins, hs, opt.ctypes.data, out.ctypes.data, None if vout is None else vout.ctypes.data,
                          lout.ctypes.data) == 0
    return out, vout, lout


def same_all(a, b):
    return all((x is None and y is None) or T.same_bits(x, y) for x, y in zip(a, b))


# ============================================================================== the three restatements agree
@pytest.mark.parametrize("name", CASE_NAMES)
@pytest.mark.parametrize("with_var", [True, False])
def test_planes_equal_the_pixel_loop(name, with_var):
    (case,) = [c for c in cases(13, 9) if c[0] == name]
    _, cam, prev, opts = case
    hdr, var, aovs = frame(cam, 1, specials=True)
    hist = history(prev, 2, specials=True) if prev is not None else None
    v = var if with_var else None
    assert same_all(T.accumulate(cam, hdr, v, aovs, hist, **opts), T.accumulate_scalar(cam, hdr, v, aovs, hist, **opts))


@pytest.mark.parametrize("name", CASE_NAMES)
@pytest.mark.parametrize("shape", [(48, 32), (1, 1), (1, 40), (40, 1), (7, 5)])
def test_host_build_of_the_header_equals_numpy(hd, name, shape):
    (case,) = [c for c in cases(*shape) if c[0] == name]
    _, cam, prev, opts = case
    for specials in (False, True):
        hdr, var, aovs = frame(cam, 3, specials)
        hist = history(prev, 4, specials) if prev is not None else None
        for v in (var, None):
            want = T.accumulate(cam, hdr, v, aovs, hist, **opts)
            assert same_all(host_temporal(hd, cam, hdr, v, aovs, hist, **{**dict(alpha_min=0.1, sigma_depth=0.02, normal_min=0.9), **opts}),
                            want), (name, shape, specials, v is None)


def test_the_cases_reach_every_rule():
    """The synthetic frames exercise what the definition distinguishes: histories kept and dropped, exact pixel centres and the image
    border reached through the general projection, points behind the previous camera, and partial bilinear footprints."""
    W, H = 48, 32
    cs = {c[0]: c for c in cases(W, H)}
    _, cam, prev, _ = cs["equal_but_not_bitwise"]
    hdr, var, aovs = frame(cam, 3)
    X = T.world_point(cam, *np.mgrid[0:H, 0:W][::-1], aovs["depth"])
    pp = T.cam_values(prev)[0]
    with np.errstate(all="ignore"):
        px, py, _ = T.project(prev, [X[k] - pp[k] for k in range(3)])
    fin = np.isfinite(px) & np.isfinite(py)
    assert (px[fin] == np.floor(px[fin])).mean() > 0.5 and (py[fin] == np.floor(py[fin])).mean() > 0.5
    assert (px[fin] == F(W - 1)).any() and (px[fin] == F(0)).any()
    for name, kept in (("identity", True), ("translation", True), ("rotation", True), ("non_orthogonal_up", True), ("behind", False)):
        _, cam, prev, opts = cs[name]
        hdr, var, aovs = frame(cam, 3)
        hist = history(prev, 4)
        _, _, l = T.accumulate(cam, hdr, var, aovs, hist, **opts)
        assert ((l > 1).any()) == kept, name
        assert (l == 1).any() or name == "identity"


# ============================================================================== module, layout, refusals
def test_module_is_built_for_sm_100a_with_only_its_own_kernel():
    lib = C.CDLL(TMP)
    assert hasattr(lib, "rbrt_temporal_launch")
    raw = C.CDLL(_abi.LIB_PATH)
    assert hasattr(raw, "rbrt_gpu_temporal_accumulate") and hasattr(raw, "rbrt_gpu_temporal_accumulate_device")
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump is not here")
    sass = subprocess.run([cuobjdump, "-sass", TMP], capture_output=True, text=True, check=True).stdout
    fns = [ln.split(":")[1].strip() for ln in sass.splitlines() if "Function :" in ln]
    assert len(fns) == 1 and "k_temporal" in fns[0]
    assert "sm_100a" in subprocess.run([cuobjdump, "-lelf", TMP], capture_output=True, text=True, check=True).stdout


def test_struct_layouts_match_header(tmp_path):
    fields = {"rbrt_temporal_opts": _abi.TemporalOptsC, "rbrt_temporal_history": _abi.TemporalHistoryC, "rbrt_aov_out": _abi.AovOutC}
    lines = ["#include <stdio.h>", "#include <stddef.h>", f'#include "{os.path.join(ROOT, "include", "rbrt_gpu.h")}"', "int main(void){"]
    for cname, ct in fields.items():
        lines.append(f'printf("{cname} %zu\\n", sizeof({cname}));')
        for fname, _ in ct._fields_:
            lines.append(f'printf("{cname}.{fname} %zu\\n", offsetof({cname}, {fname}));')
    lines.append("return 0;}")
    (tmp_path / "layout.c").write_text("\n".join(lines))
    subprocess.run(["gcc", "-std=c99", "-o", str(tmp_path / "layout"), str(tmp_path / "layout.c")], check=True)
    got = dict(l.split() for l in subprocess.run([str(tmp_path / "layout")], check=True, capture_output=True, text=True).stdout.splitlines())
    for cname, ct in fields.items():
        assert int(got[cname]) == C.sizeof(ct), cname
        for fname, _ in ct._fields_:
            assert int(got[f"{cname}.{fname}"]) == getattr(ct, fname).offset, (cname, fname)


def _call(W=8, H=6, cam=None, hdr=True, var=True, guides=True, hist=None, opts=None, outs=(True, True, True), alias=None):
    """One host call of rbrt_gpu_temporal_accumulate with planes of W x H (cam: of that size unless given)."""
    cam = cam or camera(W, H)
    keep = []

    def buf(k):
        a = np.zeros(max(W * H * k, 1), F)
        keep.append(a)
        return a.ctypes.data

    g = _abi.AovOutC(depth=buf(1), normal=buf(3), hit_kind=buf(1), elem_idx=buf(1)) if guides else None
    o = [buf(3) if outs[0] else None, buf(3) if outs[1] else None, buf(1) if outs[2] else None]
    ins = [buf(3) if hdr else None, buf(3) if var else None]
    if alias:
        alias(o, ins, g, hist)
    return _abi.lib().rbrt_gpu_temporal_accumulate(W, H, cam.to_c(), ins[0], ins[1], g, hist, opts, *o, None), keep


def test_bad_calls_are_refused_before_any_device_work():
    """Every refusal is decided from the arguments, so it needs no GPU: RBRT_E_INVALID and a message."""
    cam = camera(8, 6)
    h = _abi.TemporalHistoryC(cam=cam.to_c())
    bad = [
        dict(hdr=False), dict(guides=False), dict(outs=(False, False, False)), dict(var=False),       # var_out without var
        dict(W=0), dict(H=0), dict(cam=camera(9, 6)), dict(hist=h),                                   # a history without planes
        dict(opts=_abi.TemporalOptsC(float("nan"), 0.02, 0.9)), dict(opts=_abi.TemporalOptsC(1.5, 0.02, 0.9)),
        dict(opts=_abi.TemporalOptsC(0.1, -1.0, 0.9)), dict(opts=_abi.TemporalOptsC(0.1, 0.02, float("inf"))),
        dict(alias=lambda o, i, g, hh: o.__setitem__(0, i[0])),                                      # in place
        dict(alias=lambda o, i, g, hh: o.__setitem__(2, g.depth)),                                    # over a guide
        dict(alias=lambda o, i, g, hh: o.__setitem__(1, o[0] + 4)),                                   # two outputs overlap
    ]
    for kw in bad:
        rc, _ = _call(**kw)
        assert rc == _abi.E_INVALID, kw
        assert _abi.lib().rbrt_last_error()
    W, H = 8, 6
    with pytest.raises(R.RbrtGpuError):
        R.temporal_accumulate(camera(W, H), np.zeros((H, W, 3), F), {"depth": np.zeros((H, W), F), "normal": np.zeros((H, W, 3), F),
                                                                     "hit_kind": np.zeros((H, W), np.int32), "elem_idx": np.zeros((H, W), np.uint32)},
                              alpha_min=2.0)
    with pytest.raises(ValueError):
        R.temporal_accumulate(camera(W, H), np.zeros((H, W, 3), F), {"depth": np.zeros((H, W), F)})
