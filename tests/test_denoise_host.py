"""The guided denoiser without a GPU: the module is built for sm_100a and holds only its own kernels, rbrt_denoise_opts has one layout in
the header, ctypes and Rust, the entry points refuse bad calls without touching a device, tests/denoise_ref.py equals a plain loop
restatement and the host build of csrc/denoise.cuh bit for bit, and the CLI lists and checks --denoise."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import rbrt_b200 as R
from rbrt_b200 import _abi

from . import denoise_ref as D

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DNS = os.path.join(ROOT, "rbrt_b200", "librbrt_gpu_denoise.so")
HEADER = os.path.join(ROOT, "include", "rbrt_gpu.h")
HD = os.path.join(ROOT, "tests", "host_device")
CSRC = os.path.join(ROOT, "rbrt_b200", "csrc")
FIELDS = ["levels", "sigma_depth", "sigma_luminance"]
F = np.float32


@pytest.fixture(scope="module", autouse=True)
def denoise_module():
    if not os.path.exists(DNS) or not os.path.exists(os.path.join(ROOT, "rbrt_b200", "rbrt")):
        subprocess.run(["make", "-C", CSRC], check=True)
    return DNS


@pytest.fixture(scope="module")
def hd():
    out = os.path.join(HD, "build", "libhost_denoise.so")
    os.makedirs(os.path.dirname(out), exist_ok=True)
    srcs = [os.path.join(HD, f) for f in ("denoise_harness.cpp", "cuda_runtime.h")] + \
           [os.path.join(CSRC, f) for f in ("common.cuh", "shade.cuh", "denoise.cuh")]
    if not os.path.exists(out) or any(os.path.getmtime(s) > os.path.getmtime(out) for s in srcs):
        # the flags of tests/test_device_source_on_host.py: the stand-in cuda_runtime.h first, no contraction, no FMA
        subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-mno-fma", "-Wno-unknown-pragmas", "-fPIC", "-shared",
                        "-I", HD, "-I", CSRC, "-o", out, srcs[0]], check=True)
    lib = C.CDLL(out)
    lib.hd_denoise.argtypes = [C.c_uint32, C.c_uint32] + [C.c_void_p] * 4 + [C.c_uint32, C.c_float, C.c_float, C.c_void_p, C.c_void_p]
    return lib


def host_denoise(hd, c, a, n, z, levels=0, sigma_depth=0.0, sigma_luminance=0.0):
    L, sz, sl = D.resolve(levels, sigma_depth, sigma_luminance)
    c, a, n, z = (np.ascontiguousarray(v, F) for v in (c, a, n, z))
    H, W = z.shape
    out, rgb = np.zeros((H, W, 3), F), np.zeros((H, W, 3), np.uint8)
    assert hd.hd_denoise(W, H, c.ctypes.data, z.ctypes.data, n.ctypes.data, a.ctypes.data, L, sz, sl, out.ctypes.data, rgb.ctypes.data) == 0
    return out, rgb


def scene_like(H, W, seed):
    """Planes with the structure of real AOVs: two surfaces with smooth normals and depths, a miss region, noisy colour."""
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:H, 0:W].astype(F)
    near = (x - W / 2) ** 2 + (y - H / 2) ** 2 < (min(H, W) / 3) ** 2
    z = np.where(near, F(3.0) + F(0.01) * x, F(8.0) + F(0.05) * y).astype(F)
    n = np.stack([np.where(near, F(0.1), F(0.0)), np.where(near, F(0.2), F(1.0)), np.where(near, F(0.97), F(0.0))], -1).astype(F)
    n += rng.normal(0, 0.01, n.shape).astype(F)
    a = np.where(near[..., None], F([0.8, 0.3, 0.2]), F([0.5, 0.5, 0.5])).astype(F)
    c = (a * rng.gamma(2.0, 0.4, (H, W, 1))).astype(F)
    miss = (x < 2) & (y < 2)
    z[miss], n[miss], a[miss] = np.inf, 0.0, 0.0
    return c, a, n, z


def adversarial(H, W, seed):
    """scene_like planes with the special values of every rule: NaN / inf colour, zero and NaN albedo, misses, NaN depth, +-0,
    subnormals and huge values."""
    rng = np.random.default_rng(seed)
    c, a, n, z = scene_like(H, W, seed)
    specials = np.array([0.0, -0.0, 1e-45, -1e-45, 1e-40, np.inf, -np.inf, np.nan, 3e38, -2.5], F)
    for arr, k in ((c, 6), (a, 4), (n, 3), (z, 3)):
        flat = arr.reshape(-1)
        flat[rng.integers(0, flat.size, k)] = rng.choice(specials, k)
    c.reshape(-1)[rng.integers(0, c.size, 2)] = np.nan
    c.reshape(-1)[rng.integers(0, c.size, 2)] = np.inf
    a.reshape(-1)[rng.integers(0, a.size, 3)] = 0.0
    return c, a, n, z


# ============================================================================== module, layout, refusals
def test_module_is_built_for_sm_100a_with_only_its_own_kernels():
    lib = C.CDLL(DNS)
    assert hasattr(lib, "rbrt_denoise_launch")
    raw = C.CDLL(_abi.LIB_PATH)
    assert hasattr(raw, "rbrt_gpu_denoise") and hasattr(raw, "rbrt_gpu_denoise_device")
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump is not here")
    sass = subprocess.run([cuobjdump, "-sass", DNS], capture_output=True, text=True, check=True).stdout
    names = re.findall(r"Function : (\S+)", sass)
    assert len(names) == 3 and all("k_denoise" in n for n in names), names
    assert "arch = sm_100a" in sass
    main = subprocess.run([cuobjdump, "-sass", _abi.LIB_PATH], capture_output=True, text=True, check=True).stdout
    kernels = re.findall(r"Function : (\S+)", main)
    assert len(kernels) == 51 and not any("denoise" in k for k in kernels)


def test_opts_layout_matches_the_header_ctypes_and_rust(tmp_path):
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{HEADER}"', "int main(void){",
             'printf("size %zu\\n", sizeof(rbrt_denoise_opts));']
    lines += [f'printf("{f} %zu\\n", offsetof(rbrt_denoise_opts, {f}));' for f in FIELDS]
    lines.append("return 0;}")
    src = tmp_path / "denoise_layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "denoise_layout"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-o", str(exe), str(src)], check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    assert [f for f, _ in _abi.DenoiseOptsC._fields_] == FIELDS
    assert int(got["size"]) == C.sizeof(_abi.DenoiseOptsC) == 12
    for f in FIELDS:
        assert int(got[f]) == getattr(_abi.DenoiseOptsC, f).offset, f
    rs = open(os.path.join(ROOT, "integration", "rust", "rbrt_gpu_sys", "src", "lib.rs")).read()
    m = re.search(r"pub struct RbrtDenoiseOpts\s*\{(.*?)\}", rs, re.S)
    assert m and re.findall(r"pub (\w+)\s*:", m.group(1)) == FIELDS
    assert re.findall(r"pub \w+\s*:\s*(\w+)", m.group(1)) == ["u32", "f32", "f32"]
    for name, arity in (("rbrt_gpu_denoise", 8), ("rbrt_gpu_denoise_device", 9)):
        f = re.search(r"pub fn %s\s*\((.*?)\)\s*->" % name, rs, re.S)
        assert f and len([a for a in f.group(1).split(",") if a.strip()]) == arity, name


def test_refusals_without_a_device():
    lib = _abi.lib()
    W, H = 8, 6
    n = W * H
    hdr, alb, nrm, dep = np.ones(3 * n, F), np.ones(3 * n, F), np.ones(3 * n, F), np.ones(n, F)
    out, rgb = np.full(3 * n, 7.0, F), np.full(3 * n, 7, np.uint8)
    g = _abi.AovOutC(depth=dep.ctypes.data, normal=nrm.ctypes.data, albedo=alb.ctypes.data)
    O = _abi.DenoiseOptsC
    host = lambda *a: lib.rbrt_gpu_denoise(*a, None)
    dev = lambda *a: lib.rbrt_gpu_denoise_device(*a, None, None)
    cases = [
        ((W, H, None, g, None, out.ctypes.data, rgb.ctypes.data), b"null"),
        ((W, H, hdr.ctypes.data, None, None, out.ctypes.data, rgb.ctypes.data), b"null"),
        ((W, H, hdr.ctypes.data, _abi.AovOutC(normal=nrm.ctypes.data, albedo=alb.ctypes.data), None, out.ctypes.data, None), b"guide"),
        ((W, H, hdr.ctypes.data, _abi.AovOutC(depth=dep.ctypes.data, albedo=alb.ctypes.data), None, out.ctypes.data, None), b"guide"),
        ((W, H, hdr.ctypes.data, _abi.AovOutC(depth=dep.ctypes.data, normal=nrm.ctypes.data), None, out.ctypes.data, None), b"guide"),
        ((W, H, hdr.ctypes.data, g, None, None, None), b"no output"),
        ((0, H, hdr.ctypes.data, g, None, out.ctypes.data, None), b"empty"),
        ((W, 0, hdr.ctypes.data, g, None, out.ctypes.data, None), b"empty"),
        ((65536, 32768, hdr.ctypes.data, g, None, out.ctypes.data, None), b"too large"),
        ((W, H, hdr.ctypes.data, g, O(levels=9), out.ctypes.data, None), b"levels"),
        ((W, H, hdr.ctypes.data, g, O(sigma_depth=-1.0), out.ctypes.data, None), b"sigma"),
        ((W, H, hdr.ctypes.data, g, O(sigma_depth=float("nan")), out.ctypes.data, None), b"sigma"),
        ((W, H, hdr.ctypes.data, g, O(sigma_luminance=float("inf")), out.ctypes.data, None), b"sigma"),
        ((W, H, hdr.ctypes.data, g, O(sigma_luminance=-0.5), out.ctypes.data, None), b"sigma"),
        ((W, H, hdr.ctypes.data, g, None, hdr.ctypes.data, None), b"overlaps an input"),
        ((W, H, hdr.ctypes.data, g, None, None, alb.ctypes.data + 20), b"overlaps an input"),
        ((W, H, hdr.ctypes.data, g, None, out.ctypes.data + 4 * (3 * n - 1), dep.ctypes.data), b"overlaps an input"),
        ((W, H, hdr.ctypes.data, g, None, out.ctypes.data, out.ctypes.data + 8), b"overlap"),
    ]
    for f in (host, dev):
        for args, msg in cases:
            assert f(*args) == _abi.E_INVALID, (args, msg)
            assert msg in lib.rbrt_last_error(), (msg, lib.rbrt_last_error())
    assert (out == 7.0).all() and (rgb == 7).all()


def test_python_argument_checks():
    c, a, n, z = scene_like(6, 8, 0)
    aovs = {"depth": z, "normal": n, "albedo": a}
    bad = [(c[:, :, :2], aovs), (c, dict(aovs, depth=z.T.copy())), (c, {"depth": z, "normal": n}), (c, dict(aovs, albedo=a.astype(np.float64))),
           (c.astype(np.float64), aovs), (c[:, ::2], aovs)]
    for hdr, g in bad:
        with pytest.raises(ValueError):
            R.denoise(hdr, g)
    import torch
    with pytest.raises(ValueError):
        R.denoise_device(torch.from_numpy(c), {k: torch.from_numpy(v) for k, v in aovs.items()})


def test_denoise_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present; the refusal path is exercised on the CPU-only build box")
    c, a, n, z = scene_like(6, 8, 0)
    with pytest.raises(_abi.RbrtGpuError) as e:
        R.denoise(c, {"depth": z, "normal": n, "albedo": a})
    assert e.value.code in (_abi.E_NODEVICE, _abi.E_CUDA)


# ============================================================================== the definition: numpy, a plain loop, the host build
@pytest.mark.parametrize("shape", [(6, 8), (1, 5)])
def test_numpy_reference_equals_the_plain_loop(shape):
    H, W = shape
    for seed, opts in [(1, {}), (2, {"levels": 1}), (3, {"levels": 3, "sigma_depth": 0.5, "sigma_luminance": 3.0}), (4, {"levels": 8})]:
        planes = adversarial(H, W, seed)
        assert not np.isfinite(planes[0]).all() and (planes[1] == 0).any() and not np.isfinite(planes[3]).all()
        got, rgb = D.denoise(*planes, **opts)
        want, want_rgb = D.denoise_scalar(*planes, **opts)
        assert D.same_bits(got, want), (shape, seed, opts)
        assert np.array_equal(rgb, want_rgb)
    c, a, n, z = scene_like(H, W, 5)                                    # no special values: the filter does mix pixels
    got, _ = D.denoise(c, a, n, z, levels=2)
    assert D.same_bits(got, D.denoise_scalar(c, a, n, z, levels=2)[0]) and not D.same_bits(got, c)


def test_rules_on_hand_made_planes():
    c, a, n, z = scene_like(6, 8, 7)
    c[0, 3] = [np.nan, 1.0, 1.0]                                          # a non-finite colour: passed through, never a tap
    c[5, 7] = [np.inf, 0.0, 0.0]
    a[2, 2] = [0.0, 0.0, 0.0]                                             # zero albedo: divided by 2^-10, still valid
    out, rgb = D.denoise(c, a, n, z, levels=2)
    for y, x in [(0, 3), (5, 7), (0, 0), (1, 1)]:                         # bad colour, and the misses of scene_like
        assert D.same_bits(out[y, x], c[y, x]), (y, x)
    assert np.isfinite(out[np.isfinite(z) & np.isfinite(c).all(-1)]).all()
    assert np.array_equal(rgb, D.tonemap(out)) and rgb[5, 7, 0] == 255 and rgb[0, 3, 0] == 0
    # a miss (depth inf, normal 0) changes no other pixel: making one more pixel a miss alters only pixels that tapped it
    z2, n2 = z.copy(), n.copy()
    z2[3, 6], n2[3, 6] = np.inf, 0.0
    out2, _ = D.denoise(c, a, n2, z2, levels=1)
    ref1, _ = D.denoise(c, a, n, z, levels=1)
    far = np.ones((6, 8), bool)
    far[1:6, 4:8] = False
    assert D.same_bits(out2[far], ref1[far])


@pytest.mark.parametrize("levels", range(1, 9))
def test_host_build_equals_the_numpy_reference(hd, levels):
    for shape, seed in [((17, 33), levels), ((5, 7), 100 + levels), ((1, 9), 200 + levels), ((9, 1), 300 + levels)]:
        for opts in ({}, {"sigma_depth": 0.25, "sigma_luminance": 1.5}):
            planes = adversarial(*shape, seed)
            got, got_rgb = host_denoise(hd, *planes, levels=levels, **opts)
            want, want_rgb = D.denoise(*planes, levels=levels, **opts)
            assert D.same_bits(got, want), (shape, levels, opts, np.argwhere(~((got.view(np.uint32) == want.view(np.uint32)) | (np.isnan(got) & np.isnan(want)))))
            assert np.array_equal(got_rgb, want_rgb), (shape, levels, opts)
    c, a, n, z = scene_like(24, 40, levels)
    got, _ = host_denoise(hd, c, a, n, z, levels=levels)
    want, _ = D.denoise(c, a, n, z, levels=levels)
    assert D.same_bits(got, want) and not D.same_bits(got, c)


# ============================================================================== CLI
def test_cli_lists_and_checks_denoise():
    cli = os.path.join(ROOT, "rbrt_b200", "rbrt")
    out = subprocess.run([cli, "--help"], capture_output=True, text=True, check=True).stdout
    assert "--denoise" in out and "--aov-samples <n>" in out
    bad = subprocess.run([cli, "--denoise", "-s", "2", "--aov-samples", "3"], capture_output=True, text=True)
    assert bad.returncode != 0 and "--aov-samples" in bad.stderr and "--denoise" in bad.stderr
    bad = subprocess.run([cli, "--denoise", "--from-ppm", "x.ppm"], capture_output=True, text=True)
    assert bad.returncode != 0 and "--from-ppm" in bad.stderr
