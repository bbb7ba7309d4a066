"""Per-pixel variance and the variance-guided filter without a GPU: the module is built for sm_100a and holds only its own kernels, the entry
points refuse bad calls without touching a device, tests/variance_ref.py equals a plain loop restatement and the host build of
csrc/variance.cuh bit for bit, and the CLI lists and checks --denoise-splits."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import rbrt_b200 as R
from rbrt_b200 import _abi

from . import variance_ref as V
from .test_denoise_host import adversarial, scene_like

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
VAR = os.path.join(ROOT, "rbrt_b200", "librbrt_gpu_variance.so")
HD = os.path.join(ROOT, "tests", "host_device")
CSRC = os.path.join(ROOT, "rbrt_b200", "csrc")
F = np.float32
SPECIALS = np.array([0.0, -0.0, 1e-45, 1e-40, np.inf, -np.inf, np.nan, -1e-3, -1e-45, 3e38], F)


@pytest.fixture(scope="module", autouse=True)
def variance_module():
    if not os.path.exists(VAR) or not os.path.exists(os.path.join(ROOT, "rbrt_b200", "rbrt")):
        subprocess.run(["make", "-C", CSRC], check=True)
    return VAR


@pytest.fixture(scope="module")
def hd():
    out = os.path.join(HD, "build", "libhost_variance.so")
    os.makedirs(os.path.dirname(out), exist_ok=True)
    srcs = [os.path.join(HD, f) for f in ("variance_harness.cpp", "cuda_runtime.h")] + \
           [os.path.join(CSRC, f) for f in ("common.cuh", "shade.cuh", "denoise.cuh", "variance.cuh")]
    if not os.path.exists(out) or any(os.path.getmtime(s) > os.path.getmtime(out) for s in srcs):
        # the flags of tests/test_device_source_on_host.py: the stand-in cuda_runtime.h first, no contraction, no FMA
        subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-mno-fma", "-Wno-unknown-pragmas", "-fPIC", "-shared",
                        "-I", HD, "-I", CSRC, "-o", out, srcs[0]], check=True)
    lib = C.CDLL(out)
    lib.hd_moments.argtypes = [C.c_uint32] * 4 + [C.c_void_p] * 3
    lib.hd_denoise_variance.argtypes = [C.c_uint32, C.c_uint32] + [C.c_void_p] * 5 + [C.c_uint32, C.c_float, C.c_float, C.c_void_p, C.c_void_p]
    return lib


def host_moments(hd, acc, S):
    acc = np.ascontiguousarray(acc, F)
    K, H, W = acc.shape[:3]
    hdr, var = np.zeros((H, W, 3), F), np.zeros((H, W, 3), F)
    assert hd.hd_moments(W, H, K, S, acc.ctypes.data, hdr.ctypes.data, var.ctypes.data) == 0
    return hdr, var


def host_filter(hd, c, v, a, n, z, levels=0, sigma_depth=0.0, sigma_luminance=0.0):
    L, sz, sl = V.resolve(levels, sigma_depth, sigma_luminance)
    c, v, a, n, z = (np.ascontiguousarray(x, F) for x in (c, v, a, n, z))
    H, W = z.shape
    out, rgb = np.zeros((H, W, 3), F), np.zeros((H, W, 3), np.uint8)
    assert hd.hd_denoise_variance(W, H, c.ctypes.data, v.ctypes.data, z.ctypes.data, n.ctypes.data, a.ctypes.data, L, sz, sl,
                                  out.ctypes.data, rgb.ctypes.data) == 0
    return out, rgb


def variance_like(H, W, seed, specials=True):
    """A variance plane of the scale of a few-spp render's, with every special value when asked: ±0, subnormals, ±inf, NaN, negatives."""
    rng = np.random.default_rng(seed)
    v = rng.gamma(0.8, 0.02, (H, W, 3)).astype(F)
    v[rng.random((H, W)) < 0.1] = 0.0                                   # converged pixels
    if specials:
        k = min(len(SPECIALS), v.size)
        v.reshape(-1)[rng.choice(v.size, k, replace=False)] = SPECIALS[:k]
    return v


def adversarial_accumulators(K, H, W, seed):
    rng = np.random.default_rng(seed)
    acc = rng.gamma(1.0, 2.0, (K, H, W, 4)).astype(F)
    flat = acc[..., :3].reshape(-1)
    idx = rng.choice(flat.size, 6, replace=False)
    flat[idx] = np.array([np.nan, np.inf, -np.inf, 1e-45, 3e38, -0.0], F)
    acc[..., :3] = flat.reshape(acc[..., :3].shape)
    acc[:, 0, 0, :3] = 0.0                                               # a black pixel: variance 0
    return acc


# ============================================================================== module, refusals
def test_module_is_built_for_sm_100a_with_only_its_own_kernels():
    lib = C.CDLL(VAR)
    assert hasattr(lib, "rbrt_variance_moments_launch") and hasattr(lib, "rbrt_variance_filter_launch")
    raw = C.CDLL(_abi.LIB_PATH)
    for f in ("rbrt_gpu_render_hdr_variance", "rbrt_gpu_render_hdr_variance_device", "rbrt_gpu_denoise_variance",
              "rbrt_gpu_denoise_variance_device"):
        assert hasattr(raw, f), f
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump is not here")
    sass = subprocess.run([cuobjdump, "-sass", VAR], capture_output=True, text=True, check=True).stdout
    names = re.findall(r"Function : (\S+)", sass)
    assert len(names) == 4 and all("k_variance" in n for n in names), names
    assert sum("k_variance_level" in n for n in names) == 2
    assert "arch = sm_100a" in sass
    main = subprocess.run([cuobjdump, "-sass", _abi.LIB_PATH], capture_output=True, text=True, check=True).stdout
    kernels = re.findall(r"Function : (\S+)", main)
    assert len(kernels) == 51 and not any("variance" in k for k in kernels)


def test_render_refusals_without_a_device():
    """Every check that comes before the scene is read: a stand-in scene pointer is never dereferenced by them."""
    lib = _abi.lib()
    cam = R.Camera.new((0.0, 0.0, 0.0), (0.0, 0.0, -1.0), (0.0, 1.0, 0.0), 6, 8, 50.0).to_c()
    empty = R.Camera.new((0.0, 0.0, 0.0), (0.0, 0.0, -1.0), (0.0, 1.0, 0.0), 6, 8, 50.0).to_c()
    empty.img_width_pix = 0
    hdr, var = np.full(3 * 48, 7.0, F), np.full(3 * 48, 7.0, F)
    stand_in = C.create_string_buffer(64)
    sc = C.addressof(stand_in)
    O = R.render.make_opts
    cases = [
        ((None, cam, 8, 4, None, hdr.ctypes.data, var.ctypes.data), b"null"),
        ((sc, None, 8, 4, None, hdr.ctypes.data, var.ctypes.data), b"null"),
        ((sc, cam, 8, 4, None, None, None), b"no output"),
        ((sc, cam, 8, 1, None, hdr.ctypes.data, var.ctypes.data), b"splits"),
        ((sc, cam, 8, 0, None, hdr.ctypes.data, var.ctypes.data), b"splits"),
        ((sc, cam, 34, 17, None, hdr.ctypes.data, var.ctypes.data), b"splits"),
        ((sc, cam, 9, 4, None, hdr.ctypes.data, var.ctypes.data), b"multiple of splits"),
        ((sc, cam, 0, 4, None, hdr.ctypes.data, var.ctypes.data), b"multiple of splits"),
        ((sc, cam, 8, 4, O(shard_mode=_abi.SHARD_SAMPLES, shard_count=2), hdr.ctypes.data, var.ctypes.data), b"shard_count"),
        ((sc, empty, 8, 4, None, hdr.ctypes.data, var.ctypes.data), b"empty"),
        ((sc, cam, 8, 4, None, hdr.ctypes.data, hdr.ctypes.data + 4), b"overlap"),
    ]
    for f in (lambda *a: lib.rbrt_gpu_render_hdr_variance(*a, None), lambda *a: lib.rbrt_gpu_render_hdr_variance_device(*a, None, None)):
        for args, msg in cases:
            assert f(*args) == _abi.E_INVALID, (args, msg)
            assert msg in lib.rbrt_last_error(), (msg, lib.rbrt_last_error())
    assert (hdr == 7.0).all() and (var == 7.0).all()


def test_filter_refusals_without_a_device():
    lib = _abi.lib()
    W, H = 8, 6
    n = W * H
    hdr, var, alb, nrm, dep = np.ones(3 * n, F), np.ones(3 * n, F), np.ones(3 * n, F), np.ones(3 * n, F), np.ones(n, F)
    out, rgb = np.full(3 * n, 7.0, F), np.full(3 * n, 7, np.uint8)
    g = _abi.AovOutC(depth=dep.ctypes.data, normal=nrm.ctypes.data, albedo=alb.ctypes.data)
    O = _abi.DenoiseOptsC
    h, v = hdr.ctypes.data, var.ctypes.data
    cases = [
        ((W, H, None, v, g, None, out.ctypes.data, rgb.ctypes.data), b"null"),
        ((W, H, h, None, g, None, out.ctypes.data, rgb.ctypes.data), b"null"),
        ((W, H, h, v, None, None, out.ctypes.data, rgb.ctypes.data), b"null"),
        ((W, H, h, v, _abi.AovOutC(normal=nrm.ctypes.data, albedo=alb.ctypes.data), None, out.ctypes.data, None), b"guide"),
        ((W, H, h, v, g, None, None, None), b"no output"),
        ((0, H, h, v, g, None, out.ctypes.data, None), b"empty"),
        ((65536, 32768, h, v, g, None, out.ctypes.data, None), b"too large"),
        ((W, H, h, v, g, O(levels=9), out.ctypes.data, None), b"levels"),
        ((W, H, h, v, g, O(sigma_depth=float("nan")), out.ctypes.data, None), b"sigma"),
        ((W, H, h, v, g, O(sigma_luminance=-1.0), out.ctypes.data, None), b"sigma"),
        ((W, H, h, v, g, None, var.ctypes.data + 8, None), b"overlaps an input"),
        ((W, H, h, v, g, None, None, var.ctypes.data + 20), b"overlaps an input"),
        ((W, H, h, v, g, None, out.ctypes.data, out.ctypes.data + 8), b"overlap"),
    ]
    for f in (lambda *a: lib.rbrt_gpu_denoise_variance(*a, None), lambda *a: lib.rbrt_gpu_denoise_variance_device(*a, None, None)):
        for args, msg in cases:
            assert f(*args) == _abi.E_INVALID, (args, msg)
            assert msg in lib.rbrt_last_error(), (msg, lib.rbrt_last_error())
    assert (out == 7.0).all() and (rgb == 7).all()


def test_python_argument_checks():
    c, a, n, z = scene_like(6, 8, 0)
    v = variance_like(6, 8, 0, specials=False)
    aovs = {"depth": z, "normal": n, "albedo": a}
    for hdr, var, g in [(c, v[:, :, :2].copy(), aovs), (c, v.astype(np.float64), aovs), (c, v[:, ::2], aovs), (c, v, {"depth": z, "normal": n}),
                        (c[:, :, :2], v, aovs)]:
        with pytest.raises(ValueError):
            R.denoise_variance(hdr, var, g)
    import torch
    with pytest.raises(ValueError):
        R.denoise_variance_device(torch.from_numpy(c), torch.from_numpy(v), {k: torch.from_numpy(x) for k, x in aovs.items()})


def test_variance_calls_need_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present; the refusal path is exercised on the CPU-only build box")
    c, a, n, z = scene_like(6, 8, 0)
    with pytest.raises(_abi.RbrtGpuError) as e:
        R.denoise_variance(c, variance_like(6, 8, 0, specials=False), {"depth": z, "normal": n, "albedo": a})
    assert e.value.code in (_abi.E_NODEVICE, _abi.E_CUDA)


# ============================================================================== the definitions: numpy, a plain loop, the host build
@pytest.mark.parametrize("K", [2, 3, 4, 16])
def test_moments_numpy_equals_the_plain_loop_and_the_host_build(hd, K):
    for (H, W), seed in [((5, 7), K), ((1, 9), 10 + K), ((9, 1), 20 + K)]:
        acc = adversarial_accumulators(K, H, W, seed)
        S = K * (seed % 5 + 1)
        hdr, var = V.moments(acc, S)
        want_h, want_v = V.moments_scalar(acc, S)
        assert V.same_bits(hdr, want_h) and V.same_bits(var, want_v), (K, H, W)
        got_h, got_v = host_moments(hd, acc, S)
        assert V.same_bits(got_h, hdr) and V.same_bits(got_v, var), (K, H, W)
        assert (var[0, 0] == 0).all() and np.isnan(var).any()


@pytest.mark.parametrize("shape", [(6, 8), (1, 5), (5, 1)])
def test_filter_numpy_equals_the_plain_loop(shape):
    H, W = shape
    for seed, opts in [(1, {}), (2, {"levels": 1}), (3, {"levels": 3, "sigma_depth": 0.5, "sigma_luminance": 0.7}), (4, {"levels": 8})]:
        c, a, n, z = adversarial(H, W, seed)
        v = variance_like(H, W, seed)
        got, rgb = V.denoise_variance(c, v, a, n, z, **opts)
        want, want_rgb = V.denoise_variance_scalar(c, v, a, n, z, **opts)
        assert V.same_bits(got, want), (shape, seed, opts)
        assert np.array_equal(rgb, want_rgb)
    c, a, n, z = scene_like(H, W, 5)                                    # no special values: the filter does mix pixels
    v = variance_like(H, W, 5, specials=False)
    got, _ = V.denoise_variance(c, v, a, n, z, levels=2)
    assert V.same_bits(got, V.denoise_variance_scalar(c, v, a, n, z, levels=2)[0]) and not V.same_bits(got, c)


def test_filter_rules_on_hand_made_planes():
    c, a, n, z = scene_like(6, 8, 7)
    v = variance_like(6, 8, 7, specials=False)
    v[2, 5] = [0.01, np.nan, 0.01]                                        # invalid variance: passed through, never a tap
    v[3, 3] = [0.01, -1e-6, 0.01]
    v[4, 4] = [-0.0, 0.0, -0.0]                                           # -0 is a valid variance: the pixel is filtered
    out, rgb = V.denoise_variance(c, v, a, n, z, levels=2)
    for y, x in [(2, 5), (3, 3), (0, 0), (1, 1)]:                         # bad variance, and the misses of scene_like
        assert V.same_bits(out[y, x], c[y, x]), (y, x)
    assert np.isfinite(out).all() and np.array_equal(rgb, V.tonemap(out))
    v2 = v.copy()
    v2[4, 4] = np.nan
    assert not V.same_bits(V.denoise_variance(c, v2, a, n, z, levels=2)[0][4, 4], out[4, 4]) or V.same_bits(out[4, 4], c[4, 4])
    # zero variance everywhere: only taps of exactly the centre's luminance mix, so a constant surface stays constant and an edge stays
    c2 = np.broadcast_to(np.where(np.arange(8)[None, :, None] < 4, F(0.2), F(0.6)), (6, 8, 3)).astype(F)
    a2 = np.full((6, 8, 3), 0.5, F)
    n2 = np.tile(F([0.0, 0.0, 1.0]), (6, 8, 1))
    z2 = np.full((6, 8), 3.0, F)
    out2, _ = V.denoise_variance(c2, np.zeros_like(c2), a2, n2, z2, levels=3)
    assert V.same_bits(out2, c2)
    # with variance the same edge blurs
    out3, _ = V.denoise_variance(c2, np.full_like(c2, 0.05), a2, n2, z2, levels=3)
    assert not V.same_bits(out3, c2)


@pytest.mark.parametrize("levels", range(1, 9))
def test_filter_host_build_equals_the_numpy_reference(hd, levels):
    for shape, seed in [((17, 33), levels), ((5, 7), 100 + levels), ((1, 9), 200 + levels), ((9, 1), 300 + levels)]:
        for opts in ({}, {"sigma_depth": 0.25, "sigma_luminance": 1.5}):
            c, a, n, z = adversarial(*shape, seed)
            v = variance_like(*shape, seed)
            got, got_rgb = host_filter(hd, c, v, a, n, z, levels=levels, **opts)
            want, want_rgb = V.denoise_variance(c, v, a, n, z, levels=levels, **opts)
            assert V.same_bits(got, want), (shape, levels, opts)
            assert np.array_equal(got_rgb, want_rgb), (shape, levels, opts)
    c, a, n, z = scene_like(24, 40, levels)
    v = variance_like(24, 40, levels, specials=False)
    got, _ = host_filter(hd, c, v, a, n, z, levels=levels)
    want, _ = V.denoise_variance(c, v, a, n, z, levels=levels)
    assert V.same_bits(got, want) and not V.same_bits(got, c)


# ============================================================================== CLI
def test_cli_lists_and_checks_denoise_splits():
    cli = os.path.join(ROOT, "rbrt_b200", "rbrt")
    out = subprocess.run([cli, "--help"], capture_output=True, text=True, check=True).stdout
    assert "--denoise-splits <k>" in out
    for args, msg in [(["--denoise-splits", "4", "-s", "8"], "needs '--denoise'"),
                      (["--denoise", "--denoise-splits", "1", "-s", "8"], "2..16"),
                      (["--denoise", "--denoise-splits", "17", "-s", "34"], "2..16"),
                      (["--denoise", "--denoise-splits", "3", "-s", "8"], "divide"),
                      (["--denoise", "--denoise-splits", "4", "-s", "8", "--aov-samples", "3"], "--aov-samples"),
                      (["--denoise", "--denoise-splits", "x", "-s", "8"], "invalid value"),
                      (["--denoise", "--denoise-splits", "4", "-s", "8", "--from-ppm", "x.ppm"], "--from-ppm")]:
        r = subprocess.run([cli, "-c", "no-such-scene.yaml"] + args, capture_output=True, text=True)
        assert r.returncode != 0 and msg in r.stderr, (args, r.stderr)
