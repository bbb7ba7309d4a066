"""First-hit AOVs without a GPU: the AOV module is built for sm_100a and exports its launch interface, rbrt_aov_out has the header's layout,
the new entry points refuse bad calls without touching a device, the numpy restatement of the rules (tests/aov_ref.py) does what the
header says on hand-made hits, and the CLI lists its AOV flags."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import rbrt_b200 as R
from rbrt_b200 import _abi

from . import aov_ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
AOV = os.path.join(ROOT, "rbrt_b200", "librbrt_gpu_aov.so")
HEADER = os.path.join(ROOT, "include", "rbrt_gpu.h")
PLANES = ["depth", "normal", "albedo", "coverage", "hit_kind", "elem_idx", "tri_idx"]


@pytest.fixture(scope="module", autouse=True)
def aov_module():
    if not os.path.exists(AOV):
        subprocess.run(["make", "-C", os.path.join(ROOT, "rbrt_b200", "csrc")], check=True)
    return AOV


def test_aov_module_is_built_for_sm_100a_and_exports_its_interface():
    lib = C.CDLL(AOV)
    assert hasattr(lib, "rbrt_aov_launch")
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump is not here")
    sass = subprocess.run([cuobjdump, "-sass", AOV], capture_output=True, text=True, check=True).stdout
    names = re.findall(r"Function : (\S+)", sass)
    assert len(names) == 2 and all("k_aov" in n for n in names), names
    assert "arch = sm_100a" in sass


def test_aov_out_layout_matches_the_header(tmp_path):
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{HEADER}"', "int main(void){",
             'printf("size %zu\\n", sizeof(rbrt_aov_out));']
    lines += [f'printf("{f} %zu\\n", offsetof(rbrt_aov_out, {f}));' for f in PLANES]
    lines.append("return 0;}")
    src = tmp_path / "aov_layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "aov_layout"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-o", str(exe), str(src)], check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    assert [f for f, _ in _abi.AovOutC._fields_] == PLANES
    assert int(got["size"]) == C.sizeof(_abi.AovOutC)
    for f in PLANES:
        assert int(got[f]) == getattr(_abi.AovOutC, f).offset, f


def test_new_exports_and_refusals_without_a_device():
    lib = _abi.lib()
    raw = C.CDLL(_abi.LIB_PATH)
    assert hasattr(raw, "rbrt_gpu_render_aov") and hasattr(raw, "rbrt_gpu_render_aov_device")
    cam = R.Camera.new((0, 0, 0), (0, 0, -1), (0, 1, 0), 4, 8, 35.0).to_c()
    buf = np.full(32, 7, np.float32)
    out = _abi.AovOutC(depth=buf.ctypes.data)
    empty = _abi.AovOutC()
    for f in (lambda *a: lib.rbrt_gpu_render_aov(*a, None), lambda *a: lib.rbrt_gpu_render_aov_device(*a, None, None)):
        assert f(None, cam, 1, 0, out) == _abi.E_INVALID                 # NULL scene
        assert b"null" in lib.rbrt_last_error()
        assert f(C.c_void_p(1), None, 1, 0, out) == _abi.E_INVALID       # NULL camera (checked before the handle is touched)
        assert f(C.c_void_p(1), cam, 1, 0, None) == _abi.E_INVALID       # NULL out
        assert f(C.c_void_p(1), cam, 1, 0, empty) == _abi.E_INVALID      # every pass NULL
        assert b"no AOV" in lib.rbrt_last_error()
        assert f(C.c_void_p(1), cam, 0, 0, out) == _abi.E_INVALID        # zero samples
        cam0 = R.Camera.new((0, 0, 0), (0, 0, -1), (0, 1, 0), 0, 8, 35.0).to_c()
        assert f(C.c_void_p(1), cam0, 1, 0, out) == _abi.E_INVALID       # empty image
    assert (buf == 7).all()


def test_render_aovs_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present; the refusal path is exercised on the CPU-only build box")
    scene = R.Scene(elements=[R.Sphere((0, 0, -3), 1.0, R.Lambertian((0.5, 0.5, 0.5)))])
    cam = R.Camera.new((0, 0, 0), (0, 0, -1), (0, 1, 0), 4, 8, 35.0)
    with pytest.raises(_abi.RbrtGpuError) as e:
        R.render_aovs(cam, 1, scene)
    assert e.value.code in (_abi.E_NODEVICE, _abi.E_CUDA)
    with pytest.raises(ValueError):
        R.render_aovs(cam, 1, scene, passes=("depth", "motion"))


def _hits(rows):
    h = np.zeros(len(rows), dtype=_abi.HIT_DTYPE)
    for i, (kind, elem, tri, dist, normal) in enumerate(rows):
        h[i]["kind"], h[i]["elem_idx"], h[i]["tri_idx"], h[i]["dist"], h[i]["normal"] = kind, elem, tri, dist, normal
    return h


def test_numpy_rules_on_hand_made_hits():
    f32 = np.float32
    el = np.array([[0.5, 0.25, 0.125], [1.0, 1.0, 1.0]], f32)            # element 1: a Dielectric
    me = np.array([[0.1, 0.2, 0.3]], f32)
    M, S_, T = _abi.HIT_MESH, _abi.HIT_SPHERE, _abi.HIT_TRIANGLE
    N = _abi.HIT_NONE
    s0 = _hits([(S_, 0, 0, 2.0, (3.0, 0.0, 4.0)), (N, 0, 0, 0.0, (0, 0, 0)), (M, 0, 17, 5.0, (0.0, 1.0, 0.0)),
                (T, 1, 0, np.nan, (0.0, 0.0, -1.0)), (N, 0, 0, 0.0, (0, 0, 0))])
    s1 = _hits([(S_, 1, 0, 4.0, (0.0, -2.0, 0.0)), (N, 0, 0, 0.0, (0, 0, 0)), (N, 0, 0, 0.0, (0, 0, 0)),
                (T, 1, 0, 1.0, (0.0, 0.0, -1.0)), (M, 0, 3, 0.1, (1.0, 0.0, 0.0))])
    out = aov_ref.compose([s0, s1], el, me)
    # pixel 0: two sphere hits; normals normalised by len3 before the mean, albedo of elements 0 and 1 (Dielectric -> 1)
    assert out["depth"][0] == f32(3.0) and out["coverage"][0] == f32(1.0)
    assert np.array_equal(out["normal"][0], (np.float32([0.6, 0.0, 0.8]) + np.float32([0.0, -1.0, 0.0])) / f32(2))
    assert np.array_equal(out["albedo"][0], (el[0] + el[1]) / f32(2))
    # pixel 1: never hit -> +inf depth, zero normal / albedo / coverage, ids of a miss
    assert out["depth"][1] == np.inf and not out["normal"][1].any() and not out["albedo"][1].any() and out["coverage"][1] == 0
    assert (out["hit_kind"][1], out["elem_idx"][1], out["tri_idx"][1]) == (N, 0, 0)
    # pixel 2: one mesh hit of two samples: the mean over the hit samples only, normal used as stored
    assert out["depth"][2] == f32(5.0) and out["coverage"][2] == f32(0.5) and np.array_equal(out["normal"][2], [0, 1, 0])
    assert np.array_equal(out["albedo"][2], me[0]) and (out["hit_kind"][2], out["tri_idx"][2]) == (M, 17)
    # pixel 3: a NaN dist propagates into depth; a BasicTriangle normal is not normalised again
    assert np.isnan(out["depth"][3]) and np.array_equal(out["normal"][3], [0, 0, -1]) and out["hit_kind"][3] == T
    # pixel 4: sample 0 misses, sample 1 hits: ids come from sample 0
    assert out["depth"][4] == f32(0.1) and out["hit_kind"][4] == N and out["tri_idx"][4] == 0
    # the f32 order: sums left to right, then one division
    many = [_hits([(M, 0, 0, d, (0.0, 1.0, 0.0))]) for d in (1e8, 1.0, -1e8, 1.0)]
    assert aov_ref.compose(many, el, me)["depth"][0] == f32(((f32(1e8) + f32(1.0)) + f32(-1e8)) + f32(1.0)) / f32(4)


def test_cli_usage_lists_the_aov_flags():
    cli = os.path.join(ROOT, "rbrt_b200", "rbrt")
    if not os.path.exists(cli):
        subprocess.run(["make", "-C", os.path.join(ROOT, "rbrt_b200", "csrc")], check=True)
    out = subprocess.run([cli, "--help"], capture_output=True, text=True, check=True).stdout
    assert "--aov <prefix>" in out and "--aov-samples <n>" in out
    bad = subprocess.run([cli, "--aov-samples", "x"], capture_output=True, text=True)
    assert bad.returncode != 0 and "--aov-samples" in bad.stderr


def test_rust_crate_mirrors_aov_out_and_the_new_functions():
    rs = open(os.path.join(ROOT, "integration", "rust", "rbrt_gpu_sys", "src", "lib.rs")).read()
    m = re.search(r"pub struct RbrtAovOut\s*\{(.*?)\}", rs, re.S)
    assert m and re.findall(r"pub (\w+)\s*:", m.group(1)) == PLANES
    for name, arity in (("rbrt_gpu_render_aov", 6), ("rbrt_gpu_render_aov_device", 7)):
        f = re.search(r"pub fn %s\s*\((.*?)\)\s*->" % name, rs, re.S)
        assert f and len([a for a in f.group(1).split(",") if a.strip()]) == arity, name
