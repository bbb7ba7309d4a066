"""Nearest-surface queries without a GPU: the module is built for sm_100a, the struct matches the header, and tests/point_ref.py equals the
host build of csrc/point.cuh (the per-candidate routines and the prune bound) bit for bit: points in each of the seven Voronoi regions of a
triangle and on their boundaries, on the surface, degenerate records, ±0, subnormals, ±inf and NaN, spheres with negative and zero radius,
p = c, coordinates near 1e19.  A float64 restatement bounds the error of `dist`, and the prune bound is checked against each candidate's
own box."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from rbrt_b200 import _abi

from . import point_ref as P

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "rbrt_b200", "librbrt_gpu_point.so")
HD = os.path.join(ROOT, "tests", "host_device")
CSRC = os.path.join(ROOT, "rbrt_b200", "csrc")
F = np.float32
SPECIALS = np.array([0.0, -0.0, 1e-45, -1e-45, 1.5e-39, np.inf, -np.inf, np.nan], F)
# Largest error of `dist` against the exact distance to the same stored record, in units of u = 2^-23 * max(|p|, |v0|, |v0 + e1|, |v0 + e2|)
# plus 2^-23 * dist (test_float64_accuracy).  The prune proof (point.cuh) allows 20 u for the routine.
DIST_ERR_PIN = 1.0


@pytest.fixture(scope="module", autouse=True)
def point_module():
    if not os.path.exists(LIB):
        subprocess.run(["make", "-C", CSRC], check=True)
    return LIB


@pytest.fixture(scope="module")
def hd():
    out = os.path.join(HD, "build", "libhost_point.so")
    os.makedirs(os.path.dirname(out), exist_ok=True)
    srcs = [os.path.join(HD, f) for f in ("point_harness.cpp", "cuda_runtime.h")] + [os.path.join(CSRC, f) for f in ("common.cuh", "point.cuh")]
    if not os.path.exists(out) or any(os.path.getmtime(s) > os.path.getmtime(out) for s in srcs):
        # the flags of tests/test_device_source_on_host.py: the stand-in cuda_runtime.h first, no contraction, no FMA
        subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-mno-fma", "-Wno-unknown-pragmas", "-fPIC", "-shared",
                        "-I", HD, "-I", CSRC, "-o", out, srcs[0]], check=True)
    lib = C.CDLL(out)
    lib.hd_triangle.argtypes = [C.c_uint32] + [C.c_void_p] * 5
    lib.hd_sphere.argtypes = [C.c_uint32] + [C.c_void_p] * 4
    lib.hd_prune.argtypes = [C.c_uint32] + [C.c_void_p] * 8
    return lib


def bits_equal(a, b):
    """Bit patterns equal, any NaN equal to any NaN."""
    a, b = np.ascontiguousarray(a, F), np.ascontiguousarray(b, F)
    return (a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))


def host_triangle(hd, p, rec):
    p, rec = np.ascontiguousarray(p, F), np.ascontiguousarray(rec[:, :3, :3], F)
    n = len(p)
    d2, q, uv = np.zeros(n, F), np.zeros((n, 3), F), np.zeros((n, 2), F)
    assert hd.hd_triangle(n, p.ctypes.data, rec.ctypes.data, d2.ctypes.data, q.ctypes.data, uv.ctypes.data) == 0
    return d2, q, uv


def ref_triangle(p, rec):
    d2, q, u, v = P.closest_on_triangle([p[:, k] for k in range(3)], *([rec[:, i, k] for k in range(3)] for i in range(3)))
    return np.asarray(d2, F), np.stack(q, 1).astype(F), np.stack([u, v], 1).astype(F)


def check_triangles(hd, p, rec, what):
    got, want = host_triangle(hd, p, rec), ref_triangle(p, rec)
    for name, g, w in zip(("d2", "q", "uv"), got, want):
        ok = bits_equal(g, w).reshape(len(p), -1).all(1)
        bad = np.flatnonzero(~ok)
        assert not len(bad), f"{what}: {name}: {len(bad)} of {len(p)} differ; first p {p[bad[0]]} rec {rec[bad[0], :, :3]} got {g[bad[0]]} want {w[bad[0]]}"
    return got


def records(v0, e1, e2):
    r = np.zeros((len(v0), 3, 4), F)
    r[:, 0, :3], r[:, 1, :3], r[:, 2, :3] = v0, e1, e2
    return r


def random_triangles(n, seed, scale=1.0, centre=(0.0, 0.0, 0.0)):
    rng = np.random.default_rng(seed)
    v0 = (np.asarray(centre) + rng.normal(0, scale, (n, 3))).astype(F)
    return records(v0, rng.normal(0, scale, (n, 3)).astype(F), rng.normal(0, scale, (n, 3)).astype(F))


def region_points(rec, seed, spread=(-1.5, 2.5), height=1.0):
    """p = v0 + a e1 + b e2 + h n (n the unit normal), a and b over `spread`: every Voronoi region of the triangle."""
    rng = np.random.default_rng(seed)
    n = len(rec)
    a, b = rng.uniform(*spread, n), rng.uniform(*spread, n)
    r = rec.astype(np.float64)
    nn = np.cross(r[:, 1, :3], r[:, 2, :3])
    nn /= np.linalg.norm(nn, axis=1, keepdims=True)
    h = rng.normal(0, height, n)
    return (r[:, 0, :3] + a[:, None] * r[:, 1, :3] + b[:, None] * r[:, 2, :3] + h[:, None] * nn).astype(F)


def region_of(uv):
    u, v = uv[:, 0], uv[:, 1]
    return np.select([(u == 0) & (v == 0), (u == 1) & (v == 0), (u == 0) & (v == 1), v == 0, u == 0, u + v == 1], [0, 1, 2, 3, 4, 5], 6)


# ============================================================================== the module and the ABI
def test_module_is_built_for_sm100a_with_one_kernel_per_variant():
    cuobjdump = "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump is not here")
    out = subprocess.run([cuobjdump, "-sass", LIB], capture_output=True, text=True, check=True).stdout
    assert "sm_100a" in out
    names = sorted(set(ln.split()[-1] for ln in out.splitlines() if "Function :" in ln))
    assert len(names) == 2 and all("k_nearest" in n for n in names), names


def test_struct_matches_the_header(tmp_path):
    hdr = os.path.join(ROOT, "include", "rbrt_gpu.h")
    lines = ["#include <stdio.h>", "#include <stddef.h>", f'#include "{hdr}"', "int main(void){",
             'printf("size %zu\\n", sizeof(rbrt_nearest_out));']
    lines += [f'printf("{f} %zu\\n", offsetof(rbrt_nearest_out, {f}));' for f, _ in _abi.NearestOutC._fields_]
    src = tmp_path / "n.c"
    src.write_text("\n".join(lines + ["return 0;}"]))
    subprocess.run(["gcc", "-std=c99", "-o", str(tmp_path / "n"), str(src)], check=True)
    got = dict(l.split() for l in subprocess.run([str(tmp_path / "n")], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(got["size"]) == C.sizeof(_abi.NearestOutC)
    for f, _ in _abi.NearestOutC._fields_:
        assert int(got[f]) == getattr(_abi.NearestOutC, f).offset, f


def test_entry_point_refuses_without_touching_a_device():
    lib = _abi.lib()
    out = _abi.NearestOutC()
    st = _abi.StatsC(rays=5)
    assert lib.rbrt_gpu_query_nearest_device(None, None, 0, None, C.byref(out), None, C.byref(st)) == 0 and st.rays == 0
    assert lib.rbrt_gpu_query_nearest_device(None, None, 4, None, C.byref(out), None, None) == _abi.E_INVALID
    assert b"null" in lib.rbrt_last_error()


# ============================================================================== the triangle routine, bit for bit
def test_seven_regions_random(hd):
    rec = random_triangles(20000, 1)
    p = region_points(rec, 2)
    _, _, uv = check_triangles(hd, p, rec, "regions")
    assert set(np.unique(region_of(uv))) == set(range(7))


def boundary_cases():
    """The right triangle (0,0,0), (1,0,0), (0,1,0) and points on the planes that separate its regions, at three heights."""
    rec = records(np.zeros((1, 3), F), np.array([[1, 0, 0]], F), np.array([[0, 1, 0]], F))
    xy = [(-1, 0), (0, -1), (0, 0), (-1, -1), (1, 0), (2, 0), (1, -1), (0, 1), (0, 2), (-1, 1), (0.5, 0), (0, 0.5), (0.5, 0.5),
          (1.5, 0.5), (0.5, 1.5), (2, 1), (1, 2), (0.5, -1), (-1, 0.5), (0.25, 0.25), (1, 1)]
    p = np.array([(x, y, z) for x, y in xy for z in (0.0, -0.0, 0.75)], F)
    return p, np.repeat(rec, len(p), 0)


def test_region_boundaries(hd):
    p, rec = boundary_cases()
    d2, q, uv = check_triangles(hd, p, rec, "boundaries")
    assert np.isfinite(d2).all()
    # the boundary points' exact answers: their distance is |z| plus the planar offset, never below it
    assert (d2 >= (p[:, 2].astype(F) ** 2) * F(1 - 1e-6)).all()


def test_points_on_the_surface(hd):
    rec = random_triangles(5000, 3, centre=(3.0, -2.0, 7.0))
    rng = np.random.default_rng(4)
    a, b = rng.random(5000).astype(F), rng.random(5000).astype(F)
    flip = a + b > 1
    a[flip], b[flip] = F(1) - a[flip], F(1) - b[flip]
    p = ((rec[:, 0, :3] + a[:, None] * rec[:, 1, :3]) + b[:, None] * rec[:, 2, :3]).astype(F)
    d2, _, _ = check_triangles(hd, p, rec, "on the surface")
    scale = np.abs(rec[:, :, :3]).max((1, 2)) + np.abs(p).max(1)
    assert (np.sqrt(d2) <= 32 * 2.0 ** -23 * scale).all(), float((np.sqrt(d2) / (2.0 ** -23 * scale)).max())


def test_degenerate_records_never_give_nan(hd):
    rng = np.random.default_rng(5)
    n = 3000
    v0 = rng.normal(0, 2, (n, 3)).astype(F)
    d = rng.normal(0, 1, (n, 3)).astype(F)
    kinds = []
    kinds.append(records(v0, d, (F(2) * d).astype(F)))                  # collinear, exactly parallel edges
    kinds.append(records(v0, np.zeros_like(d), d))                      # e1 = 0
    kinds.append(records(v0, d, np.zeros_like(d)))                      # e2 = 0
    kinds.append(records(v0, d, d))                                     # b = c
    kinds.append(records(v0, np.zeros_like(d), np.zeros_like(d)))       # three equal vertices
    kinds.append(records(v0, d, (F(-0.5) * d).astype(F)))               # collinear, v0 between b and c
    rec = np.concatenate(kinds, 0)
    p = np.concatenate([region_points(records(v0, d, rng.normal(0, 1, (n, 3)).astype(F)), 6 + k) for k in range(len(kinds))], 0)
    d2, q, uv = check_triangles(hd, p, rec, "degenerate")
    assert np.isfinite(d2).all() and np.isfinite(q).all() and np.isfinite(uv).all()
    # the distance is that of the segment (or point) the record collapses to, in float64
    want = segment_set_dist64(p, rec)
    assert np.allclose(np.sqrt(d2), want, rtol=1e-5, atol=1e-5)


def segment_set_dist64(p, rec):
    r = rec.astype(np.float64)
    a, b, c = r[:, 0, :3], r[:, 0, :3] + r[:, 1, :3], r[:, 0, :3] + r[:, 2, :3]
    p = p.astype(np.float64)
    out = np.full(len(p), np.inf)
    for x, y in ((a, b), (a, c), (b, c)):
        e = y - x
        ee = (e * e).sum(1)
        t = np.where(ee > 0, np.clip(((p - x) * e).sum(1) / np.where(ee > 0, ee, 1), 0, 1), 0)
        out = np.minimum(out, np.linalg.norm(p - (x + t[:, None] * e), axis=1))
    return out


def test_special_values(hd):
    rng = np.random.default_rng(7)
    base = random_triangles(4000, 8)
    p = region_points(base, 9)
    rec = base.copy()
    # one special value in one coordinate of the point or the record
    where = rng.integers(0, 12, 4000)
    val = SPECIALS[rng.integers(0, len(SPECIALS), 4000)]
    for i in range(4000):
        if where[i] < 3:
            p[i, where[i]] = val[i]
        else:
            rec[i, (where[i] - 3) // 3, (where[i] - 3) % 3] = val[i]
    d2, _, _ = check_triangles(hd, p, rec, "specials")
    finite_in = np.isfinite(p).all(1) & np.isfinite(rec[:, :, :3]).all((1, 2))
    assert not np.isnan(d2[finite_in]).any()
    assert not np.isfinite(d2[~np.isfinite(p).all(1)]).any()             # a point with an inf or NaN coordinate has no finite d2
    # whole records of subnormals, ±0 and tiny points
    tiny = (rng.normal(0, 1, (2000, 3, 4)) * 1e-41).astype(F)
    check_triangles(hd, (rng.normal(0, 1, (2000, 3)) * 1e-40).astype(F), tiny, "subnormal")
    zeros = np.where(rng.random((2000, 3, 4)) < 0.5, F(0), F(-0.0)).astype(F)
    check_triangles(hd, np.where(rng.random((2000, 3)) < 0.5, F(0), F(-0.0)).astype(F), zeros, "signed zeros")


def test_coordinates_near_1e19(hd):
    rec = random_triangles(3000, 10, scale=1e18, centre=(1e19, -1e19, 5e18))
    p = region_points(rec, 11, height=1e18)
    d2, _, _ = check_triangles(hd, p, rec, "1e19")
    # near 1.8e19 the squares overflow: d2 = inf, which is never recorded
    far = p.copy()
    far[:, 0] = F(-3e19)
    d2f, _, _ = check_triangles(hd, far, rec, "overflow")
    assert np.isinf(d2f).all()


# ============================================================================== the sphere routine
def test_spheres(hd):
    rng = np.random.default_rng(12)
    n = 6000
    s = np.zeros((n, 4), F)
    s[:, :3] = rng.normal(0, 3, (n, 3))
    s[:, 3] = rng.uniform(-2, 2, n)
    s[::7, 3] = 0.0
    s[1::7, 3] = -0.0
    s[2::7, 3] *= -1
    p = (s[:, :3] + rng.normal(0, 2, (n, 3))).astype(F)
    p[::5] = s[::5, :3]                                                   # p = c
    p[3::11, 1] = SPECIALS[rng.integers(0, len(SPECIALS), len(p[3::11]))]
    s[4::13, 0] = SPECIALS[rng.integers(0, len(SPECIALS), len(s[4::13]))]
    d2, q = np.zeros(n, F), np.zeros((n, 3), F)
    sc, pc = np.ascontiguousarray(s), np.ascontiguousarray(p)
    assert hd.hd_sphere(n, pc.ctypes.data, sc.ctypes.data, d2.ctypes.data, q.ctypes.data) == 0
    wd, wq = P.closest_on_sphere([p[:, k] for k in range(3)], [s[:, k] for k in range(3)], s[:, 3])
    assert bits_equal(d2, wd).all() and bits_equal(q, np.stack(wq, 1)).all()
    at_c = (p == s[:, :3]).all(1) & np.isfinite(s).all(1)
    assert np.array_equal(q[at_c, 0], (s[at_c, 0] + np.abs(s[at_c, 3])).astype(F))
    assert np.allclose(np.sqrt(d2[at_c]), np.abs(s[at_c, 3]), rtol=1e-6, atol=1e-6)


# ============================================================================== accuracy against float64
def exact_dist64(p, rec):
    """The distance from p to the real triangle {v0 + u e1 + v e2} of each record, in float64 (Ericson's regions in exact-enough
    arithmetic: the records are well-shaped, so float64 rounding is far below the float32 error measured)."""
    p64, r = p.astype(np.float64), rec.astype(np.float64)
    d2, _, _, _ = P.closest_on_triangle([p64[:, k] for k in range(3)], *([r[:, i, k] for k in range(3)] for i in range(3)))
    return np.sqrt(d2)


def test_float64_accuracy(hd):
    worst = 0.0
    for seed, (scale, centre) in enumerate([(1.0, (0, 0, 0)), (1.0, (1000.0, -500.0, 20.0)), (1e-3, (0, 0, 0)), (50.0, (0, 0, 0)),
                                            (1e-2, (1e5, 0, 0))]):
        rec = random_triangles(20000, 20 + seed, scale, centre)
        p = region_points(rec, 40 + seed, height=scale)
        d2, _, _ = host_triangle(hd, p, rec)
        d = np.sqrt(d2.astype(np.float64))
        dist = np.sqrt(d2).astype(np.float64)                             # the plane `dist` = sqrt_rn(d2)
        exact = exact_dist64(p, rec)
        r = rec.astype(np.float64)
        s = np.maximum.reduce([np.abs(p).max(1), np.abs(r[:, 0, :3]).max(1), np.abs(r[:, 0, :3] + r[:, 1, :3]).max(1),
                               np.abs(r[:, 0, :3] + r[:, 2, :3]).max(1)])
        err = np.abs(dist - exact) / (2.0 ** -23 * s + 2.0 ** -23 * exact)
        worst = max(worst, float(err.max()))
        assert np.isfinite(d).all()
    assert worst <= DIST_ERR_PIN, worst
    print(f"largest dist error: {worst:.3f} u")


# ============================================================================== the prune bound
def test_prune_bound_never_drops_a_candidates_own_box(hd):
    """For each triangle, its exact vertex box (the tightest box the tree can hold it in), with best d2 = the candidate's own d2: the box
    bound must not exceed the prune bound.  Also with max_dist = the candidate's dist (the acceptance bound) and at every scale."""
    for seed, (scale, centre) in enumerate([(1.0, (0, 0, 0)), (1e-3, (1e3, 0, 0)), (1e-2, (1e6, -1e6, 0)), (1e4, (0, 0, 0)),
                                            (1e-30, (0, 0, 0)), (1e17, (1e18, 0, 0))]):
        rec = random_triangles(20000, 60 + seed, scale, centre)
        p = region_points(rec, 80 + seed, height=scale)
        p[::3] = rec[::3, 0, :3]                                          # on a vertex
        d2, _, _ = host_triangle(hd, p, rec)
        r = rec[:, :, :3]
        verts = np.stack([r[:, 0], (r[:, 0] + r[:, 1]).astype(F), (r[:, 0] + r[:, 2]).astype(F)], 1)
        # the raw vertices the box is built from: v0 and the f32 sums are within one rounding of them; both kinds of box are checked
        for box in (np.concatenate([verts.min(1), verts.max(1)], 1).astype(F),):
            n = len(p)
            md = np.full(n, np.inf, F)
            for best, mdv in ((d2, md), (np.full(n, np.inf, F), np.nextafter(np.sqrt(d2), F(np.inf)).astype(F))):
                bd, pd, acc = np.zeros(n, F), np.zeros(n, F), np.zeros(n, np.int32)
                args = [np.ascontiguousarray(a, F) for a in (p, box, mdv, best, box)]
                assert hd.hd_prune(n, *[a.ctypes.data for a in args], bd.ctypes.data, pd.ctypes.data, acc.ctypes.data) == 0
                bad = np.flatnonzero(bd > pd)
                assert not len(bad), f"scale {scale}: {len(bad)} boxes pruned; first p {p[bad[0]]} d2 {d2[bad[0]]} box {bd[bad[0]]} prune {pd[bad[0]]}"


def test_prune_bound_special_values(hd):
    n = 6
    p = np.zeros((n, 3), F)
    box = np.tile(np.array([[1, 1, 1, 2, 2, 2]], F), (n, 1))
    box[1, [0, 3]] = np.nan                                                # a qstep = NaN axis: contributes 0
    mesh = np.tile(np.array([[1, 1, 1, 2, 2, 2]], F), (n, 1))
    mesh[2, 3] = np.inf                                                    # a mesh with an inf coordinate: nothing is pruned
    md = np.array([np.inf, np.inf, np.inf, np.nan, 0.0, -1.0], F)
    best = np.array([1.0, 1.0, 1.0, np.inf, np.inf, np.inf], F)
    bd, pd, acc = np.zeros(n, F), np.zeros(n, F), np.zeros(n, np.int32)
    args = [np.ascontiguousarray(a, F) for a in (p, box, md, best, mesh)]
    assert hd.hd_prune(n, *[a.ctypes.data for a in args], bd.ctypes.data, pd.ctypes.data, acc.ctypes.data) == 0
    assert bd[0] == 3.0 and bd[1] == 2.0 and not np.isnan(bd).any()
    assert np.isinf(pd[2]) and bd[0] > pd[0]
    assert list(acc) == [1, 1, 1, 0, 0, 0]                                 # a NaN, zero or negative bound accepts nothing
