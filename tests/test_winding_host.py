"""Winding numbers without a GPU: the module is built for sm_100a, and the host build of csrc/winding.cuh (the triangle and sphere terms,
the far test, the expansion and the moments with their merge) is checked against the float64 restatements of tests/winding_ref.py: random
triangles at scales 1e-30 ... 1e18, points on a vertex, on an edge, in the plane and at the centroid, degenerate records, ±0,
subnormals, ±inf and NaN; the sphere rule at d2 == r2, for a negative radius and r = 0; merges over random trees against the direct
moments, with R bounding every vertex; and the expansion error on a random patch as the distance grows."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from . import winding_ref as W

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "rbrt_b200", "librbrt_gpu_wind.so")
HD = os.path.join(ROOT, "tests", "host_device")
CSRC = os.path.join(ROOT, "rbrt_b200", "csrc")
F = np.float32
U = 4.0 * np.pi * 2.0 ** -24                                              # an ulp of 4 pi's neighbourhood, halved: 2^-24 * 4 pi
# Largest |Omega32 - Omega64| of a triangle term over the random triangles of test_triangle_random_scales, in units of U
# (22.1 measured there, 33.5 in test_special_values).
TRI_ERR_PIN = 64
# Relative errors of the merged moments against the direct float64 ones (test_merges_over_random_trees).
MOM_ERR_PIN = 1e-5


@pytest.fixture(scope="module", autouse=True)
def wind_module():
    if not os.path.exists(LIB):
        subprocess.run(["make", "-C", CSRC], check=True)
    return LIB


@pytest.fixture(scope="module")
def hd():
    out = os.path.join(HD, "build", "libhost_winding.so")
    os.makedirs(os.path.dirname(out), exist_ok=True)
    srcs = [os.path.join(HD, f) for f in ("winding_harness.cpp", "cuda_runtime.h")] + [os.path.join(CSRC, f) for f in ("common.cuh", "winding.cuh")]
    if not os.path.exists(out) or any(os.path.getmtime(s) > os.path.getmtime(out) for s in srcs):
        # the flags of tests/test_device_source_on_host.py: the stand-in cuda_runtime.h first, no contraction, no FMA
        subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-mno-fma", "-Wno-unknown-pragmas", "-fPIC", "-shared",
                        "-I", HD, "-I", CSRC, "-o", out, srcs[0]], check=True)
    lib = C.CDLL(out)
    lib.hd_tri.argtypes = [C.c_uint32] + [C.c_void_p] * 3
    lib.hd_sphere.argtypes = [C.c_uint32] + [C.c_void_p] * 3
    lib.hd_leaf.argtypes = [C.c_uint32] + [C.c_void_p] * 3
    lib.hd_merge.argtypes = [C.c_void_p] * 4
    lib.hd_far.argtypes = [C.c_uint32, C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.c_void_p]
    return lib


def host_tri(hd, p, rec):
    p, rec = np.ascontiguousarray(p, F), np.ascontiguousarray(np.asarray(rec, F)[:, :3, :3])
    om = np.zeros(len(p), F)
    assert hd.hd_tri(len(p), p.ctypes.data, rec.ctypes.data, om.ctypes.data) == 0
    return om


def ref_tri(p, rec):
    p, r = np.asarray(p, np.float64), np.asarray(rec, F).astype(np.float64)
    return W.omega([p[:, k] for k in range(3)], *([r[:, i, k] for k in range(3)] for i in range(3)))


def records(tris):
    """[N,3,4] float32 records of triangles [N,3,3] as the scene stores them (v0, e1 = b - a, e2 = c - a)."""
    t = np.asarray(tris, F)
    r = np.zeros((len(t), 3, 4), F)
    r[:, 0, :3], r[:, 1, :3], r[:, 2, :3] = t[:, 0], t[:, 1] - t[:, 0], t[:, 2] - t[:, 0]
    return r


# ============================================================================== triangle terms
def test_triangle_random_scales(hd):
    """Random triangles and points at every scale from 1e-30 to 1e18 (p within a few triangle sizes): the f32 term is within TRI_ERR_PIN
    units of 2^-24 * 4 pi of the exact solid angle of the stored record."""
    rng = np.random.default_rng(1)
    worst = 0.0
    for scale in 10.0 ** np.arange(-30, 19, 4):
        n = 4000
        c = rng.normal(size=(n, 3)) * scale * rng.choice([1.0, 1e3], n)[:, None]
        tris = c[:, None, :] + rng.normal(size=(n, 3, 3)) * scale
        rec = records(tris)
        p = (c + rng.normal(size=(n, 3)) * scale * 2).astype(F)
        got, want = host_tri(hd, p, rec), ref_tri(p, rec)
        assert np.isfinite(got).all() and (np.abs(got) <= 2 * np.pi * (1 + 1e-6)).all()
        err = np.abs(got - want) / U
        worst = max(worst, err.max())
        assert err.max() <= TRI_ERR_PIN, (scale, err.max(), p[err.argmax()], rec[err.argmax()])
    print("largest triangle term error", worst, "x 2^-24 * 4 pi")
    assert worst > 0


def test_triangle_special_positions(hd):
    """On a vertex, on an edge, in the plane: 0.  Just above and below the centroid: -2 pi and +2 pi (the sign of the corner order)."""
    tri = np.array([[(0.0, 0.0, 0.0), (4.0, 0.0, 0.0), (0.0, 4.0, 0.0)]], F)          # counter-clockwise seen from +z: normal +z
    rec = records(tri)
    for v in range(3):                                                               # each corner as v0, p on it
        rot = records(np.roll(tri, -v, axis=1))
        assert host_tri(hd, tri[:, v], rot)[0] == 0.0
    in_plane = np.array([(2.0, 0.0, 0.0), (2.0, 2.0, 0.0), (4.0 / 3, 4.0 / 3, 0.0), (9.0, -3.0, 0.0), (1.0, 1.0, 0.0)], F)
    assert (host_tri(hd, in_plane, np.repeat(rec, len(in_plane), 0)) == 0.0).all()
    c = np.array([4.0 / 3, 4.0 / 3, 0.0])
    for h in (1e-3, 1e-6, 1e-20):
        p = np.array([c + (0, 0, h), c - (0, 0, h)], F)
        got, want = host_tri(hd, p, np.repeat(rec, 2, 0)), ref_tri(p, np.repeat(rec, 2, 0))
        assert got[0] < 0 < got[1] and np.allclose(np.abs(got), 2 * np.pi, atol=1e-2), (h, got)
        assert np.abs(got - want).max() <= TRI_ERR_PIN * U


def test_degenerate_records(hd):
    """Collinear corners, a zero-length edge and three equal corners have no solid angle: the f32 term is within the pin of 0, and
    exactly 0 where det vanishes exactly (three equal corners, and a point on the line of a collinear record)."""
    rng = np.random.default_rng(2)
    n = 3000
    a = rng.normal(size=(n, 3)) * 10
    d = rng.normal(size=(n, 3))
    kinds = [np.stack([a, a + d, a + 2.5 * d], 1), np.stack([a, a, a + d], 1), np.stack([a, a + d, a + d], 1), np.stack([a, a, a], 1)]
    p = (a + rng.normal(size=(n, 3)) * 5).astype(F)
    for i, t in enumerate(kinds):
        rec = records(t)
        got = host_tri(hd, p, rec)
        assert np.isfinite(got).all() and np.abs(got).max() <= TRI_ERR_PIN * U, (i, np.abs(got).max())
    assert (host_tri(hd, p, records(kinds[3])) == 0).all()
    line = np.array([[(0.0, 0.0, 0.0), (1.0, 0.0, 0.0), (3.0, 0.0, 0.0)]], F)
    assert (host_tri(hd, np.array([(5.0, 0.0, 0.0), (-2.0, 0.0, 0.0)], F), np.repeat(records(line), 2, 0)) == 0).all()


def test_special_values(hd):
    """±0, subnormals, ±inf and NaN in the point or the record: never a non-finite term; inf and NaN give 0; subnormal geometry keeps its
    solid angle (the power-of-two scaling)."""
    S = np.array([0.0, -0.0, 1e-45, -1e-45, 1.5e-39, np.inf, -np.inf, np.nan], F)
    rng = np.random.default_rng(3)
    n = 20000
    base = records(rng.normal(size=(n, 3, 3)))
    p = rng.normal(size=(n, 3)).astype(F)
    where = rng.integers(0, 12, n)                                         # 0..2: a point component; 3..11: a record component
    val = S[rng.integers(0, len(S), n)]
    for i in range(n):
        w = where[i]
        if w < 3:
            p[i, w] = val[i]
        else:
            base[i, (w - 3) // 3, (w - 3) % 3] = val[i]
    got = host_tri(hd, p, base)
    assert np.isfinite(got).all()
    bad = ~np.isfinite(p).all(1) | ~np.isfinite(base[:, :, :3]).all((1, 2))
    assert (got[bad] == 0).all()
    want = ref_tri(p[~bad], base[~bad])
    assert np.abs(got[~bad] - want).max() <= TRI_ERR_PIN * U
    tiny = records(np.array([[(1e-45, 0, 2e-45), (4e-45, 0, 2e-45), (1e-45, 3e-45, 2e-45)]], F))   # subnormal corners
    got = host_tri(hd, np.array([(1.5e-45, 1.5e-45, 0.0)], F), tiny)
    want = ref_tri(np.array([(1.5e-45, 1.5e-45, 0.0)], F), tiny)
    assert got[0] != 0 and abs(got[0] - want[0]) <= TRI_ERR_PIN * U, (got, want)


# ============================================================================== spheres
def test_sphere_rule(hd):
    p = np.array([(3.0, 4.0, 0.0), (3.0, 4.0, 0.0), (0.0, 0.0, 0.0), (0.0, 0.0, 0.0), (1.0, 1.0, 1.0), (6.0, 0.0, 0.0), (0.0, 0.0, 0.0),
                  (np.nan, 0.0, 0.0), (np.inf, 0.0, 0.0), (0.0, 0.0, 0.0)], F)
    s = np.array([(0, 0, 0, 5.0), (0, 0, 0, -5.0), (0, 0, 0, 0.0), (0, 0, 0, -0.0), (0, 0, 0, -2.0), (0, 0, 0, 5.0), (0, 0, 0, 1e-30),
                  (0, 0, 0, 1.0), (0, 0, 0, 1.0), (0, 0, 0, np.inf)], F)
    got = np.zeros(len(p), np.int32)
    assert hd.hd_sphere(len(p), p.ctypes.data, s.ctypes.data, got.ctypes.data) == 0
    # on the surface for either sign; r = 0 (also at p = c); inside; outside; r2 = 1e-60 underflows to 0 = d2 at p = c: on the surface;
    # NaN and inf points; an infinite radius
    assert got.tolist() == [1, 1, 0, 0, 2, 0, 1, 0, 0, 2]
    rng = np.random.default_rng(4)
    p = rng.normal(size=(5000, 3)).astype(F)
    s = np.concatenate([rng.normal(size=(5000, 3)), rng.normal(size=(5000, 1)) * 2], 1).astype(F)
    got = np.zeros(len(p), np.int32)
    hd.hd_sphere(len(p), p.ctypes.data, s.ctypes.data, got.ctypes.data)
    assert np.array_equal(got, W.sphere_halves(p, s[:, :3], s[:, 3]))


# ============================================================================== moments
def leaf(hd, rec):
    r = np.ascontiguousarray(rec, F)
    out, area = np.zeros(16, F), C.c_double()
    hd.hd_leaf(len(r), r.ctypes.data, out.ctypes.data, C.byref(area))
    return out, area.value


def merge(hd, kids):
    recs = np.zeros((4, 16), F)
    recs[:, 3] = -1.0
    areas = np.zeros(4, np.float64)
    for k, (r, a) in enumerate(kids):
        recs[k], areas[k] = r, a
    out, area = np.zeros(16, F), C.c_double()
    assert hd.hd_merge(recs.ctypes.data, areas.ctypes.data, out.ctypes.data, C.byref(area)) == 1
    return out, area.value


def build(hd, rec, rng):
    """The record of a random tree over rec: leaves of 1..8 triangles, nodes of 2..4 children."""
    if len(rec) <= 8 and (len(rec) == 1 or rng.random() < 0.5):
        return leaf(hd, rec)
    k = int(rng.integers(2, 5)) if len(rec) >= 4 else 2
    cuts = np.sort(rng.choice(np.arange(1, len(rec)), min(k, len(rec)) - 1, replace=False))
    return merge(hd, [build(hd, part, rng) for part in np.split(rec, cuts)])


def unpack(r):
    T = np.array([r[7], r[8], r[9], r[10], r[11], r[12], r[13], r[14], r[15]], np.float64).reshape(3, 3)
    return r[:3].astype(np.float64), float(r[3]), r[4:7].astype(np.float64), T


@pytest.mark.parametrize("seed", range(6))
def test_merges_over_random_trees(hd, seed):
    """The root record of a random tree equals the direct float64 moments: c within MOM_ERR_PIN of the patch's size, N within
    MOM_ERR_PIN of sum |N_t|, T (about the stored c) within MOM_ERR_PIN of sum |N_t| times the size; R bounds every vertex."""
    rng = np.random.default_rng(seed)
    n = int(rng.integers(1, 400))
    centre = rng.normal(size=3) * 10.0 ** rng.uniform(-3, 6)
    size = 10.0 ** rng.uniform(-3, 3)
    tris = centre + rng.normal(size=(n, 1, 3)) * size + rng.normal(size=(n, 3, 3)) * size * 0.1
    rec = records(tris)
    r, area = build(hd, rec, rng)
    c, R, N, T = unpack(r)
    c64, R64, N64, _ = W.moments(rec)
    rr = rec.astype(np.float64)
    Nt = 0.5 * np.cross(rr[:, 1, :3], rr[:, 2, :3])
    ct = rr[:, 0, :3] + (rr[:, 1, :3] + rr[:, 2, :3]) / 3.0
    T64 = np.einsum("ti,tj->ij", Nt, ct - c)                                   # about the stored centre
    scale_n = np.abs(Nt).sum()
    ext = np.ptp(rr[:, 0, :3], 0).max() + size
    assert np.abs(c - c64).max() <= MOM_ERR_PIN * ext
    assert np.abs(N - N64).max() <= MOM_ERR_PIN * scale_n
    assert np.abs(T - T64).max() <= MOM_ERR_PIN * scale_n * ext
    assert abs(area - np.linalg.norm(Nt, axis=1).sum()) <= 1e-9 * area
    verts = np.concatenate([rr[:, 0, :3], rr[:, 0, :3] + rr[:, 1, :3], rr[:, 0, :3] + rr[:, 2, :3]], 0)
    assert np.linalg.norm(verts - c, axis=1).max() <= R and R <= 4 * R64 + 1e-30


def test_merge_without_the_shift_would_differ(hd):
    """Two children far apart: T of their merge carries N_k (x) (c_k - c), which the children's own T (about their own centres) lacks."""
    a = records(np.array([[(0, 0, 0), (1, 0, 0), (0, 1, 0)]], F))
    b = records(np.array([[(10, 0, 0), (10, 1, 0), (10, 0, 1)]], F))            # facing +x
    r, _ = merge(hd, [leaf(hd, a), leaf(hd, b)])
    _, _, _, T = unpack(r)
    c64, _, _, T64 = W.moments(np.concatenate([a, b]))
    assert np.allclose(T, T64, rtol=1e-6, atol=1e-6) and abs(T64[0, 0]) > 1.0


def test_non_finite_moments_are_always_descended(hd):
    """A NaN or inf corner makes R = +inf, and a merge over such a child too: the far test never takes it."""
    good = records(np.array([[(0, 0, 0), (1, 0, 0), (0, 1, 0)]], F))
    for v in (np.nan, np.inf):
        bad = records(np.array([[(0, 0, 0), (1, v, 0), (0, 1, 0)]], F))
        r, _ = leaf(hd, bad)
        assert r[3] == np.inf
        m, _ = merge(hd, [leaf(hd, good), (r, 0.5)])
        assert m[3] == np.inf
        far, om = np.zeros(1, np.int32), np.zeros(1, F)
        p = np.array([(1e6, 1e6, 1e6)], F)
        hd.hd_far(1, p.ctypes.data, np.ascontiguousarray(m).ctypes.data, 2.0, far.ctypes.data, om.ctypes.data)
        assert far[0] == 0


# ============================================================================== the far field
def test_expansion_error_falls_with_distance(hd):
    """A random patch of 8 triangles within R of its centre: the f32 expansion's error against the exact float64 sum of its solid angles
    falls at least like (R / d)^3 (the first term left out is of order (R / d)^4), and the far test is |p - c| > beta R."""
    rng = np.random.default_rng(5)
    v = rng.normal(size=(8, 3, 3)) * 0.5 + np.array([3.0, -1.0, 2.0])
    rec = records(v)
    r, _ = leaf(hd, rec)
    c, R, _, _ = unpack(r)
    dirs = rng.normal(size=(64, 3))
    dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    ds = R * np.array([2.5, 5.0, 10.0, 20.0, 40.0])
    errs = []
    for d in ds:
        p = (c + dirs * d).astype(F)
        far, om = np.zeros(len(p), np.int32), np.zeros(len(p), F)
        hd.hd_far(len(p), p.ctypes.data, r.ctypes.data, 2.0, far.ctypes.data, om.ctypes.data)
        exact = sum(ref_tri(p, rec[t:t + 1]) for t in range(len(rec)))
        dist = np.linalg.norm(p.astype(np.float64) - c, axis=1)
        assert np.array_equal(far.astype(bool), dist > 2.0 * R)
        errs.append(np.abs(om - exact).max())
    slopes = np.diff(np.log2(errs))
    print("expansion errors", errs, "log2 slopes", slopes)
    assert (slopes <= -3.0).all(), (errs, slopes)
    assert errs[-1] < 1e-6
