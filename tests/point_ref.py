"""Nearest-surface queries of include/rbrt_gpu.h (rbrt_gpu_query_nearest_device, DESIGN.md section 17) restated in float32.

Every float32 operation below is one IEEE operation, correctly rounded, in the order rbrt_b200/csrc/point.cuh writes it, so the results equal
the kernel and the host build of point.cuh bit for bit.  The functions take numpy arrays or CUDA torch tensors (`X` = NP or TORCH): the
torch form is the same op sequence, one elementwise kernel per operation, and lets the GPU tests brute-force C3's 1.31 M triangles.

  closest_on_triangle  the routine of one triangle record (Ericson's regions, degenerate records as their segments), over arrays;
  closest_on_sphere    the routine of one sphere;
  candidates           a scene's candidates in scene order (elements, then each mesh's tested triangles by original index);
  nearest              the brute-force query: the least (d2, scene order) of the accepted candidates, and every output plane.
"""
import numpy as np

from . import motion_ref as M

F = np.float32
FLT_MAX = 3.40282347e+38
HIT_NONE, HIT_SPHERE, HIT_MESH, HIT_TRIANGLE = -1, 0, 1, 2


class NP:
    where, sqrt, abs = staticmethod(np.where), staticmethod(np.sqrt), staticmethod(np.abs)


class TORCH:
    @staticmethod
    def where(c, a, b):
        import torch
        return torch.where(c, a, b)

    @staticmethod
    def sqrt(a):
        import torch
        return torch.sqrt(a)

    @staticmethod
    def abs(a):
        import torch
        return torch.abs(a)


def dot(a, b):
    return (a[0] * b[0] + a[1] * b[1]) + a[2] * b[2]


def cross(a, b):
    return [a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]]


def sub(a, b):
    return [a[k] - b[k] for k in range(3)]


def d2_of(p, q):
    w = sub(p, q)
    return dot(w, w)


def _sel(X, c, a, b):
    return [X.where(c, a[k], b[k]) for k in range(3)]


def _zero(X, like):
    if X is TORCH:
        import torch
        return torch.zeros_like(like)
    return np.zeros(np.shape(like), F)


def _bcast(X, a, like):                                                  # a itself (no arithmetic: -0 stays -0), broadcast to like's shape
    if X is TORCH:
        import torch
        return torch.broadcast_to(a, like.shape)
    return np.broadcast_to(a, np.shape(like))


def _clamp01(X, x):                                                      # x > 0 ? (x < 1 ? x : 1) : 0 (a NaN gives 0)
    return X.where(x > 0.0, X.where(x < 1.0, x, 1.0), 0.0)


def _seg_t(X, ap, e):
    ee = dot(e, e)
    x = X.where(ee > 0.0, dot(ap, e) / ee, 0.0)
    return _clamp01(X, x)


def _pq(v0, e1, e2, u, v):                                               # (v0 + u*e1) + v*e2
    return [(v0[k] + u * e1[k]) + v * e2[k] for k in range(3)]


def _segments(X, p, v0, e1, e2, ap):
    t = _seg_t(X, ap, e1)
    qa = [v0[k] + t * e1[k] for k in range(3)]
    best, bu, bv, q = d2_of(p, qa), t, _zero(X, t), qa
    t = _seg_t(X, ap, e2)
    qa = [v0[k] + t * e2[k] for k in range(3)]
    d = d2_of(p, qa)
    c = d < best
    best, bu, bv, q = X.where(c, d, best), X.where(c, 0.0, bu), X.where(c, t, bv), _sel(X, c, qa, q)
    bc, bp = sub(e2, e1), sub(ap, e1)
    t = _seg_t(X, bp, bc)
    w1 = 1.0 - t
    qa = _pq(v0, e1, e2, w1, t)
    d = d2_of(p, qa)
    c = d < best
    return X.where(c, d, best), X.where(c, w1, bu), X.where(c, t, bv), _sel(X, c, qa, q)


def closest_on_triangle(p, v0, e1, e2, X=NP):
    """p, v0, e1, e2: 3-lists of broadcastable float32 arrays (components).  Returns (d2, q 3-list, u, v)."""
    with np.errstate(all="ignore"):
        ap = sub(p, v0)
        n = cross(e1, e2)
        deg = (n[0] == 0.0) & (n[1] == 0.0) & (n[2] == 0.0)
        d1, d2 = dot(e1, ap), dot(e2, ap)
        bp = sub(ap, e1)
        d3, d4 = dot(e1, bp), dot(e2, bp)
        vc = d1 * d4 - d3 * d2
        cp = sub(ap, e2)
        d5, d6 = dot(e1, cp), dot(e2, cp)
        vb = d5 * d2 - d1 * d6
        va = d3 * d6 - d5 * d4
        x, y = d4 - d3, d5 - d6
        s_ab, s_ac, s_bc = d1 - d3, d2 - d6, x + y
        u_ab = X.where(s_ab > 0.0, d1 / s_ab, 0.0)
        v_ac = X.where(s_ac > 0.0, d2 / s_ac, 0.0)
        w_bc = X.where(s_bc > 0.0, x / s_bc, 0.0)
        s = (va + vb) + vc
        u_f, v_f = vb / s, vc / s
        regions = [deg,
                   (d1 <= 0.0) & (d2 <= 0.0),                                          # a
                   (d3 >= 0.0) & (d4 <= d3),                                           # b
                   (vc <= 0.0) & (d1 >= 0.0) & (d3 <= 0.0),                            # ab
                   (d6 >= 0.0) & (d5 <= d6),                                           # c
                   (vb <= 0.0) & (d2 >= 0.0) & (d6 <= 0.0),                            # ac
                   (va <= 0.0) & (x >= 0.0) & (y >= 0.0),                              # bc
                   (va >= 0.0) & (vb >= 0.0) & (vc >= 0.0) & (s > 0.0)]                # face
        zero = _zero(X, d1)
        one = zero + 1.0
        sd, su, sv, sq = _segments(X, p, v0, e1, e2, ap)
        w1 = 1.0 - w_bc
        cand = [(su, sv, sq),
                (zero, zero, [_bcast(X, v0[k], d1) for k in range(3)]),
                (one, zero, [v0[k] + e1[k] for k in range(3)]),
                (u_ab, zero, [v0[k] + u_ab * e1[k] for k in range(3)]),
                (zero, one, [v0[k] + e2[k] for k in range(3)]),
                (zero, v_ac, [v0[k] + v_ac * e2[k] for k in range(3)]),
                (w1, w_bc, _pq(v0, e1, e2, w1, w_bc)),
                (u_f, v_f, _pq(v0, e1, e2, u_f, v_f))]
        # the first region that holds decides; none: the segments
        u, v, q = su, sv, sq
        for r in range(len(regions) - 1, -1, -1):
            cu, cv, cq = cand[r]
            u, v, q = X.where(regions[r], cu, u), X.where(regions[r], cv, v), _sel(X, regions[r], cq, q)
        return d2_of(p, q), q, u, v


def closest_on_sphere(p, c, r, X=NP):
    """p, c: 3-lists; r: radius array.  Returns (d2, q)."""
    with np.errstate(all="ignore"):
        ra = X.abs(r)
        w = sub(p, c)
        l = X.sqrt(dot(w, w))
        k = ra / l
        at_c = l == 0.0
        q = [X.where(at_c, c[0] + ra, c[0] + w[0] * k), X.where(at_c, c[1] + 0.0, c[1] + w[1] * k), X.where(at_c, c[2] + 0.0, c[2] + w[2] * k)]
        return d2_of(p, q), q


def accept(d2, max_dist, X=NP):
    with np.errstate(all="ignore"):
        return (d2 <= FLT_MAX) & (X.sqrt(d2) < max_dist)


def unit_normals(rec):
    """[N,3] stored unit normals of records [N,3,4]: norm(cross(e1, e2)), three true divisions (k_prepare, BasicTriangle::new)."""
    e1, e2 = [rec[:, 1, k] for k in range(3)], [rec[:, 2, k] for k in range(3)]
    with np.errstate(all="ignore"):
        n = cross(e1, e2)
        l = np.sqrt(dot(n, n))
        return np.stack([n[k] / l for k in range(3)], 1).astype(F)


def n_tested(n, lanes):
    """N_eff of a mesh of n triangles under the SIMD tail rule (mesh.rs:136-144)."""
    r = n % lanes
    return n if (r == 0 or 2 * r >= lanes) else n - r


def scene_geometry(scene):
    """(elements, meshes) of an rbrt_b200.Scene host mirror, as motion_ref.element_records and the mesh triangle arrays take them."""
    from rbrt_b200.triangle import BasicTriangle
    from rbrt_b200.vec3 import Vec3
    els = []
    for e in scene.elements:
        if isinstance(e, BasicTriangle):
            els.append(("triangle", np.array([[Vec3.from_any(c).x, Vec3.from_any(c).y, Vec3.from_any(c).z] for c in e.corners], F)))
        else:
            c = Vec3.from_any(e.center)
            els.append(("sphere", (c.x, c.y, c.z), e.radius))
    return els, [np.asarray(m.triangles, F).reshape(-1, 3, 3) for m in scene.triangle_meshes]


def candidates(scene=None, elements=None, meshes=None, lanes=None):
    """The scene's candidates in scene order: a dict of float32 records rec [C,3,4] (a sphere: row 0 = {c, r}), is_tri [C], kind [C]
    (HIT_*), elem_idx [C], tri_idx [C] and normal [C,3] (a triangle's stored unit normal; unused for spheres)."""
    if scene is not None:
        elements, meshes = scene_geometry(scene)
        lanes = scene.simd_lanes
    lanes = lanes or 8
    er = M.element_records(elements) if elements else np.zeros((0, 3, 4), F)
    e_tri = np.array([e[0] == "triangle" for e in elements], bool)
    recs, is_tri, kind, elem, tri = [er], [e_tri], [np.where(e_tri, HIT_TRIANGLE, HIT_SPHERE)], [np.arange(len(elements))], [np.zeros(len(elements), np.int64)]
    for mi, t in enumerate(meshes):
        k = n_tested(len(t), lanes)
        recs.append(M.tri_records(t[:k]))
        is_tri.append(np.ones(k, bool))
        kind.append(np.full(k, HIT_MESH))
        elem.append(np.full(k, mi))
        tri.append(np.arange(k))
    rec = np.concatenate(recs, 0).astype(F)
    is_tri = np.concatenate(is_tri)
    nrm = np.zeros((len(rec), 3), F)
    nrm[is_tri] = unit_normals(rec[is_tri])
    return {"rec": rec, "is_tri": is_tri, "kind": np.concatenate(kind).astype(np.int32), "elem_idx": np.concatenate(elem).astype(np.uint32),
            "tri_idx": np.concatenate(tri).astype(np.uint32), "normal": nrm}


def _pair_d2(X, P, rec, is_tri):
    """d2 [n, C] of points P [n,3] against candidate records [C,3,4]."""
    p = [P[:, k:k + 1] for k in range(3)]
    v0, e1, e2 = ([rec[:, i, k][None, :] for k in range(3)] for i in range(3))
    dt = closest_on_triangle(p, v0, e1, e2, X)[0]
    ds = closest_on_sphere(p, v0, rec[:, 0, 3][None, :], X)[0]
    return X.where(is_tri[None, :], dt, ds)


def nearest(cand, points, max_dist=None, X=NP, chunk=None):
    """The brute-force query of points [N,3] against candidates(...): a dict of the output planes (numpy) dist, kind, elem_idx, tri_idx,
    point, normal, uv, and the winner's candidate index `which` (-1: none).  With X = TORCH every pair is evaluated on the GPU."""
    P = np.ascontiguousarray(points, F).reshape(-1, 3)
    n, C = len(P), len(cand["rec"])
    md = np.full(n, np.inf, F) if max_dist is None else np.ascontiguousarray(max_dist, F)
    which = np.full(n, -1, np.int64)
    if C:
        if X is TORCH:
            import torch
            rec_d = torch.from_numpy(cand["rec"]).cuda()
            tri_d = torch.from_numpy(cand["is_tri"]).cuda()
            chunk = chunk or max(1, (1 << 24) // C)
            for s in range(0, n, chunk):
                Pd = torch.from_numpy(P[s:s + chunk]).cuda()
                d2 = _pair_d2(X, Pd, rec_d, tri_d)
                ok = accept(d2, torch.from_numpy(md[s:s + chunk]).cuda()[:, None], X)
                d2 = torch.where(ok, d2, torch.full_like(d2, float("inf")))
                mn = d2.min(1)
                # first minimum: the lowest index among the equal minima
                idx = torch.where(d2 == mn.values[:, None], torch.arange(C, device="cuda")[None, :], C).min(1).values
                idx = torch.where(ok.any(1), idx, -1)
                which[s:s + chunk] = idx.cpu().numpy()
        else:
            chunk = chunk or max(1, (1 << 22) // C)
            for s in range(0, n, chunk):
                d2 = _pair_d2(X, P[s:s + chunk], cand["rec"], cand["is_tri"])
                ok = accept(d2, md[s:s + chunk, None])
                d2 = np.where(ok, d2, np.inf)
                idx = np.argmin(d2, 1)                                   # the first minimum
                which[s:s + chunk] = np.where(ok.any(1), idx, -1)
    return planes(cand, P, which)


def planes(cand, P, which):
    """The output planes of the winners `which` [N] (candidate index, -1 none) of points P."""
    n = len(P)
    out = {"dist": np.full(n, np.inf, F), "kind": np.full(n, HIT_NONE, np.int32), "elem_idx": np.zeros(n, np.uint32),
           "tri_idx": np.zeros(n, np.uint32), "point": np.zeros((n, 3), F), "normal": np.zeros((n, 3), F), "uv": np.zeros((n, 2), F),
           "which": which}
    h = which >= 0
    if h.any():
        w = which[h]
        rec, tri = cand["rec"][w], cand["is_tri"][w]
        p = [P[h, k] for k in range(3)]
        v0, e1, e2 = ([rec[:, i, k] for k in range(3)] for i in range(3))
        dt, qt, ut, vt = closest_on_triangle(p, v0, e1, e2)
        ds, qs = closest_on_sphere(p, v0, rec[:, 0, 3])
        d2 = np.where(tri, dt, ds)
        q = np.stack([np.where(tri, qt[k], qs[k]) for k in range(3)], 1).astype(F)
        with np.errstate(all="ignore"):
            out["dist"][h] = np.sqrt(d2)
            out["point"][h] = q
            out["uv"][h] = np.stack([np.where(tri, ut, F(0)), np.where(tri, vt, F(0))], 1)
            sn = np.stack([q[:, k] - v0[k] for k in range(3)], 1)           # a sphere's normal: q - c, un-normalised
            out["normal"][h] = np.where(tri[:, None], cand["normal"][w], sn)
        out["kind"][h] = cand["kind"][w]
        out["elem_idx"][h] = cand["elem_idx"][w]
        out["tri_idx"][h] = np.where(cand["kind"][w] == HIT_MESH, cand["tri_idx"][w], 0)
    return out
