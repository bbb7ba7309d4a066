"""Generalized winding numbers of include/rbrt_gpu.h (rbrt_gpu_query_winding_device, DESIGN.md section 18) restated in float64.

The candidates are tests/point_ref.candidates (every element and every tested mesh triangle, as the scene stores them).  A triangle's term is
the exact solid angle of its stored record {v0, v0 + e1, v0 + e2} in float64; a sphere's is the rule of the header, whose comparison of
d2 and r2 is float32 (as the kernel decides it).  The functions take numpy arrays or, with X = TORCH, CUDA float64 tensors (the same
code), which lets the GPU tests brute-force C3's 1.31 M triangles.

  omega         the solid angle of triangle records seen from points, float64;
  sphere_halves the sphere rule in halves of a full turn (2 inside, 1 on the surface, 0 outside or r = 0);
  winding       the exact sum over a scene's candidates, / 4 pi: w64 per point (NaN for a point with a NaN coordinate);
  moments       the moments of a set of triangles (c, R, N, T) computed directly, and expand: their far-field expansion.
"""
import numpy as np

F = np.float32
FOUR_PI = 4.0 * np.pi


class NP:
    where, sqrt, arctan2, isfinite = staticmethod(np.where), staticmethod(np.sqrt), staticmethod(np.arctan2), staticmethod(np.isfinite)


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
    def arctan2(a, b):
        import torch
        return torch.atan2(a, b)

    @staticmethod
    def isfinite(a):
        import torch
        return torch.isfinite(a)


def _dot(a, b):
    return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]


def _cross(a, b):
    return [a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]]


def omega(p, v0, e1, e2, X=NP):
    """Solid angles (float64) of the triangles {v0, v0 + e1, v0 + e2} seen from p: 3-lists of broadcastable float64 arrays.  det exactly
    0, a non-finite corner vector (an inf or NaN point or vertex) and a non-finite result give 0, as the kernel's rule."""
    with np.errstate(all="ignore"):
        a = [v0[k] - p[k] for k in range(3)]
        b = [a[k] + e1[k] for k in range(3)]
        c = [a[k] + e2[k] for k in range(3)]
        det = _dot(a, _cross(b, c))
        la, lb, lc = (X.sqrt(_dot(x, x)) for x in (a, b, c))
        den = la * lb * lc + _dot(a, b) * lc + _dot(a, c) * lb + _dot(b, c) * la
        om = 2.0 * X.arctan2(det, den)
        fin = X.isfinite(a[0]) & X.isfinite(a[1]) & X.isfinite(a[2]) & X.isfinite(b[0]) & X.isfinite(b[1]) & X.isfinite(b[2])
        fin = fin & X.isfinite(c[0]) & X.isfinite(c[1]) & X.isfinite(c[2])
        return X.where((det != 0) & fin & X.isfinite(om), om, 0.0)


def sphere_halves(p, c, r):
    """The sphere rule (numpy float32, as the kernel computes it): 2 when d2 < r2, 1 when equal, 0 otherwise or for r = 0."""
    with np.errstate(all="ignore"):
        p, c, r = np.asarray(p, F), np.asarray(c, F), np.asarray(r, F)
        d = [p[..., k] - c[..., k] for k in range(3)]
        d2 = (d[0] * d[0] + d[1] * d[1]) + d[2] * d[2]
        r2 = r * r
        return np.where(r == 0, 0, np.where(d2 < r2, 2, np.where(d2 == r2, 1, 0)))


def winding(cand, points, X=NP, chunk=None):
    """w64 [N] (numpy float64) of points [N,3] against point_ref.candidates(...): the exact sum of every candidate's term / 4 pi."""
    Pn = np.ascontiguousarray(points, F).reshape(-1, 3)
    n = len(Pn)
    rec, tri = cand["rec"], cand["is_tri"]
    total = np.zeros(n, np.float64)
    trec = rec[tri]
    if (~tri).any():                                                     # spheres, in float32 as the kernel decides them
        s = rec[~tri][:, 0, :]
        h = sphere_halves(Pn[:, None, :], s[None, :, :3], s[None, :, 3])
        total += 2.0 * np.pi * h.sum(1)
    if len(trec):
        C = len(trec)
        if X is TORCH:
            import torch
            r = torch.from_numpy(trec.astype(np.float64)).cuda()
            v0, e1, e2 = ([r[:, i, k][None, :] for k in range(3)] for i in range(3))
            chunk = chunk or max(1, (1 << 25) // C)
            for s in range(0, n, chunk):
                Pd = torch.from_numpy(Pn[s:s + chunk].astype(np.float64)).cuda()
                om = omega([Pd[:, k:k + 1] for k in range(3)], v0, e1, e2, X)
                total[s:s + chunk] += om.sum(1).cpu().numpy()
        else:
            r = trec.astype(np.float64)
            v0, e1, e2 = ([r[:, i, k][None, :] for k in range(3)] for i in range(3))
            chunk = chunk or max(1, (1 << 22) // C)
            for s in range(0, n, chunk):
                Pd = Pn[s:s + chunk].astype(np.float64)
                total[s:s + chunk] += omega([Pd[:, k:k + 1] for k in range(3)], v0, e1, e2).sum(1)
    w = total / FOUR_PI
    w[np.isnan(Pn).any(1)] = np.nan
    return w


def moments(rec):
    """Direct float64 moments of triangle records [M,3,4] about their area-weighted centroid: (c [3], R, N [3], T [3,3]); R is the
    largest distance from c to a vertex."""
    r = np.asarray(rec, np.float64)[:, :, :3]
    v0, e1, e2 = r[:, 0], r[:, 1], r[:, 2]
    Nt = 0.5 * np.cross(e1, e2)
    a = np.linalg.norm(Nt, axis=1)
    ct = v0 + (e1 + e2) / 3.0
    c = (a[:, None] * ct).sum(0) / a.sum() if a.sum() > 0 else ct.mean(0)
    T = np.einsum("ti,tj->ij", Nt, ct - c)
    verts = np.concatenate([v0, v0 + e1, v0 + e2], 0)
    return c, np.linalg.norm(verts - c, axis=1).max(), Nt.sum(0), T


def expand(p, c, N, T):
    """The far-field expansion of the solid angle (float64) of moments (c, N, T) seen from points p [K,3]."""
    r = np.asarray(c, np.float64)[None, :] - np.asarray(p, np.float64)
    l = np.linalg.norm(r, axis=1)
    u = r / l[:, None]
    utu = np.einsum("ki,ij,kj->k", u, T, u)
    return (u @ N) / l ** 2 + (np.trace(T) - 3.0 * utu) / l ** 3
