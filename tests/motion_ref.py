"""Per-object motion vectors of include/rbrt_gpu.h (rbrt_gpu_render_motion*, rbrt_gpu_temporal_accumulate_motion*; DESIGN.md section 16)
restated in numpy float32.

Every numpy float32 operation below is one IEEE operation, correctly rounded, in the order the header writes it, so the results equal the
kernels and the host build of rbrt_b200/csrc/motion.cuh bit for bit (NaN payloads aside).  The camera arithmetic (projection, camera
values) is tests/temporal_ref.py's.

  pixel_dirs      step 1: the pixel-centre ray directions of a camera;
  motion          steps 3-5 for hits given as (tri, o, d, t, current record, snapshot record);
  motion_from_hits  the same from rbrt_hit records (Scene.hit) and the geometry a test fed to the scene before and after an update;
  accumulate_motion  the temporal accumulation with the motion variant of step 3.
"""
import numpy as np

from . import temporal_ref as T

F = np.float32


def pixel_dirs(cam):
    """[H,W,3] float32: the direction of each pixel's centre ray (temporal step 3's d)."""
    pos, right, up, center, mmh, mmv, W, H = T.cam_values(cam)
    y, x = np.mgrid[0:H, 0:W]
    col_mm = ((x.astype(F) - F(W // 2) + F(0.5)) - F(0.5)) * mmh
    row_mm = ((y.astype(F) - F(H // 2) + F(0.5)) - F(0.5)) * mmv
    ch, cv = T.MM * col_mm, T.MM * row_mm
    v = [((center[k] + ch * right[k]) - cv * up[k]) - pos[k] for k in range(3)]
    l = np.sqrt(T.dot(v, v))
    return np.stack([v[k] / l for k in range(3)], -1).astype(F)


def camera_rays(cam):
    """[H*W,6] float32 rays (origin, direction) of the motion pass, for Scene.hit."""
    d = pixel_dirs(cam).reshape(-1, 3)
    o = np.broadcast_to(T.cam_values(cam)[0], d.shape)
    return np.ascontiguousarray(np.concatenate([o, d], 1), F)


def _bits(a):
    return np.ascontiguousarray(a, F).view(np.uint32)


def motion(cam, prev, tri, o, d, t, cur, old):
    """Steps 3-5 for N hits: tri [N] bool (a mesh triangle or BasicTriangle; else a sphere), o, d [N,3], t [N], cur / old [N,3,4]
    records (triangle: rows v0, e1, e2, xyz used; sphere: row 0 = {c, r}).  Returns (motion [N,2], prev_dist [N]) float32."""
    tri = np.asarray(tri, bool)
    o, d, t = np.asarray(o, F), np.asarray(d, F), np.asarray(t, F)
    cur, old = np.asarray(cur, F), np.asarray(old, F)
    with np.errstate(all="ignore"):
        P = [o[:, k] + t * d[:, k] for k in range(3)]
        same_tri = (_bits(cur[:, :, :3]) == _bits(old[:, :, :3])).all((1, 2))
        same_sph = (_bits(cur[:, 0, :]) == _bits(old[:, 0, :])).all(1)
        v0, e1, e2 = ([cur[:, i, k] for k in range(3)] for i in range(3))
        w0, w1, w2 = ([old[:, i, k] for k in range(3)] for i in range(3))
        ds = [d[:, k] for k in range(3)]
        h = T.cross(ds, e2)
        f = F(1) / T.dot(e1, h)
        s = [o[:, k] - v0[k] for k in range(3)]
        u = f * T.dot(s, h)
        v = f * T.dot(ds, T.cross(s, e1))
        Pt = [(w0[k] + u * w1[k]) + v * w2[k] for k in range(3)]
        kr = old[:, 0, 3] / cur[:, 0, 3]
        Ps = [old[:, 0, k] + (P[k] - cur[:, 0, k]) * kr for k in range(3)]
        Pp = [np.where(tri, np.where(same_tri, P[k], Pt[k]), np.where(same_sph, P[k], Ps[k])).astype(F) for k in range(3)]
        pos, ppos = T.cam_values(cam)[0], T.cam_values(prev)[0]
        D = [P[k] - pos[k] for k in range(3)]
        Dp = [Pp[k] - ppos[k] for k in range(3)]
        qx, qy, okq = T.project(cam, D)
        px, py, okp = T.project(prev, Dp)
        ok = okq & okp & np.isfinite(qx) & np.isfinite(qy) & np.isfinite(px) & np.isfinite(py)
        m = np.stack([np.where(ok, px - qx, F(np.nan)), np.where(ok, py - qy, F(np.nan))], -1).astype(F)
        pd = np.sqrt(T.dot(Dp, Dp)).astype(F)
    return m, pd


def tri_records(tris):
    """[N,3,4] records v0, e1 = b - a, e2 = c - a of triangles [N,3,3] (as the scene stores them, float32)."""
    tris = np.asarray(tris, F).reshape(-1, 3, 3)
    r = np.zeros((len(tris), 3, 4), F)
    r[:, 0, :3] = tris[:, 0]
    r[:, 1, :3] = tris[:, 1] - tris[:, 0]
    r[:, 2, :3] = tris[:, 2] - tris[:, 0]
    return r


def element_records(elements):
    """[E,3,4] records of Scene.elements given as ("sphere", centre xyz, radius) or ("triangle", corners [3,3])."""
    out = np.zeros((len(elements), 3, 4), F)
    for i, e in enumerate(elements):
        if e[0] == "sphere":
            out[i, 0] = [e[1][0], e[1][1], e[1][2], e[2]]
        else:
            out[i] = tri_records(np.asarray(e[1], F)[None])[0]
    return out


def motion_from_hits(cam, prev, hits, geometry, snapshot):
    """The motion pass from Scene.hit records of camera_rays(cam) ([H*W] HIT_DTYPE).  geometry / snapshot: the scene now and at the
    snapshot, each a dict with "elements" (element_records' input) and "meshes" (a list of triangle arrays [N,3,3] in original order).
    Returns (motion [H,W,2], prev_dist [H,W])."""
    W, H = cam.img_width_pix, cam.img_height_pix
    d = pixel_dirs(cam).reshape(-1, 3)
    o = np.broadcast_to(T.cam_values(cam)[0], d.shape)
    kind = hits["kind"]
    n = len(kind)
    cur = np.zeros((n, 3, 4), F)
    old = np.zeros((n, 3, 4), F)
    ecur, eold = element_records(geometry["elements"]), element_records(snapshot["elements"])
    el = (kind == 0) | (kind == 2)
    cur[el], old[el] = ecur[hits["elem_idx"][el]], eold[hits["elem_idx"][el]]
    for mi, (mc, mo) in enumerate(zip(geometry["meshes"], snapshot["meshes"])):
        sel = (kind == 1) & (hits["elem_idx"] == mi)
        if sel.any():
            cur[sel] = tri_records(np.asarray(mc, F)[hits["tri_idx"][sel]])
            old[sel] = tri_records(np.asarray(mo, F)[hits["tri_idx"][sel]])
    m, pd = motion(cam, prev, kind != 0, o, d, hits["t"], cur, old)
    hit = kind >= 0
    m[~hit] = np.nan
    pd[~hit] = np.inf
    return m.reshape(H, W, 2), pd.reshape(H, W)


def accumulate_motion(cam, hdr, var, aovs, history, motion_plane, prev_dist, alpha_min=T.ALPHA_MIN, sigma_depth=T.SIGMA_DEPTH,
                      normal_min=T.NORMAL_MIN):
    """rbrt_gpu_temporal_accumulate_motion: T.accumulate with step 3 taken along motion_plane [H,W,2] where both components are finite
    (r = prev_dist [H,W]).  Returns (hdr_out, var_out or None, len_out)."""
    am, sz, nm = F(alpha_min), F(sigma_depth), F(normal_min)
    c = np.asarray(hdr, F)
    H, W = c.shape[:2]
    z = np.asarray(aovs["depth"], F)
    v = None if var is None else np.asarray(var, F)
    with np.errstate(all="ignore"):
        valid = np.isfinite(c).all(-1) & np.isfinite(z)
        if v is not None:
            valid &= (np.isfinite(v) & (v >= F(0))).all(-1)
        out = c.copy()
        vout = None if v is None else v.copy()
        lout = np.where(valid, F(1), F(0)).astype(F)
        if history is None:
            return out, vout, lout
        prev = history["cam"]
        yy, xx = np.mgrid[0:H, 0:W].astype(np.int64)
        # step 3, camera reprojection (temporal_ref's)
        X = T.world_point(cam, xx, yy, z)
        ppos = T.cam_values(prev)[0]
        D = [X[k] - ppos[k] for k in range(3)]
        r_cam = np.sqrt(T.dot(D, D))
        if T.same_camera(cam, prev):
            px_cam, py_cam = xx.astype(F), yy.astype(F)
            ok_cam = np.ones((H, W), bool)
        else:
            px_cam, py_cam, ok_cam = T.project(prev, D)
        # step 3 along the motion
        mp = np.asarray(motion_plane, F)
        use = np.isfinite(mp[..., 0]) & np.isfinite(mp[..., 1])
        px = np.where(use, xx.astype(F) + mp[..., 0], px_cam).astype(F)
        py = np.where(use, yy.astype(F) + mp[..., 1], py_cam).astype(F)
        r = np.where(use, np.asarray(prev_dist, F), r_cam).astype(F)
        ok = valid & np.isfinite(r) & np.where(use, True, ok_cam)
        ok &= (px >= F(0)) & (px <= F(W - 1)) & (py >= F(0)) & (py <= F(H - 1))
        fx0 = np.where(ok, np.floor(px), F(0)).astype(F)
        fy0 = np.where(ok, np.floor(py), F(0)).astype(F)
        x0, y0 = fx0.astype(np.int64), fy0.astype(np.int64)
        fx, fy = np.where(ok, px - fx0, F(0)).astype(F), np.where(ok, py - fy0, F(0)).astype(F)
        # steps 4 and 5, as temporal_ref.accumulate
        n = np.asarray(aovs["normal"], F)
        ns = [n[..., k] for k in range(3)]
        ln = np.sqrt(T.dot(ns, ns))
        kp, ep = np.asarray(aovs["hit_kind"]), np.asarray(aovs["elem_idx"])
        ha = history["aovs"]
        hc, hl = np.asarray(history["hdr"], F), np.asarray(history["length"], F)
        hz, hn = np.asarray(ha["depth"], F), np.asarray(ha["normal"], F)
        hk, he = np.asarray(ha["hit_kind"]), np.asarray(ha["elem_idx"])
        hv = None if v is None else np.asarray(history["var"], F)
        tol = sz * r
        gx, gy = F(1) - fx, F(1) - fy
        sw = np.zeros((H, W), F)
        s = np.zeros((H, W, 3), F)
        sv = np.zeros((H, W, 3), F)
        sl = np.zeros((H, W), F)
        for t in range(4):
            qx, qy = x0 + (t & 1), y0 + (t >> 1)
            w = (fx if t & 1 else gx) * (fy if t >> 1 else gy)
            inside = (qx < W) & (qy < H)
            qxc, qyc = np.minimum(qx, W - 1), np.minimum(qy, H - 1)
            lq = hl[qyc, qxc]
            cons = ok & (w != F(0)) & inside & (lq > F(0)) & (hk[qyc, qxc] == kp) & (he[qyc, qxc] == ep)
            cons &= np.abs(hz[qyc, qxc] - r) <= tol
            nq = hn[qyc, qxc]
            nqs = [nq[..., k] for k in range(3)]
            cons &= T.dot(ns, nqs) >= nm * (ln * np.sqrt(T.dot(nqs, nqs)))
            sw = np.where(cons, sw + w, sw)
            s = np.where(cons[..., None], s + w[..., None] * hc[qyc, qxc], s)
            sl = np.where(cons, sl + w * lq, sl)
            if v is not None:
                sv = np.where(cons[..., None], sv + (w * w)[..., None] * hv[qyc, qxc], sv)
        has = ok & (sw >= T.MIN_WEIGHT)
        nh = sl / sw
        a1 = F(1) / (nh + F(1))
        al = np.where(a1 > am, a1, am).astype(F)
        ch = s / sw[..., None]
        out = np.where(has[..., None], ch + al[..., None] * (c - ch), out)
        if v is not None:
            om = F(1) - al
            k1, k2 = om * om, al * al
            vout = np.where(has[..., None], k1[..., None] * (sv / (sw * sw)[..., None]) + k2[..., None] * v, vout)
        lout = np.where(has, nh + F(1), lout).astype(F)
    return out.astype(F), None if vout is None else vout.astype(F), lout
