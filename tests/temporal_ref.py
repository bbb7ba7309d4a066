"""Temporal accumulation of include/rbrt_gpu.h (rbrt_gpu_temporal_accumulate*, DESIGN.md section 15) restated in numpy float32.

Every numpy float32 operation below is one IEEE operation, correctly rounded, in the order the header writes it, so the results equal the
kernel and the host build of rbrt_b200/csrc/temporal.cuh bit for bit (NaN payloads aside).  `accumulate` works on whole planes and
`accumulate_scalar` is the same definition as a plain loop over pixels; the tests check the pair against each other.

Cameras are rbrt_b200.Camera values; planes are [H,W,3] / [H,W] arrays; `aovs` and a history's `aovs` are dicts with depth, normal,
hit_kind and elem_idx.  A history is a dict with cam, hdr, var (with var), length and aovs, as rbrt_b200.temporal_accumulate takes it.
"""
import numpy as np

F = np.float32
ALPHA_MIN, SIGMA_DEPTH, NORMAL_MIN = F(0.1), F(0.02), F(0.9)
MIN_WEIGHT = F(2.0 ** -6)
MM = F(0.001)


def cam_values(cam):
    """The fields the definition reads, as float32: pos, right, up, center (3 each), mm_h, mm_v, and W, H."""
    v3 = lambda v: np.array([v.x, v.y, v.z], F)
    return (v3(cam.position), v3(cam.right), v3(cam.up), v3(cam.img_center_point), F(cam.mm_per_pix_hor), F(cam.mm_per_pix_vert),
            int(cam.img_width_pix), int(cam.img_height_pix))


def same_camera(a, b):
    return bytes(a.to_c()) == bytes(b.to_c())


def dot(a, b):
    return (a[0] * b[0] + a[1] * b[1]) + a[2] * b[2]


def cross(a, b):
    return [a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]]


def world_point(cam, x, y, z):
    """pos + z * d for pixel (x, y) (arrays or scalars), d the pixel centre's camera-ray direction; a list of three components."""
    pos, right, up, center, mmh, mmv, W, H = cam_values(cam)
    col_off = F(x) - F(W // 2) if np.isscalar(x) else x.astype(F) - F(W // 2)
    row_off = F(y) - F(H // 2) if np.isscalar(y) else y.astype(F) - F(H // 2)
    col_mm = ((col_off + F(0.5)) - F(0.5)) * mmh
    row_mm = ((row_off + F(0.5)) - F(0.5)) * mmv
    ch, cv = MM * col_mm, MM * row_mm
    v = [((center[k] + ch * right[k]) - cv * up[k]) - pos[k] for k in range(3)]
    l = np.sqrt(dot(v, v))
    return [pos[k] + z * (v[k] / l) for k in range(3)]


def project(cam, D):
    """(px, py, s > 0) of the point pos + D in camera cam, Cramer's rule in the header's order."""
    pos, right, up, center, mmh, mmv, W, H = cam_values(cam)
    C = [center[k] - pos[k] for k in range(3)]
    ru = cross(right, up)
    det = dot(D, ru)
    s = dot(C, ru) / det
    a = dot(D, cross(up, C)) / det
    b = dot(D, cross(right, C)) / det
    return (a / MM) / mmh + F(W // 2), (b / MM) / mmv + F(H // 2), s > F(0)


def _opts(alpha_min, sigma_depth, normal_min):
    return F(alpha_min), F(sigma_depth), F(normal_min)


def accumulate(cam, hdr, var, aovs, history=None, alpha_min=ALPHA_MIN, sigma_depth=SIGMA_DEPTH, normal_min=NORMAL_MIN):
    """-> (hdr_out [H,W,3], var_out [H,W,3] or None, len_out [H,W]) float32, whole planes."""
    am, sz, nm = _opts(alpha_min, sigma_depth, normal_min)
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
        X = world_point(cam, xx, yy, z)
        ppos = cam_values(prev)[0]
        D = [X[k] - ppos[k] for k in range(3)]
        r = np.sqrt(dot(D, D))
        ok = valid & np.isfinite(r)
        if same_camera(cam, prev):
            x0, y0 = xx, yy
            fx = fy = np.zeros((H, W), F)
        else:
            px, py, s_ok = project(prev, D)
            ok &= s_ok & (px >= F(0)) & (px <= F(W - 1)) & (py >= F(0)) & (py <= F(H - 1))
            fx0 = np.where(ok, np.floor(px), F(0)).astype(F)
            fy0 = np.where(ok, np.floor(py), F(0)).astype(F)
            x0, y0 = fx0.astype(np.int64), fy0.astype(np.int64)
            fx, fy = np.where(ok, px - fx0, F(0)).astype(F), np.where(ok, py - fy0, F(0)).astype(F)
        n = np.asarray(aovs["normal"], F)
        ns = [n[..., k] for k in range(3)]
        ln = np.sqrt(dot(ns, ns))
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
            cons &= dot(ns, nqs) >= nm * (ln * np.sqrt(dot(nqs, nqs)))
            sw = np.where(cons, sw + w, sw)
            s = np.where(cons[..., None], s + w[..., None] * hc[qyc, qxc], s)
            sl = np.where(cons, sl + w * lq, sl)
            if v is not None:
                sv = np.where(cons[..., None], sv + (w * w)[..., None] * hv[qyc, qxc], sv)
        has = ok & (sw >= MIN_WEIGHT)
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


def accumulate_scalar(cam, hdr, var, aovs, history=None, alpha_min=ALPHA_MIN, sigma_depth=SIGMA_DEPTH, normal_min=NORMAL_MIN):
    """The same definition as a loop over pixels in float32 scalars."""
    am, sz, nm = _opts(alpha_min, sigma_depth, normal_min)
    c = np.asarray(hdr, F)
    H, W = c.shape[:2]
    out = c.copy()
    vout = None if var is None else np.asarray(var, F).copy()
    lout = np.zeros((H, W), F)
    fin = lambda a: bool(np.isfinite(a))
    with np.errstate(all="ignore"):
        same = history is not None and same_camera(cam, history["cam"])
        for y in range(H):
            for x in range(W):
                cp = c[y, x]
                z = F(aovs["depth"][y, x])
                vp = None if var is None else np.asarray(var, F)[y, x]
                if not (all(fin(e) for e in cp) and fin(z) and (vp is None or all(fin(e) and e >= F(0) for e in vp))):
                    continue
                lout[y, x] = F(1)
                if history is None:
                    continue
                prev = history["cam"]
                X = world_point(cam, x, y, z)
                ppos = cam_values(prev)[0]
                D = [X[k] - ppos[k] for k in range(3)]
                r = np.sqrt(dot(D, D))
                if not fin(r):
                    continue
                if same:
                    x0, y0, fx, fy = x, y, F(0), F(0)
                else:
                    px, py, s_ok = project(prev, D)
                    if not (s_ok and px >= F(0) and px <= F(W - 1) and py >= F(0) and py <= F(H - 1)):
                        continue
                    fx0, fy0 = np.floor(px), np.floor(py)
                    x0, y0, fx, fy = int(fx0), int(fy0), px - fx0, py - fy0
                ha = history["aovs"]
                n = np.asarray(aovs["normal"], F)[y, x]
                sw, sl = F(0), F(0)
                s = [F(0)] * 3
                sv = [F(0)] * 3
                for t in range(4):
                    qx, qy = x0 + (t & 1), y0 + (t >> 1)
                    w = (fx if t & 1 else F(1) - fx) * (fy if t >> 1 else F(1) - fy)
                    if w == F(0) or qx >= W or qy >= H:
                        continue
                    lq = F(history["length"][qy, qx])
                    if not (lq > F(0)) or ha["hit_kind"][qy, qx] != aovs["hit_kind"][y, x] or ha["elem_idx"][qy, qx] != aovs["elem_idx"][y, x]:
                        continue
                    if not (abs(F(ha["depth"][qy, qx]) - r) <= sz * r):
                        continue
                    nq = np.asarray(ha["normal"], F)[qy, qx]
                    if not (dot(n, nq) >= nm * (np.sqrt(dot(n, n)) * np.sqrt(dot(nq, nq)))):
                        continue
                    cq = np.asarray(history["hdr"], F)[qy, qx]
                    sw = sw + w
                    s = [s[k] + w * cq[k] for k in range(3)]
                    sl = sl + w * lq
                    if var is not None:
                        vq = np.asarray(history["var"], F)[qy, qx]
                        sv = [sv[k] + (w * w) * vq[k] for k in range(3)]
                if not (sw >= MIN_WEIGHT):
                    continue
                nh = sl / sw
                a1 = F(1) / (nh + F(1))
                al = a1 if a1 > am else am
                for k in range(3):
                    ch = s[k] / sw
                    out[y, x, k] = ch + al * (cp[k] - ch)
                    if var is not None:
                        om = F(1) - al
                        vout[y, x, k] = (om * om) * (sv[k] / (sw * sw)) + (al * al) * vp[k]
                lout[y, x] = nh + F(1)
    return out, vout, lout


def same_bits(a, b):
    """Equal bit for bit, any NaN equal to any NaN."""
    a, b = np.ascontiguousarray(a, F), np.ascontiguousarray(b, F)
    if a.shape != b.shape:
        return False
    na, nb = np.isnan(a), np.isnan(b)
    return bool(np.array_equal(na, nb) and np.array_equal(a[~na].view(np.uint32), b[~nb].view(np.uint32)))
