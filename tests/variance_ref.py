"""Per-pixel variance from sample-range shards and the variance-guided à-trous filter of include/rbrt_gpu.h (rbrt_gpu_render_hdr_variance*,
rbrt_gpu_denoise_variance*, DESIGN.md section 14) restated in numpy float32.

Every numpy float32 operation below is one IEEE operation, correctly rounded, in the order the header writes it, so the results equal the
kernels and the host build of rbrt_b200/csrc/variance.cuh bit for bit (NaN payloads aside).  `moments` and `denoise_variance` work on whole
planes; `moments_scalar` and `denoise_variance_scalar` are the same definitions as plain loops over pixels, and the tests check the pairs
against each other.
"""
import numpy as np

from .denoise_ref import (ALBEDO_FLOOR, CENTRE, H_B3, MAX_LEVELS, _inside, _shift, luminance, same_bits,  # noqa: F401
                          tonemap)

F = np.float32
MAX_SPLITS = 16
DEFAULT_LEVELS = 5
SIGMA_DEPTH = F(0.01)
SIGMA_LUMINANCE = F(4.0)
EPS_LUMINANCE = F(2.0 ** -10)
K3 = (F(0.25), F(0.5), F(0.25))


def resolve(levels=0, sigma_depth=0.0, sigma_luminance=0.0):
    """0 = the default, as rbrt_denoise_opts for the variance-guided filter."""
    return (int(levels) or DEFAULT_LEVELS, F(sigma_depth) if sigma_depth else SIGMA_DEPTH,
            F(sigma_luminance) if sigma_luminance else SIGMA_LUMINANCE)


# ============================================================================== moments of K shard accumulators
def moments(acc, S):
    """acc: [K, H, W, >=3] float32 per-pixel sums of shard k's S/K samples -> (hdr [H,W,3], var [H,W,3]) float32."""
    a = np.asarray(acc, F)[..., :3]
    K = a.shape[0]
    inv_S, inv_n = F(1.0) / F(S), F(1.0) / F(S // K)
    with np.errstate(all="ignore"):
        s = a[0]
        for k in range(1, K):
            s = s + a[k]
        hdr = s * inv_S
        q = np.zeros_like(hdr)
        for k in range(K):
            d = a[k] * inv_n - hdr
            q = q + d * d
        var = q / F(K * (K - 1))
    return hdr, var


def moments_scalar(acc, S):
    a = np.asarray(acc, F)
    K, H, W = a.shape[:3]
    inv_S, inv_n = F(1.0) / F(S), F(1.0) / F(S // K)
    kk = F(K * (K - 1))
    hdr, var = np.zeros((H, W, 3), F), np.zeros((H, W, 3), F)
    with np.errstate(all="ignore"):
        for y in range(H):
            for x in range(W):
                for c in range(3):
                    s = a[0, y, x, c]
                    for k in range(1, K):
                        s = s + a[k, y, x, c]
                    m = s * inv_S
                    q = F(0.0)
                    for k in range(K):
                        d = a[k, y, x, c] * inv_n - m
                        q = q + d * d
                    hdr[y, x, c], var[y, x, c] = m, q / kk
    return hdr, var


# ============================================================================== the variance-guided filter
def _pack(c, v, a, z):
    d = np.where(a > ALBEDO_FLOOR, a, ALBEDO_FLOOR)
    e = c / d
    l = luminance(e[..., 0], e[..., 1], e[..., 2])
    valid = np.isfinite(c).all(-1) & np.isfinite(d).all(-1) & np.isfinite(z) & ((v >= F(0.0)) & np.isfinite(v)).all(-1)
    sd = ((F(0.2126) / d[..., 0]) * np.sqrt(v[..., 0]) + (F(0.7152) / d[..., 1]) * np.sqrt(v[..., 1])) + \
        (F(0.0722) / d[..., 2]) * np.sqrt(v[..., 2])
    return d, e, l, valid, sd * sd


def denoise_variance(hdr, var, albedo, normal, depth, levels=0, sigma_depth=0.0, sigma_luminance=0.0):
    """hdr, var, albedo, normal [H,W,3] and depth [H,W] float32 -> (hdr_out [H,W,3] float32, rgb_out [H,W,3] uint8)."""
    L, sz, sl = resolve(levels, sigma_depth, sigma_luminance)
    c, v, a, n, z = (np.asarray(x, F) for x in (hdr, var, albedo, normal, depth))
    H, W = z.shape
    one = F(1.0)
    with np.errstate(all="ignore"):
        d, e, l, valid, s2 = _pack(c, v, a, z)
        for i in range(L):
            s = 1 << i
            gs, gw = np.zeros((H, W), F), np.zeros((H, W), F)
            for dy in (-1, 0, 1):
                for dx in (-1, 0, 1):
                    ok = _inside(H, W, dy, dx) & _shift(valid, dy, dx)
                    k = K3[dx + 1] * K3[dy + 1]
                    gs = np.where(ok, gs + k * _shift(s2, dy, dx), gs)
                    gw = np.where(ok, gw + k, gw)
            r_z = one / ((sz * z) * F(s))
            r_l = one / (sl * np.sqrt(gs / gw) + EPS_LUMINANCE)
            sw = np.zeros((H, W), F)
            se = np.zeros((H, W, 3), F)
            sv = np.zeros((H, W), F)
            for dy in range(-2, 3):
                for dx in range(-2, 3):
                    oy, ox = dy * s, dx * s
                    ok = _inside(H, W, oy, ox)
                    if dy == 0 and dx == 0:
                        w, eq, vq = np.full((H, W), CENTRE), e, s2
                    else:
                        nq, zq, eq, lq, vq = _shift(n, oy, ox), _shift(z, oy, ox), _shift(e, oy, ox), _shift(l, oy, ox), _shift(s2, oy, ox)
                        ok &= _shift(valid, oy, ox)
                        dot = (n[..., 0] * nq[..., 0] + n[..., 1] * nq[..., 1]) + n[..., 2] * nq[..., 2]
                        wn = np.where(dot > F(0.0), dot, F(0.0))
                        for _ in range(7):
                            wn = wn * wn
                        ok &= wn != F(0.0)
                        xz = np.abs(z - zq) * r_z
                        xl = (l - lq) * r_l
                        dl = one + xl * xl
                        w = (H_B3[dx + 2] * H_B3[dy + 2] * wn) / ((one + xz * xz) * (dl * dl))
                    sw = np.where(ok, sw + w, sw)
                    se = np.where(ok[..., None], se + w[..., None] * eq, se)
                    sv = np.where(ok, sv + (w * w) * vq, sv)
            o = se / sw[..., None]
            e = np.where(valid[..., None], o, e)
            l = np.where(valid, luminance(o[..., 0], o[..., 1], o[..., 2]), l)
            s2 = np.where(valid, sv / (sw * sw), s2)
        out = np.where(valid[..., None], e * d, c)
    return out, tonemap(out)


def denoise_variance_scalar(hdr, var, albedo, normal, depth, levels=0, sigma_depth=0.0, sigma_luminance=0.0):
    """The same definition as a loop over pixels and taps with numpy float32 scalars (slow: for small images)."""
    L, sz, sl = resolve(levels, sigma_depth, sigma_luminance)
    c, v, a, n, z = (np.asarray(x, F) for x in (hdr, var, albedo, normal, depth))
    H, W = z.shape
    one = F(1.0)
    fin = lambda t: bool(np.isfinite(t))
    with np.errstate(all="ignore"):
        d = [[[a[y, x, k] if a[y, x, k] > ALBEDO_FLOOR else ALBEDO_FLOOR for k in range(3)] for x in range(W)] for y in range(H)]
        e = [[[c[y, x, k] / d[y][x][k] for k in range(3)] for x in range(W)] for y in range(H)]
        lum = [[luminance(*e[y][x]) for x in range(W)] for y in range(H)]
        valid = [[all(fin(c[y, x, k]) and fin(d[y][x][k]) and v[y, x, k] >= F(0.0) and fin(v[y, x, k]) for k in range(3)) and fin(z[y, x])
                  for x in range(W)] for y in range(H)]
        sig = [[None] * W for _ in range(H)]
        for y in range(H):
            for x in range(W):
                dd = d[y][x]
                sd = ((F(0.2126) / dd[0]) * np.sqrt(v[y, x, 0]) + (F(0.7152) / dd[1]) * np.sqrt(v[y, x, 1])) + \
                    (F(0.0722) / dd[2]) * np.sqrt(v[y, x, 2])
                sig[y][x] = sd * sd
        for i in range(L):
            s = 1 << i
            ne = [[list(e[y][x]) for x in range(W)] for y in range(H)]
            nl = [[lum[y][x] for x in range(W)] for y in range(H)]
            ns = [[sig[y][x] for x in range(W)] for y in range(H)]
            for y in range(H):
                for x in range(W):
                    if not valid[y][x]:
                        continue
                    gs, gw = F(0.0), F(0.0)
                    for dy in (-1, 0, 1):
                        for dx in (-1, 0, 1):
                            qy, qx = y + dy, x + dx
                            if 0 <= qy < H and 0 <= qx < W and valid[qy][qx]:
                                k = K3[dx + 1] * K3[dy + 1]
                                gs = gs + k * sig[qy][qx]
                                gw = gw + k
                    zp, lp, np_ = z[y, x], lum[y][x], n[y, x]
                    r_z = one / ((sz * zp) * F(s))
                    r_l = one / (sl * np.sqrt(gs / gw) + EPS_LUMINANCE)
                    sw, sv, s3 = F(0.0), F(0.0), [F(0.0)] * 3
                    for dy in range(-2, 3):
                        for dx in range(-2, 3):
                            qy, qx = y + dy * s, x + dx * s
                            if not (0 <= qy < H and 0 <= qx < W):
                                continue
                            if dy == 0 and dx == 0:
                                w = CENTRE
                            else:
                                if not valid[qy][qx]:
                                    continue
                                nq = n[qy, qx]
                                dot = (np_[0] * nq[0] + np_[1] * nq[1]) + np_[2] * nq[2]
                                wn = dot if dot > F(0.0) else F(0.0)
                                for _ in range(7):
                                    wn = wn * wn
                                if wn == F(0.0):
                                    continue
                                xz = abs(zp - z[qy, qx]) * r_z
                                xl = (lp - lum[qy][qx]) * r_l
                                dl = one + xl * xl
                                w = (H_B3[dx + 2] * H_B3[dy + 2] * wn) / ((one + xz * xz) * (dl * dl))
                            sw = sw + w
                            s3 = [s3[k] + w * e[qy][qx][k] for k in range(3)]
                            sv = sv + (w * w) * sig[qy][qx]
                    ne[y][x] = [s3[k] / sw for k in range(3)]
                    nl[y][x] = luminance(*ne[y][x])
                    ns[y][x] = sv / (sw * sw)
            e, lum, sig = ne, nl, ns
        out = np.array([[[e[y][x][k] * d[y][x][k] if valid[y][x] else c[y, x, k] for k in range(3)] for x in range(W)] for y in range(H)],
                       F).reshape(H, W, 3)
    return out, tonemap(out)
