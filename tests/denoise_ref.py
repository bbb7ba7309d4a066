"""The guided à-trous denoiser of include/rbrt_gpu.h (rbrt_gpu_denoise*, DESIGN.md section 13) restated in numpy float32.

Every numpy float32 operation below is one IEEE operation, correctly rounded, in the order the header writes it, so the result equals the
kernels and the host build of rbrt_b200/csrc/denoise.cuh bit for bit (NaN payloads aside).  `denoise` works on whole planes, one shifted
copy per tap; `denoise_scalar` is the same definition as a plain loop over pixels and taps, and the tests check the two against each other.
"""
import numpy as np

F = np.float32
DEFAULT_LEVELS = 4
MAX_LEVELS = 8
SIGMA_DEPTH = F(0.01)
SIGMA_LUMINANCE = F(0.25)
EPS_LUMINANCE = F(2.0 ** -7)
ALBEDO_FLOOR = F(2.0 ** -10)
H_B3 = (F(1 / 16), F(0.25), F(0.375), F(0.25), F(1 / 16))
CENTRE = F(9 / 64)


def resolve(levels=0, sigma_depth=0.0, sigma_luminance=0.0):
    """0 = the default, as rbrt_denoise_opts."""
    return (int(levels) or DEFAULT_LEVELS, F(sigma_depth) if sigma_depth else SIGMA_DEPTH,
            F(sigma_luminance) if sigma_luminance else SIGMA_LUMINANCE)


def luminance(r, g, b):
    return (F(0.2126) * r + F(0.7152) * g) + F(0.0722) * b


def tonemap(c):
    """(sqrt(c) * 256) as u8, saturating, NaN -> 0: k_finalize's (lib.rs:116-122)."""
    with np.errstate(all="ignore"):
        v = np.sqrt(np.asarray(c, F)) * F(256.0)
        t = np.where(v >= F(255.0), F(255.0), np.where(v > F(0.0), v, F(0.0)))   # NaN fails both compares -> 0
    return np.trunc(t).astype(np.uint8)


def _shift(a, oy, ox):
    """a[y + oy, x + ox] where that is inside the image (anything elsewhere: the caller masks it)."""
    H, W = a.shape[:2]
    out = np.zeros_like(a)
    if abs(oy) >= H or abs(ox) >= W:
        return out
    ys, yd = slice(max(0, oy), min(H, H + oy)), slice(max(0, -oy), min(H, H - oy))
    xs, xd = slice(max(0, ox), min(W, W + ox)), slice(max(0, -ox), min(W, W - ox))
    out[yd, xd] = a[ys, xs]
    return out


def _inside(H, W, oy, ox):
    y = np.arange(H)[:, None] + oy
    x = np.arange(W)[None, :] + ox
    return (y >= 0) & (y < H) & (x >= 0) & (x < W)


def denoise(hdr, albedo, normal, depth, levels=0, sigma_depth=0.0, sigma_luminance=0.0):
    """hdr, albedo, normal [H,W,3] and depth [H,W] float32 -> (hdr_out [H,W,3] float32, rgb_out [H,W,3] uint8)."""
    L, sz, sl = resolve(levels, sigma_depth, sigma_luminance)
    c, a, n, z = (np.asarray(v, F) for v in (hdr, albedo, normal, depth))
    H, W = z.shape
    with np.errstate(all="ignore"):
        d = np.where(a > ALBEDO_FLOOR, a, ALBEDO_FLOOR)
        e = c / d
        l = luminance(e[..., 0], e[..., 1], e[..., 2])
        valid = np.isfinite(c).all(-1) & np.isfinite(d).all(-1) & np.isfinite(z)
        for i in range(L):
            s = 1 << i
            r_z = F(1.0) / ((sz * z) * F(s))
            r_l = F(1.0) / (sl * l + EPS_LUMINANCE)
            sw = np.zeros((H, W), F)
            se = np.zeros((H, W, 3), F)
            for dy in range(-2, 3):
                for dx in range(-2, 3):
                    oy, ox = dy * s, dx * s
                    ok = _inside(H, W, oy, ox)
                    if dy == 0 and dx == 0:
                        w, eq = np.full((H, W), CENTRE), e
                    else:
                        nq, zq, eq, lq = _shift(n, oy, ox), _shift(z, oy, ox), _shift(e, oy, ox), _shift(l, oy, ox)
                        ok &= _shift(valid, oy, ox)
                        dot = (n[..., 0] * nq[..., 0] + n[..., 1] * nq[..., 1]) + n[..., 2] * nq[..., 2]
                        wn = np.where(dot > F(0.0), dot, F(0.0))
                        for _ in range(7):
                            wn = wn * wn
                        ok &= wn != F(0.0)
                        xz = np.abs(z - zq) * r_z
                        xl = (l - lq) * r_l
                        w = (H_B3[dx + 2] * H_B3[dy + 2] * wn) / ((F(1.0) + xz * xz) * (F(1.0) + xl * xl))
                    sw = np.where(ok, sw + w, sw)
                    se = np.where(ok[..., None], se + w[..., None] * eq, se)
            o = se / sw[..., None]
            e = np.where(valid[..., None], o, e)
            l = np.where(valid, luminance(o[..., 0], o[..., 1], o[..., 2]), l)
        out = np.where(valid[..., None], e * d, c)
    return out, tonemap(out)


def denoise_scalar(hdr, albedo, normal, depth, levels=0, sigma_depth=0.0, sigma_luminance=0.0):
    """The same definition as a loop over pixels and taps with numpy float32 scalars (slow: for small images)."""
    L, sz, sl = resolve(levels, sigma_depth, sigma_luminance)
    c, a, n, z = (np.asarray(v, F) for v in (hdr, albedo, normal, depth))
    H, W = z.shape
    one = F(1.0)
    with np.errstate(all="ignore"):
        d = [[[a[y, x, k] if a[y, x, k] > ALBEDO_FLOOR else ALBEDO_FLOOR for k in range(3)] for x in range(W)] for y in range(H)]
        e = [[[c[y, x, k] / d[y][x][k] for k in range(3)] for x in range(W)] for y in range(H)]
        lum = [[luminance(*e[y][x]) for x in range(W)] for y in range(H)]
        fin = lambda v: bool(np.isfinite(v))
        valid = [[all(fin(c[y, x, k]) and fin(d[y][x][k]) for k in range(3)) and fin(z[y, x]) for x in range(W)] for y in range(H)]
        for i in range(L):
            s = 1 << i
            ne = [[list(e[y][x]) for x in range(W)] for y in range(H)]
            nl = [[lum[y][x] for x in range(W)] for y in range(H)]
            for y in range(H):
                for x in range(W):
                    if not valid[y][x]:
                        continue
                    zp, lp, np_ = z[y, x], lum[y][x], n[y, x]
                    r_z = one / ((sz * zp) * F(s))
                    r_l = one / (sl * lp + EPS_LUMINANCE)
                    sw, s3 = F(0.0), [F(0.0)] * 3
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
                                w = (H_B3[dx + 2] * H_B3[dy + 2] * wn) / ((one + xz * xz) * (one + xl * xl))
                            sw = sw + w
                            s3 = [s3[k] + w * e[qy][qx][k] for k in range(3)]
                    ne[y][x] = [s3[k] / sw for k in range(3)]
                    nl[y][x] = luminance(*ne[y][x])
            e, lum = ne, nl
        out = np.array([[[e[y][x][k] * d[y][x][k] if valid[y][x] else c[y, x, k] for k in range(3)] for x in range(W)] for y in range(H)],
                       F).reshape(H, W, 3)
    return out, tonemap(out)


def same_bits(a, b):
    """Bit-identical float32 arrays, any NaN equal to any NaN."""
    a, b = np.asarray(a, F), np.asarray(b, F)
    nan = np.isnan(a) & np.isnan(b)
    return a.shape == b.shape and bool(((a.view(np.uint32) == b.view(np.uint32)) | nan).all())
