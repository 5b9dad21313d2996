"""Independent numpy restatement of rtiow_denoise (include/rtiow_cuda.h), bit for bit.

Every step is numpy float32 arithmetic, which rounds each +, -, *, / correctly and keeps denormals, in the order the header pins:
demodulation by max(albedo, 2^-8), `levels` a-trous levels of 5x5 taps at step 2^i with Cauchy edge-stopping weights, and
remodulation.  The RGBA8 bytes are the frame epilogue's to_rgba at spp = 1, in float64.  denoise() works on whole sub-images per
tap; denoise_scalar() is the same filter as a plain per-pixel loop over np.float32 scalars, which tests compare it against.
"""
import numpy as np

F = np.float32
H1 = (F(1 / 16), F(1 / 4), F(3 / 8), F(1 / 4), F(1 / 16))
ALBEDO_FLOOR = F(2.0 ** -8)
DEPTH_FLOOR = F(2.0 ** -16)


def _k(sigma):
    """1 / (s s) in float32 (0 for s = +inf)"""
    s = F(sigma)
    return F(1) / (s * s)


def level_ks(sigma_color, sigma_normal, sigma_depth, i):
    """the inverse squared widths of level i: the colour width is sigma_color 2^-i"""
    return _k(F(sigma_color) * F(2.0 ** -i)), _k(sigma_normal), _k(sigma_depth)


def _cauchy(d, k):
    return F(1) / (F(1) + d * k)


def quantise(y):
    """to_rgba<double>(y, alpha, spp = 1) per channel (rt_device.cuh): sqrt in double, clamp to [0, 0.999], x256, truncate"""
    c = np.sqrt(np.asarray(y, np.float64) * 1.0)
    c = np.clip(c, 0.0, 0.999)
    v = 256.0 * c
    return np.where(v >= 255.0, 255, np.floor(v)).astype(np.uint8)


def _rgba(y, alpha):
    h, w = y.shape[:2]
    out = np.empty((h, w, 4), np.uint8)
    out[..., :3] = quantise(y)
    out[..., 3] = alpha
    return out


def denoise(color, albedo, normal, depth, levels, sigma_color, sigma_normal, sigma_depth, alpha=255):
    """-> (out_color float32[H,W,3], out_rgba uint8[H,W,4]); inputs as rtiow_render_aov writes them"""
    color, albedo, normal = (np.asarray(a, F).reshape(np.shape(depth) + (3,)) for a in (color, albedo, normal))
    depth = np.asarray(depth, F)
    H, W = depth.shape
    with np.errstate(over="ignore", under="ignore", divide="ignore", invalid="ignore"):
        a = np.maximum(albedo, ALBEDO_FLOOR)
        x = color / a
        zinf = np.isinf(depth)
        for i in range(levels):
            s = 1 << i
            sf = F(s)
            kc, kn, kz = level_ks(sigma_color, sigma_normal, sigma_depth, i)
            num = np.zeros_like(x)
            den = np.zeros((H, W), F)
            for dy in range(-2, 3):
                for dx in range(-2, 3):
                    oy, ox = dy * s, dx * s
                    y0, y1, x0, x1 = max(0, -oy), min(H, H - oy), max(0, -ox), min(W, W - ox)
                    if y0 >= y1 or x0 >= x1:
                        continue
                    P = (slice(y0, y1), slice(x0, x1))
                    Q = (slice(y0 + oy, y1 + oy), slice(x0 + ox, x1 + ox))
                    d = x[P] - x[Q]
                    dc = d[..., 0] * d[..., 0]
                    dc = dc + d[..., 1] * d[..., 1]
                    dc = dc + d[..., 2] * d[..., 2]
                    d = normal[P] - normal[Q]
                    dn = d[..., 0] * d[..., 0]
                    dn = dn + d[..., 1] * d[..., 1]
                    dn = dn + d[..., 2] * d[..., 2]
                    zp, zq = depth[P], depth[Q]
                    t = (zp - zq) / (sf * np.maximum(np.maximum(zp, zq), DEPTH_FLOOR))
                    wz = _cauchy(t * t, kz)
                    ip, iq = zinf[P], zinf[Q]
                    wz = np.where(ip | iq, np.where(ip & iq, F(1), F(0)), wz).astype(F)
                    h = H1[dy + 2] * H1[dx + 2]
                    w = ((h * _cauchy(dc, kc)) * _cauchy(dn, kn)) * wz
                    num[P] = num[P] + w[..., None] * x[Q]
                    den[P] = den[P] + w
            x = num / den[..., None]
        y = x * a
    return y, _rgba(y, alpha)


def denoise_scalar(color, albedo, normal, depth, levels, sigma_color, sigma_normal, sigma_depth, alpha=255):
    """the same filter as a plain loop over pixels and taps on np.float32 scalars (slow: small images only)"""
    depth = np.asarray(depth, F)
    H, W = depth.shape
    color, albedo, normal = (np.asarray(a, F).reshape(H, W, 3) for a in (color, albedo, normal))
    with np.errstate(over="ignore", under="ignore", divide="ignore", invalid="ignore"):
        a = np.empty((H, W, 3), F)
        x = np.empty((H, W, 3), F)
        for py in range(H):
            for px in range(W):
                for c in range(3):
                    a[py, px, c] = max(albedo[py, px, c], ALBEDO_FLOOR)
                    x[py, px, c] = color[py, px, c] / a[py, px, c]
        for i in range(levels):
            s = 1 << i
            kc, kn, kz = level_ks(sigma_color, sigma_normal, sigma_depth, i)
            nxt = np.empty_like(x)
            for py in range(H):
                for px in range(W):
                    num = [F(0), F(0), F(0)]
                    den = F(0)
                    zp = depth[py, px]
                    for dy in range(-2, 3):
                        qy = py + dy * s
                        if not 0 <= qy < H:
                            continue
                        for dx in range(-2, 3):
                            qx = px + dx * s
                            if not 0 <= qx < W:
                                continue
                            dc = F(0)
                            dn = F(0)
                            for c in range(3):
                                d = x[py, px, c] - x[qy, qx, c]
                                dc = d * d if c == 0 else dc + d * d
                                d = normal[py, px, c] - normal[qy, qx, c]
                                dn = d * d if c == 0 else dn + d * d
                            zq = depth[qy, qx]
                            if np.isinf(zp) or np.isinf(zq):
                                wz = F(1) if (np.isinf(zp) and np.isinf(zq)) else F(0)
                            else:
                                t = (zp - zq) / (F(s) * max(max(zp, zq), DEPTH_FLOOR))
                                wz = _cauchy(t * t, kz)
                            w = ((H1[dy + 2] * H1[dx + 2] * _cauchy(dc, kc)) * _cauchy(dn, kn)) * wz
                            for c in range(3):
                                num[c] = num[c] + w * x[qy, qx, c]
                            den = den + w
                    for c in range(3):
                        nxt[py, px, c] = num[c] / den
            x = nxt
        y = np.empty_like(x)
        for py in range(H):
            for px in range(W):
                for c in range(3):
                    y[py, px, c] = x[py, px, c] * a[py, px, c]
    return y, _rgba(y, alpha)
