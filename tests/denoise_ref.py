"""Float64 NumPy restatement of pt_denoise (csrc/denoise.cu, DESIGN.md "Denoising"), and of pt_render_features'
surface attributes, for the tests.

The guide record (depth, its screen-space gradient, the normal) is rounded exactly as the kernel rounds it: the kernel
computes it with explicitly rounded fp32 operations, so the float32 steps below give the same bits; everything after
that is float64 here and fp32 on the device."""
import numpy as np

LUM = np.array([0.2126, 0.7152, 0.0722])
H5 = np.array([1 / 16, 1 / 4, 3 / 8, 1 / 4, 1 / 16])
DEFAULTS = (4.0, 128.0, 1.0)  # sigma_l, sigma_n, sigma_z


def _grad(z, axis):
    """central differences of fp32 z along `axis`, one-sided at the borders, 0 across an axis of one pixel (fp32)."""
    z = np.moveaxis(z, axis, -1)
    g = np.zeros_like(z)
    n = z.shape[-1]
    if n >= 2:
        g[..., 0] = z[..., 1] - z[..., 0]
        g[..., -1] = z[..., -1] - z[..., -2]
    if n >= 3:
        g[..., 1:-1] = (z[..., 2:] - z[..., :-2]) * np.float32(0.5)
    return np.moveaxis(g, -1, axis)


def guides(feat, W, H):
    """(z, gx, gy, n[H,W,3], has_n) as the kernel's 16-byte guide record decodes them."""
    f = np.asarray(feat, np.float32).reshape(2, H, W, 4)
    f0, f1 = f[0], f[1]
    z = f0[..., 3] / np.maximum(f1[..., 3], np.float32(1.0))
    gx = np.clip(_grad(z, 1), -65504, 65504).astype(np.float16).astype(np.float64)
    gy = np.clip(_grad(z, 0), -65504, 65504).astype(np.float16).astype(np.float64)
    x, y, w = f0[..., 0], f0[..., 1], f0[..., 2]
    ln = np.sqrt((x * x + y * y) + w * w)
    has = (f1[..., 3] > 0) & (ln >= np.float32(1e-6))
    safe = np.where(has, ln, np.float32(1.0))
    q = np.stack([np.clip(np.rint((c / safe) * np.float32(32767.0)), -32767, 32767) for c in (x, y, w)], -1)
    q = np.where(has[..., None], q, 0.0)
    has = np.any(q != 0, -1)
    return z.astype(np.float64), gx, gy, q / 32767.0, has


def albedo(feat, W, H, spp):
    f1 = np.asarray(feat, np.float32).reshape(2, H, W, 4)[1].astype(np.float64)
    return np.maximum(f1[..., :3] / spp, 1e-3)


def _shift(a, dy, dx, fill=0.0):
    """out[j, i] = a[j + dy, i + dx] where that is inside the image, `fill` elsewhere; plus the inside mask."""
    H, W = a.shape[:2]
    out = np.full_like(a, fill)
    ok = np.zeros((H, W), bool)
    ys, xs = slice(max(0, -dy), min(H, H - dy)), slice(max(0, -dx), min(W, W - dx))
    ysrc, xsrc = slice(max(0, dy), min(H, H + dy)), slice(max(0, dx), min(W, W + dx))
    if ys.start < ys.stop and xs.start < xs.stop:
        out[ys, xs] = a[ysrc, xsrc]
        ok[ys, xs] = True
    return out, ok


def denoise(accum, accum_sq, feat, W, H, spp, iterations=5, sigma_l=0.0, sigma_n=0.0, sigma_z=0.0):
    """pt_denoise: float64 [H*W, 3] denoised mean.  accum, accum_sq: [H*W, 4]; feat: [2, H*W, 4] (device layouts)."""
    sl, sn, sz = (s if s > 0 else d for s, d in zip((sigma_l, sigma_n, sigma_z), DEFAULTS))
    N = float(spp)
    s = np.asarray(accum, np.float32).reshape(H, W, 4)[..., :3].astype(np.float64)
    if iterations == 0:
        return (s / N).reshape(-1, 3)
    q = np.asarray(accum_sq, np.float32).reshape(H, W, 4)[..., :3].astype(np.float64)
    v = np.maximum(0.0, q - s * s / N) / (N * max(N - 1.0, 1.0))
    a = albedo(feat, W, H, N)
    c = s / N / a
    var = (v / (a * a)) @ LUM
    z, gx, gy, n, has = guides(feat, W, H)
    for it in range(iterations):
        step = 1 << it
        gv = np.zeros((H, W))
        gw = np.zeros((H, W))
        for dy in (-1, 0, 1):
            for dx in (-1, 0, 1):
                vq, ok = _shift(var, dy, dx)
                w = (0.5 if dx == 0 else 0.25) * (0.5 if dy == 0 else 0.25) * ok
                gv += w * vq
                gw += w
        denom_l = sl * np.sqrt(gv / gw) + 1e-4
        lp = c @ LUM
        sw = np.full((H, W), 9 / 64)
        sc = 9 / 64 * c
        sv = (9 / 64) ** 2 * var
        for dy in range(-2, 3):
            for dx in range(-2, 3):
                if dx == 0 and dy == 0:
                    continue
                cq, ok = _shift(c, dy * step, dx * step)
                vq, _ = _shift(var, dy * step, dx * step)
                zq, _ = _shift(z, dy * step, dx * step)
                nq, _ = _shift(n, dy * step, dx * step)
                hq, _ = _shift(has, dy * step, dx * step, False)
                wz = np.exp(-np.abs(z - zq) / (sz * np.abs(gx * (dx * step) + gy * (dy * step)) + 1e-4))
                wn = np.where(has & hq, np.maximum(0.0, np.sum(n * nq, -1)) ** sn, np.where(~has & ~hq, 1.0, 0.0))
                wl = np.exp(-np.abs(lp - cq @ LUM) / denom_l)
                w = H5[dx + 2] * H5[dy + 2] * wz * wn * wl * ok
                sw += w
                sc += w[..., None] * cq
                sv += w * w * vq
        c = sc / sw[..., None]
        var = sv / (sw * sw)
    return (c * a).reshape(-1, 3)


# ---- surface attributes (pt_render_features) -------------------------------------------------------------------------
def sky(d):
    t = 0.5 * (d[:, 1] + 1.0)
    return np.stack([(1 - t) + t * 0.5, (1 - t) + t * 0.7, (1 - t) + t], -1)


def _lut():
    x = np.arange(256) / 255.0
    return (x ** 2.2).astype(np.float32).astype(np.float64), (x * 2.0 - 1.0).astype(np.float32).astype(np.float64)


def bilinear_texture(texels, areas, tex_flags, tid, u, v):
    """sample_texture (15_module.py:238-258 with its quirks: truncating cast after -0.5, v wraps with the area WIDTH,
    taps outside the atlas weigh 0): (albedo [n,3], normal [n,3], |texel coordinates| [n]) as float64."""
    la, ln = _lut()
    TW, TH = texels.shape[:2]
    ar = np.asarray(areas)[tid]
    w, h = ar[:, 2] - ar[:, 0], ar[:, 3] - ar[:, 1]
    uu = u * w - 0.5
    vv = v * h - 0.5
    l = np.trunc(uu).astype(np.int64)
    b = np.trunc(vv).astype(np.int64)
    r, t = l + 1, b + 1
    taps = [(l, b, (r - uu) * (t - vv)), (l, t, (r - uu) * (vv - b)), (r, b, (uu - l) * (t - vv)), (r, t, (uu - l) * (vv - b))]
    alb = np.zeros((len(u), 3))
    nrm = np.zeros((len(u), 3))
    for x, y, wt in taps:
        X = ar[:, 0] + np.mod(x, w)
        Y = ar[:, 1] + np.mod(y, w)
        ok = (X >= 0) & (Y >= 0) & (X < TW) & (Y < TH)
        tx = texels[np.where(ok, X, 0), np.where(ok, Y, 0)]
        wt = np.where(ok, wt, 0.0)[:, None]
        alb += wt * la[tx[:, :3]]
        nrm += wt * ln[tx[:, 4:7]]
    plain = (np.asarray(tex_flags)[tid] & 1) != 0
    nrm[plain] = (0.0, 0.0, 1.0)
    return alb, nrm, np.abs(uu) + np.abs(vv)


def _normalize(x):
    return x / np.linalg.norm(x, axis=-1, keepdims=True)


def legacy_surfaces(world, prim, point, u, v, want_texel_coords=False):
    """(normal, albedo) of the legacy scatter code at device primitive ids `prim` (spheres first, then the faces in the
    device order of World.device_scene), outward (not yet turned to face the ray); want_texel_coords adds the magnitude
    |u * width - 0.5| + |v * height - 0.5| of each lookup's texel coordinates."""
    texels, areas, flags = world._atlas
    n_sph = len(world.spheres)
    normal = np.zeros((len(prim), 3))
    alb = np.zeros((len(prim), 3))
    tc = np.zeros(len(prim))
    sph = prim < n_sph
    if sph.any():
        cr, _, tex = world.sphere_arrays()
        N = _normalize(point[sph] - cr[prim[sph], :3].astype(np.float64))
        r = np.sqrt(N[:, 0] ** 2 + N[:, 2] ** 2)
        T = np.stack([N[:, 2] / r, np.zeros_like(r), -N[:, 0] / r], -1)
        B = np.stack([N[:, 0] * N[:, 1], -r, N[:, 2] * N[:, 1]], -1)
        phi = np.arcsin(np.clip(N[:, 1], -1, 1))
        theta = np.arctan2(-N[:, 0], -N[:, 2])
        uu = (theta / np.pi + 1.0) * 0.5
        vv = phi / np.pi + 0.5
        a, tn, tc[sph] = bilinear_texture(texels, areas, flags, tex[prim[sph]], 2.0 * uu, vv)
        normal[sph] = _normalize(tn[:, :1] * T + tn[:, 1:2] * B + tn[:, 2:3] * N)
        alb[sph] = a
    tri = ~sph
    if tri.any():
        faces, nrm, uv = [], [], []
        nb = ub = 0
        for m in world.meshes:
            f = np.asarray(m["indices"], np.int64)[m["_visit_order"]].copy()
            f[:, [1, 4, 7]] += nb
            f[:, [2, 5, 8]] += ub
            faces.append(f)
            nrm.append(np.asarray(m["normals"], np.float32).reshape(-1, 3))
            uv.append(np.asarray(m["texture_coords"], np.float32).reshape(-1, 2))
            nb += len(nrm[-1])
            ub += len(uv[-1])
        F = np.concatenate(faces)[prim[tri] - n_sph]
        nrm = np.concatenate(nrm).astype(np.float64)
        uv = np.concatenate(uv).astype(np.float64)
        w1, w2, w3 = (1.0 - u[tri] - v[tri])[:, None], u[tri][:, None], v[tri][:, None]
        normal[tri] = _normalize(w1 * nrm[F[:, 1]] + w2 * nrm[F[:, 4]] + w3 * nrm[F[:, 7]])
        t = w1 * uv[F[:, 2]] + w2 * uv[F[:, 5]] + w3 * uv[F[:, 8]]
        alb[tri], _, tc[tri] = bilinear_texture(texels, areas, flags, F[:, 9], t[:, 0], t[:, 1])
    return (normal, alb, tc) if want_texel_coords else (normal, alb)
