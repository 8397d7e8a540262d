"""Restatement of b2pt_denoise_views (include/b2pt.h, DESIGN.md 8e) in numpy, written from its formulas.

prep() is the per-pixel arithmetic in float32, in the kernel's operation order, so its means and variances can be
compared bit for bit; the filter levels run in float64.  Arrays use the C-ABI layout [K, nViews, H*W, 4]."""
import numpy as np

LUM = np.array([0.2126, 0.7152, 0.0722])
LUM32 = LUM.astype(np.float32)
B3 = np.array([1.0, 4.0, 6.0, 4.0, 1.0]) / 16.0
DEFAULTS = dict(levels=5, sigma_lum=4.0, sigma_albedo=0.1, sigma_normal=0.3, sigma_depth=2.0)


def dn(x):
    return np.where(np.isnan(x), np.float32(0), x).astype(np.float32)


def prep(color, moment2, albedo, normal_depth, checkpoints):
    """float32 (m [K,V,N,3], V0 [K,V,N], g_a [K,V,N,4], g_n [K,V,N,3], z [K,V,N]); V0 is 0 where it does not exist
    (no moment2, or c < 2)."""
    c = np.asarray(checkpoints, np.float32).reshape(-1, 1, 1)
    S = np.asarray(color, np.float32)
    m = np.stack([dn(S[..., ch]) / c for ch in range(3)], -1)
    V0 = np.zeros(S.shape[:-1], np.float32)
    if moment2 is not None:
        Q = np.asarray(moment2, np.float32)
        var = [np.maximum(np.float32(0), dn(Q[..., ch]) / c - m[..., ch] * m[..., ch]) for ch in range(3)]
        with np.errstate(divide="ignore", invalid="ignore"):  # c = 1: no variance, masked below
            v = (LUM32[0] * var[0] + LUM32[1] * var[1] + LUM32[2] * var[2]) / (c - np.float32(1))
        V0 = np.where(c >= 2, v, np.float32(0)).astype(np.float32)
    A, ND = np.asarray(albedo, np.float32), np.asarray(normal_depth, np.float32)
    ga = A / c[..., None]
    gn = ND[..., :3] / c[..., None]
    with np.errstate(divide="ignore", invalid="ignore"):
        z = np.where(A[..., 3] > 0, ND[..., 3] / np.where(A[..., 3] > 0, A[..., 3], 1), np.float32(0))
    return m, V0, ga, gn, z.astype(np.float32)


def atrous_level(x, V, ga, gn, z, H, W, step, use_lum, sigma_lum, sigma_albedo, sigma_normal, sigma_depth):
    """One level on float64 images [..., H, W, ch]; use_lum broadcasts over the leading axes."""
    j, i = np.meshgrid(np.arange(H), np.arange(W), indexing="ij")
    Lp = x @ LUM
    hit = ga[..., 3] > 0
    sw = np.zeros(x.shape[:-1])
    sx = np.zeros(x.shape)
    sv = np.zeros(x.shape[:-1])
    for dy in range(-2, 3):
        for dx in range(-2, 3):
            jj, ii = j + step * dy, i + step * dx
            ok = (jj >= 0) & (jj < H) & (ii >= 0) & (ii < W)
            jc, ic = np.clip(jj, 0, H - 1), np.clip(ii, 0, W - 1)
            xq, Vq, aq, nq, zq = (a[..., jc, ic, :] if a.ndim == x.ndim else a[..., jc, ic] for a in (x, V, ga, gn, z))
            e = np.zeros(sw.shape)
            if np.isfinite(sigma_lum):
                el = np.abs(Lp - xq @ LUM) / (sigma_lum * np.sqrt(V) + 1e-6)
                e = e + np.where(use_lum, el, 0.0)
            if np.isfinite(sigma_albedo):
                e = e + ((ga - aq) ** 2).sum(-1) / sigma_albedo ** 2
            if np.isfinite(sigma_normal):
                e = e + ((gn - nq) ** 2).sum(-1) / sigma_normal ** 2
            if np.isfinite(sigma_depth):
                both = hit & (aq[..., 3] > 0)
                with np.errstate(divide="ignore", invalid="ignore"):
                    ez = np.abs(z - zq) * H / (sigma_depth * z * step * np.hypot(dx, dy) + 1e-6)
                e = e + np.where(both, ez, 0.0)
            w = B3[dx + 2] * B3[dy + 2] * np.exp(-e) * ok
            sw += w
            sx += w[..., None] * xq
            sv += w * w * Vq
    return sx / sw[..., None], sv / (sw * sw)


def denoise(color, moment2, albedo, normal_depth, W, H, checkpoints, levels=None, sigma_lum=None, sigma_albedo=None,
            sigma_normal=None, sigma_depth=None):
    """(x_L [K,V,N,3], V_L [K,V,N]) in float64 for inputs [K,V,H*W,4]; unset parameters take the defaults."""
    p = dict(DEFAULTS)
    for k, v in dict(levels=levels, sigma_lum=sigma_lum, sigma_albedo=sigma_albedo, sigma_normal=sigma_normal,
                     sigma_depth=sigma_depth).items():
        if v is not None:
            p[k] = v
    m, V0, ga, gn, z = prep(color, moment2, albedo, normal_depth, checkpoints)
    K, nv = m.shape[:2]
    img = lambda a: a.astype(np.float64).reshape((K, nv, H, W) + a.shape[3:])
    x, V, ga, gn, z = img(m), img(V0), img(ga), img(gn), img(z)
    c = np.asarray(checkpoints).reshape(-1, 1, 1, 1)
    use_lum = np.broadcast_to((moment2 is not None) & (c >= 2), V.shape)
    for lev in range(p["levels"]):
        x, V = atrous_level(x, V, ga, gn, z, H, W, 1 << lev, use_lum, p["sigma_lum"], p["sigma_albedo"],
                            p["sigma_normal"], p["sigma_depth"])
    return x.reshape(K, nv, H * W, 3), V.reshape(K, nv, H * W)
