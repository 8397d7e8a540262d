"""Restatement of the temporal step of b2pt_denoise_views_temporal (include/b2pt.h, DESIGN.md 8j) in numpy float32.

Every operation is an elementwise float32 + - * / sqrt floor or comparison, each IEEE-rounded and without FMA, in the
order the header fixes, so the result can be compared bit for bit.  The per-pixel inputs come from denoise_ref.prep and
the camera basis from the oracle's camera (as tests/motion_ref.py takes it).  Arrays use the C-ABI layout
[K, nViews, H*W, ch]; the a-trous levels that follow are denoise_ref's."""
import numpy as np

import denoise_ref as R
from oracle import oracle as O

f = np.float32
DEFAULTS = dict(alpha=0.1, min_visible=0.5, normal_tol=0.3, albedo_tol=0.03, depth_tol=0.05)


def centre_directions(row, W, H):
    """raygen's pinhole direction of every pixel at jitter (0.5, 0.5): float32 [H*W, 3]."""
    cam = O.Camera(W, H, pos=row[:3], lookAt=row[3:6], up=tuple(row[6:9]), fov=float(row[9]))
    nlook, dx, dy = cam.basis()
    j, i = np.divmod(np.arange(W * H), W)
    i, j = i.astype(f), j.astype(f)
    sx = (f(2) * (i + f(0.5)) - f(W)) / f(2)
    sy = (f(2) * (j + f(0.5)) - f(H)) / f(2)
    d = [(nlook[c] + dx[c] * sx) + dy[c] * sy for c in range(3)]
    d = [np.where(x == 0, x + f(0.0000001), x).astype(f) for x in d]
    m = np.sqrt((d[0] * d[0] + d[1] * d[1]) + d[2] * d[2])
    return np.stack([x / m for x in d], -1).astype(f)


def step(m, V0, ga, gn, z, M, prev, row, prev_row, W, H, alpha, min_visible, normal_tol, albedo_tol, depth_tol):
    """One view of every slice: (x_bar [K,N,3], V_bar [K,N], n [K,N]) from its prep values (m [K,N,3], V0 [K,N],
    ga [K,N,4], gn [K,N,3], z [K,N]), its motion sums M [K,N,4] and the previous view's state prev = (x_bar, V_bar, n,
    ga, gn, z) or None."""
    K, N = V0.shape
    xb, Vb, n = m.copy(), V0.copy(), np.ones((K, N), f)
    if prev is None or not f(alpha) < f(1):
        return xb, Vb, n
    px, pV, pn, pga, pgn, pz = prev
    Sx, Sy, Svis, Sval = (M[..., c] for c in range(4))
    take = (ga[..., 3] > 0) & (Sval > 0) & (Svis >= f(min_visible) * Sval)
    j, i = np.divmod(np.arange(N), W)
    with np.errstate(divide="ignore", invalid="ignore"):
        u = i.astype(f) + Sx / Sval
        y = j.astype(f) + Sy / Sval
    u0, y0 = np.floor(u), np.floor(y)
    with np.errstate(invalid="ignore"):
        fu, fy = u - u0, y - y0
    d = centre_directions(row, W, H)
    pos, ppos = np.asarray(row[:3], f), np.asarray(prev_row[:3], f)
    e = [(pos[c] + d[:, c] * z) - ppos[c] for c in range(3)]
    dprev = np.sqrt((e[0] * e[0] + e[1] * e[1]) + e[2] * e[2])
    sb, sv, sn = np.zeros((K, N), f), np.zeros((K, N), f), np.zeros((K, N), f)
    sx = np.zeros((K, N, 3), f)
    kk = np.arange(K)[:, None]
    for dx, dy in ((0, 0), (1, 0), (0, 1), (1, 1)):
        cu, cy = u0 + f(dx), y0 + f(dy)
        with np.errstate(invalid="ignore"):
            ok = take & (cu >= 0) & (cu <= f(W - 1)) & (cy >= 0) & (cy <= f(H - 1))
        q = np.where(ok, np.where(ok, cy, 0).astype(np.int64) * W + np.where(ok, cu, 0).astype(np.int64), 0)
        aq, nq, zq = pga[kk, q], pgn[kk, q], pz[kk, q]
        ok &= aq[..., 3] > 0
        with np.errstate(invalid="ignore", over="ignore"):
            if np.isfinite(normal_tol):
                dn = gn - nq
                ok &= (dn[..., 0] * dn[..., 0] + dn[..., 1] * dn[..., 1]) + dn[..., 2] * dn[..., 2] <= \
                    f(normal_tol) * f(normal_tol)
            if np.isfinite(albedo_tol):
                da = ga - aq
                ok &= ((da[..., 0] * da[..., 0] + da[..., 1] * da[..., 1]) + da[..., 2] * da[..., 2]) + \
                    da[..., 3] * da[..., 3] <= f(albedo_tol) * f(albedo_tol)
            if np.isfinite(depth_tol):
                ok &= np.abs(zq - dprev) <= f(depth_tol) * dprev
        b = (fu if dx else f(1) - fu) * (fy if dy else f(1) - fy)
        with np.errstate(invalid="ignore", over="ignore"):
            sb = np.where(ok, sb + b, sb)
            sx = np.where(ok[..., None], sx + b[..., None] * px[kk, q], sx)
            sv = np.where(ok, sv + (b * b) * pV[kk, q], sv)
            sn = np.where(ok, sn + b * pn[kk, q], sn)
    take &= sb > 0
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        nn = sn / sb + f(1)
        a = np.maximum(f(alpha), f(1) / nn)
        r = f(1) - a
        xt = r[..., None] * (sx / sb[..., None]) + a[..., None] * m
        Vt = (r * r) * (sv / (sb * sb)) + (a * a) * V0
    return (np.where(take[..., None], xt, xb).astype(f), np.where(take, Vt, Vb).astype(f),
            np.where(take, nn, n).astype(f))


def temporal(color, moment2, albedo, normal_depth, motion, views, W, H, checkpoints, **params):
    """(x_bar [K,V,N,3], V_bar [K,V,N], n [K,V,N]) float32 for inputs [K,V,H*W,4] and views [V,10]; unset parameters
    take the defaults.  With levels = 0, b2pt_denoise_views_temporal's output is (x_bar, V_bar) bit for bit."""
    p = dict(DEFAULTS)
    p.update(params)
    m, V0, ga, gn, z = R.prep(color, moment2, albedo, normal_depth, checkpoints)
    M = np.asarray(motion, f)
    views = np.asarray(views, f).reshape(-1, 10)
    xs, Vs, ns = [], [], []
    prev = None
    for v in range(m.shape[1]):
        xb, Vb, n = step(m[:, v], V0[:, v], ga[:, v], gn[:, v], z[:, v], M[:, v], prev, views[v],
                         views[max(v - 1, 0)], W, H, **p)
        xs.append(xb), Vs.append(Vb), ns.append(n)
        prev = (xb, Vb, n, ga[:, v], gn[:, v], z[:, v])
    return np.stack(xs, 1), np.stack(Vs, 1), np.stack(ns, 1)


def filtered(color, moment2, albedo, normal_depth, motion, views, W, H, checkpoints, temporal_params=None,
             **denoise_params):
    """float64 (x_L [K,V,N,3], V_L [K,V,N]): the restated temporal result through denoise_ref's a-trous levels."""
    xb, Vb, _ = temporal(color, moment2, albedo, normal_depth, motion, views, W, H, checkpoints,
                         **(temporal_params or {}))
    p = dict(R.DEFAULTS)
    p.update({k: v for k, v in denoise_params.items() if v is not None})
    _, _, ga, gn, z = R.prep(color, moment2, albedo, normal_depth, checkpoints)
    K, nv = Vb.shape[:2]
    img = lambda a: a.astype(np.float64).reshape((K, nv, H, W) + a.shape[3:])
    x, V, ga, gn, z = img(xb), img(Vb), img(ga), img(gn), img(z)
    c = np.asarray(checkpoints).reshape(-1, 1, 1, 1)
    use_lum = np.broadcast_to((moment2 is not None) & (c >= 2), V.shape)
    for lev in range(p["levels"]):
        x, V = R.atrous_level(x, V, ga, gn, z, H, W, 1 << lev, use_lum, p["sigma_lum"], p["sigma_albedo"],
                              p["sigma_normal"], p["sigma_depth"])
    return x.reshape(K, nv, H * W, 3), V.reshape(K, nv, H * W)
