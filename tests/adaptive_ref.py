"""numpy float32 restatement of the selection rule of b2pt_render_views_adaptive (DESIGN.md 8f), in the operation order
the kernels use (no FMA): the tests replay it on the slices of a checkpointed render and compare the counts."""
import numpy as np

f32 = np.float32


def unconverged(S, Q, c, tau, eps):
    """Bool [...] of sums S and sums of squares Q ([..., 4] float32) of c samples: the variance test fails."""
    cf = f32(c)
    with np.errstate(all="ignore"):
        m = np.where(np.isnan(S[..., :3]), f32(0), S[..., :3]).astype(f32) / cf
        q = np.where(np.isnan(Q[..., :3]), f32(0), Q[..., :3]).astype(f32) / cf
        v = np.fmax(f32(0), q - m * m)
        V = ((f32(0.2126) * v[..., 0] + f32(0.7152) * v[..., 1]) + f32(0.0722) * v[..., 2]) / f32(c - 1)
        L = (f32(0.2126) * m[..., 0] + f32(0.7152) * m[..., 1]) + f32(0.0722) * m[..., 2]
        e = f32(tau) * (L + f32(eps))
        converged = (f32(tau) > 0) & (V <= e * e)  # NaN compares false
    return ~converged


def dilate(flags, W, H, radius):
    """flags [V, H*W] bool -> any flag within Chebyshev distance radius in the same view."""
    f = flags.reshape(-1, H, W)
    out = np.zeros_like(f)
    for dy in range(-radius, radius + 1):
        for dx in range(-radius, radius + 1):
            src = f[:, max(0, dy):H + min(0, dy), max(0, dx):W + min(0, dx)]
            out[:, max(0, -dy):H + min(0, -dy), max(0, -dx):W + min(0, -dx)] |= src
    return out.reshape(flags.shape)


def replay(S, Q, rounds, W, H, tau, eps, radius):
    """Counts [V, H*W] and active [K] of an adaptive render whose pixels' sums at rounds[k] samples are S[k], Q[k]
    ([K, V, H*W, 4], e.g. b2pt_render_views_checkpoints(rounds) with moments)."""
    counts = np.full(S.shape[1:3], rounds[0], np.int32)
    active = [counts.size]
    for k in range(len(rounds) - 1):
        at = counts == rounds[k]
        act = at & dilate(at & unconverged(S[k], Q[k], rounds[k], tau, eps), W, H, radius)
        counts[act] = rounds[k + 1]
        active.append(int(act.sum()))
    return counts, np.array(active, np.int64)
