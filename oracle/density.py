"""NumPy oracle of the number density at sample points (ModelDensity, K7).

A saved row (float32 x, y, z widened to float64) is a member of the ball (p, r) when
    d2 = (dx*dx + dy*dy) + dz*dz <= r*r,    dx = x - p_x, ...
every operation a float64 op rounded to nearest (NumPy's order, no FMA).  Per ball:
S1 = sum frac, S2 = sum frac**2, count = members.

Two candidate generators give the same members: a cKDTree ball query with the radius
inflated by 1e-9 (it must not miss a row whose rounded d2 just makes it), and brute force
over all rows in chunks (small cases).
"""
import numpy as np


def _as_rows(X):
    X = np.asarray(X)
    return X.astype(np.float32).astype(np.float64)


def member_mask(P, p, r):
    """Exact rule for rows P (n, 3) float64 (float32 values) against one ball."""
    d = P - np.asarray(p, dtype=np.float64)
    d2 = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
    return d2 <= np.float64(r) * np.float64(r)


def ball_sums_kdtree(X, frac, points, radius, chunk=256):
    """(S1, S2, count) per point; candidates from scipy's cKDTree."""
    from scipy.spatial import cKDTree
    P = _as_rows(X)
    f = np.asarray(frac, dtype=np.float32).astype(np.float64)
    pts = np.asarray(points, dtype=np.float64).reshape(-1, 3)
    rad = np.broadcast_to(np.asarray(radius, dtype=np.float64), (len(pts),))
    s1, s2 = np.zeros(len(pts)), np.zeros(len(pts))
    cnt = np.zeros(len(pts), dtype=np.int64)
    if len(P) == 0 or len(pts) == 0:
        return s1, s2, cnt
    tree = cKDTree(P)
    for c0 in range(0, len(pts), chunk):
        sl = slice(c0, c0 + chunk)
        cand = tree.query_ball_point(pts[sl], rad[sl] * (1 + 1e-9), return_sorted=False)
        for k, idx in enumerate(cand):
            i = c0 + k
            idx = np.asarray(idx, dtype=np.int64)
            m = idx[member_mask(P[idx], pts[i], rad[i])]
            fm = f[m]
            s1[i], s2[i], cnt[i] = fm.sum(), (fm * fm).sum(), len(m)
    return s1, s2, cnt


def ball_sums_brute(X, frac, points, radius, chunk=1 << 22):
    """Same sums by testing every row against every ball (chunks of rows x points)."""
    P = _as_rows(X)
    f = np.asarray(frac, dtype=np.float32).astype(np.float64)
    pts = np.asarray(points, dtype=np.float64).reshape(-1, 3)
    rad = np.broadcast_to(np.asarray(radius, dtype=np.float64), (len(pts),))
    s1, s2 = np.zeros(len(pts)), np.zeros(len(pts))
    cnt = np.zeros(len(pts), dtype=np.int64)
    if len(P) == 0 or len(pts) == 0:
        return s1, s2, cnt
    per = max(1, chunk // len(P))
    for c0 in range(0, len(pts), per):
        p = pts[c0:c0 + per]
        d = P[None, :, :] - p[:, None, :]
        d2 = (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]
        m = d2 <= (rad[c0:c0 + per] * rad[c0:c0 + per])[:, None]
        s1[c0:c0 + per] = np.where(m, f[None, :], 0.0).sum(axis=1)
        s2[c0:c0 + per] = np.where(m, (f * f)[None, :], 0.0).sum(axis=1)
        cnt[c0:c0 + per] = m.sum(axis=1)
    return s1, s2, cnt


def lens_volume(d, r):
    """Volume of the ball (centre at distance d from the origin, radius r) outside the unit
    sphere, in units of R_p**3."""
    d = np.asarray(d, dtype=np.float64)
    r = np.asarray(r, dtype=np.float64)
    d, r = np.broadcast_arrays(d, r)
    full = 4.0 / 3.0 * np.pi * r**3
    out = np.empty(d.shape)
    with np.errstate(divide='ignore', invalid='ignore'):
        cap = (np.pi * (r + 1 - d)**2 * (d * d + 2 * d * (r + 1) - 3 * (r - 1)**2) / (12 * d))
    out[...] = np.maximum(full - cap, 0.0)
    out[d >= r + 1] = full[d >= r + 1]
    inside = d + r <= 1
    out[inside] = 0.0
    cover = (d + 1 <= r) & ~inside
    out[cover] = 4.0 / 3.0 * np.pi * (r[cover]**3 - 1)
    return out
