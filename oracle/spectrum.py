"""NumPy oracle of the Doppler line profiles along lines of sight (LOSSpectrum).

TEST INFRASTRUCTURE -- see oracle/__init__.py for who may import this.

The members of spectrum i and their weights are the hits of the reference's compute_iteration
(compute_iteration.py:151-222): ``los_hits`` below is ``imaging.los_iteration`` statement by
statement, returning per line of sight the hit indices and weights that function only sums.
tests/test_spectrum.py pins it to ``imaging.los_iteration`` (hit counts, included masks and
`used` sets equal, radiance bit for bit) and, summed over the columns, to the reference's own
output (tests/golden/los.npz).  A hit's velocity along the boresight b, in km/s,

    v = ((vx*bx + vy*by) + vz*bz) * vscale

is computed elementwise, every operation a float64 op rounded to nearest (no np.dot /
einsum, whose summation order and contraction are unspecified).  Columns: 0 for v < vmin,
1 + searchsorted(edges, v, 'right') - 1 on edges = np.linspace(vmin, vmax, nbins + 1) for
vmin <= v <= vmax (vmax in the last bin, np.histogram's rule), nbins + 1 above vmax.
"""
import numpy as np

from .imaging import packet_weighting


def los_hits(x, y, z, vy, frac, los, *, vrplanet, dphi, outeredge, rp_cm, gtables):
    """Per line of sight (packet indices, weights) of every hit, weight 0 included, for
    quantity == 'radiance': the membership and weighting of ``imaging.los_iteration``
    (reference compute_iteration.py:98-222) in the same operations.  los: (nlos, 6) rows
    x, y, z, xbore, ybore, zbore."""
    from sklearn.neighbors import KDTree
    los = np.asarray(los, dtype=np.float64)
    sx, sy, sz, bx, by, bz = (los[:, k] for k in range(6))
    dist_from_plan = np.sqrt(sx**2 + sy**2 + sz**2)
    ang = np.arccos((-sx * bx - sy * by - sz * bz) / dist_from_plan)
    asize_plan = np.arcsin(1. / dist_from_plan)
    dist_from_plan = dist_from_plan.copy()
    dist_from_plan[ang > asize_plan] = 1e30

    pts = np.stack([x, y, z], axis=1)
    radvel_sun = vy + vrplanet
    tree = KDTree(pts)
    hits = []
    for i in range(los.shape[0]):
        x_sc = los[i, 0:3].astype(float)
        bore = los[i, 3:6].astype(float)
        b = 2 * np.sum(x_sc * bore)
        c = np.linalg.norm(x_sc)**2 - outeredge**2
        dd = (-b + np.sqrt(b**2 - 4 * 1 * c)) / 2
        t = [np.sin(dphi)]
        while t[-1] < dd:
            t.append(t[-1] + t[-1] * np.sin(dphi))
        t = np.array(t)
        xbore = x_sc[np.newaxis, :] + bore[np.newaxis, :] * t[:, np.newaxis]
        wid = t * np.sin(dphi * 2)
        ind = np.concatenate(tree.query_radius(xbore, wid))
        ilocs = np.unique(ind).astype(int)

        rel = pts[ilocs] - x_sc[np.newaxis, :]
        dist_sc = np.linalg.norm(rel, axis=1)
        losrad = np.sum(rel * bore[np.newaxis, :], axis=1)
        cosang = np.sum(rel * bore[np.newaxis, :], axis=1) / dist_sc
        cosang[cosang > 1] = 1
        angp = np.arccos(cosang)
        inview = (losrad < dist_from_plan[i]) & (angp <= dphi)
        if np.any(inview):
            sel = ilocs[inview]
            d_in = dist_sc[inview]
            l_in = losrad[inview]
            w = packet_weighting('radiance', frac[sel], radvel_sun[sel], gtables)
            apix = np.pi * (d_in * np.sin(dphi))**2 * rp_cm**2
            wtemp = w / apix
            hit = x_sc[np.newaxis, :] + bore[np.newaxis, :] * l_in[:, np.newaxis]
            rhohit = np.linalg.norm(hit[:, [0, 2]], axis=1)
            wtemp = wtemp * ((rhohit > 1) | (hit[:, 1] < 0))
            hits.append((sel, wtemp))
        else:
            hits.append((np.zeros(0, dtype=int), np.zeros(0)))
    return hits


def doppler(vx, vy, vz, bx, by, bz, vscale):
    """Velocity along the boresight [km/s], NumPy's elementwise order."""
    return ((vx * bx + vy * by) + vz * bz) * vscale


def columns(v, vmin, vmax, nbins):
    """Spectrum column (0 .. nbins + 1) of every velocity."""
    v = np.asarray(v, dtype=np.float64)
    edges = np.linspace(vmin, vmax, nbins + 1)
    k = np.minimum(np.searchsorted(edges, v, 'right') - 1, nbins - 1)
    return np.where(v < vmin, 0, np.where(v <= vmax, k + 1, nbins + 1))


def los_spectrum(vx, vy, vz, los, hits, vmin, vmax, nbins, vscale):
    """(spectrum, counts), each (nlos, nbins + 2): per line of sight the sum of the hits'
    weights and their number per column.  ``hits`` as ``los_hits`` returns them;
    ``los`` (nlos, 6) rows x, y, z, xbore, ybore, zbore."""
    los = np.asarray(los, dtype=np.float64)
    nlos = los.shape[0]
    spec = np.zeros((nlos, nbins + 2))
    cnt = np.zeros((nlos, nbins + 2), dtype=np.int64)
    for i, (sel, w) in enumerate(hits):
        if len(sel) == 0:
            continue
        v = doppler(vx[sel], vy[sel], vz[sel], los[i, 3], los[i, 4], los[i, 5], vscale)
        c = columns(v, vmin, vmax, nbins)
        np.add.at(spec[i], c, w)
        cnt[i] = np.bincount(c, minlength=nbins + 2)
    return spec, cnt
