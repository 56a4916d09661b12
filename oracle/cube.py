"""NumPy oracle of the Doppler-resolved image cubes (ModelImageCube).

TEST INFRASTRUCTURE -- see oracle/__init__.py for who may import this.

The rows, pixels and weights are those of the reference's ModelImage.create_image
(ModelImage.py:229-274), restated here as ``imaging.create_image`` has them: rotation by
np.matmul, occultation, sunlight mask and ``packet_weighting``.  The pixel of a row follows
np.histogram2d's rule on edges = np.linspace(lo, hi, n + 1): searchsorted(edges, v, 'right') - 1,
with the right edge in the last bin and rows outside the range dropped.  A row's velocity is
``spectrum.doppler`` along row 1 of M (the observer direction maps to (0, -1, 0), so v > 0
recedes) and its column ``spectrum.columns``.  tests/test_image_cube.py pins the sum over the
velocity axis to the reference's own create_image() output (tests/golden/image.npz).
"""
import numpy as np

from .imaging import packet_weighting
from .spectrum import columns, doppler


def hist_bin(v, lo, hi, n):
    """np.histogram2d's bin of every value on linspace(lo, hi, n + 1), -1 outside."""
    edges = np.linspace(lo, hi, n + 1)
    k = np.searchsorted(edges, v, 'right') - 1
    k[v == edges[-1]] = n - 1
    return np.where((k >= 0) & (k < n), k, -1)


def create_cube(x, y, z, vx, vy, vz, frac, *, vrplanet, M, dims, xrange, zrange, apix, quantity,
                vmin, vmax, nbins, vscale, gtables=()):
    """(cube, counts), both (nx, nz, nbins + 2), BEFORE the atoms_per_packet scaling: per pixel
    and velocity column the sum of the rows' weights and their number.  Column 0 holds v < vmin,
    nbins + 1 v > vmax (NaN included)."""
    M = np.asarray(M)
    radvel_sun = vy + vrplanet
    pts_sun = np.stack([x, y, z], axis=1)
    pts_obs = np.array(np.matmul(M, pts_sun.transpose()).transpose())
    rho_obs = np.linalg.norm(pts_obs[:, [0, 2]], axis=1)
    inview = (rho_obs > 1) | (pts_obs[:, 1] < 0)
    frac = frac * inview
    rho_sun = np.linalg.norm(pts_sun[:, [0, 2]], axis=1)
    out_of_shadow = (rho_sun > 1) | (pts_sun[:, 1] < 0)
    weight = packet_weighting(quantity, frac, radvel_sun, gtables, out_of_shadow)
    weight = weight / apix
    nx, nz = int(dims[0]), int(dims[1])
    ix = hist_bin(pts_obs[:, 0], xrange[0], xrange[1], nx)
    iz = hist_bin(pts_obs[:, 2], zrange[0], zrange[1], nz)
    v = doppler(vx, vy, vz, M[1, 0], M[1, 1], M[1, 2], vscale)
    col = columns(v, vmin, vmax, nbins)
    sel = (ix >= 0) & (iz >= 0)
    cell = (ix[sel] * nz + iz[sel]) * (nbins + 2) + col[sel]
    ncell = nx * nz * (nbins + 2)
    cube = np.zeros(ncell)
    np.add.at(cube, cell, weight[sel])
    counts = np.bincount(cell, minlength=ncell).astype(np.int64)
    return cube.reshape(nx, nz, nbins + 2), counts.reshape(nx, nz, nbins + 2)
