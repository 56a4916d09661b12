"""``ModelDensity``: number density of the modelled exosphere at sample points.

The reference's ``ModelDensity.py`` is unfinished and not exported; this product defines the
semantics itself.  For every sample point p_i (model frame: planet-centred, R_p, Sun at -y,
the frame of ``Output.X``) and ball radius r_i, the saved rows of every output file of the
``Input`` (float32, frac == 0 rows dropped: what ``Output.save`` keeps) are tested with

    d2 = (dx*dx + dy*dy) + dz*dz <= r_i*r_i,   dx = x - p_x, ...  (float64, rounded to nearest)

and summed on the GPU (K7, ``nx_density_accumulate``): S1 = sum frac, S2 = sum frac**2 and
the member count.  With ``atoms_per_packet = 1e23 / (totalsource / endtime)`` (as
``ModelImage`` / ``LOSResult``) and V_i the volume of ball i outside the planet:

    density     = atoms_per_packet * S1 / V_i          [cm^-3]
    density_err = atoms_per_packet * sqrt(S2) / V_i    (Monte-Carlo standard error)

A ball entirely inside the planet has V = 0: its density is NaN.  Moons' bodies are not
taken out of V.
"""
import numpy as np
import pandas as pd

from . import catalogue
from .engine import get_engine
from .ModelResult import ModelResult
from .sharding import combine_ranks, local_device
from .units import Quantity, value_of


def lens_volume(d, r):
    """Volume of a ball of radius r (centre at distance d from the planet's centre) that lies
    outside the planet, in R_p**3.  Closed form; a sliver just outside d + r = 1 loses its
    relative accuracy to cancellation and is never negative."""
    d = np.asarray(d, dtype=np.float64)
    r = np.asarray(r, dtype=np.float64)
    d, r = np.broadcast_arrays(d, r)
    full = 4.0 / 3.0 * np.pi * r**3
    with np.errstate(divide='ignore', invalid='ignore'):
        lens = full - np.pi * (r + 1 - d)**2 * (d * d + 2 * d * (r + 1) - 3 * (r - 1)**2) / (12 * d)
    return np.select([d >= r + 1, d + r <= 1, d + 1 <= r],
                     [full, 0.0, 4.0 / 3.0 * np.pi * (r**3 - 1)], np.maximum(lens, 0.0))


def sample_points(points, radius):
    """(points (N, 3) float64, radius (N,) float64, index) from an (N, 3) array or a DataFrame
    with columns x, y, z; raises ValueError for a bad shape, a non-finite value or a radius
    <= 0."""
    if isinstance(points, pd.DataFrame):
        missing = [c for c in ('x', 'y', 'z') if c not in points.columns]
        if missing:
            raise ValueError(f'points DataFrame lacks columns {missing}')
        index = points.index
        pts = points[['x', 'y', 'z']].to_numpy(dtype=np.float64)
    else:
        pts = np.asarray(points, dtype=np.float64)
        if pts.ndim != 2 or pts.shape[1] != 3:
            raise ValueError(f'points must be an (N, 3) array, not shape {pts.shape}')
        index = pd.RangeIndex(len(pts))
    pts = np.ascontiguousarray(pts)
    rad = np.asarray(radius, dtype=np.float64)
    if rad.ndim == 0:
        rad = np.full(len(pts), float(rad))
    if rad.shape != (len(pts),):
        raise ValueError(f'radius must be a scalar or one value per point, not shape {rad.shape}')
    if not np.all(np.isfinite(pts)):
        raise ValueError('points must be finite')
    if not (np.all(np.isfinite(rad)) and np.all(rad > 0)):
        raise ValueError('radius must be finite and > 0')
    return pts, np.ascontiguousarray(rad), index


class ModelDensity(ModelResult):
    def __init__(self, inputs, points, radius, params=None, device=None):
        pts, rad, index = sample_points(points, radius)
        if params is None:
            params = {'quantity': 'density'}
        if params.get('quantity', 'density') != 'density':
            raise ValueError("ModelDensity computes quantity = 'density'")
        params = dict(params, quantity='density')
        super().__init__(inputs, params)
        self.type = 'density'
        self._device = local_device() if device is None else device
        self.points = pd.DataFrame(pts, columns=['x', 'y', 'z'], index=index)
        self.radius = pd.Series(rad, index=index)
        self.density_unit = 'cm-3'

        npts = len(pts)
        s1, s2 = np.zeros(npts), np.zeros(npts)
        count = np.zeros(npts, dtype=np.int64)
        self.outid, self.outputfiles, _, _ = self.inputs.search()
        totalsource = 0.
        npackets = 0
        for fname in self.outputfiles:
            output = catalogue.fetch(fname)
            if npts:
                eng = get_engine(self._device)
                # resident rows, or -- recipe-only constant-step runs -- the same rows
                # regenerated chunk by chunk
                for table, _ in output.tables():
                    eng.bind_packets(table)
                    try:
                        eng.density_accumulate(pts, rad, s1, s2, count, n=table.n)
                    finally:
                        eng.bind_packets(None)
            totalsource += output.totalsource
            npackets += output.npackets
        self.totalsource, = combine_ranks((s1, s2, count), totalsource)
        self.npackets_total = npackets

        endtime = float(value_of(self.inputs.options.endtime))
        self.atoms_per_packet = (1e23 / (self.totalsource / endtime) if self.totalsource > 0
                                 else np.nan)
        self.sourcerate = Quantity(1e23, '1/s')
        r_cm = float(self.inputs.geometry.planet.radius.value) * 1e5
        vol = lens_volume(np.sqrt((pts * pts).sum(axis=1)), rad) * r_cm**3
        with np.errstate(divide='ignore', invalid='ignore'):
            dens = np.where(vol > 0, self.atoms_per_packet * s1 / vol, np.nan)
            err = np.where(vol > 0, self.atoms_per_packet * np.sqrt(s2) / vol, np.nan)
        self.volume = pd.Series(vol, index=index)                 # cm^3 outside the planet
        self.density = pd.Series(dens, index=index)
        self.density_err = pd.Series(err, index=index)
        self.npackets = pd.Series(count, index=index)
        self.s1 = pd.Series(s1, index=index)
        self.s2 = pd.Series(s2, index=index)

    def __repr__(self):
        return self.__str__()

    def __str__(self):
        return f'''Model Density
quantity = {self.quantity}
points = {len(self.density)}
totalsource = {self.totalsource}
atoms per packet = {self.atoms_per_packet}
density unit = {self.density_unit}'''
