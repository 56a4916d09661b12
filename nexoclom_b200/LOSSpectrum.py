"""``LOSSpectrum``: Doppler-resolved emission line profiles along lines of sight.

The reference has no such product; this one defines the semantics on top of the line-of-sight
membership that ``LOSResult`` reproduces from the reference's ``compute_iteration``.  For
spectrum i (observer ``x_sc``, unit boresight ``b``) the members are exactly ``LOSResult``'s
hits for that line: the same cone / KD-ball / planet test on the same rows (float32, frac == 0
dropped), each with the same radiance weight ``w`` (``packet_weighting`` summed over the
selected emission lines, and 0 for a hit whose foot-point is in the planet's shadow).  A
hit's Doppler velocity is

    v = ((vx*bx + vy*by) + vz*bz) * R_p[km]      [km/s], every op float64 rounded to nearest

in the planet's rest frame, positive away from the observer (a red shift).  The observer's
own velocity relative to the planet is not part of ``scdata``: shift ``velocity`` by it.
Bins are ``edges = np.linspace(vmin, vmax, nbins + 1)`` with ``np.histogram``'s rule (vmax
belongs to the last bin); hits below vmin and above vmax are kept in ``outside``.  So, per
spectrum, the hit counts over all columns equal ``LOSResult``'s ``npackets_los`` and the
weights sum to its radiance before the fit.

The sums run on the GPU (``nx_los_spectrum``: K5's candidate search, then the exact test with
the velocity binning).  As in ``ModelImage`` the source rate is 1e23 atoms/s
(``atoms_per_packet = 1e23 / (totalsource / endtime)``) and nothing is fitted to the data: to
put a spectrum on the scale of a fitted ``LOSResult`` multiply it by that result's
``sourcerate``.

Attributes (rows indexed like ``scdata.data``): ``edges`` and ``velocity`` (bin centres),
km/s; ``spectrum`` (kR per km/s); ``npackets`` (hits per bin); ``outside`` (kR below / above
the range); ``radiance`` (kR, all hits).
"""
import numbers

import numpy as np
import pandas as pd

from . import catalogue
from .engine import get_engine
from .LOSResult import cone_half_angle, dist_from_planet_cut
from .ModelResult import ModelResult
from .runsetup import get_setup
from .sharding import combine_ranks, local_device
from ._lib import LosParams
from .units import Quantity, value_of

MAX_CELLS = 2**31          # nspec * (nbins + 2) must stay below (32-bit cell index)


def velocity_bins(velocity, nspec):
    """(vmin, vmax, nbins) from ``velocity = (vmin, vmax, nbins)`` in km/s; raises ValueError
    unless it is a 3-sequence of finite vmin < vmax and an integer nbins >= 1 with
    nspec * (nbins + 2) < 2**31."""
    if isinstance(velocity, (str, bytes)) or not hasattr(velocity, '__len__') or len(velocity) != 3:
        raise ValueError('velocity must be a sequence (vmin, vmax, nbins)')
    vmin, vmax, nbins = velocity
    try:
        vmin, vmax = float(vmin), float(vmax)
    except (TypeError, ValueError):
        raise ValueError('vmin and vmax must be numbers (km/s)') from None
    if not (np.isfinite(vmin) and np.isfinite(vmax)):
        raise ValueError('vmin and vmax must be finite')
    if not vmin < vmax:
        raise ValueError('vmin must be < vmax')
    if isinstance(nbins, bool) or not isinstance(nbins, numbers.Integral) or nbins < 1:
        raise ValueError('nbins must be an integer >= 1')
    nbins = int(nbins)
    if nspec * (nbins + 2) >= MAX_CELLS:
        raise ValueError(f'{nspec} spectra x {nbins + 2} columns is more than 2**31 cells')
    return vmin, vmax, nbins


class LOSSpectrum(ModelResult):
    def __init__(self, scdata, inputs, velocity, params=None, dphi=Quantity(1., 'deg'),
                 device=None):
        if params is None:
            params = {'quantity': 'radiance'}
        if not isinstance(params, dict) or params.get('quantity', None) != 'radiance':
            raise ValueError("LOSSpectrum computes quantity = 'radiance' only")
        nspec = len(scdata)
        vmin, vmax, nbins = velocity_bins(velocity, nspec)
        dphi = cone_half_angle(dphi)
        scdata.set_frame('Model')
        super().__init__(inputs, params)
        self.type = 'LineOfSightSpectrum'
        self.species = scdata.species
        self.query = scdata.query
        self.dphi = dphi
        self._device = local_device() if device is None else device
        self.edges = np.linspace(vmin, vmax, nbins + 1)
        self.velocity = 0.5 * (self.edges[:-1] + self.edges[1:])
        self.velocity_unit = 'km/s'
        self.radiance_unit = 'kR'

        data = scdata.data
        los = np.stack([data[c].values.astype(float) for c in
                        ('x', 'y', 'z', 'xbore', 'ybore', 'zbore')])
        dist_from_plan = dist_from_planet_cut(data).values if nspec else np.zeros(0)
        spec = np.zeros((nspec, nbins + 2))
        cnt = np.zeros((nspec, nbins + 2), dtype=np.int64)
        self.outid, self.outputfiles, _, _ = self.inputs.search()
        totalsource, npackets = 0., 0
        self.kernel_ms = 0.0
        for fname in self.outputfiles:
            output = catalogue.fetch(fname)
            if nspec:
                eng = get_engine(self._device)
                setup = get_setup(self.inputs, strict_math=getattr(output, 'strict_math', False))
                lp = LosParams()
                lp.dphi = self.dphi
                lp.outeredge = float(self.inputs.options.outeredge)
                lp.vrplanet = setup.vrplanet
                lp.rp_cm = setup.radius_km * 1e5
                lp.quantity = 1
                # resident rows, or -- recipe-only constant-step runs -- the same rows
                # regenerated chunk by chunk
                for table, _ in output.tables():
                    self._upload_weighting_tables(eng, setup)
                    eng.bind_packets(table)
                    try:
                        s_, c_ = eng.los_spectrum(los, dist_from_plan, lp, vmin, vmax, nbins,
                                                  setup.radius_km, n=table.n)
                        self.kernel_ms += eng.last_kernel_ms()
                    finally:
                        eng.bind_packets(None)
                    spec += s_
                    cnt += c_
            totalsource += output.totalsource
            npackets += output.npackets
        self.totalsource, npackets = combine_ranks((spec, cnt), totalsource, npackets)
        npackets = int(round(npackets))

        endtime = float(value_of(self.inputs.options.endtime))
        self.atoms_per_packet = (1e23 / (self.totalsource / endtime) if self.totalsource > 0
                                 else np.nan)
        self.sourcerate = Quantity(1e23, '1/s')
        kR = spec * (self.atoms_per_packet / 1e3)
        width = np.diff(self.edges)
        cols = pd.Index(self.velocity, name='velocity')
        self.spectrum = pd.DataFrame(kR[:, 1:-1] / width, index=data.index, columns=cols)
        self.npackets = pd.DataFrame(cnt[:, 1:-1], index=data.index, columns=cols)
        self.outside = pd.DataFrame({'below': kR[:, 0], 'above': kR[:, -1]}, index=data.index)
        self.npackets_outside = pd.DataFrame({'below': cnt[:, 0], 'above': cnt[:, -1]},
                                             index=data.index)
        self.radiance = pd.Series(kR.sum(axis=1), index=data.index)
        self.npackets_los = pd.Series(cnt.sum(axis=1), index=data.index)
        self.npackets_total = npackets

    def __repr__(self):
        return self.__str__()

    def __str__(self):
        return f'''LOS Spectrum
quantity = {self.quantity}
spectra = {len(self.radiance)}
velocity = {self.edges[0]} .. {self.edges[-1]} km/s in {len(self.velocity)} bins
totalsource = {self.totalsource}
atoms per packet = {self.atoms_per_packet}
dphi = {self.dphi}'''
