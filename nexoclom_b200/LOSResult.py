"""``LOSResult``: model radiance along spacecraft lines of sight.

Drop-in for the reference ``data_simulation/LOSResult.py:75-308`` and
``data_simulation/compute_iteration.py:90-240``.  The per-spectrum Python loop
(KD-tree ball query, cone test, planet truncation, weighting, foot-point shadow
test; compute_iteration.py:151-222) is one CUDA kernel (K5,
``nx_los_accumulate``) that evaluates every (line of sight, packet) pair with
the same membership rule.  The SQL model cache is replaced by an in-memory one.

``scdata`` is duck-typed exactly as in the reference: ``.data`` DataFrame with
``x, y, z, xbore, ybore, zbore, radiance, sigma, alttan``; ``.species``;
``.query``; ``.set_frame('Model')``; ``len()``; ``.subslong``.
"""
import numpy as np
import pandas as pd

from . import catalogue
from .engine import get_engine
from .ModelResult import ModelResult
from .Output import Output
from .runsetup import get_setup
from ._lib import LosParams
from .units import Quantity, value_of


class IterationResult:
    """Per-outputfile LOS result (reference compute_iteration.py:15-35)."""

    def __init__(self, iteration, losresult):
        self.radiance = iteration['radiance']
        self.npackets = iteration['npackets']
        self.totalsource = iteration['totalsource']
        self.outputfile = iteration['outputfile']
        self.out_idnum = iteration['out_idnum']
        self.included = iteration['included']
        self.modelfile = None
        self.model_idnum = None
        self.used_packets = iteration.get('used', None)
        self.used_packets0 = iteration.get('used0', None)
        self.quantity = losresult.quantity
        self.query = losresult.query
        self.dphi = losresult.dphi
        self.mechanism = losresult.mechanism
        self.wavelength = losresult.wavelength
        self.fitted = losresult.fitted
        self.used_csr = None
        self.spectrum_index = None

    def used_sets(self):
        """(used, used0) as pandas Series of sets, exactly what the reference stores
        (row labels of the output's X and values of its 'Index' column)."""
        if self.used_csr is None:
            return None, None
        off, idx0, labels = self.used_csr
        n = len(off) - 1
        used = pd.Series([set(labels[off[i]:off[i + 1]].tolist()) for i in range(n)],
                         index=self.spectrum_index)
        used0 = pd.Series([set(idx0[off[i]:off[i + 1]].tolist()) for i in range(n)],
                          index=self.spectrum_index)
        return used, used0


def dist_from_planet_cut(data):
    """LOS truncation distance: |x_sc| if the boresight hits the planet, else
    1e30 (reference compute_iteration.py:105-115)."""
    dist_from_plan = np.sqrt(data.x**2 + data.y**2 + data.z**2)
    ang = np.arccos((-data.x * data.xbore - data.y * data.ybore -
                     data.z * data.zbore) / dist_from_plan)
    asize_plan = np.arcsin(1. / dist_from_plan)
    dist_from_plan = dist_from_plan.copy()
    dist_from_plan.loc[ang > asize_plan] = 1e30
    return dist_from_plan


def cone_half_angle(dphi):
    """The lines of sight's cone half-angle in radians, from a Quantity or a number of
    degrees.  ValueError unless it is finite, > 0 and < 90 degrees (the same rule the C ABI
    applies), so a bad angle fails before any device work."""
    rad = (float(dphi.to('rad').value) if isinstance(dphi, Quantity)
           else float(np.radians(dphi)))
    if not 0.0 < rad < np.pi / 2:
        raise ValueError(f'dphi = {dphi}: the cone half-angle must be finite, > 0 and < 90 deg')
    return rad


def compute_iteration(self, outputfile, scdata, delay=False):
    """One output file against all spectra (reference compute_iteration.py:90-240).  The
    packets are the Output's resident table (the rows the reference reads back from its
    pickle); a constant-step run that was too large to keep its rows regenerates them chunk
    by chunk (``Output.tables``), so ANY Output works here, as in the reference."""
    data = scdata.data
    dist_from_plan = dist_from_planet_cut(data)

    output = catalogue.fetch(outputfile)
    totalsource = output.totalsource
    idnum = output.idnum

    eng = get_engine(self._device)
    setup = get_setup(self.inputs, strict_math=getattr(output, 'strict_math', False))
    lp = LosParams()
    lp.dphi = self.dphi
    lp.outeredge = float(self.inputs.options.outeredge)
    lp.vrplanet = setup.vrplanet
    lp.rp_cm = setup.radius_km * 1e5
    if self.quantity != 'radiance':
        assert False, 'Other quantities not set up.'          # compute_iteration.py:213
    lp.quantity = 1
    los = np.stack([data[c].values.astype(float) for c in
                    ('x', 'y', 'z', 'xbore', 'ybore', 'zbore')])
    print(f'{data.shape[0]} spectra taken.')

    rad_ = np.zeros(len(data))
    npack_ = np.zeros(len(data), dtype=np.int64)
    included_ = np.zeros(output.npackets, dtype=bool)
    used_csr = None
    resident = getattr(output, 'trajectory_kept', True)
    self.kernel_ms = 0.0
    for table, first in output.tables():
        # (re)upload per chunk: regenerating a chunk re-uploads the run tables
        self._upload_weighting_tables(eng, setup)
        eng.bind_packets(table)
        try:
            want_used = resident and getattr(self, 'keep_used', True)
            # `used` / `used0` (compute_iteration.py:143-144, 210-211): packets with weight
            # > 0 per spectrum, as CSR (the sets the reference stores are built on demand by
            # IterationResult.used_sets()).  Their counts come out of the accumulate pass, the
            # indices from the candidate pairs that pass left on the device (nothing may touch
            # the engine in between).
            if want_used:
                r_, n_, inc_, cnt_ = eng.los_accumulate(los, dist_from_plan.values, lp,
                                                        n=table.n, count_used=True)
                self.kernel_ms += eng.last_kernel_ms()
                off, idx = eng.los_used_fill(los, dist_from_plan.values, lp, cnt_, n=table.n)
            else:
                r_, n_, inc_ = eng.los_accumulate(los, dist_from_plan.values, lp, n=table.n)
            self.kernel_ms += eng.last_kernel_ms()
            index = table.index_host() + first
            included_[index[inc_]] = True
            rad_ += r_
            npack_ += n_
            if want_used:
                used_csr = (off, index[idx], output.row_labels()[idx])
        finally:
            eng.bind_packets(None)
    assert np.all(np.isfinite(rad_))

    rad = pd.Series(rad_, index=data.index)
    npack = pd.Series(npack_, index=data.index, dtype=int)
    included = pd.Series(included_, index=pd.RangeIndex(output.npackets), dtype=bool)
    iteration_ = {'radiance': rad, 'npackets': npack, 'totalsource': totalsource,
                  'outputfile': outputfile, 'out_idnum': idnum, 'query': scdata.query,
                  'used': None, 'used0': None, 'included': included}
    result = IterationResult(iteration_, self)
    result.used_csr = used_csr
    result.spectrum_index = data.index
    return result


class LOSResult(ModelResult):
    def __init__(self, scdata, inputs, params=None, dphi=Quantity(1., 'deg'), device=None,
                 **kwargs):
        dphi = cone_half_angle(dphi)
        if params is None:
            params = {'quantity': 'radiance'}
        scdata.set_frame('Model')
        super().__init__(inputs, params)
        self.species = scdata.species
        self.query = scdata.query
        self.type = 'LineOfSight'
        self.dphi = dphi
        self._oedge = np.min([self.inputs.options.outeredge * 2, 100])
        self.fitted = self.inputs.options.fitted
        nspec = len(scdata)
        self.radiance = pd.Series(np.zeros(nspec), index=scdata.data.index)
        self.radiance_unit = 'kR'
        self.sourcemap = None
        self.modelfiles = None
        self.goodness_of_fit = None
        self.mask = None
        self.masking = kwargs.get('masking', None)
        self.fit_method = kwargs.get('fit_method', None)
        self.label = kwargs.get('label', 'LOSResult')
        # True: make_mask / determine_source_rate behave exactly like the reference
        self.reference_exact = kwargs.get('reference_exact', True)
        from .sharding import local_device
        self._device = local_device() if device is None else device
        self._iterations = {}

    def __repr__(self):
        return self.__str__()

    def __str__(self):
        return f'''Model Label = {self.label}
quantity = {self.quantity}
npackets = {self.npackets}
totalsource = {self.totalsource}
atoms per packet = {self.atoms_per_packet}
sourcerate = {self.sourcerate}
dphi = {self.dphi}
fit_method = {self.fit_method}
fitted = {self.fitted}'''

    def make_mask(self, data):
        """reference LOSResult.py:171-200, keyword by keyword.

        `middleNN` as the reference does it (``reference_exact``, the default): the WHOLE
        data frame goes to astropy's ``PercentileInterval.get_limits`` (:181-182), which
        ravel()s every column -- positions, boresights, sigma, ... -- into one sample, drops
        the non-finite values and takes the two percentiles; the radiances are then compared
        with those limits (:183-185).  A frame with a non-numeric column fails there, as it
        does in the reference.  ``reference_exact=False`` takes the percentiles of the
        radiances themselves.  Pinned by tests/golden/source_rate.npz (the unmodified method)."""
        mask = np.array([True for _ in data.radiance])
        sigmalimit = None
        if self.masking is not None:
            for masktype in self.masking.split(';'):
                masktype = masktype.strip().lower()
                if masktype.startswith('middle'):
                    perinterval = float(masktype[6:])
                    lower = (100 - perinterval) * 0.5
                    if getattr(self, 'reference_exact', True):
                        values = np.asarray(data).ravel()
                        values = values[np.isfinite(values)]
                    else:
                        values = np.asarray(data.radiance)
                    lim = np.percentile(values, (lower, 100 - lower))
                    mask = mask & (data.radiance >= lim[0]) & (data.radiance <= lim[1])
                elif masktype.startswith('minalt'):
                    mask = mask & (data.alttan >= float(masktype[6:]))
                elif masktype.startswith('minsnr'):
                    snr = data.radiance / data.sigma
                    mask = mask & (snr > float(masktype[6:]))
                elif masktype.startswith('siglimit'):
                    sigmalimit = float(masktype[8:])
                else:
                    raise ValueError('nexoclom.math.fit_model',
                                     f'masking = {masktype} not defined.')
        return np.asarray(mask), sigmalimit

    def simulate_data_from_inputs(self, scdata, distribute=None):
        """reference LOSResult.py:202-276."""
        if ((self.inputs.spatialdist.type == 'surface map') and
                (self.inputs.spatialdist.coordinate_system == 'planet-fixed')):
            self.inputs.spatialdist.subsolarlon = Quantity(scdata.subslong.median(), 'rad')

        (self.outid, self.outputfiles, self.npackets, self.totalsource) = self.inputs.search()
        print(f'LOSResult: {len(self.outid)} output files found.')
        from .sharding import rank_world
        if self.npackets == 0 and rank_world()[1] == 1:
            raise RuntimeError('No packets found for these Inputs.')
        if distribute in (True, 'delay', 'delayed'):
            assert False, "Don't do this"                       # LOSResult.py:230

        data = scdata.data
        iteration_results = []
        for outputfile in self.outputfiles:
            if outputfile not in self._iterations:
                self._iterations[outputfile] = compute_iteration(self, outputfile, scdata)
            it = self._iterations[outputfile]
            assert len(it.radiance) == len(data)
            iteration_results.append(it)

        self.modelfiles = {}
        self.npackets_los = pd.Series(np.zeros(len(data), dtype=int), index=data.index)
        for it in iteration_results:
            self.radiance += it.radiance
            self.npackets_los += it.npackets
            self.modelfiles[it.outputfile] = it.modelfile

        # sharded run: every rank holds the columns of its own packets; ONE all-reduce per
        # product (radiance, hit counts, packet / source totals) makes them complete
        from .sharding import allreduce_sum, rank_world
        if rank_world()[1] > 1:
            rad = np.ascontiguousarray(self.radiance.values, dtype=np.float64)
            cnt = np.ascontiguousarray(self.npackets_los.values, dtype=np.int64)
            tot = np.array([float(self.totalsource), float(self.npackets)])
            allreduce_sum(rad, cnt, tot)
            self.radiance = pd.Series(rad, index=data.index)
            self.npackets_los = pd.Series(cnt, index=data.index)
            self.totalsource, self.npackets = float(tot[0]), int(round(tot[1]))

        model_rate = self.totalsource / float(value_of(self.inputs.options.endtime))
        self.atoms_per_packet = 1e23 / model_rate
        self.radiance *= self.atoms_per_packet / 1e3  # kR
        self.determine_source_rate(scdata, use_weight=False)
        self.outputfiles = list(self.modelfiles.keys())
        print(self.totalsource, self.atoms_per_packet)

    def determine_source_rate(self, scdata, use_weight=True):
        """Linear least-squares scale factor model -> data (reference LOSResult.py:278-308).
        astropy's LinearLSQFitter (5.3, pinned by the reference's poetry.lock) multiplies both
        sides of the design equation by `weights` before np.linalg.lstsq, i.e. it minimises
        sum((w (d - f m))**2): on a Multiply model that is the closed form
        f = sum(w^2 m d) / sum(w^2 m m).  The reference passes w = 1/sigma**2 (:281), so its
        weighted fit is a 1/sigma^4 fit -- kept.

        `siglimit`: the reference refits the clipped points with the weights of the FIRST
        mask (:296-298); astropy raises on the length mismatch whenever a point was clipped.
        ``reference_exact`` (default) does the same -- ValueError, message of the NumPy
        broadcast that fails inside astropy --; ``reference_exact=False`` lets the weights
        follow the clipped mask.  Pinned by tests/golden/source_rate.npz."""
        mask, sigmalimit = self.make_mask(scdata.data)
        d = scdata.data.radiance.values
        m = self.radiance.values
        sigma = scdata.data.sigma.values
        exact = getattr(self, 'reference_exact', True)

        def weights_of(msk):
            return 1. / sigma[msk]**2 if use_weight else np.ones_like(sigma[msk])

        def fit(msk, w):
            if len(w) != int(np.sum(msk)):
                raise ValueError(f'operands could not be broadcast together with shapes '
                                 f'({int(np.sum(msk))},1) ({len(w)},1) (ufunc \'multiply\')')
            return np.sum(w * w * m[msk] * d[msk]) / np.sum(w * w * m[msk] * m[msk])

        if not np.all(m == 0):
            weights = weights_of(mask)
            factor = fit(mask, weights)
            if sigmalimit is not None:
                diff = np.abs((d - factor * m) / sigma)
                mask = mask & (diff < sigmalimit)
                factor = fit(mask, weights if exact else weights_of(mask))
            self.radiance *= factor
            self.sourcerate = Quantity(factor, '')      # x 10**23 atoms/s
        else:
            self.sourcerate = Quantity(0., '')
        self.goodness_of_fit = None
        self.mask = mask

    def make_source_map(self, grid_params=None, normalize=True, do_source=True,
                        do_available=True, distribute=None):
        """Source maps of the modelled (`source`) and of all launched (`available`) packets,
        summed over the output files of this result and optionally converted to fluxes
        (reference LOSResult.py:310-491).  The per-file maps come from K6
        (``make_source_map.make_source_map``); what is done here is the reference's host
        arithmetic, statement by statement -- including its habit of adding ``speed_dist`` of
        the file with the largest speed range twice (:349-353).  Quantities are plain arrays:
        abundance in atoms cm^-2 s^-1, speed distributions per km/s, angular ones per rad."""
        from .make_source_map import make_source_map
        from .sourcemap import SourceMap
        if distribute in (True, 'delay', 'delayed'):
            assert False, "Don't do this"                              # :328
        sourcemap = availablemap = None
        todo = (['source'] if do_source else []) + (['available'] if do_available else [])
        rate_per_s = float(value_of(self.sourcerate)) * 1e23         # sourcerate.to(1/u.s)
        r_cm = float(self.inputs.geometry.planet.radius.value) * 1e5
        for todo_ in todo:
            sources = [make_source_map(outputfile, grid_params, todo=todo_, device=self._device)
                       for outputfile in self.modelfiles]
            sources = [{k: np.asarray(value_of(v), dtype=float) for k, v in s_.items()}
                       for s_ in sources]
            dist = {key: np.zeros_like(value) for key, value in sources[0].items()}
            vmaxes = [s_['speed'].max() for s_ in sources]
            vmax = max(vmaxes)
            dist['speed'] = sources[int(np.where(np.asarray(vmaxes) == vmax)[0][0])]['speed']
            for s_ in sources:
                for key in ('abundance_uncor', 'n_included', 'n_total', 'altitude_dist',
                            'altitude_dist_map', 'azimuth_dist', 'azimuth_dist_map',
                            'speed_dist', 'speed_dist_map'):
                    dist[key] += s_[key]
                if s_['speed'].max() == vmax:
                    dist['speed_dist'] += s_['speed_dist']
                    dist['speed_dist_map'] += s_['speed_dist_map']
                else:
                    dist['speed_dist'] += np.interp(dist['speed'], s_['speed'], s_['speed_dist'])
                    for i in range(len(dist['longitude'])):
                        for j in range(len(dist['latitude'])):
                            dist['speed_dist_map'] += np.interp(dist['speed'], s_['speed'],
                                                                s_['speed_dist_map'][i, j, :])
            for key in ('longitude', 'latitude', 'azimuth', 'altitude'):
                dist[key] = sources[0][key]
            with np.errstate(divide='ignore', invalid='ignore'):
                dist['fraction_observed'] = dist['n_included'] / dist['n_total']
                q = np.isnan(dist['fraction_observed'])
                dist['fraction_observed'][q] = 1
                dist['abundance'] = dist['abundance_uncor'] / dist['fraction_observed']
            dist['fraction_observed'][q] = 0
            dist['abundance'][np.isnan(dist['abundance'])] = 0

            if normalize:
                dx = dist['longitude'][1] - dist['longitude'][0]
                dy = dist['latitude'][1] - dist['latitude'][0]
                _, gridlatitude = np.meshgrid(dist['longitude'], dist['latitude'])
                d_area = np.abs(dx * (np.sin(gridlatitude + dy / 2) - np.sin(gridlatitude - dy / 2)))
                area = r_cm**2 * d_area
                with np.errstate(divide='ignore', invalid='ignore'):
                    dist['abundance'] = dist['abundance'] / dist['abundance'].sum() / area.T * rate_per_s
                    dist['abundance_uncor'] = (dist['abundance_uncor'] /
                                               dist['abundance_uncor'].sum() / area.T * rate_per_s)
                    dv = dist['speed'][1] - dist['speed'][0]
                    dist['speed_dist'] = (rate_per_s * dist['speed_dist'] /
                                          dist['speed_dist'].sum() / dv)
                    dist['speed_dist_map'] = (dist['abundance'][:, :, np.newaxis] *
                                              dist['speed_dist_map'] /
                                              dist['speed_dist_map'].sum(axis=2)[:, :, np.newaxis] / dv)
                    # the reference normalises the AXES 'altitude' / 'azimuth' here, not the
                    # distributions (:452-455, :464-467); kept
                    dalt = dist['altitude'][1] - dist['altitude'][0]
                    dist['altitude_dist_map'] = (dist['abundance'][:, :, np.newaxis] *
                                                 dist['altitude_dist_map'] /
                                                 dist['altitude_dist_map'].sum(axis=2)[:, :, np.newaxis] / dalt)
                    dist['altitude'] = rate_per_s * dist['altitude'] / dist['altitude'].sum() / dalt
                    daz = dist['azimuth'][1] - dist['azimuth'][0]
                    dist['azimuth_dist_map'] = (dist['abundance'][:, :, np.newaxis] *
                                                dist['azimuth_dist_map'] /
                                                dist['azimuth_dist_map'].sum(axis=2)[:, :, np.newaxis] / daz)
                    dist['azimuth'] = rate_per_s * dist['azimuth'] / dist['azimuth'].sum() / daz
            source_ = SourceMap(dist)
            for key in ('abundance_uncor', 'n_included', 'n_total', 'speed_dist_map',
                        'altitude_dist_map', 'azimuth_dist_map'):
                setattr(source_, key, dist[key])
            if todo_ == 'source':
                sourcemap = source_
            else:
                availablemap = source_
        return sourcemap, availablemap
