"""``ModelDeposition``: where the source's atoms go -- the surface deposition map and the loss
budget of the adaptive driver's runs.

The reference records neither; this product defines the semantics (DESIGN.md section 8).  It
regenerates every output file of the ``Input`` with the deposition sink of the adaptive driver
(``nx_integrate_adaptive_deposit``): an adaptive ``Output`` is a pure function of (seed,
first_id, npackets), or of the X0 it holds, so the regenerated run is the run the user made,
bit for bit.  Per accepted step:

* SURFACE: a step that ends inside the planet deposits the packet's whole frac (perfect
  sticking, at the post-step point) or ``frac before - frac after`` a bounce (at the bounce
  point).  One event per such step, whatever its amount.  The point goes on the map at
  ``lon = (atan2(x, -y) + 2 pi) mod 2 pi``, ``lat = atan2(z, sqrt(x*x + y*y))``, binned like
  ``np.histogram2d`` on ``linspace(0, 2 pi, nlon + 1) x linspace(-pi/2, pi/2, nlat + 1)``, the
  axes of ``make_source_map``;
* MOON, ESCAPED (r^2 > outeredge), VANISHED (frac < 1e-10): the frac the first of these tests
  sets to zero;
* REMAINING: the frac of packets still in flight when they retire (or never integrated);
* LOST (photo-ionisation or lifetime loss in flight): SOURCE minus all of the above, where
  SOURCE is the initial frac.

The map is the deposition over the run window of the steady-state snapshot: packets are
released uniformly over ``endtime``, so the atoms released late have not landed yet and are in
REMAINING.  As in ``ModelImage``, rates are for a source of 1e23 atoms/s
(``atoms_per_packet = 1e23 / (totalsource / endtime)``).

Attributes: ``deposition`` (nlon, nlat) atoms cm^-2 s^-1; ``packet_map`` (nlon, nlat) int64
surface events per cell; ``deposited`` (nlon, nlat) deposited frac; ``longitude`` /
``latitude`` bin centres (rad) and ``lon_edges`` / ``lat_edges``; ``budget`` (a Series of
surface, moon, escaped, vanished, remaining, lost as fractions of the source); ``rates``
(atoms/s, same index); ``event_counts`` (events per bucket, and the source packets);
``buckets`` (frac sums, with source); ``totalsource``, ``atoms_per_packet``, ``sourcerate``,
``attempted_steps``, ``accepted_steps``, ``bounces``.
"""
import copy

import numpy as np
import pandas as pd

from . import catalogue
from .engine import Engine, get_engine
from .runsetup import get_setup
from .sharding import combine_ranks, local_device, nccl_comm
from .units import Quantity, value_of

BUCKETS = Engine.DEPOSIT_BUCKETS                    # nx_deposit_bucket order
BUDGET = ('surface', 'moon', 'escaped', 'vanished', 'remaining', 'lost')


def map_bins(params):
    """(nlon, nlat) from ``params`` (``nlonbins`` / ``nlatbins``, defaults 180 / 90 as
    ``make_source_map``); ValueError unless both are positive integers with nlon * nlat <
    2**31."""
    out = []
    for key, default in (('nlonbins', 180), ('nlatbins', 90)):
        v = params.get(key, default)
        try:
            ok = float(v) == int(float(v)) and int(float(v)) >= 1
        except (TypeError, ValueError):
            ok = False
        if isinstance(v, bool) or not ok:
            raise ValueError(f'{key} must be a positive integer, got {v!r}')
        out.append(int(float(v)))
    if out[0] * out[1] >= 2**31:
        raise ValueError(f'{out[0]} x {out[1]} cells is more than 2**31')
    return tuple(out)


def cell_area(nlon, nlat, radius_cm):
    """(nlon, nlat) cm^2 of the map's cells: R^2 dlon (sin lat_hi - sin lat_lo)."""
    lon = np.linspace(0, 2 * np.pi, nlon + 1)
    lat = np.linspace(-np.pi / 2, np.pi / 2, nlat + 1)
    return radius_cm**2 * np.outer(np.diff(lon), np.diff(np.sin(lat)))


def regeneration(output):
    """('seed', seed) or ('x0', columns): how to re-create an adaptive Output's initial
    state; ValueError when it cannot be (a bounce run without a seed, or no X0 held)."""
    seed = getattr(output, 'seed', None)
    if getattr(output, 'imported_x0', False):
        cols = getattr(output, '_imported_cols', None)
        if cols is None:
            raise ValueError('an output file holds no initial state (X0) to regenerate its run')
        return 'x0', cols
    if seed is None:
        raise ValueError('an output file has neither a seed nor an X0 to regenerate its run')
    return 'seed', seed


def regeneration_plan(inputs):
    """(outid, outputfiles, outputs, recipes) of every output file of ``inputs``, with the
    ``regeneration`` recipe of each; ValueError before any device work when one cannot be
    regenerated (a bounce run needs the seed of its deviates)."""
    outid, outputfiles, _, _ = inputs.search()
    outputs = [catalogue.fetch(f) for f in outputfiles]
    si = inputs.surfaceinteraction
    bounce = not (si.sticktype == 'constant' and si.stickcoef == 1.0)
    recipes = []
    for output in outputs:
        how = regeneration(output)
        if bounce and getattr(output, 'seed', None) is None:
            raise ValueError('a bounce run needs the seed of its deviates, and an output file '
                             'has none (written by the reference?)')
        recipes.append(how)
    return outid, outputfiles, outputs, recipes


def regenerate(model, eng, outputs, recipes, integrate):
    """Re-run every Output on ``eng`` from its recipe through ``integrate(eng, seed, first_id,
    n)``, a sink entry of the adaptive driver returning (attempted, accepted, bounces).  Adds
    the step totals and the kernel time to ``model``; returns the summed totalsource."""
    totalsource = 0.
    for output, (kind, what) in zip(outputs, recipes):
        setup = get_setup(model.inputs, strict_math=getattr(output, 'strict_math', False))
        setup.upload(eng)
        n = int(output.npackets)
        if kind == 'x0':
            eng.import_state(what)
        else:
            eng.init_state(setup.source_params(eng), what, output.first_id, n)
        att, acc, bnc = integrate(eng, getattr(output, 'seed', None) or 0, output.first_id, n)
        model.kernel_ms += eng.last_kernel_ms()
        model.attempted_steps += att
        model.accepted_steps += acc
        model.bounces += bnc
        totalsource += float(output.totalsource)
    return totalsource


class ModelDeposition:
    def __init__(self, inputs, params=None, device=None):
        params = {} if params is None else params
        if not isinstance(params, dict):
            raise ValueError('params must be a dict')
        if inputs.options.step_size != 0:
            raise ValueError('ModelDeposition needs the adaptive driver (options.step_size = 0); '
                             'constant-step runs do not define the fate of a packet')
        nlon, nlat = map_bins(params)
        self.inputs = copy.deepcopy(inputs)
        self.params = params
        self.type = 'deposition'
        self._device = local_device() if device is None else device
        self.nlon, self.nlat = nlon, nlat
        self.lon_edges = np.linspace(0, 2 * np.pi, nlon + 1)
        self.lat_edges = np.linspace(-np.pi / 2, np.pi / 2, nlat + 1)
        self.longitude = 0.5 * (self.lon_edges[:-1] + self.lon_edges[1:])
        self.latitude = 0.5 * (self.lat_edges[:-1] + self.lat_edges[1:])

        self.outid, self.outputfiles, outputs, recipes = regeneration_plan(self.inputs)

        comm = nccl_comm()
        dmap = np.zeros((nlon, nlat))
        cnt = np.zeros((nlon, nlat), dtype=np.int64)
        sums = np.zeros(len(BUCKETS))
        counts = np.zeros(len(BUCKETS), dtype=np.int64)
        totalsource = 0.
        self.attempted_steps = self.accepted_steps = self.bounces = 0
        self.kernel_ms = 0.0
        if outputs or comm is not None:
            eng = get_engine(self._device)
            eng.deposit_begin(nlon, nlat)
            try:
                totalsource = regenerate(self, eng, outputs, recipes,
                                         Engine.integrate_adaptive_deposit)
                if comm is not None:          # one collective; totalsource rides with the sink
                    totalsource = eng.deposit_allreduce(comm[1], totalsource)
                dmap, cnt, sums, counts = eng.deposit_fetch(nlon, nlat)
            finally:
                eng.deposit_end()
        if comm is None:
            totalsource, = combine_ranks((dmap, cnt, sums, counts), totalsource)
        self._finish(dmap, cnt, sums, counts, totalsource)

    def _finish(self, dmap, cnt, sums, counts, totalsource):
        self.totalsource = totalsource
        endtime = float(value_of(self.inputs.options.endtime))
        self.atoms_per_packet = 1e23 / (totalsource / endtime) if totalsource > 0 else np.nan
        self.sourcerate = Quantity(1e23, '1/s')
        r_cm = float(value_of(self.inputs.geometry.planet.radius)) * 1e5
        self.deposited = dmap
        self.packet_map = cnt
        self.deposition = dmap * self.atoms_per_packet / endtime / cell_area(self.nlon, self.nlat,
                                                                             r_cm)
        self.deposition_unit = 'cm-2 s-1'
        b = dict(zip(BUCKETS, sums))
        self.buckets = pd.Series(b)
        source = b['source']
        amounts = {k: b[k] for k in BUDGET[:-1]}
        amounts['lost'] = source - sum(amounts[k] for k in BUDGET[:-1])
        amounts = pd.Series(amounts)[list(BUDGET)]
        self.budget = amounts / source if source > 0 else amounts * np.nan
        self.rates = amounts * self.atoms_per_packet / endtime
        self.event_counts = pd.Series(dict(zip(BUCKETS, counts)))

    def __repr__(self):
        return self.__str__()

    def __str__(self):
        budget = ', '.join(f'{k} {v:.4g}' for k, v in self.budget.items())
        return f'''Model Deposition
map = {self.nlon} x {self.nlat} (lon x lat)
totalsource = {self.totalsource}
atoms per packet = {self.atoms_per_packet}
budget = {budget}'''
