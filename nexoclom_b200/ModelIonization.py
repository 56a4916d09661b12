"""``ModelIonization``: where the source's atoms are lost in flight -- 3-D ion production maps
from the adaptive driver.

The reference has no such product; this one defines the semantics (DESIGN.md section 8).  Like
``ModelDeposition`` it regenerates every output file of the ``Input`` (K1 from the seed and
``first_id``, or the imported X0) through a sink build of the adaptive driver
(``nx_integrate_adaptive_ionize``), so the run is the run the user made, bit for bit.  Where
``ModelDeposition`` reports the frac lost in flight as one number (LOST), this product says
where it was lost.  For every accepted step, before any surface, moon, escape or vanish
handling:

* ``loss = frac before - frac of the Runge-Kutta step``; a step with ``loss == 0`` is not
  recorded, a negative one (a step across the shadow edge can raise the frac slightly) is
  recorded as it is, so the totals are exact;
* it is recorded at the midpoint of the step's chord, ``(x + x_rk) * 0.5`` per axis (before a
  bounce moves the packet), in the planet frame of ``Output.X`` (R_p, Sun toward -y);
* binned like ``np.histogramdd`` on ``linspace(lo_k, hi_k, n_k + 1)`` per axis, the last right
  edge in the last cell; a midpoint outside the box (or NaN) goes to OUTSIDE.

The grid plus OUTSIDE is ``ModelDeposition``'s LOST up to rounding.  Every accepted step is a
sample, so the map has far less Monte-Carlo noise than the saved rows weighted by a loss rate.

Caveats: like the deposition map this is the production over the run window.  Packets are
released uniformly over ``endtime``, so the map approaches the steady state only when
``endtime`` is long compared with the lifetimes and the flight times.  With
``options.lifetime > 0`` it is the lifetime loss (unshadowed), not strictly photo-ionisation.
A step's loss goes to the one cell of its chord's midpoint, not split over the cells the chord
crosses.

Parameters (``params``, all in R_p as for ``ModelImage``): ``dims = 'nx,ny,nz'`` (default
``'100,100,100'``), ``center = 'x,y,z'`` (default ``'0,0,0'``), ``width = 'wx,wy,wz'`` (default
``'8,8,8'``).

Attributes: ``production`` (nx, ny, nz) ions cm^-3 s^-1 for a source of 1e23 atoms/s,
``ionized * atoms_per_packet / endtime / V_ext``, where ``V_ext`` is the part of the cell's volume
outside the planet (NaN for a cell wholly inside it; moons' bodies are not excluded, as in
``ModelDensity``); ``ionized`` (nx, ny, nz) frac sums; ``packet_grid`` (nx, ny, nz) int64
recorded steps; ``outside`` / ``outside_count``; ``exterior_fraction`` (nx, ny, nz); ``rate``
(ions/s, grid plus OUTSIDE); ``xaxis`` / ``yaxis`` / ``zaxis`` (bin centres) and ``edges``;
``totalsource``, ``atoms_per_packet``, ``sourcerate``, ``attempted_steps``, ``accepted_steps``,
``bounces``, ``kernel_ms``.
"""
import copy

import numpy as np

from .engine import Engine, get_engine
from .ModelDeposition import regenerate, regeneration_plan
from .runsetup import get_setup
from .sharding import combine_ranks, local_device, nccl_comm
from .units import Quantity, value_of

SUBCELLS = 16              # sub-cell midpoints per axis of a cell the planet's surface cuts


def _triple(params, key, default, kind):
    text = params.get(key, default)
    try:
        parts = [kind(float(v)) if kind is int else float(v) for v in str(text).split(',')]
        ok = len(parts) == 3 and all(np.isfinite(parts))
        if kind is int:
            ok = ok and all(float(v) == int(float(v)) and int(float(v)) >= 1
                            for v in str(text).split(','))
    except (TypeError, ValueError):
        ok = False
    if isinstance(text, bool) or not ok:
        raise ValueError(f'{key} must be three comma-separated '
                         f"{'positive integers' if kind is int else 'finite numbers'}, got {text!r}")
    return parts


def grid_params(params):
    """(dims, lo, hi) of the grid from ``params``: three cells counts, the box's lower and upper
    corners in R_p; ValueError for malformed values, a width <= 0 or nx*ny*nz + 1 >= 2**31."""
    dims = _triple(params, 'dims', '100,100,100', int)
    center = _triple(params, 'center', '0,0,0', float)
    width = _triple(params, 'width', '8,8,8', float)
    if min(width) <= 0:
        raise ValueError(f'width must be > 0 on every axis, got {params.get("width")!r}')
    if dims[0] * dims[1] * dims[2] + 1 >= 2**31:
        raise ValueError(f'{dims[0]} x {dims[1]} x {dims[2]} cells plus OUTSIDE is 2**31 or more')
    lo = [c - w / 2 for c, w in zip(center, width)]
    hi = [c + w / 2 for c, w in zip(center, width)]
    for a, b in zip(lo, hi):
        if not a < b:
            raise ValueError('the box has no width in floating point')
    return dims, lo, hi


def exterior_fraction(edges, sub=SUBCELLS):
    """(nx, ny, nz) fraction of each cell's volume at r >= 1 (outside the planet) for the cell
    edges (ex, ey, ez): 1 when the cell's nearest point is at r >= 1, 0 when its farthest corner
    is at r <= 1, otherwise the fraction of its sub**3 sub-cell midpoints at r >= 1."""
    near2, far2 = [], []
    for e in edges:
        a, b = e[:-1], e[1:]
        near = np.where((a <= 0) & (b >= 0), 0.0, np.minimum(np.abs(a), np.abs(b)))
        near2.append(near * near)
        far = np.maximum(np.abs(a), np.abs(b))
        far2.append(far * far)
    n2 = near2[0][:, None, None] + near2[1][None, :, None] + near2[2][None, None, :]
    f2 = far2[0][:, None, None] + far2[1][None, :, None] + far2[2][None, None, :]
    out = np.where(n2 >= 1.0, 1.0, 0.0)
    cut = np.nonzero((n2 < 1.0) & (f2 > 1.0))
    t = (np.arange(sub) + 0.5) / sub
    step = 4096
    for s in range(0, len(cut[0]), step):
        r2 = 0.
        for k, e in enumerate(edges):
            idx = cut[k][s:s + step]
            c = e[idx][:, None] + t[None, :] * (e[idx + 1] - e[idx])[:, None]
            shape = [len(idx), 1, 1, 1]
            shape[k + 1] = sub
            r2 = r2 + (c * c).reshape(shape)
        out[tuple(c[s:s + step] for c in cut)] = (r2 >= 1.0).mean(axis=(1, 2, 3))
    return out


class ModelIonization:
    def __init__(self, inputs, params=None, device=None):
        params = {} if params is None else params
        if not isinstance(params, dict):
            raise ValueError('params must be a dict')
        if inputs.options.step_size != 0:
            raise ValueError('ModelIonization needs the adaptive driver (options.step_size = 0); '
                             'constant-step runs do not define the loss of a packet per step')
        dims, lo, hi = grid_params(params)
        self.inputs = copy.deepcopy(inputs)
        if get_setup(self.inputs).params.loss_mode == 0:
            raise ValueError('ModelIonization needs a loss process (a lifetime or a photo rate); '
                             'this input loses nothing in flight, the map would be zero')
        self.params = params
        self.type = 'ionization'
        self._device = local_device() if device is None else device
        self.dims = tuple(dims)
        self.edges = tuple(np.linspace(a, b, n + 1) for a, b, n in zip(lo, hi, dims))
        self.xaxis, self.yaxis, self.zaxis = (0.5 * (e[:-1] + e[1:]) for e in self.edges)

        self.outid, self.outputfiles, outputs, recipes = regeneration_plan(self.inputs)
        comm = nccl_comm()
        grid = np.zeros(self.dims)
        cnt = np.zeros(self.dims, dtype=np.int64)
        outside, outside_count = np.zeros(1), np.zeros(1, dtype=np.int64)
        totalsource = 0.
        self.attempted_steps = self.accepted_steps = self.bounces = 0
        self.kernel_ms = 0.0
        if outputs or comm is not None:
            eng = get_engine(self._device)
            eng.ionize_begin(lo, hi, dims)
            try:
                totalsource = regenerate(self, eng, outputs, recipes,
                                         Engine.integrate_adaptive_ionize)
                if comm is not None:          # one collective; totalsource rides with the grid
                    totalsource = eng.ionize_allreduce(comm[1], totalsource)
                grid, cnt, o_sum, o_cnt = eng.ionize_fetch(dims)
                outside[0], outside_count[0] = o_sum, o_cnt
            finally:
                eng.ionize_end()
        if comm is None:
            totalsource, = combine_ranks((grid, cnt, outside, outside_count), totalsource)
        self._finish(grid, cnt, float(outside[0]), int(outside_count[0]), totalsource)

    def _finish(self, grid, cnt, outside, outside_count, totalsource):
        self.totalsource = totalsource
        endtime = float(value_of(self.inputs.options.endtime))
        self.atoms_per_packet = 1e23 / (totalsource / endtime) if totalsource > 0 else np.nan
        self.sourcerate = Quantity(1e23, '1/s')
        r_cm = float(value_of(self.inputs.geometry.planet.radius)) * 1e5
        self.ionized = grid
        self.packet_grid = cnt
        self.outside, self.outside_count = outside, outside_count
        self.exterior_fraction = exterior_fraction(self.edges)
        cell = np.prod([e[1] - e[0] for e in self.edges]) * r_cm**3
        v_ext = self.exterior_fraction * cell
        with np.errstate(divide='ignore', invalid='ignore'):
            self.production = np.where(v_ext > 0, grid * self.atoms_per_packet / endtime / v_ext,
                                       np.nan)
        self.production_unit = 'cm-3 s-1'
        self.rate = (grid.sum() + outside) * self.atoms_per_packet / endtime

    def __repr__(self):
        return self.__str__()

    def __str__(self):
        nx, ny, nz = self.dims
        box = ' x '.join(f'[{e[0]:.4g}, {e[-1]:.4g}]' for e in self.edges)
        return f'''Model Ionization
grid = {nx} x {ny} x {nz} (x, y, z) over {box} R_p
totalsource = {self.totalsource}
atoms per packet = {self.atoms_per_packet}
rate = {self.rate:.4g} ions/s (outside the grid {self.outside:.4g} of frac)'''
