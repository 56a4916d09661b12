"""``ModelTrajectoryImage`` and ``ModelTrajectoryDensity``: images and number-density grids
from every accepted step of the adaptive driver, not only from the state it saves.

The snapshot products (``ModelImage``, ``ModelDensity``, ...) bin the one row per packet an
adaptive ``Output`` keeps, and in a bound exosphere most packets have retired by then.  These
products regenerate every output file of the ``Input`` exactly as ``ModelIonization`` does
(``regeneration_plan`` / ``regenerate``: K1 from the seed and ``first_id``, or the imported X0)
through the trajectory sink of the adaptive driver (``nx_integrate_adaptive_trace``), so the run
is the run the user made, bit for bit.  The reference has no such product; DESIGN.md section 8
states the semantics.  For every accepted step, with ``T = endtime``, ``t0`` the packet's
initial time remaining, ``t`` the time remaining before the step and ``h`` the step:

* the step is represented by the midpoint ``m = (s + s_rk) * 0.5`` of the state before it and
  the Runge-Kutta state (before any surface, moon, escape or vanish handling);
* its weight is the age-weighted dwell ``a = h * T / ((T - t0) + (t - h / 2))``: the packets are
  released uniformly over ``(0, T]``, so a packet is still in flight at age ``a`` with
  probability ``(T - a) / T``; dividing by it (at the midpoint's age ``t0 - t + h / 2``) makes
  the sums estimate the same steady state as the snapshot at ``time = 0``;
* the image adds ``w(m) * a`` at ``m``'s pixel, ``w`` being ``ModelImage``'s weight (frac,
  occultation, and for radiance the sunlit mask and g-values) of the midpoint; the grid adds
  ``frac(m) * a`` at ``m``'s cell (``np.histogramdd``'s rule, OUTSIDE beyond the box);
* ``image = sums * atoms_per_packet / T``, in ``ModelImage.image``'s units and with its
  expectation; ``density = dwell * atoms_per_packet / T / V_ext`` in atoms cm^-3 for a source
  of 1e23 atoms/s, ``V_ext`` the part of the cell outside the planet (NaN for a cell wholly
  inside it), as in ``ModelIonization``.

Every accepted step is a sample, so for the same packets the noise is several times to tens of
times lower than the snapshot's.  Caveats: a step goes to the one pixel or cell of its
midpoint, not split over the ones its chord crosses; a step that ends inside the planet counts
its full ``h``.  The age weight assumes the reference's release law, ``t0 ~ U(0, T]``, which K1
follows for adaptive runs: an imported X0 must have every ``time`` finite and in ``[0, T]``.

Refused with ``ValueError`` before any device work: constant-step inputs (``ModelImage`` already
samples every step of those), inputs with moons (the moon's phase makes the forces depend on
the time, so a sample at age ``a`` does not show the snapshot's state), imported X0 times
outside ``[0, T]`` or not finite, malformed params, and output files that cannot be regenerated.
"""
import copy

import numpy as np

from .engine import Engine, get_engine
from .ModelDeposition import regenerate, regeneration_plan
from .ModelImage import ModelImage
from .ModelIonization import exterior_fraction, grid_params
from .ModelResult import ModelResult
from .runsetup import get_setup
from .sharding import combine_ranks, local_device, nccl_comm
from .units import Quantity, value_of


def _numbers(params, key, default, count, positive_int=False):
    text = params.get(key, default)
    try:
        parts = [float(v) for v in str(text).split(',')]
        ok = len(parts) == count and all(np.isfinite(parts)) and not isinstance(text, bool)
        if positive_int:
            ok = ok and all(v == int(v) and v >= 1 for v in parts)
    except (TypeError, ValueError):
        ok = False
    if not ok:
        what = 'positive integers' if positive_int else 'finite numbers'
        raise ValueError(f'{key} must be {count} comma-separated {what}, got {text!r}')
    return parts


def image_trace_params(params):
    """Validate ``ModelImage``'s params for a trajectory image: ``quantity`` column or radiance,
    ``dims`` two positive integers (nx * nz < 2**30), ``center`` two finite numbers, ``width``
    two finite numbers > 0, the sub-observer point finite; ValueError otherwise."""
    if not isinstance(params, dict):
        raise ValueError('params must be a dict')
    if params.get('quantity') not in ('column', 'radiance'):
        raise ValueError(f"quantity must be 'column' or 'radiance', got {params.get('quantity')!r}")
    dims = _numbers(params, 'dims', '800,800', 2, positive_int=True)
    if dims[0] * dims[1] >= 2**30:
        raise ValueError(f'{int(dims[0])} x {int(dims[1])} pixels is 2**30 or more')
    _numbers(params, 'center', '0,0', 2)
    if min(_numbers(params, 'width', '8,8', 2)) <= 0:
        raise ValueError(f'width must be > 0 on both axes, got {params.get("width")!r}')
    _numbers(params, 'subobslongitude', '0', 1)
    _numbers(params, 'subobslatitude', repr(np.pi / 2), 1)


def check_trace_inputs(inputs, outputs, recipes):
    """The refusals both products share (ValueError): constant-step inputs, moons, and imported
    X0 times outside [0, endtime] or not finite."""
    if inputs.options.step_size != 0:
        raise ValueError('the trajectory products need the adaptive driver (options.step_size = 0); '
                         'ModelImage already samples every step of a constant-step run')
    if get_setup(inputs).params.nmoons != 0:
        raise ValueError('the trajectory products do not support moons: the moon moves, so a '
                         "step's sample at age a shows the forces of another time than the image")
    endtime = float(value_of(inputs.options.endtime))
    for kind, what in recipes:
        if kind != 'x0':
            continue
        t = np.asarray(what[:, 0] if isinstance(what, np.ndarray) and what.ndim == 2 else what[0],
                       dtype=np.float64)
        if not (np.all(np.isfinite(t)) and np.all((t >= 0) & (t <= endtime))):
            raise ValueError('an imported X0 has a time outside [0, endtime] or not finite; the '
                             "age weight assumes the reference's release law t0 ~ U(0, endtime]")


def run_trace(model, image_params, grid):
    """Regenerate every output file of ``model`` through the trajectory sink (one NCCL
    all-reduce per product, totalsource riding along; gloo through ``combine_ranks``).  Sets the
    step totals and ``kernel_ms``; returns (totalsource, trace_fetch's six values)."""
    comm = nccl_comm()
    npix = (0, 0) if image_params is None else (image_params.nx, image_params.nz)
    img = np.zeros(npix) if image_params is not None else None
    img_n = np.zeros(npix, dtype=np.int64) if image_params is not None else None
    g = gn = None
    if grid is not None:
        g, gn = np.zeros(grid[2]), np.zeros(grid[2], dtype=np.int64)
    outside, outside_n = np.zeros(1), np.zeros(1, dtype=np.int64)
    totalsource = 0.
    model.attempted_steps = model.accepted_steps = model.bounces = 0
    model.kernel_ms = 0.0
    if model._outputs or comm is not None:
        eng = get_engine(model._device)
        eng.trace_begin(image_params, grid)

        def integrate(eng, seed, first_id, n):
            model._upload_tables(eng)
            return Engine.integrate_adaptive_trace(eng, seed, first_id, n)
        try:
            totalsource = regenerate(model, eng, model._outputs, model._recipes, integrate)
            if comm is not None:
                totalsource = eng.trace_allreduce(comm[1], totalsource)
            fi, fin, fg, fgn, fo, fon = eng.trace_fetch()
        finally:
            eng.trace_end()
        if fi is not None:
            img, img_n = fi, fin
        if fg is not None:
            g, gn = fg, fgn
            outside[0], outside_n[0] = fo, fon
    if comm is None:
        arrays = [a for a in (img, img_n, g, gn) if a is not None]
        if grid is not None:
            arrays += [outside, outside_n]
        totalsource, = combine_ranks(tuple(arrays), totalsource)
    return totalsource, img, img_n, g, gn, float(outside[0]), int(outside_n[0])


def _scale(totalsource, endtime):
    return 1e23 / (totalsource / endtime) if totalsource > 0 else np.nan


class ModelTrajectoryImage(ModelImage):
    """Column or radiance image from every accepted step (see the module docstring).  Takes
    ``ModelImage``'s params (``quantity``, ``dims``, ``center``, ``width``, ``subobslongitude``,
    ``subobslatitude``, ``wavelength``, ``g``).

    Attributes: ``image`` (nx, nz) in ``ModelImage.image``'s units; ``step_image`` (nx, nz)
    int64 recorded steps per pixel; ``xaxis`` / ``zaxis``, ``Apix``, ``atoms_per_packet``,
    ``totalsource``, ``sourcerate``, ``attempted_steps``, ``accepted_steps``, ``bounces``,
    ``kernel_ms``."""

    def __init__(self, inputs, params, device=None):
        image_trace_params(params)
        ModelResult.__init__(self, inputs, params)
        self.type = 'trajectory image'
        self._image_geometry(self.inputs, device)
        self.outid, self.outputfiles, self._outputs, self._recipes = regeneration_plan(self.inputs)
        check_trace_inputs(self.inputs, self._outputs, self._recipes)
        ip = self.image_params(get_setup(self.inputs))
        totalsource, img, cnt, _, _, _, _ = run_trace(self, ip, None)
        self.totalsource = totalsource
        endtime = float(value_of(self.inputs.options.endtime))
        self.atoms_per_packet = _scale(totalsource, endtime)
        self.sourcerate = Quantity(1e23, '1/s')
        self.image = img * self.atoms_per_packet / endtime
        self.step_image = cnt

    def _upload_tables(self, eng):
        self._upload_weighting_tables(eng, eng._uploaded_setup)


class ModelTrajectoryDensity:
    """Number density on a box grid from every accepted step (see the module docstring).  Takes
    ``ModelIonization``'s grid params (``dims``, ``center``, ``width``, in R_p).

    Attributes: ``density`` (nx, ny, nz) atoms cm^-3 for a source of 1e23 atoms/s (NaN for cells
    wholly inside the planet); ``dwell`` (nx, ny, nz) sums of ``frac * a`` (s); ``step_grid``
    (nx, ny, nz) int64 recorded steps; ``outside`` / ``outside_count``; ``exterior_fraction``;
    ``xaxis`` / ``yaxis`` / ``zaxis`` (bin centres) and ``edges``; ``totalsource``,
    ``atoms_per_packet``, ``sourcerate``, ``attempted_steps``, ``accepted_steps``, ``bounces``,
    ``kernel_ms``."""

    def __init__(self, inputs, params=None, device=None):
        params = {} if params is None else params
        if not isinstance(params, dict):
            raise ValueError('params must be a dict')
        dims, lo, hi = grid_params(params)
        self.inputs = copy.deepcopy(inputs)
        self.params = params
        self.type = 'trajectory density'
        self._device = local_device() if device is None else device
        self.dims = tuple(dims)
        self.edges = tuple(np.linspace(a, b, n + 1) for a, b, n in zip(lo, hi, dims))
        self.xaxis, self.yaxis, self.zaxis = (0.5 * (e[:-1] + e[1:]) for e in self.edges)
        self.outid, self.outputfiles, self._outputs, self._recipes = regeneration_plan(self.inputs)
        check_trace_inputs(self.inputs, self._outputs, self._recipes)
        totalsource, _, _, grid, cnt, outside, outside_count = run_trace(
            self, None, (lo, hi, self.dims))
        self.totalsource = totalsource
        endtime = float(value_of(self.inputs.options.endtime))
        self.atoms_per_packet = _scale(totalsource, endtime)
        self.sourcerate = Quantity(1e23, '1/s')
        self.dwell = grid
        self.step_grid = cnt
        self.outside, self.outside_count = outside, outside_count
        self.exterior_fraction = exterior_fraction(self.edges)
        r_cm = float(value_of(self.inputs.geometry.planet.radius)) * 1e5
        v_ext = self.exterior_fraction * np.prod([e[1] - e[0] for e in self.edges]) * r_cm**3
        with np.errstate(divide='ignore', invalid='ignore'):
            self.density = np.where(v_ext > 0, grid * self.atoms_per_packet / endtime / v_ext,
                                    np.nan)
        self.density_unit = 'cm-3'

    def _upload_tables(self, eng):
        pass

    def __repr__(self):
        return self.__str__()

    def __str__(self):
        nx, ny, nz = self.dims
        box = ' x '.join(f'[{e[0]:.4g}, {e[-1]:.4g}]' for e in self.edges)
        return f'''Model Trajectory Density
grid = {nx} x {ny} x {nz} (x, y, z) over {box} R_p
totalsource = {self.totalsource}
atoms per packet = {self.atoms_per_packet}'''
