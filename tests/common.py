"""Shared helpers for the tests: workload loading, oracle constants from a
RunSetup, comparison metrics."""
import os
import sys

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

WORKLOADS = os.path.join(REPO, 'nexoclom_b200', 'workloads')
GOLDEN = os.path.join(REPO, 'tests', 'golden')


def workload(name):
    from nexoclom_b200.Input import Input
    return Input(os.path.join(WORKLOADS, name))


def oracle_constants(setup):
    """oracle.tracking.RunConstants carrying the same numbers as setup.params."""
    from oracle.tracking import RunConstants
    p = setup.params
    sint = setup.inputs.surfaceinteraction
    return RunConstants(
        GM=p.GM, vrplanet=p.vrplanet, gravity=bool(p.gravity), radpres=bool(p.radpres),
        radpres_v=setup.radpres_v, radpres_a=setup.radpres_a,
        lifetime=(1.0 / p.loss_rate if p.loss_mode == 1 else 0.0),
        photo=(p.loss_rate if p.loss_mode == 2 else None),
        resolution=p.resolution if p.resolution > 0 else 1e-4, outeredge=p.outeredge,
        step_size=p.step_size, endtime=p.endtime, sticktype=sint.sticktype,
        stickcoef=getattr(sint, 'stickcoef', 1.0),
        accomfactor=sint.accomfactor, A=tuple(p.stick_A),
        taa=float(np.asarray(setup.inputs.geometry.taa)),
        planet_radius_km=p.planet_radius_km,
        v_interp=(setup.surfaceint.v_interp if setup.surfaceint is not None and
                  setup.surfaceint.tck is not None else None),
        moons=list(getattr(setup, 'moons', [])))


def vec_rel(a, b):
    """|a-b| / |b| per row for (N,3) arrays."""
    return np.linalg.norm(a - b, axis=1) / np.maximum(np.linalg.norm(b, axis=1), 1e-300)


def state_parity(X_gpu, X_ref):
    """Relative differences between two (N,8) packet tables.  `pos` / `vel` (vector norms)
    and `time` cover EVERY packet whose alive flag agrees -- the dead ones too: their last
    position decides a pixel of `packet_image` when compress=False -- `frac` the packets
    alive in both (it is exactly 0 for the dead).  Returns maxima and mismatch counts."""
    alive_g, alive_r = X_gpu[:, 7] > 0, X_ref[:, 7] > 0
    both = alive_g & alive_r
    same = alive_g == alive_r
    out = dict(alive_mismatch=int((~same).sum()), n_both=int(both.sum()),
               n_dead_both=int((same & ~alive_g).sum()))
    if same.any():
        out['pos'] = float(vec_rel(X_gpu[same, 1:4], X_ref[same, 1:4]).max())
        out['vel'] = float(vec_rel(X_gpu[same, 4:7], X_ref[same, 4:7]).max())
        out['time'] = float(np.abs(X_gpu[same, 0] - X_ref[same, 0]).max())
        out['frac'] = 0.0
    if both.any():
        out['frac'] = float((np.abs(X_gpu[both, 7] - X_ref[both, 7]) / X_ref[both, 7]).max())
    return out


# ---------------------------------------------------------------------------- kernel builds
# The integrators have no runtime force flags on the fast path: nx_kernels.cu sends each run to
# a build whose forces and loss are template arguments, MODE = gravity*8 + radpres*4 + loss_mode
# (+16 with one moon).  A cell of the matrix below is one such choice, set through the real
# knobs of an Input, so that every build can be run against the oracle.
LOSSES = ('none', 'lifetime', 'photo')          # loss_mode 0, 1, 2


class Cell:
    """One force x loss x moon choice on a base workload.  `driver` is 'adaptive' or
    'constant'; `bounce`: sticking 0.5 with accommodation (Na.bounce.stick05.input's surface)
    instead of perfect sticking."""

    def __init__(self, driver, bounce, moon, gravity, radpres, loss):
        assert driver in ('adaptive', 'constant') and loss in LOSSES
        assert not (driver == 'constant' and not bounce)
        self.driver, self.bounce, self.moon = driver, bool(bounce), bool(moon)
        self.gravity, self.radpres, self.loss = bool(gravity), bool(radpres), loss

    @property
    def id(self):
        return (f"{self.driver[0]}{'b' if self.bounce else ''}{'m' if self.moon else ''}-"
                f"g{int(self.gravity)}r{int(self.radpres)}-{self.loss}")

    def __repr__(self):
        return self.id

    @property
    def endtime(self):
        # long enough that packets land, escape and survive; the loss time is the run length
        return 10000. if self.moon and not self.bounce else 1500. if self.bounce else 3000.

    def inputs(self):
        from nexoclom_b200.units import Quantity
        if self.moon:
            inputs = workload('Na.Io.Jupiter.input')
            # Io passes through Jupiter's shadow during the run, so the packets around it see
            # lit and shadowed stages
            inputs.geometry.phi = (Quantity(0.2, 'rad'),)
            if self.bounce:
                # packets from Io hardly ever reach Jupiter: start them on the planet, where
                # they hop and bounce while the moon's gravity still acts on every stage.
                # Sticking 0.5 without accommodation: Jupiter has no surface temperature model.
                # Speeds 1-3 km/s: a packet launched near 0 km/s comes to rest on the surface,
                # where its velocity has no relative accuracy.
                inputs.surfaceinteraction = workload('Na.bounce.stick05.input').surfaceinteraction
                inputs.surfaceinteraction.accomfactor = 0.
                inputs.speeddist.vprob = Quantity(2., 'km/s')
                inputs.speeddist.delv = Quantity(1., 'km/s')
                inputs.geometry.startpoint = inputs.geometry.planet.object
        else:
            inputs = workload('Na.bounce.stick05.input' if self.bounce
                              else 'Na.maxwellian.radpres.input')
        if self.driver == 'adaptive':
            inputs.options.step_size = 0.
            inputs.options.resolution = 1e-4
        inputs.forces.gravity = self.gravity
        inputs.forces.radpres = self.radpres
        inputs.options.endtime = Quantity(self.endtime, 's')
        if self.loss == 'lifetime':                       # loss_mode 1: constant lifetime
            inputs.options.lifetime = Quantity(self.endtime, 's')
        elif self.loss == 'photo':                        # loss_mode 2: generic photo rate,
            inputs.options.lifetime = Quantity(-self.endtime, 's')        # shadowed
        else:
            inputs.options.lifetime = Quantity(0., 's')
        return inputs

    def setup(self, strict_math=False):
        from nexoclom_b200.runsetup import RunSetup
        setup = RunSetup(self.inputs(), strict_math=strict_math)
        p = setup.params
        if self.loss == 'none':
            # No Input selects loss_mode 0 for a species with a tabulated photo rate (lifetime 0
            # looks the rate up in RunSetup.__init__); the C ABI takes RunParams as they are.
            p.loss_mode, p.loss_rate = 0, 0.0
        assert p.loss_mode == LOSSES.index(self.loss)
        assert (bool(p.gravity), bool(p.radpres), p.nmoons) == (self.gravity, self.radpres,
                                                                int(self.moon))
        return setup

    def x0(self, setup, n, seed):
        """(n, 8) initial states.  With bounce, every 16th packet starts with frac 3e-10, so
        that it vanishes after a bounce or two: a bounce run has dead packets too."""
        from oracle import initial_state
        X0 = initial_state.draw_x0(setup, n, seed)[:, :8]
        if self.bounce:
            X0[::16, 7] = 3e-10
        return X0


def _kernel_cells():
    from itertools import product
    fr = list(product((True, False), (True, False), LOSSES))
    adaptive = [Cell('adaptive', False, False, g, r, loss) for g, r, loss in fr]
    adaptive += [Cell('adaptive', False, True, True, r, loss) for _, r, loss in fr[:6]]
    adaptive += [Cell('adaptive', True, m, True, r, loss) for m in (False, True)
                 for _, r, loss in fr[:6]]
    # the strict builds a run falls back to: a moon without gravity, bounce without gravity
    adaptive += [Cell('adaptive', False, True, False, True, 'photo'),
                 Cell('adaptive', True, False, False, True, 'photo')]
    constant = [Cell('constant', True, False, g, r, loss) for g, r, loss in fr]
    return adaptive + constant


# every fast build of the three dispatchers, and the strict fallbacks (test_kernel_builds.py)
KERNEL_CELLS = _kernel_cells()


def adaptive_mode(p, bounce=False):
    """MODE of the k_integrate_adaptive build dispatch_adaptive (nx_kernels.cu) selects for
    RunParams p; -1 is the strict (generic) build.  The bounce builds need gravity."""
    if p.strict_math or p.nmoons > 1:
        return -1
    if (bounce or p.nmoons == 1) and not p.gravity:
        return -1
    return (8 if p.gravity else 0) | (4 if p.radpres else 0) | (p.loss_mode & 3) | \
        (16 if p.nmoons == 1 else 0)


def stream_mode(p):
    """MODE of k_integrate_adaptive_stream (launch_integrate_adaptive_stream)."""
    if p.strict_math or p.nmoons > 1 or (p.nmoons == 1 and not p.gravity):
        return -1
    return (8 if p.gravity else 0) | (4 if p.radpres else 0) | (p.loss_mode & 3) | \
        (16 if p.nmoons == 1 else 0)


def constant_mode(p):
    """MODE of k_integrate_constant (launch_integrate_constant): no fast build with moons."""
    if p.strict_math or p.nmoons > 0:
        return -1
    return (8 if p.gravity else 0) | (4 if p.radpres else 0) | (p.loss_mode & 3)


def kernel_builds(p, driver, bounce):
    """The kernel builds a run with RunParams p makes through every entry of its driver, as
    (kernel, template arguments): the adaptive driver's resident run (K2 / K2b), its deposition
    sink (K2d) and, without bounce, its host-buffer stream (K2s); the constant-step driver with
    and without the row sink (K3)."""
    if driver == 'constant':
        m = constant_mode(p)
        return {('k_integrate_constant', (m, False)), ('k_integrate_constant', (m, True))}
    m = adaptive_mode(p, bounce)
    out = {('k_integrate_adaptive', (m, bounce, False)), ('k_integrate_adaptive', (m, bounce, True))}
    if not bounce:
        out.add(('k_integrate_adaptive_stream', (stream_mode(p),)))
    return out


def source_case_input(tag):
    """Parsed tests/golden/source_cases/<tag>.input; table files named relative to the repo
    root are made absolute so the tests run from any directory."""
    from nexoclom_b200.Input import Input
    inputs = Input(os.path.join(GOLDEN, 'source_cases', tag + '.input'))
    for group, attr in ((inputs.spatialdist, 'mapfile'), (inputs.speeddist, 'vdistfile')):
        path = getattr(group, attr, None)
        if isinstance(path, str) and path != 'default' and not os.path.isabs(path):
            setattr(group, attr, os.path.join(REPO, path))
    return inputs
