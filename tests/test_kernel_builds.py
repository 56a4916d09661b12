"""Every integrator kernel build against the oracle.  nx_kernels.cu sends each run to a build
with its forces and loss as template arguments (MODE = gravity*8 + radpres*4 + loss_mode, +16
with one moon), so a build that no workload selects is never run by the other tests.  The cells
of common.KERNEL_CELLS set the real knobs of an Input for every build; here (CPU) they are shown
to cover every build the dispatchers can select, and (GPU) every family a cell selects is run:

  K2   k_integrate_adaptive<MODE>                  resident run, perfect sticking
  K2b  k_integrate_adaptive<MODE, BOUNCE>          sticking 0.5 (bounce cells)
  K2d  k_integrate_adaptive<MODE, BOUNCE, SINK>    the same runs through the deposition sink
  K2s  k_integrate_adaptive_stream<MODE>           the host-buffer stream of a K2 run
  K3   k_integrate_constant<MODE, ROWS>            constant step with bounce, with the row sink

The oracle runs once per cell: oracle.deposition gives the states, the step counts and the
events of one run (pinned bit for bit to oracle.tracking / oracle.adaptive_bounce in
test_deposition.py)."""
import os
import re

import numpy as np
import pytest

from common import (REPO, KERNEL_CELLS, adaptive_mode, constant_mode, kernel_builds,
                    oracle_constants, state_parity, stream_mode)
from nexoclom_b200._lib import RunParams
from oracle import adaptive_bounce, deposition, initial_state, tracking

ADAPTIVE = [c for c in KERNEL_CELLS if c.driver == 'adaptive']
CONSTANT = [c for c in KERNEL_CELLS if c.driver == 'constant']
N, SEED, FIRST = 2000, 17, 123
NLON, NLAT = 72, 36
K2_TOL = 1e-11               # the host build's gate (test_hostcheck.py)
STATE_TOL = 1e-8             # with bounce (test_adaptive_bounce.py) and for K3 (test_gpu_parity.py)
KERNELS = os.path.join(REPO, 'nexoclom_b200', 'csrc', 'nx_kernels.cu')


def cell_builds(cells):
    out = set()
    for c in cells:
        out |= kernel_builds(c.setup().params, c.driver, c.bounce)
    return out


def dispatch_cases():
    """(kernel, template arguments, case label) of every `case N: return launch_..._mode<...>`
    line of nx_kernels.cu's dispatchers.  launch_adaptive_mode's SINK argument stands for both
    builds; launch_constant_mode launches k_integrate_constant with and without ROWS."""
    src = open(KERNELS).read()
    out = []
    for label, fn, args in re.findall(r'case\s+(\d+):\s*return\s+(launch_\w+_mode)<([^>]*)>', src):
        a = [x.strip() for x in args.split(',')]
        if fn == 'launch_adaptive_mode':
            assert a[2] == 'SINK', args
            out += [('k_integrate_adaptive', (int(a[0]), a[1] == 'true', s), int(label))
                    for s in (False, True)]
        elif fn == 'launch_adaptive_stream_mode':
            out.append(('k_integrate_adaptive_stream', (int(a[0]),), int(label)))
        elif fn == 'launch_constant_mode':
            out += [('k_integrate_constant', (int(a[0]), r), int(label)) for r in (False, True)]
        else:
            raise AssertionError(f'unknown dispatch target {fn}')
    return out


def test_matrix_covers_every_dispatched_build():
    """The fast builds the cells select are exactly those the dispatchers' case lines launch:
    a build added to nx_kernels.cu without a cell fails here."""
    cases = dispatch_cases()
    source = {(k, a) for k, a, _ in cases}
    # K2s; K3 with and without ROWS; K2 and K2b with and without SINK
    assert len(source) == 18 + 2 * 12 + 2 * 18 + 2 * 12
    builds = cell_builds(KERNEL_CELLS)
    assert {b for b in builds if b[1][0] >= 0} == source
    # and the cells reach the strict fallbacks of the adaptive dispatchers
    assert {b for b in builds if b[1][0] < 0} == {
        ('k_integrate_adaptive', (-1, False, False)), ('k_integrate_adaptive', (-1, False, True)),
        ('k_integrate_adaptive', (-1, True, False)), ('k_integrate_adaptive', (-1, True, True)),
        ('k_integrate_adaptive_stream', (-1,))}


def test_dispatch_restatement_matches_case_labels():
    """common.adaptive_mode / stream_mode / constant_mode against the case tables: RunParams
    with the label's forces select the build the case launches.  The bounce switch's key
    leaves gravity out (its builds all have it)."""
    for kernel, args, label in dispatch_cases():
        p = RunParams()
        p.gravity = int(bool(label & 8) or (kernel == 'k_integrate_adaptive' and args[1]))
        p.radpres, p.loss_mode, p.nmoons = int(bool(label & 4)), label & 3, (label >> 4) & 1
        if kernel == 'k_integrate_adaptive':
            assert adaptive_mode(p, bounce=args[1]) == args[0], (kernel, args, label)
        elif kernel == 'k_integrate_adaptive_stream':
            assert stream_mode(p) == args[0], (kernel, args, label)
        else:
            assert constant_mode(p) == args[0], (kernel, args, label)
    # the strict fallbacks
    p = RunParams()
    p.gravity, p.radpres, p.loss_mode = 1, 1, 2
    assert (adaptive_mode(p), adaptive_mode(p, True), stream_mode(p), constant_mode(p)) == \
        (14, 14, 14, 14)
    p.strict_math = 1
    assert (adaptive_mode(p), adaptive_mode(p, True), stream_mode(p), constant_mode(p)) == \
        (-1, -1, -1, -1)
    p.strict_math, p.nmoons = 0, 2
    assert (adaptive_mode(p), adaptive_mode(p, True), stream_mode(p), constant_mode(p)) == \
        (-1, -1, -1, -1)
    p.nmoons = 1
    assert (adaptive_mode(p), adaptive_mode(p, True), stream_mode(p), constant_mode(p)) == \
        (30, 30, 30, -1)
    p.gravity = 0
    assert (adaptive_mode(p), adaptive_mode(p, True), stream_mode(p)) == (-1, -1, -1)
    p.nmoons = 0
    assert (adaptive_mode(p), adaptive_mode(p, True), stream_mode(p), constant_mode(p)) == \
        (6, -1, 6, 6)


def shadowed(X):
    """Rows (time, x, y, z, ...) inside the planet's shadow (the sun is toward -y)."""
    return (X[:, 1] ** 2 + X[:, 3] ** 2 <= 1.0) & (X[:, 2] >= 0.0)


# ---------------------------------------------------------------------------- GPU
def run_adaptive(engine, cell, setup, X0, nlon=NLON, nlat=NLAT):
    """The cell's K2 / K2b run, its K2s stream (perfect sticking only) and its K2d run.
    Returns (state, (attempted, accepted, bounces), (attempted, accepted) per packet), the
    stream's run (or None) and the sink's run with the sink's contents."""
    setup.upload(engine)
    engine.import_state(X0)
    if cell.bounce:
        tot = engine.integrate_adaptive_bounce(SEED, FIRST)
    else:
        tot = engine.integrate_adaptive() + (0,)
    resident = (engine.export_state().T, tot, engine.export_stats())
    stream = None
    if not cell.bounce:
        t = engine.integrate_adaptive_host(X0, nchunks=3)
        stream = (engine.export_state().T, t + (0,), engine.export_stats())
    engine.import_state(X0)
    engine.deposit_begin(nlon, nlat)
    try:
        t = engine.integrate_adaptive_deposit(SEED, FIRST)
        got = engine.deposit_fetch(nlon, nlat)
    finally:
        engine.deposit_end()
    sink = (engine.export_state().T, t, engine.export_stats())
    return resident, stream, sink, got


def run_constant(engine, setup, X0):
    """K3 with the dense trajectory, then with the row sink, on the same packets."""
    setup.upload(engine)
    engine.import_state(X0)
    traj, nsteps, steps = engine.integrate_constant(seed=SEED, first_id=FIRST, trajectory=True)
    engine.import_state(X0)
    tab, nsteps_r, steps_r = engine.integrate_constant_rows(seed=SEED, first_id=FIRST,
                                                            skip_dead=True)
    try:
        cols, index, step = tab.export(with_step=True)
    finally:
        tab.free()
    return traj, nsteps, steps, (cols, index, step, nsteps_r, steps_r)


def same_run(a, b):
    return (np.array_equal(a[0], b[0]) and a[1] == b[1] and np.array_equal(a[2][0], b[2][0])
            and np.array_equal(a[2][1], b[2][1]))


@pytest.mark.gpu
@pytest.mark.parametrize('cell', ADAPTIVE, ids=str)
def test_adaptive_builds_match_oracle(engine, cell):
    setup = cell.setup()
    p = setup.params
    mode = adaptive_mode(p, cell.bounce)
    X0 = cell.x0(setup, N, 21)
    Xo, a_o, c_o, b_o, ev, _ = deposition.integrate_adaptive(
        X0, oracle_constants(setup), adaptive_bounce.bounce_uniforms(SEED, FIRST))
    resident, stream, sink, got = run_adaptive(engine, cell, setup, X0)

    # K2 / K2b against the oracle
    Xg, tot, (a_g, c_g) = resident
    par = state_parity(Xg, Xo)
    print(cell, 'MODE', mode, par, 'bounces', tot[2])
    assert par['alive_mismatch'] == 0, par
    assert np.array_equal(a_g, a_o) and np.array_equal(c_g, c_o)
    assert tot == (int(a_o.sum()), int(c_o.sum()), int(b_o.sum()))
    assert max(par['pos'], par['vel'], par['frac']) < (STATE_TOL if cell.bounce else K2_TOL), par
    assert np.all(Xg[Xo[:, 7] == 0, 0] == 0)                      # dead => time = 0
    # K2s: the stream of the host buffers is the resident run, bit for bit
    if stream is not None:
        assert same_run(stream, resident)
    # K2d: the sink leaves the run as it was, and its contents are the oracle's events
    assert same_run(sink, resident)
    from test_deposition import compare_sink
    compare_sink(got, ev, NLON, NLAT, exact_cells=mode < 0)
    if cell.bounce:
        assert got[3][deposition.SURFACE] == int(b_o.sum())

    # the cell exercised what its build compiles in
    alive = Xo[:, 7] > 0
    assert alive.any()
    if cell.gravity or cell.radpres or cell.moon:                 # something ends a flight
        assert (~alive).any()
    if cell.loss != 'none':
        assert (Xo[alive, 7] < 0.9).any()
    if cell.bounce and (cell.gravity or cell.radpres):
        assert b_o.sum() > 0
    if cell.radpres or cell.loss == 'photo':
        rows = np.concatenate([X0[a_o > 0], Xo[alive]])
        sh = shadowed(rows)
        assert sh.any() and (~sh).any()


@pytest.mark.gpu
@pytest.mark.parametrize('cell', CONSTANT, ids=str)
def test_constant_builds_match_oracle(engine, cell):
    setup = cell.setup()
    X0 = cell.x0(setup, N, 9)
    hits = []
    uniforms = initial_state.bounce_uniforms(SEED, FIRST)

    def counted(ct, idx):
        hits.append(len(idx))
        return uniforms(ct, idx)

    ref, nsteps, natt = tracking.integrate_constant(X0, oracle_constants(setup), uniforms=counted)
    traj, ns, steps, (cols, index, step, ns_r, steps_r) = run_constant(engine, setup, X0)
    assert ns == nsteps and traj.shape == ref.shape
    assert np.array_equal(traj[:, 7, :] > 0, ref[:, 7, :] > 0)
    err = np.max(np.abs(traj - ref) / np.maximum(np.abs(ref), 1e-3))
    print(cell, 'MODE', constant_mode(setup.params), 'max rel', err, 'bounces', sum(hits))
    assert err < STATE_TOL
    assert steps == int(natt.sum())
    # ROWS: the sink keeps the live rows of the same trajectory, float32
    assert ns_r == nsteps and steps_r == steps
    pk, st = np.nonzero(traj[:, 7, :] > 0)
    order = np.lexsort((step, index))
    assert len(index) == len(pk)
    assert np.array_equal(index[order], pk) and np.array_equal(step[order], st)
    for k, c in enumerate(('time', 'x', 'y', 'z', 'vx', 'vy', 'vz', 'frac')):
        assert np.array_equal(cols[c][order], traj[pk, k, st].astype(np.float32)), c

    final = ref[:, 7, -1]
    assert (final > 0).any()
    if cell.gravity:               # without it the run is too short for a packet to vanish
        assert (final == 0).any()
    if cell.loss != 'none':
        assert (final[final > 0] < 0.9).any()
    if cell.gravity or cell.radpres:
        assert sum(hits) > 0
    if cell.radpres or cell.loss == 'photo':
        sh = shadowed(traj.transpose(0, 2, 1)[pk, st])
        assert sh.any() and (~sh).any()


_KERNEL_NAME = re.compile(r'(k_integrate_(?:adaptive_stream|adaptive|constant))<([^>]*)>')


def build_of(name):
    """('k_integrate_adaptive', (14, False, False)) from a demangled kernel name, or None."""
    m = _KERNEL_NAME.search(name)
    if not m:
        return None
    args = []
    for a in m.group(2).split(','):
        a = re.sub(r'^\((?:int|bool)\)', '', a.strip())
        args.append(a == 'true' if a in ('true', 'false') else int(a))
    return m.group(1), tuple(args)


def test_kernel_name_parser():
    assert build_of('void nx::k_integrate_adaptive<14, false, true>(nx::StateCols, long long)') == \
        ('k_integrate_adaptive', (14, False, True))
    assert build_of('void k_integrate_adaptive_stream<-1>(double const*)') == \
        ('k_integrate_adaptive_stream', (-1,))
    assert build_of('void nx::k_integrate_constant<(int)9, true>(x)') == \
        ('k_integrate_constant', (9, True))
    assert build_of('void nx::k_cost_histogram(nx::StateCols)') is None


@pytest.mark.gpu
def test_profiler_sees_every_build(engine):
    """The matrix once under torch.profiler: the integrator kernels that ran are exactly the
    builds the cells select (common.kernel_builds), so the restatement of the dispatch, and
    with it the coverage test above, is what the library does."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for cell in KERNEL_CELLS:
            setup = cell.setup()
            X0 = cell.x0(setup, 256, 3)
            if cell.driver == 'adaptive':
                run_adaptive(engine, cell, setup, X0, 8, 4)
            else:
                run_constant(engine, setup, X0)
        engine.sync()
    names = {e.name for e in prof.events() if 'k_integrate_' in e.name}
    print('kernels seen:', sorted(names))
    seen = {build_of(n) for n in names} - {None}
    assert seen == cell_builds(KERNEL_CELLS)
