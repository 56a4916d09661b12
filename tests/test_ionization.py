"""3-D ion production maps of the adaptive driver (K2i: k_ionize_adaptive,
nx_integrate_adaptive_ionize, Engine.integrate_adaptive_ionize, ModelIonization).  The oracle
is oracle/ionization.py: the deposition oracle's adaptive driver with a recorder, pinned here to
oracle.deposition bit for bit, that sees every accepted step's loss, ``frac before - frac of the
Runge-Kutta step``, at the midpoint of its chord.

A step whose frac does not change is not recorded.  In the planet's shadow (photo-loss) the
fast path's frac is unchanged exactly, while the strict path and the oracle form
exp(log f), which may differ from f by an ulp: those steps record a loss of about 1e-16 or
nothing, depending on the implementation's libm.  The comparisons below therefore take an
oracle step of |loss| <= AMBIGUOUS as one an implementation may or may not record, and a strict
implementation may also record (with a loss of an ulp) one of the oracle's accepted steps whose
frac came back unchanged: each cell's count lies between the oracle's count of larger steps and
that plus its ambiguous ones, plus for the strict path the oracle's unrecorded accepted steps
(all three equal for a lifetime loss, where every step loses frac).  The sums bound what those
steps can carry."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from common import REPO, KERNEL_CELLS, Cell, adaptive_mode, oracle_constants, state_parity, workload
from nexoclom_b200._lib import dptr
from oracle import adaptive_bounce, deposition, initial_state, ionization

U32P = C.POINTER(C.c_uint32)
U64P = C.POINTER(C.c_uint64)
EDGE_TOL = 1e-12             # R_p: midpoints this close to a cell edge may bin either side
SUM_TOL = 1e-12              # x SOURCE
AMBIGUOUS = 1e-15            # |loss| of a step that may or may not be recorded (see above)
EXTERIOR_TOL = 0.01          # |16^3 - 64^3| exterior fraction of a cut cell (see below)
# a non-cubic, off-centre box
LO, HI, DIMS = (-3.1, -2.7, -2.2), (3.3, 4.1, 2.6), (23, 31, 17)
WORKLOADS = ['Ca.isotropic.flat.input', 'Na.maxwellian.radpres.input', 'Na.bounce.adaptive.input',
             'Na.bounce.stick05.input']
LIFETIME = [Cell('adaptive', False, False, True, True, 'lifetime'),
            Cell('adaptive', True, False, True, False, 'lifetime')]
ION_CELLS = [c for c in KERNEL_CELLS if c.driver == 'adaptive' and c.loss != 'none']


def setup_of(wl, strict_math=False):
    if isinstance(wl, Cell):
        return wl.setup(strict_math=strict_math)
    from test_deposition import setup_of as dep_setup
    return dep_setup(wl, strict_math)


def x0_of(wl, setup, n, seed):
    if isinstance(wl, Cell):
        return wl.x0(setup, n, seed)
    return initial_state.draw_x0(setup, n, seed)[:, :8]


def is_bounce(setup):
    p = setup.params
    return not (p.sticktype == 0 and p.stickcoef == 1.0)


def run_oracle(setup, X0, seed, first_id=0):
    """(X, attempted, accepted, bounces, events, loss) and the recorder of the same run."""
    rec = ionization.Recorder()
    out = ionization.integrate_adaptive(X0, oracle_constants(setup),
                                        adaptive_bounce.bounce_uniforms(seed, first_id),
                                        recorder=rec)
    return out, rec


def silent_steps(accepted, rec):
    """The oracle's accepted steps that recorded nothing (frac unchanged)."""
    return int(accepted.sum()) - len(rec.arrays()[1])


def edge_cells(mid, lo, hi, dims, tol=EDGE_TOL):
    """Cells (and -1 for OUTSIDE) a midpoint within `tol` of a cell edge may bin into."""
    e = ionization.edges(lo, hi, dims)
    near = np.zeros(len(mid), bool)
    for k in range(3):
        i = np.clip(np.searchsorted(e[k], mid[:, k]), 1, len(e[k]) - 1)
        d = np.minimum(np.abs(mid[:, k] - e[k][i - 1]), np.abs(mid[:, k] - e[k][i]))
        near |= d < tol
    pts = mid[near]
    out = set()
    for dx in (-2 * tol, 0, 2 * tol):
        for dy in (-2 * tol, 0, 2 * tol):
            for dz in (-2 * tol, 0, 2 * tol):
                out |= set(ionization.cell(pts + [dx, dy, dz], lo, hi, dims).tolist())
    return out


def compare_grid(got, rec, source, lo=LO, hi=HI, dims=DIMS, silent=0):
    """got = (sums, counts, outside, outside_count) against the oracle's recorded steps: counts
    exact (up to the ambiguous steps, and `silent` unrecorded accepted steps of the oracle for
    a strict implementation) in every cell but those a midpoint next to an edge touches, total
    count exact (same), sums within SUM_TOL x SOURCE.  Returns the number of ambiguous steps."""
    sums, cnt, out, out_n = got
    _, loss, mid = rec.arrays()
    ncell = int(np.prod(dims))
    c = ionization.cell(mid, lo, hi, dims)
    slot = np.where(c >= 0, c, ncell)                  # OUTSIDE last, as in the accumulator
    amb = np.abs(loss) <= AMBIGUOUS
    firm = np.bincount(slot[~amb], minlength=ncell + 1)
    maybe = np.bincount(slot[amb], minlength=ncell + 1)
    osum = np.bincount(slot, weights=loss, minlength=ncell + 1)
    g_cnt = np.append(np.asarray(cnt).ravel(), out_n)
    g_sum = np.append(np.asarray(sums).ravel(), out)
    ok = np.ones(ncell + 1, bool)
    for k in edge_cells(mid, lo, hi, dims):
        ok[k if k >= 0 else ncell] = False
    assert np.all(firm[ok] <= g_cnt[ok]) and np.all(g_cnt[ok] <= firm[ok] + maybe[ok] + silent)
    assert firm.sum() <= g_cnt.sum() <= firm.sum() + maybe.sum() + silent
    tol = SUM_TOL * max(source, 1.0)
    assert np.max(np.abs(g_sum[ok] - osum[ok]), initial=0) <= tol
    assert abs(g_sum.sum() - osum.sum()) <= tol
    # and the oracle's binning is np.histogramdd's
    hs, hc, ho, hon = ionization.bin_steps(loss, mid, lo, hi, dims)
    assert np.array_equal(hc.ravel(), firm[:ncell] + maybe[:ncell]) and hon == firm[-1] + maybe[-1]
    assert np.allclose(hs.ravel(), osum[:ncell], rtol=0, atol=1e-15 * max(source, 1.0))
    return int(amb.sum())


# ---------------------------------------------------------------------------- host build
@pytest.fixture(scope='module')
def hci(built):
    return C.CDLL(os.path.join(REPO, 'tests', '_hostcheck', 'libnexo_ionization_hostcheck.so'))


def _grid_args(lo, hi, dims):
    return ((C.c_double * 3)(*lo), (C.c_double * 3)(*hi), (C.c_int * 3)(*dims))


def run_host(hci, setup, X0, seed, first_id, strict, lo=LO, hi=HI, dims=DIMS):
    p = setup.params
    n = len(X0)
    X = np.ascontiguousarray(X0, dtype=np.float64).copy()
    att, acc = (np.zeros(n, np.uint32) for _ in range(2))
    rv = ra = np.zeros(1)
    nrp = 0
    if setup.radpres_v is not None:
        rv, ra = np.ascontiguousarray(setup.radpres_v), np.ascontiguousarray(setup.radpres_a)
        nrp = len(rv)
    tck = setup.spline_tck or (np.zeros(8), np.zeros(8), np.zeros(16))
    tx, ty, c = (np.ascontiguousarray(a, dtype=np.float64) for a in tck)
    ncell = int(np.prod(dims))
    sums = np.zeros(ncell + 1)
    cnt = np.zeros(ncell + 1, np.uint64)
    st = hci.hc_integrate_adaptive_ionize(
        C.c_long(n), dptr(X), att.ctypes.data_as(U32P), acc.ctypes.data_as(U32P), C.byref(p),
        dptr(rv), dptr(ra), C.c_int(nrp), dptr(tx), C.c_int(len(tx)), dptr(ty), C.c_int(len(ty)),
        dptr(c), C.c_ulonglong(seed), C.c_ulonglong(first_id), C.c_int(strict),
        C.c_int(int(is_bounce(setup))), *_grid_args(lo, hi, dims), dptr(sums),
        cnt.ctypes.data_as(U64P))
    assert st == 0
    cnt = cnt.astype(np.int64)
    return X, att, acc, (sums[:ncell].reshape(dims), cnt[:ncell].reshape(dims), sums[ncell],
                         int(cnt[ncell]))


# ---------------------------------------------------------------------------- CPU
@pytest.mark.parametrize('wl', WORKLOADS + LIFETIME, ids=str)
def test_oracle_recorder_changes_nothing(wl):
    """ionization.integrate_adaptive is oracle.deposition's driver: with the recorder on or off,
    its states, step counts, events and loss are deposition.integrate_adaptive's, bit for bit.
    Per packet the recorded loss sums (in step order) to the returned `loss` exactly, and
    recorded loss + the deposition buckets close on SOURCE."""
    setup = setup_of(wl)
    X0 = x0_of(wl, setup, 300, 8)
    seed, first = 13, 500
    rc = oracle_constants(setup)
    plain = deposition.integrate_adaptive(X0, rc, adaptive_bounce.bounce_uniforms(seed, first))
    off = ionization.integrate_adaptive(X0, rc, adaptive_bounce.bounce_uniforms(seed, first))
    (X, att, acc, bnc, ev, loss), rec = run_oracle(setup, X0, seed, first)
    for run in (off, (X, att, acc, bnc, ev, loss)):
        for a, b in zip(plain[:4] + (plain[5],), run[:4] + (run[5],)):
            assert np.array_equal(a, b)
        for k in plain[4]:
            assert np.array_equal(run[4][k], plain[4][k], equal_nan=True)
    packet, dl, mid = rec.arrays()
    assert len(packet) > 0 and np.all(dl != 0) and mid.shape == (len(packet), 3)
    assert np.array_equal(rec.per_packet(len(X0)), loss)
    b = ev['bucket']
    source = ev['amount'][b == deposition.SOURCE].sum()
    fates = ev['amount'][b != deposition.SOURCE].sum()
    assert abs(dl.sum() + fates - source) <= 1e-13 * source


def test_cell_helper_matches_histogramdd(hci):
    """ion_cell against np.histogramdd's rule: every edge value, one ulp either side, hi
    exactly, just below lo, NaN and +-inf, on non-cubic grids and an off-centre box."""
    rng = np.random.default_rng(4)
    for lo, hi, dims in ((LO, HI, DIMS), ((0.3, -5.0, 1.0), (0.9, -1.25, 7.5), (1, 9, 4)),
                         ((-4., -4., -4.), (4., 4., 4.), (100, 100, 100)),
                         ((-1e-3, 2., -7.), (3e-3, 2.5, 11.), (7, 1, 13))):
        e = ionization.edges(lo, hi, dims)
        special = [np.concatenate([x, np.nextafter(x, -np.inf), np.nextafter(x, np.inf),
                                   [np.nan, np.inf, -np.inf]]) for x in e]
        pts = []
        for k in range(3):          # every special value of one axis, the others anywhere
            m = len(special[k])
            p = np.column_stack([rng.uniform(l - 0.1 * (h - l), h + 0.1 * (h - l), m)
                                 for l, h in zip(lo, hi)])
            p[:, k] = special[k]
            pts.append(p)
            q = np.column_stack([rng.choice(s, m) for s in special])   # and corners
            pts.append(q)
        pts = np.concatenate(pts)
        want = ionization.cell(pts, lo, hi, dims)
        args = _grid_args(lo, hi, dims)
        hci.hc_ion_cell.restype = C.c_longlong
        got = np.array([hci.hc_ion_cell(C.c_double(x), C.c_double(y), C.c_double(z), *args)
                        for x, y, z in pts])
        assert np.array_equal(got, want)
        assert (want >= 0).any() and (want < 0).any()
        fin = np.all(np.isfinite(pts), axis=1)
        h, _ = np.histogramdd(pts[fin], bins=e)
        inside = want >= 0
        assert np.array_equal(np.bincount(want[inside], minlength=int(np.prod(dims))),
                              h.astype(np.int64).ravel())


@pytest.mark.parametrize('wl', WORKLOADS + LIFETIME, ids=str)
@pytest.mark.parametrize('strict', [1, 0])
def test_host_build_matches_oracle(hci, wl, strict):
    from test_hostcheck import host_strict
    setup = setup_of(wl, strict_math=bool(strict))
    X0 = x0_of(wl, setup, 300, 21)
    seed, first = 5, 1000
    (Xo, a_o, c_o, b_o, ev, loss), rec = run_oracle(setup, X0, seed, first)
    hs = host_strict(setup, strict, is_bounce(setup))
    _, a_h, c_h, got = run_host(hci, setup, X0, seed, first, hs)
    assert np.array_equal(a_h, a_o) and np.array_equal(c_h, c_o)
    source = float(X0[X0[:, 7] > 0, 7].sum())
    namb = compare_grid(got, rec, source, silent=silent_steps(c_o, rec) if hs else 0)
    if isinstance(wl, Cell):                 # a lifetime loss: every step loses frac
        assert namb == 0
    print(wl, 'strict', strict, 'steps', got[1].sum() + got[3], 'ambiguous', namb)


def test_exterior_fraction():
    """Exactly 1 / 0 for cells wholly outside / inside the planet; on cut cells the product's
    16^3 sub-cells agree with the 64^3 reference to EXTERIOR_TOL; the exterior volume of a box
    around the planet is V_box - 4 pi / 3 to that bound over its cut cells.

    The bound: only a sub-cell the sphere cuts can be misclassified, so the error of a cut
    cell is at most the share of its 16^3 sub-cells the surface crosses (about 3 * 16^2 / 16^3
    = 0.19 for a flat cut), and far less in practice because the errors on the two sides of the
    surface cancel.  EXTERIOR_TOL = 0.01 is about twice the largest difference measured on the
    grids below (0.0053, on the 11 x 6 x 8 grid).
    """
    from nexoclom_b200.ModelIonization import exterior_fraction
    for lo, hi, dims in (((-1.5, -1.5, -1.5), (1.5, 1.5, 1.5), (9, 9, 9)),
                         ((-1.3, -0.2, -2.0), (2.1, 1.6, 0.7), (11, 6, 8)),
                         ((-4., -4., -4.), (4., 4., 4.), (16, 16, 16))):
        e = ionization.edges(lo, hi, dims)
        f = exterior_fraction(e)
        ref = ionization.exterior_fraction_reference(e)
        whole = (ref == 0) | (ref == 1)
        cut = ~whole
        assert np.array_equal(f[whole], ref[whole])
        assert cut.any() and np.max(np.abs(f[cut] - ref[cut])) <= EXTERIOR_TOL
        print(dims, 'max |16^3 - 64^3|', np.max(np.abs(f[cut] - ref[cut])))
        cell = np.prod([x[1] - x[0] for x in e])
        vol = np.prod(np.subtract(hi, lo))
        if all(l < -1 and h > 1 for l, h in zip(lo, hi)):
            assert abs(f.sum() * cell - (vol - 4 * np.pi / 3)) <= EXTERIOR_TOL * cut.sum() * cell
    # cells wholly inside / outside, by the nearest point and the farthest corner
    e = ionization.edges((0.0, 0.0, 0.0), (0.5, 0.5, 2.0), (1, 1, 4))
    assert np.array_equal(exterior_fraction(e).ravel()[[0, 2, 3]], [0.0, 1.0, 1.0])


def test_grid_params_and_validation():
    from nexoclom_b200 import ModelIonization
    from nexoclom_b200.ModelIonization import grid_params
    dims, lo, hi = grid_params({})
    assert dims == [100, 100, 100] and lo == [-4.0] * 3 and hi == [4.0] * 3
    dims, lo, hi = grid_params({'dims': '3,4,5', 'center': '1,-2,0.5', 'width': '2,4,1'})
    assert dims == [3, 4, 5] and lo == [0.0, -4.0, 0.0] and hi == [2.0, 0.0, 1.0]
    for bad in ({'dims': '0,1,1'}, {'dims': '2,2'}, {'dims': '2.5,2,2'}, {'dims': 'a,b,c'},
                {'dims': True}, {'center': '0,0'}, {'center': 'nan,0,0'}, {'width': '1,1,0'},
                {'width': '1,-1,1'}, {'width': '1,inf,1'}, {'dims': '1291,1291,1291'}):
        with pytest.raises(ValueError):
            grid_params(bad)
    # nx*ny*nz + 1 < 2**31: the largest grid passes, one more cell does not
    assert grid_params({'dims': f'{2**31 - 2},1,1'})[0] == [2**31 - 2, 1, 1]
    with pytest.raises(ValueError, match='2\\*\\*31'):
        grid_params({'dims': f'{2**31 - 1},1,1'})
    # the two refusals, before any device work
    with pytest.raises(ValueError, match='adaptive driver'):
        ModelIonization(workload('Na.bounce.input'))
    with pytest.raises(ValueError):
        ModelIonization(workload('Na.maxwellian.radpres.input'), {'dims': '10,10'})


def test_no_loss_process_is_refused(monkeypatch):
    """loss_mode 0 (no lifetime and no photo rate): the map would be identically zero."""
    import sys
    from nexoclom_b200 import ModelIonization
    mod = sys.modules['nexoclom_b200.ModelIonization']

    class P:
        loss_mode = 0

    class S:
        params = P()

    monkeypatch.setattr(mod, 'get_setup', lambda inputs, strict_math=False: S())
    with pytest.raises(ValueError, match='loss process'):
        ModelIonization(workload('Na.maxwellian.radpres.input'))


def test_ion_grid_struct_matches_header():
    from nexoclom_b200._lib import IonGrid
    header = open(os.path.join(REPO, 'include', 'nexoclom_b200.h')).read()
    body = re.search(r'typedef struct nx_ion_grid \{(.*?)\} nx_ion_grid;', header, re.S).group(1)
    assert re.search(r'double lo\[3\], hi\[3\];', body) and re.search(r'int32_t n\[3\];', body)
    assert C.sizeof(IonGrid) == 6 * 8 + 4 * 4 == 64
    assert [f[0] for f in IonGrid._fields_] == ['lo', 'hi', 'n', 'reserved']


def test_units_and_rate():
    """The product's host arithmetic: production in cm^-3 s^-1 over the exterior volume, NaN
    inside the planet, the rate over grid + OUTSIDE."""
    from nexoclom_b200.ModelIonization import ModelIonization
    inputs = workload('Na.maxwellian.radpres.input')
    m = ModelIonization.__new__(ModelIonization)
    m.inputs, m.dims = inputs, (8, 8, 8)
    m.edges = ionization.edges((-2, -2, -2), (2, 2, 2), (8, 8, 8))     # cells of 0.5 R_p
    grid = np.zeros((8, 8, 8))
    grid[0, 0, 0] = 3.0
    grid[3, 3, 3] = 1.0                       # [-0.5, 0]^3, wholly inside the planet: NaN
    m._finish(grid, np.ones((8, 8, 8), np.int64), 0.5, 2, 10.0)
    endtime = float(np.asarray(inputs.options.endtime))
    assert m.atoms_per_packet == pytest.approx(1e23 * endtime / 10.0)
    assert m.rate == pytest.approx(4.5 * m.atoms_per_packet / endtime)
    r_cm = float(np.asarray(inputs.geometry.planet.radius.value)) * 1e5
    assert m.exterior_fraction[0, 0, 0] == 1.0 and m.exterior_fraction[3, 3, 3] == 0.0
    assert m.production[0, 0, 0] == pytest.approx(3.0 * m.atoms_per_packet / endtime /
                                                  (0.125 * r_cm**3))
    assert np.isnan(m.production[3, 3, 3]) and m.production[7, 7, 7] == 0.0
    assert 'Model Ionization' in str(m)


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank),
                      WORLD_SIZE=str(world))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        from nexoclom_b200.sharding import combine_ranks
        grid = np.full((3, 2, 2), rank + 1.0)
        cnt = np.full((3, 2, 2), rank + 1, np.int64)
        out, out_n = np.array([0.5 * (rank + 1)]), np.array([rank + 1], np.int64)
        tot, = combine_ranks((grid, cnt, out, out_n), 10.0 * (rank + 1))
        q.put((rank, grid.tolist(), cnt.tolist(), float(out[0]), int(out_n[0]), tot))
    finally:
        dist.destroy_process_group()


def test_gloo_two_rank_reduction():
    import multiprocessing as mp
    import socket
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        port = s.getsockname()[1]
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for _, grid, cnt, out, out_n, tot in res:
        assert np.all(np.array(grid) == 3.0) and np.all(np.array(cnt) == 3)
        assert out == 1.5 and out_n == 3 and tot == 30.0


def ion_builds(cells):
    """The k_ionize_adaptive builds (MODE, BOUNCE) the ion runs of `cells` select: the build
    of the plain run (common.adaptive_mode)."""
    return {(adaptive_mode(c.setup().params, c.bounce), c.bounce) for c in cells}


def test_cells_reach_every_ion_build():
    """The cells with a loss term select exactly the 22 ion builds nx_kernels.cu instantiates:
    every dispatched (MODE, BOUNCE) with MODE & 3 in {1, 2}, and the two strict kernels."""
    from test_kernel_builds import dispatch_cases
    src = {(a[0], a[1]) for k, a, _ in dispatch_cases()
           if k == 'k_integrate_adaptive' and (a[0] & 3) in (1, 2)}
    assert len(src) == 20
    want = src | {(-1, False), (-1, True)}
    assert ion_builds(ION_CELLS) == want and len(want) == 22


# ---------------------------------------------------------------------------- GPU
def grid_of(setup):
    """A non-cubic grid around the planet, wide enough for a moon's orbit."""
    p = setup.params
    r = 6.0 if p.nmoons == 0 else float(p.moon_a[0]) + 2.0
    return (-r, -1.1 * r, -0.8 * r), (r, 1.2 * r, 0.9 * r), (37, 41, 29)


def gpu_ionize(engine, setup, X0, seed, first_id, grid):
    lo, hi, dims = grid
    setup.upload(engine)
    engine.import_state(X0)
    engine.ionize_begin(lo, hi, dims)
    try:
        tot = engine.integrate_adaptive_ionize(seed, first_id)
        got = engine.ionize_fetch(dims)
    finally:
        engine.ionize_end()
    return engine.export_state().T, tot, engine.export_stats(), got


@pytest.mark.gpu
@pytest.mark.parametrize('cell', ION_CELLS, ids=str)
def test_ion_builds_match_oracle(engine, cell):
    """Every ion build against the oracle; the ion run is the plain (and the deposition) run
    bit for bit: final state, attempted / accepted per packet and in total, bounces."""
    from test_kernel_builds import (FIRST, K2_TOL, N, SEED, STATE_TOL, run_adaptive, same_run)
    setup = cell.setup()
    X0 = cell.x0(setup, N, 21)
    (Xo, a_o, c_o, b_o, ev, loss), rec = run_oracle(setup, X0, SEED, FIRST)
    resident, _, sink, _ = run_adaptive(engine, cell, setup, X0)
    grid = grid_of(setup)
    ion = gpu_ionize(engine, setup, X0, SEED, FIRST, grid)
    assert same_run(ion, resident) and same_run(ion, sink)
    Xg, tot, (a_g, c_g), got = ion
    par = state_parity(Xg, Xo)
    assert par['alive_mismatch'] == 0, par
    assert np.array_equal(a_g, a_o) and np.array_equal(c_g, c_o)
    assert tot == (int(a_o.sum()), int(c_o.sum()), int(b_o.sum()))
    assert max(par['pos'], par['vel'], par['frac']) < (STATE_TOL if cell.bounce else K2_TOL), par
    source = float(X0[X0[:, 7] > 0, 7].sum())
    mode = adaptive_mode(setup.params, cell.bounce)
    namb = compare_grid(got, rec, source, *grid, silent=silent_steps(c_o, rec) if mode < 0 else 0)
    print(cell, 'MODE', mode, 'steps', got[1].sum() + got[3],
          'outside', got[3], 'ambiguous', namb)
    assert got[1].sum() > 0


_ION_NAME = re.compile(r'k_ionize_adaptive<([^>]*)>')


def ion_build_of(name):
    m = _ION_NAME.search(name)
    if not m:
        return None
    a = [re.sub(r'^\((?:int|bool)\)', '', x.strip()) for x in m.group(1).split(',')]
    return int(a[0]), a[1] == 'true'


@pytest.mark.gpu
def test_profiler_sees_every_ion_build(engine):
    """The ion runs of the cells under torch.profiler: the k_ionize_adaptive kernels that ran
    are exactly the builds the cells predict."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    assert ion_build_of('void nx::k_ionize_adaptive<(int)-1, true>(nx::StateCols)') == (-1, True)
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for cell in ION_CELLS:
            setup = cell.setup()
            gpu_ionize(engine, setup, cell.x0(setup, 256, 3), 1, 0, grid_of(setup))
        engine.sync()
    names = {e.name for e in prof.events() if 'k_ionize_adaptive' in e.name}
    print('kernels seen:', sorted(names))
    assert {ion_build_of(n) for n in names} == ion_builds(ION_CELLS)


@pytest.mark.gpu
@pytest.mark.parametrize('wl', ['Na.maxwellian.radpres.input', 'Na.bounce.adaptive.input',
                                'Na.Io.Jupiter.input'])
def test_closure_with_deposition(wl):
    """ModelIonization's grid + OUTSIDE is ModelDeposition's LOST on the same Input (perfect
    sticking, bounce, a moon), and its rate the deposition's lost rate, to 1e-12 of the source;
    the two regenerate the same runs."""
    from nexoclom_b200 import ModelDeposition, ModelIonization
    inputs = workload(wl)
    inputs.delete_files()
    n = 1_000_000 if wl == 'Na.maxwellian.radpres.input' else 50_000
    params = {'dims': '80,80,80', 'width': '8,8,8'}
    if wl == 'Na.Io.Jupiter.input':
        params = {'dims': '60,60,30', 'width': '16,16,8'}
    try:
        inputs.run(n, seed=3)
        dep = ModelDeposition(inputs)
        ion = ModelIonization(inputs, params)
    finally:
        inputs.delete_files()
    b = dep.buckets
    lost = b['source'] - sum(b[k] for k in ('surface', 'moon', 'escaped', 'vanished', 'remaining'))
    assert ion.totalsource == dep.totalsource == n
    assert abs(ion.ionized.sum() + ion.outside - lost) <= 1e-12 * b['source']
    assert abs(ion.rate - dep.rates['lost']) <= 1e-12 * 1e23
    assert (ion.attempted_steps, ion.accepted_steps, ion.bounces) == \
        (dep.attempted_steps, dep.accepted_steps, dep.bounces)
    assert ion.production.shape == ion.dims and np.nanmax(ion.production) > 0
    assert ion.packet_grid.sum() > 0 and lost > 0
    if wl == 'Na.bounce.adaptive.input':
        assert ion.bounces > 0
    print(wl, ion)


@pytest.mark.gpu
def test_shard_invariance(engine):
    """Two first_id halves summed are the whole run: counts exact, sums to 1e-12 x SOURCE."""
    setup = setup_of('Na.bounce.adaptive.input')
    n, seed, h = 40000, 77, 15000
    X0 = initial_state.draw_x0(setup, n, 3)[:, :8]
    grid = ((-6., -6., -6.), (6., 7., 5.), (60, 65, 55))
    whole = gpu_ionize(engine, setup, X0, seed, 0, grid)[3]
    s0 = gpu_ionize(engine, setup, X0[:h], seed, 0, grid)[3]
    s1 = gpu_ionize(engine, setup, X0[h:], seed, h, grid)[3]
    assert np.array_equal(s0[1] + s1[1], whole[1]) and s0[3] + s1[3] == whole[3]
    assert np.allclose(s0[0] + s1[0], whole[0], rtol=0, atol=1e-12 * n)
    assert abs(s0[2] + s1[2] - whole[2]) <= 1e-12 * n
    assert whole[1].sum() > 0


ANALYTIC_INPUT = '''geometry.planet = Mercury
geometry.taa = 0.
forces.gravity = False
forces.radpres = False
SpatialDist.type = uniform
SpeedDist.type = flat
SpeedDist.vprob = {v}
SpeedDist.delv = {dv}
AngularDist.type = radial
options.endtime = {T}
options.species = Na
options.lifetime = {tau}
options.outeredge = 100
'''


@pytest.mark.gpu
def test_analytic_radial_outflow(engine, tmp_path):
    """An expectation independent of the oracle.  No forces, lifetime loss nu = 1/tau, radial
    ejection at a speed uniform in [v - dv, v + dv], endtime T.  A packet released at t0
    uniform in [0, T] flies radially, r = 1 + v t, for D = T - t0 ~ U[0, T] seconds, so its
    expected loss between flight times t and t + dt is nu e^(-nu t) P(D > t) dt =
    nu e^(-nu t) (1 - t/T) dt, with the antiderivative F(t) = e^(-nu t) (1/(nu T) - 1 + t/T).
    A shell [r_a, r_b) then expects mu = < F(t_b) - F(t_a) >_v per packet, t = (r - 1) / v
    clipped to [0, T].

    The grid is summed into shells several cells wide, each cell by its centre.  The steps are
    far shorter than a cell (no forces: the step is set by the frac's error alone, h < 0.004
    tau), so every recorded midpoint lies on its packet's path; a cell whose centre is in one
    shell may hold loss from the other side of a boundary only within half a cell diagonal d
    of it.  Bound per shell: |G - N mu| <= 5 sigma + N (B(r_a) + B(r_b)), where B(r) is the
    expected loss per packet in (r - d/2, r + d/2) and sigma^2 = N Var(X) <= N m mu, X being a
    packet's loss in the shell (0 <= X <= m = max_v of e^(-nu t_a) - e^(-nu t_b))."""
    from nexoclom_b200.Input import Input
    from nexoclom_b200.runsetup import RunSetup
    v_kms, dv_kms, T, tau = 3.0, 0.02, 4000.0, 2000.0
    path = tmp_path / 'radial.input'
    path.write_text(ANALYTIC_INPUT.format(v=v_kms, dv=dv_kms, T=T, tau=tau))
    setup = RunSetup(Input(str(path)))
    assert setup.params.loss_mode == 1 and not setup.params.gravity and not setup.params.radpres
    nu = 1.0 / tau
    vs = np.linspace(v_kms - dv_kms, v_kms + dv_kms, 401) / setup.radius_km       # R_p / s

    def F(t):
        t = np.clip(t, 0.0, T)
        return np.exp(-nu * t) * (1.0 / (nu * T) - 1.0 + t / T)

    def expect(ra, rb):
        """(mean, max) per packet of the loss between radii ra and rb."""
        ta, tb = np.maximum(ra - 1.0, 0.0) / vs, np.maximum(rb - 1.0, 0.0) / vs
        m = np.exp(-nu * np.clip(ta, 0, T)) - np.exp(-nu * np.clip(tb, 0, T))
        return float(np.mean(F(tb) - F(ta))), float(m.max())

    n, width, ncell = 2_000_000, 14.0, 140
    lo, hi = (-width / 2,) * 3, (width / 2,) * 3
    setup.upload(engine)
    engine.init_state(setup.source_params(engine), 11, 0, n)
    engine.ionize_begin(lo, hi, (ncell,) * 3)
    try:
        engine.integrate_adaptive_ionize(0, 0)
        grid, cnt, out, out_n = engine.ionize_fetch((ncell,) * 3)
    finally:
        engine.ionize_end()
    assert out_n == 0 and out == 0.0
    c = 0.5 * (np.linspace(lo[0], hi[0], ncell + 1)[:-1] + np.linspace(lo[0], hi[0], ncell + 1)[1:])
    r = np.sqrt(c[:, None, None]**2 + c[None, :, None]**2 + c[None, None, :]**2)
    d = np.sqrt(3) * width / ncell
    shells = [0.0, 2.0, 3.0, 4.0, 5.0, 7.0]
    total_mu, _ = expect(1.0, 1.0 + v_kms * 2 * T)
    assert abs(grid.sum() - n * total_mu) < 1e-2 * n * total_mu
    for ra, rb in zip(shells[:-1], shells[1:]):
        g = grid[(r >= ra) & (r < rb)].sum()
        mu, m = expect(ra, rb)
        sigma = np.sqrt(n * m * mu)
        band = sum(expect(b - d / 2, b + d / 2)[0] for b in (ra, rb) if b > 1.0)
        print(f'shell [{ra}, {rb}): grid {g:.6g}, expected {n * mu:.6g}, 5 sigma {5 * sigma:.3g}, '
              f'boundary {n * band:.3g}')
        assert abs(g - n * mu) <= 5 * sigma + n * band
