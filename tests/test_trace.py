"""Images and density grids from every accepted step of the adaptive driver (K2t:
k_trace_adaptive, nx_integrate_adaptive_trace, Engine.integrate_adaptive_trace,
ModelTrajectoryImage, ModelTrajectoryDensity).  The oracle is oracle/trace.py: the ionization
oracle's driver, pinned here to it bit for bit, with a recorder of every accepted step (packet,
h, the state before it, the Runge-Kutta state), from which it forms the midpoints and the
age-weighted dwells a = (h T) / ((T - t0) + (t - h / 2)) with the product's arithmetic.

Counts are compared exactly except in the pixels and cells a midpoint within EDGE_TOL of an edge
may fall in; sums within SUM_TOL of the total."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from common import REPO, KERNEL_CELLS, Cell, adaptive_mode, oracle_constants, state_parity, workload
from nexoclom_b200._lib import ImageParams, dptr
from oracle import adaptive_bounce, imaging, initial_state, ionization, trace

U32P = C.POINTER(C.c_uint32)
U64P = C.POINTER(C.c_uint64)
EDGE_TOL = 1e-12             # R_p: midpoints this close to a pixel or cell edge may bin either side
SUM_TOL = 1e-12              # x the total
LO, HI, DIMS = (-3.1, -2.7, -2.2), (3.3, 4.1, 2.6), (23, 31, 17)
WORKLOADS = ['Ca.isotropic.flat.input', 'Na.maxwellian.radpres.input', 'Na.bounce.adaptive.input',
             'Na.bounce.stick05.input']
LIFETIME = [Cell('adaptive', False, False, True, True, 'lifetime'),
            Cell('adaptive', True, False, True, False, 'lifetime')]
TRACE_CELLS = [c for c in KERNEL_CELLS if c.driver == 'adaptive' and not c.moon]
# (cell, strict_math): without moons only strict_math selects the strict kernel without bounce
TRACE_RUNS = [(c, False) for c in TRACE_CELLS] + [(LIFETIME[0], True)]
RUN_IDS = [f"{c}{'-strict' if s else ''}" for c, s in TRACE_RUNS]


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
    rec = trace.Recorder()
    out = trace.integrate_adaptive(X0, oracle_constants(setup),
                                   adaptive_bounce.bounce_uniforms(seed, first_id), recorder=rec)
    return out, rec


def image_params(setup, quantity, dims=(37, 29), x=(-5.3, 4.7), z=(-4.1, 5.9), subobs=(0.7, 0.4)):
    from nexoclom_b200.ModelImage import image_rotation
    M = np.asarray(image_rotation(*subobs))
    ip = ImageParams()
    for k in range(9):
        ip.M[k] = float(M.flat[k])
    ip.x0, ip.x1 = x
    ip.z0, ip.z1 = z
    ip.nx, ip.nz = dims
    rcm = setup.radius_km * 1e5
    ip.apix = ((x[1] - x[0]) / dims[0] * rcm) * ((z[1] - z[0]) / dims[1] * rcm)
    ip.vrplanet = setup.vrplanet
    ip.quantity = 1 if quantity == 'radiance' else 0
    ip.round_f32 = ip.skip_dead = 0
    return ip


def image_kw(ip, quantity, gt):
    M = np.array(ip.M[:]).reshape(3, 3)
    return dict(vrplanet=ip.vrplanet, M=M, dims=[ip.nx, ip.nz], xrange=(ip.x0, ip.x1),
                zrange=(ip.z0, ip.z1), apix=ip.apix, quantity=quantity, gtables=gt)


def _edge_near(v, e, tol):
    i = np.clip(np.searchsorted(e, v), 1, len(e) - 1)
    return np.minimum(np.abs(v - e[i - 1]), np.abs(v - e[i])) < tol


def image_edge_pixels(mid, ip):
    """Pixels (and -1) a midpoint whose observer coordinates lie within EDGE_TOL of a pixel edge
    may fall in."""
    M = np.array(ip.M[:]).reshape(3, 3)
    obs = mid[:, 1:4] @ M.T
    ex, ez = np.linspace(ip.x0, ip.x1, ip.nx + 1), np.linspace(ip.z0, ip.z1, ip.nz + 1)
    near = _edge_near(obs[:, 0], ex, EDGE_TOL) | _edge_near(obs[:, 2], ez, EDGE_TOL)
    out = set()
    for dx in (-2 * EDGE_TOL, 0, 2 * EDGE_TOL):
        for dz in (-2 * EDGE_TOL, 0, 2 * EDGE_TOL):
            ix = np.searchsorted(ex, obs[near, 0] + dx, side='right') - 1
            iz = np.searchsorted(ez, obs[near, 2] + dz, side='right') - 1
            ok = (ix >= 0) & (ix < ip.nx) & (iz >= 0) & (iz < ip.nz)
            out |= set(np.where(ok, ix * ip.nz + iz, -1).tolist())
    return out


def grid_edge_cells(mid, lo, hi, dims):
    e = ionization.edges(lo, hi, dims)
    near = np.zeros(len(mid), bool)
    for k in range(3):
        near |= _edge_near(mid[:, 1 + k], e[k], EDGE_TOL)
    out = set()
    for dx in (-2 * EDGE_TOL, 0, 2 * EDGE_TOL):
        for dy in (-2 * EDGE_TOL, 0, 2 * EDGE_TOL):
            for dz in (-2 * EDGE_TOL, 0, 2 * EDGE_TOL):
                out |= set(ionization.cell(mid[near, 1:4] + [dx, dy, dz], lo, hi, dims).tolist())
    return out


def compare_image(got, mid, a, ip, quantity, gt):
    """got = (sums (nx, nz), counts) against the oracle's binning of the recorded steps."""
    want, wcnt = trace.bin_image(mid, a, **image_kw(ip, quantity, gt))
    ok = np.ones(ip.nx * ip.nz, bool)
    for k in image_edge_pixels(mid, ip):
        if k >= 0:
            ok[k] = False
    g, gc = np.asarray(got[0]).ravel(), np.asarray(got[1]).ravel()
    assert np.array_equal(gc[ok], wcnt.ravel()[ok])
    tol = SUM_TOL * max(abs(want).sum(), 1e-300)
    assert np.max(np.abs(g[ok] - want.ravel()[ok]), initial=0) <= tol
    assert abs(g.sum() - want.sum()) <= tol + np.abs(want.ravel()[~ok]).sum()
    return int(wcnt.sum())


def compare_grid(got, mid, a, lo=LO, hi=HI, dims=DIMS):
    """got = (sums, counts, outside, outside count) against the oracle's binning."""
    sums, cnt, out, out_n = got
    ws, wc, wo, won = trace.bin_grid(mid, a, lo, hi, dims)
    ncell = int(np.prod(dims))
    ok = np.ones(ncell + 1, bool)
    for k in grid_edge_cells(mid, lo, hi, dims):
        ok[k if k >= 0 else ncell] = False
    g_cnt = np.append(np.asarray(cnt).ravel(), out_n)
    w_cnt = np.append(wc.ravel(), won)
    g_sum = np.append(np.asarray(sums).ravel(), out)
    w_sum = np.append(ws.ravel(), wo)
    assert np.array_equal(g_cnt[ok], w_cnt[ok]) and g_cnt.sum() == w_cnt.sum()
    tol = SUM_TOL * max(w_sum.sum(), 1e-300)
    assert np.max(np.abs(g_sum[ok] - w_sum[ok]), initial=0) <= tol
    assert abs(g_sum.sum() - w_sum.sum()) <= tol
    return int(w_cnt.sum())


# ---------------------------------------------------------------------------- host build
@pytest.fixture(scope='module')
def hct(built):
    return C.CDLL(os.path.join(REPO, 'tests', '_hostcheck', 'libnexo_trace_hostcheck.so'))


def _gt_args(gt):
    if not gt:
        return C.c_int(0), None, dptr(np.zeros(1)), dptr(np.zeros(1))
    sizes = np.array([len(v) for v, _ in gt], np.int32)
    v = np.ascontiguousarray(np.concatenate([v for v, _ in gt]), np.float64)
    g = np.ascontiguousarray(np.concatenate([g for _, g in gt]), np.float64)
    _gt_args.keep = (sizes, v, g)
    return C.c_int(len(gt)), sizes.ctypes.data_as(C.POINTER(C.c_int)), dptr(v), dptr(g)


def run_host(hct, setup, X0, seed, first_id, strict, ip, gt, grid=(LO, HI, DIMS)):
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
    img = np.zeros(ip.nx * ip.nz)
    icnt = np.zeros(ip.nx * ip.nz, np.uint64)
    lo, hi, dims = grid
    ncell = int(np.prod(dims))
    sums, cnt = np.zeros(ncell + 1), np.zeros(ncell + 1, np.uint64)
    st = hct.hc_integrate_adaptive_trace(
        C.c_long(n), dptr(X), att.ctypes.data_as(U32P), acc.ctypes.data_as(U32P), C.byref(p),
        dptr(rv), dptr(ra), C.c_int(nrp), dptr(tx), C.c_int(len(tx)), dptr(ty), C.c_int(len(ty)),
        dptr(c), C.c_ulonglong(seed), C.c_ulonglong(first_id), C.c_int(strict),
        C.c_int(int(is_bounce(setup))), C.byref(ip), *_gt_args(gt), dptr(img),
        icnt.ctypes.data_as(U64P), (C.c_double * 3)(*lo), (C.c_double * 3)(*hi),
        (C.c_int * 3)(*dims), dptr(sums), cnt.ctypes.data_as(U64P))
    assert st == 0
    cnt = cnt.astype(np.int64)
    return X, att, acc, (img.reshape(ip.nx, ip.nz), icnt.astype(np.int64).reshape(ip.nx, ip.nz)), \
        (sums[:ncell].reshape(dims), cnt[:ncell].reshape(dims), sums[ncell], int(cnt[ncell]))


# ---------------------------------------------------------------------------- CPU
@pytest.mark.parametrize('wl', WORKLOADS + LIFETIME, ids=str)
def test_oracle_recorder_changes_nothing(wl):
    """trace.integrate_adaptive is oracle.ionization's driver: with the recorder on or off its
    states, step counts, events and loss are ionization.integrate_adaptive's, bit for bit, and
    the recorder sees every accepted step once, with h and the time it started from."""
    setup = setup_of(wl)
    X0 = x0_of(wl, setup, 300, 8)
    seed, first = 13, 500
    rc = oracle_constants(setup)
    plain = ionization.integrate_adaptive(X0, rc, adaptive_bounce.bounce_uniforms(seed, first))
    off = trace.integrate_adaptive(X0, rc, adaptive_bounce.bounce_uniforms(seed, first))
    on, rec = run_oracle(setup, X0, seed, first)
    for run in (off, on):
        for a, b in zip(plain[:4] + (plain[5],), run[:4] + (run[5],)):
            assert np.array_equal(a, b)
        for k in plain[4]:
            assert np.array_equal(run[4][k], plain[4][k], equal_nan=True)
    packet, h, s, s_rk = rec.arrays()
    assert len(packet) == int(on[2].sum()) > 0
    assert np.array_equal(np.bincount(packet, minlength=len(X0)), on[2])
    assert np.all(h > 0) and np.all(h <= s[:, 0])
    endtime = float(setup.params.endtime)
    mid, a = trace.steps(rec, X0[:, 0], endtime)
    assert np.all(a >= h) and np.all(np.isfinite(a))           # T / (T - age) >= 1
    assert np.array_equal(mid, (s + s_rk) * 0.5)


@pytest.mark.parametrize('wl', WORKLOADS + LIFETIME, ids=str)
@pytest.mark.parametrize('strict', [1, 0])
def test_host_build_matches_oracle(hct, wl, strict):
    """trace_record and the TRACE attempts, host build, against the oracle: a column image and
    the grid (radiance for the Na workloads); the state and step counts as the oracle's."""
    from test_hostcheck import host_strict
    setup = setup_of(wl, strict_math=bool(strict))
    X0 = x0_of(wl, setup, 300, 21)
    seed, first = 5, 1000
    (Xo, a_o, c_o, b_o, ev, loss), rec = run_oracle(setup, X0, seed, first)
    hs = host_strict(setup, strict, is_bounce(setup))
    quantity = 'radiance' if 'Na.' in str(wl) else 'column'
    gt = setup.gtables([5891, 5897]) if quantity == 'radiance' else []
    ip = image_params(setup, quantity)
    _, a_h, c_h, img, grid = run_host(hct, setup, X0, seed, first, hs, ip, gt)
    assert np.array_equal(a_h, a_o) and np.array_equal(c_h, c_o)
    mid, a = trace.steps(rec, X0[:, 0], float(setup.params.endtime))
    nimg = compare_image(img, mid, a, ip, quantity, gt)
    nstep = compare_grid(grid, mid, a)
    assert nimg > 0 and nstep == int(c_o.sum())
    print(wl, 'strict', strict, 'steps', nstep, 'in the image', nimg)


def test_params_validation():
    from nexoclom_b200.ModelTrajectory import image_trace_params
    from nexoclom_b200 import ModelTrajectoryDensity, ModelTrajectoryImage
    image_trace_params({'quantity': 'column'})
    image_trace_params({'quantity': 'radiance', 'dims': '40,30', 'center': '1,-1', 'width': '4,3'})
    bad = [{'quantity': 'colum'}, {}, {'quantity': 'column', 'dims': '40'},
           {'quantity': 'column', 'dims': '0,4'}, {'quantity': 'column', 'dims': '4.5,4'},
           {'quantity': 'column', 'dims': '40000,40000'}, {'quantity': 'column', 'center': 'a,b'},
           {'quantity': 'column', 'width': '4,-1'}, {'quantity': 'column', 'width': 'nan,1'},
           {'quantity': 'column', 'subobslongitude': 'inf'}]
    for params in bad:
        with pytest.raises(ValueError):
            image_trace_params(params)
    with pytest.raises(ValueError):
        image_trace_params('quantity=column')
    inputs = workload('Na.maxwellian.radpres.input')
    for params in bad[2:5]:
        with pytest.raises(ValueError):
            ModelTrajectoryImage(inputs, params)
    for params in ({'dims': '4,4'}, {'width': '1,1,0'}, {'center': '0,0,nan'}, 'dims=4,4,4'):
        with pytest.raises(ValueError):
            ModelTrajectoryDensity(inputs, params)


def test_refusals():
    """Constant-step inputs, moons and imported X0 times outside [0, T] are refused before any
    device work (no GPU is touched here)."""
    from nexoclom_b200 import ModelTrajectoryDensity, ModelTrajectoryImage
    from nexoclom_b200.ModelTrajectory import check_trace_inputs
    for cls, params in ((ModelTrajectoryImage, {'quantity': 'column'}), (ModelTrajectoryDensity, {})):
        with pytest.raises(ValueError, match='adaptive driver'):
            cls(workload('Na.bounce.input'), params)
        moon = workload('Na.Io.Jupiter.input')
        assert moon.options.step_size == 0
        with pytest.raises(ValueError, match='moons'):
            cls(moon, params)
    inputs = workload('Na.maxwellian.radpres.input')
    T = float(inputs.options.endtime.value)
    good = [np.array([0.0, T, 0.5 * T])] + [np.zeros(3)] * 7
    check_trace_inputs(inputs, [None], [('x0', good)])
    check_trace_inputs(inputs, [None], [('x0', np.column_stack(good))])
    check_trace_inputs(inputs, [None], [('seed', 3)])
    for t in ([-1.0, 0.0, 1.0], [0.0, T * (1 + 1e-15) + 1.0, 1.0], [np.nan, 1.0, 1.0],
              [np.inf, 1.0, 1.0]):
        cols = [np.array(t)] + [np.zeros(3)] * 7
        with pytest.raises(ValueError, match='imported X0'):
            check_trace_inputs(inputs, [None], [('x0', cols)])
        with pytest.raises(ValueError, match='imported X0'):
            check_trace_inputs(inputs, [None], [('x0', np.column_stack(cols))])


def test_abi_matches_header():
    """nx_trace_begin takes the existing nx_image_params and nx_ion_grid; the product enum and
    the bindings agree with the header."""
    from nexoclom_b200 import _lib
    header = open(os.path.join(REPO, 'include', 'nexoclom_b200.h')).read()
    assert re.search(r'NX_PRODUCT_TRACE = 4', header) and _lib.NX_PRODUCT_TRACE == 4
    assert re.search(r'int nx_trace_begin\(nx_ctx\* ctx, const nx_image_params\* image, '
                     r'const nx_ion_grid\* grid\);', header)
    assert re.search(r'int nx_integrate_adaptive_trace\(nx_ctx\* ctx, long long n, uint64_t seed, '
                     r'uint64_t first_id,', header)
    assert C.sizeof(ImageParams) == 9 * 8 + 6 * 8 + 6 * 4 == 144
    src = open(os.path.join(REPO, 'nexoclom_b200', '_lib.py')).read()
    assert "'nx_trace_begin': [vp, C.POINTER(ImageParams), C.POINTER(IonGrid)]" in src


class _FakeEngine:
    """The trajectory sink of one rank without a device: fixed sums, recording the calls."""

    def __init__(self, rank, npix, dims):
        self.rank, self.npix, self.dims, self.calls = rank, npix, dims, []
        self._uploaded_setup = None

    def trace_begin(self, ip, grid):
        self.calls.append(('begin', ip is not None, grid is not None))

    def trace_fetch(self):
        r = self.rank + 1.0
        img = np.full(self.npix, r) if self.npix else None
        imgn = np.full(self.npix, self.rank + 1, np.int64) if self.npix else None
        g = np.full(self.dims, 2 * r) if self.dims else None
        gn = np.full(self.dims, 2 * (self.rank + 1), np.int64) if self.dims else None
        return img, imgn, g, gn, (0.5 * r if self.dims else None), (self.rank + 1 if self.dims else None)

    def trace_end(self):
        self.calls.append(('end',))


def _fake_model(rank):
    import nexoclom_b200.ModelTrajectory as mt

    class M:
        _device = 0
        _outputs = ['out']
        _recipes = [('seed', 1)]

        def _upload_tables(self, eng):
            pass
    mt.regenerate = lambda model, eng, outputs, recipes, integrate: 10.0 * (rank + 1)
    return M()


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank),
                      WORLD_SIZE=str(world))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        import nexoclom_b200.ModelTrajectory as mt
        ip = ImageParams()
        ip.nx, ip.nz = 3, 2
        res = []
        for image, grid in ((ip, None), (None, ((0, 0, 0), (1, 1, 1), (2, 2, 2)))):
            eng = _FakeEngine(rank, (3, 2) if image is not None else None,
                              (2, 2, 2) if grid is not None else None)
            mt.get_engine = lambda device: eng
            model = _fake_model(rank)
            out = mt.run_trace(model, image, grid)
            res.append([None if v is None else np.asarray(v).tolist() for v in out])
        q.put((rank, res))
    finally:
        dist.destroy_process_group()


def test_gloo_two_rank_reduction():
    """run_trace's host reduction over two gloo ranks: the image, the grid, OUTSIDE and the
    totalsource riding along are summed once over the ranks."""
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
    for _, (img_run, grid_run) in res:
        tot, img, imgn, g, gn, out, outn = img_run
        assert tot == 30.0 and np.all(np.array(img) == 3.0) and np.all(np.array(imgn) == 3)
        assert g is None and gn is None
        tot, img, imgn, g, gn, out, outn = grid_run
        assert tot == 30.0 and img is None and imgn is None
        assert np.all(np.array(g) == 6.0) and np.all(np.array(gn) == 6)
        assert out == 1.5 and outn == 3


def test_units_and_normalisation(monkeypatch):
    """The host arithmetic: image = sums * atoms_per_packet / T (ModelImage's units); density
    = dwell * atoms_per_packet / T / V_ext in cm^-3, NaN inside the planet."""
    import nexoclom_b200.ModelTrajectory as mt
    inputs = workload('Na.maxwellian.radpres.input')
    T = float(inputs.options.endtime.value)
    monkeypatch.setattr(mt, 'regeneration_plan', lambda inputs: (0, [], [], []))
    dims = (8, 8, 8)
    grid = np.zeros(dims)
    grid[0, 0, 0] = 3.0
    grid[3, 3, 3] = 1.0                       # [-0.5, 0]^3, wholly inside the planet: NaN
    img = np.arange(6.0).reshape(3, 2)

    def fake_run(model, ip, g):
        model.attempted_steps = model.accepted_steps = model.bounces = 0
        model.kernel_ms = 0.0
        if ip is not None:
            assert (ip.nx, ip.nz) == (3, 2) and ip.round_f32 == 0 and ip.quantity == 0
            return 10.0, img, np.ones((3, 2), np.int64), None, None, 0.0, 0
        assert tuple(g[2]) == dims
        return 10.0, None, None, grid, np.ones(dims, np.int64), 0.5, 2
    monkeypatch.setattr(mt, 'run_trace', fake_run)
    im = mt.ModelTrajectoryImage(inputs, {'quantity': 'column', 'dims': '3,2'})
    apk = 1e23 * T / 10.0
    assert im.atoms_per_packet == pytest.approx(apk)
    assert np.allclose(im.image, img * apk / T, rtol=1e-15)
    assert im.step_image.shape == (3, 2) and len(im.xaxis) == 3 and len(im.zaxis) == 2
    d = mt.ModelTrajectoryDensity(inputs, {'dims': '8,8,8', 'width': '4,4,4'})
    r_cm = float(np.asarray(inputs.geometry.planet.radius.value)) * 1e5
    assert d.exterior_fraction[0, 0, 0] == 1.0 and d.exterior_fraction[3, 3, 3] == 0.0
    assert d.density[0, 0, 0] == pytest.approx(3.0 * apk / T / (0.125 * r_cm**3))
    assert np.isnan(d.density[3, 3, 3]) and d.density[7, 7, 7] == 0.0
    assert d.outside == 0.5 and d.outside_count == 2 and d.dwell is grid
    assert 'Model Trajectory Density' in str(d)


def _shells(r, w, edges):
    return np.array([w[(r >= a) & (r < b)].sum() for a, b in zip(edges[:-1], edges[1:])])


@pytest.mark.parametrize('wl, n, seeds', [('Na.maxwellian.radpres.input', 2000, 3),
                                          ('Ca.isotropic.flat.input', 300, 2)])
def test_trajectory_agrees_with_snapshot(wl, n, seeds):
    """Oracle level: radial shell profiles of the age-weighted trajectory (sum of frac(m) a / T
    per shell) and of the snapshot (sum of the final rows' frac) agree within 5 combined sigma,
    each sigma from per-packet sums (packets are independent, steps of one packet are not), in
    every shell where the snapshot has at least 10 rows.  The trajectory's noise is the lower."""
    setup = setup_of(wl)
    T = float(setup.params.endtime)
    edges = np.array([1.0, 1.05, 1.2, 1.4, 2.0, 3.0, 4.0])
    snap_s = snap_v = snap_n = traj_s = traj_v = 0.0
    for seed in range(seeds):
        X0 = initial_state.draw_x0(setup, n, 100 + seed)[:, :8]
        (X, _, acc, _, _, _), rec = run_oracle(setup, X0, 1, 0)
        live = X[:, 7] > 0
        rs = np.sqrt((X[:, 1:4] ** 2).sum(axis=1))
        per = np.zeros((len(edges) - 1, n))
        for k, (a, b) in enumerate(zip(edges[:-1], edges[1:])):
            m = live & (rs >= a) & (rs < b)
            per[k, m] = X[m, 7]
        snap_s = snap_s + per.sum(axis=1)
        snap_v = snap_v + (per ** 2).sum(axis=1)
        snap_n = snap_n + (per > 0).sum(axis=1)
        packet = rec.arrays()[0]
        mid, a = trace.steps(rec, X0[:, 0], T)
        rm = np.sqrt((mid[:, 1:4] ** 2).sum(axis=1))
        tp = np.zeros((len(edges) - 1, n))
        for k, (lo, hi) in enumerate(zip(edges[:-1], edges[1:])):
            m = (rm >= lo) & (rm < hi)
            tp[k] = np.bincount(packet[m], weights=mid[m, 7] * a[m] / T, minlength=n)
        traj_s = traj_s + tp.sum(axis=1)
        traj_v = traj_v + (tp ** 2).sum(axis=1)
    checked = 0
    for k in range(len(edges) - 1):
        print(f'shell [{edges[k]}, {edges[k + 1]}): snapshot {snap_s[k]:.4g} +- {np.sqrt(snap_v[k]):.3g} '
              f'({int(snap_n[k])} rows), trajectory {traj_s[k]:.4g} +- {np.sqrt(traj_v[k]):.3g}')
        if snap_n[k] >= 10:
            assert abs(traj_s[k] - snap_s[k]) <= 5 * np.sqrt(snap_v[k] + traj_v[k])
            assert traj_v[k] < snap_v[k]
            checked += 1
    assert checked >= 2


def trace_builds(runs):
    """The k_trace_adaptive builds (MODE, BOUNCE) the trace runs of `runs` ((cell, strict_math)
    pairs) select: the build of the plain run (common.adaptive_mode)."""
    return {(adaptive_mode(c.setup(strict_math=s).params, c.bounce), c.bounce) for c, s in runs}


def test_cells_reach_every_trace_build():
    """The cells without a moon, and one strict_math run, select exactly the 20 trace builds
    nx_kernels.cu instantiates: every dispatched (MODE, BOUNCE) without MODE bit 16, and the two
    strict kernels."""
    from test_kernel_builds import dispatch_cases
    src = {(a[0], a[1]) for k, a, _ in dispatch_cases()
           if k == 'k_integrate_adaptive' and a[0] >= 0 and not (a[0] & 16)}
    assert len(src) == 18
    want = src | {(-1, False), (-1, True)}
    assert trace_builds(TRACE_RUNS) == want and len(want) == 20


# ---------------------------------------------------------------------------- GPU
def grid_of(setup):
    return (-6.0, -6.6, -4.8), (6.0, 7.2, 5.4), (37, 41, 29)


def gpu_trace(engine, setup, X0, seed, first_id, ip=None, grid=None, gt=()):
    setup.upload(engine)
    if gt:
        engine.upload_gtables(gt)
    engine.import_state(X0)
    engine.trace_begin(ip, grid)
    try:
        tot = engine.integrate_adaptive_trace(seed, first_id)
        got = engine.trace_fetch()
    finally:
        engine.trace_end()
    return engine.export_state().T, tot, engine.export_stats(), got


@pytest.mark.gpu
@pytest.mark.parametrize('cell, strict', TRACE_RUNS, ids=RUN_IDS)
def test_trace_builds_match_oracle(engine, cell, strict):
    """Every trace build against the oracle, a column image plus the grid and a radiance image;
    both trace runs are the plain run bit for bit: final state, attempted / accepted per packet
    and in total, bounces."""
    from test_kernel_builds import FIRST, K2_TOL, N, SEED, STATE_TOL, run_adaptive, same_run
    setup = cell.setup(strict_math=strict)
    X0 = cell.x0(setup, N, 21)
    (Xo, a_o, c_o, b_o, _, _), rec = run_oracle(setup, X0, SEED, FIRST)
    resident, _, _, _ = run_adaptive(engine, cell, setup, X0)
    grid = grid_of(setup)
    mid, a = trace.steps(rec, X0[:, 0], float(setup.params.endtime))
    col = image_params(setup, 'column')
    t1 = gpu_trace(engine, setup, X0, SEED, FIRST, col, grid)
    gt = setup.gtables([5891, 5897])
    rad = image_params(setup, 'radiance', dims=(41, 23))
    t2 = gpu_trace(engine, setup, X0, SEED, FIRST, rad, None, gt)
    assert same_run(t1, resident) and same_run(t2, resident)
    Xg, tot, (a_g, c_g), got = t1
    par = state_parity(Xg, Xo)
    assert par['alive_mismatch'] == 0, par
    assert np.array_equal(a_g, a_o) and np.array_equal(c_g, c_o)
    assert tot == (int(a_o.sum()), int(c_o.sum()), int(b_o.sum()))
    assert max(par['pos'], par['vel'], par['frac']) < (STATE_TOL if cell.bounce else K2_TOL), par
    nimg = compare_image(got[:2], mid, a, col, 'column', [])
    nstep = compare_grid(got[2:], mid, a, *grid)
    compare_image(t2[3][:2], mid, a, rad, 'radiance', gt)
    assert t2[3][2] is None and nstep == int(c_o.sum()) and nimg > 0
    print(cell, 'MODE', adaptive_mode(setup.params, cell.bounce), 'steps', nstep, 'image', nimg)


_TRACE_NAME = re.compile(r'k_trace_adaptive<([^>]*)>')


def trace_build_of(name):
    m = _TRACE_NAME.search(name)
    if not m:
        return None
    a = [re.sub(r'^\((?:int|bool)\)', '', x.strip()) for x in m.group(1).split(',')]
    return int(a[0]), a[1] == 'true'


@pytest.mark.gpu
def test_profiler_sees_every_trace_build(engine):
    import torch
    from torch.profiler import ProfilerActivity, profile
    assert trace_build_of('void nx::k_trace_adaptive<(int)-1, true>(nx::StateCols)') == (-1, True)
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for cell, strict in TRACE_RUNS:
            setup = cell.setup(strict_math=strict)
            gpu_trace(engine, setup, cell.x0(setup, 256, 3), 1, 0, None, grid_of(setup))
        engine.sync()
    names = {e.name for e in prof.events() if 'k_trace_adaptive' in e.name}
    print('kernels seen:', sorted(names))
    assert {trace_build_of(n) for n in names} == trace_builds(TRACE_RUNS)


@pytest.mark.gpu
def test_moons_and_missing_gtables_are_refused(engine):
    setup = setup_of('Na.Io.Jupiter.input')
    setup.upload(engine)
    engine.import_state(initial_state.draw_x0(setup, 64, 3)[:, :8])
    engine.trace_begin(None, ((-1, -1, -1), (1, 1, 1), (2, 2, 2)))
    try:
        with pytest.raises(RuntimeError, match='moons'):
            engine.integrate_adaptive_trace(0, 0)
    finally:
        engine.trace_end()
    with pytest.raises(RuntimeError, match='neither'):
        engine.trace_begin(None, None)


@pytest.mark.gpu
def test_shard_invariance(engine):
    """Two first_id halves summed are the whole run: counts exact, sums to 1e-12 of the total."""
    setup = setup_of('Na.bounce.adaptive.input')
    n, seed, h = 40000, 77, 15000
    X0 = initial_state.draw_x0(setup, n, 3)[:, :8]
    grid = ((-6., -6., -6.), (6., 7., 5.), (60, 65, 55))
    ip = image_params(setup, 'column', dims=(80, 70))
    whole = gpu_trace(engine, setup, X0, seed, 0, ip, grid)[3]
    s0 = gpu_trace(engine, setup, X0[:h], seed, 0, ip, grid)[3]
    s1 = gpu_trace(engine, setup, X0[h:], seed, h, ip, grid)[3]
    for k in (1, 3):
        assert np.array_equal(s0[k] + s1[k], whole[k]) and whole[k].sum() > 0
    assert s0[5] + s1[5] == whole[5]
    for k in (0, 2):
        assert np.allclose(s0[k] + s1[k], whole[k], rtol=0, atol=1e-12 * whole[k].sum())
    assert abs(s0[4] + s1[4] - whole[4]) <= 1e-12 * whole[2].sum()


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
    """An expectation independent of the oracle.  No forces, lifetime tau, radial ejection at a
    speed uniform in [v - dv, v + dv], T comparable to tau.  The snapshot's steady state has, per
    packet, (1/T) e^(-t/tau) dt atoms at flight times [t, t + dt), t = (r - 1)/v < T, so a shell
    [r_a, r_b) expects mu = <(tau/T)(e^(-t_a/tau) - e^(-t_b/tau))>_v, t clipped to [0, T].  The
    grid (each cell by its centre) sums frac(m) a / T per shell; the bound is 5 sigma plus the
    expectation in a band of half a cell diagonal around each shell boundary.  A packet's
    contribution is X = int e^(-t/tau) / (T - t) dt over its flight in the shell (t0 ~ U(0, T]
    limits the flight), and sigma^2 = N E[X^2], computed here by quadrature.  The same sums
    without the age factor (the run-window quantity, (1 - t/T) e^(-t/tau)) fail the bound in
    some shell, so the age weight is what passes it.  The column image in annuli of projected
    radius b >= 1.2 (no occultation) matches the Abel projection of the same profile: an atom at
    r has b < B with probability 1 - sqrt(1 - B^2/r^2)."""
    from nexoclom_b200.Input import Input
    from nexoclom_b200.runsetup import RunSetup
    v_kms, dv_kms, T, tau = 3.0, 0.02, 4000.0, 2000.0
    path = tmp_path / 'radial.input'
    path.write_text(ANALYTIC_INPUT.format(v=v_kms, dv=dv_kms, T=T, tau=tau))
    setup = RunSetup(Input(str(path)))
    assert setup.params.loss_mode == 1 and not setup.params.gravity and not setup.params.radpres
    vs = np.linspace(v_kms - dv_kms, v_kms + dv_kms, 41) / setup.radius_km       # R_p / s
    tq = np.linspace(0.0, T, 8001)[:-1] + T / 16000        # flight times (midpoint rule)
    dt = T / 8000

    def occupancy(ra, rb, weight):
        """(mean per packet, E[X^2] per packet) of int weight(t) dt over the flight in the shell."""
        means, sq = [], []
        t0 = np.linspace(0.0, T, 401)[1:] - T / 800
        for v in vs:
            r = 1.0 + v * tq
            f = np.where((r >= ra) & (r < rb), weight(tq), 0.0) * dt
            cum = np.concatenate([[0.0], np.cumsum(f)])
            x = cum[np.minimum((t0 / dt).astype(int), len(f))]        # flight limited to t0
            means.append(x.mean())
            sq.append((x * x).mean())
        return float(np.mean(means)), float(np.mean(sq))

    aged = lambda t: np.exp(-t / tau) / (T - t)                       # noqa: E731
    window = lambda t: np.exp(-t / tau) / T                           # noqa: E731

    def mu_snapshot(ra, rb):
        ta = np.clip(np.maximum(ra - 1.0, 0.0) / vs, 0, T)
        tb = np.clip(np.maximum(rb - 1.0, 0.0) / vs, 0, T)
        return float(np.mean(tau / T * (np.exp(-ta / tau) - np.exp(-tb / tau))))

    n, width, ncell = 2_000_000, 14.0, 140
    lo, hi = (-width / 2,) * 3, (width / 2,) * 3
    npix = 140
    ip = image_params(setup, 'column', dims=(npix, npix), x=(-7.0, 7.0), z=(-7.0, 7.0),
                      subobs=(0.0, np.pi / 2))
    setup.upload(engine)
    engine.init_state(setup.source_params(engine), 11, 0, n)
    engine.trace_begin(ip, (lo, hi, (ncell,) * 3))
    try:
        engine.integrate_adaptive_trace(0, 0)
        img, img_n, grid, cnt, out, out_n = engine.trace_fetch()
    finally:
        engine.trace_end()
    assert out_n == 0 and out == 0.0
    c = 0.5 * (np.linspace(lo[0], hi[0], ncell + 1)[:-1] + np.linspace(lo[0], hi[0], ncell + 1)[1:])
    r = np.sqrt(c[:, None, None]**2 + c[None, :, None]**2 + c[None, None, :]**2)
    d = np.sqrt(3) * width / ncell
    shells = [1.0, 2.0, 3.0, 4.0, 5.0, 6.0]
    window_fails = False
    for ra, rb in zip(shells[:-1], shells[1:]):
        g = grid[(r >= ra) & (r < rb)].sum() / T
        mu = mu_snapshot(ra, rb)
        _, ex2 = occupancy(ra, rb, aged)
        sigma = np.sqrt(n * ex2)
        band = sum(mu_snapshot(b - d / 2, b + d / 2) for b in (ra, rb) if b > 1.0)
        bound = 5 * sigma + n * band
        mu_w, _ = occupancy(ra, rb, window)
        print(f'shell [{ra}, {rb}): grid {g:.6g}, snapshot {n * mu:.6g}, run window {n * mu_w:.6g}, '
              f'5 sigma {5 * sigma:.3g}, boundary {n * band:.3g}')
        assert abs(g - n * mu) <= bound
        window_fails |= abs(g - n * mu_w) > bound
    assert window_fails
    # column image: sum of w a over an annulus, times apix / T, is the expected atoms there
    pc = 0.5 * (np.linspace(-7, 7, npix + 1)[:-1] + np.linspace(-7, 7, npix + 1)[1:])
    b = np.sqrt(pc[:, None] ** 2 + pc[None, :] ** 2)
    dp = np.sqrt(2) * 14.0 / npix
    rq = 1.0 + vs[:, None] * tq[None, :]
    dens = np.exp(-tq / tau)[None, :] * dt / T                         # per packet per flight time

    def projected(ba, bb):
        def cdf(B):
            return 1.0 - np.sqrt(np.clip(1.0 - (B / rq) ** 2, 0.0, 1.0))
        return float(np.mean((dens * (cdf(bb) - cdf(ba))).sum(axis=1)))
    _, ex2_all = occupancy(1.0, 100.0, aged)
    for ba, bb in ((1.2, 2.0), (2.0, 3.0), (3.0, 4.5)):
        s = img[(b >= ba) & (b < bb)].sum() * ip.apix / T
        mu = projected(ba, bb)
        band = sum(projected(x - dp / 2, x + dp / 2) for x in (ba, bb))
        bound = 5 * np.sqrt(n * ex2_all) + n * band
        print(f'annulus [{ba}, {bb}): image {s:.6g}, Abel {n * mu:.6g}, bound {bound:.3g}')
        assert abs(s - n * mu) <= bound


@pytest.mark.gpu
def test_agrees_with_model_image():
    """configs[1] at 1e7 packets: a coarse column image from the trajectories agrees with
    ModelImage's snapshot per pixel within 5 sigma, sigma from the saved rows' sum of w^2
    (independent packets), in every pixel with at least 50 rows."""
    from nexoclom_b200 import ModelImage, ModelTrajectoryImage
    inputs = workload('Na.maxwellian.radpres.input')
    inputs.delete_files()
    params = {'quantity': 'column', 'dims': '16,16', 'center': '0,0', 'width': '8,8'}
    try:
        inputs.run(10_000_000, seed=5)
        snap = ModelImage(inputs, params)
        traj = ModelTrajectoryImage(inputs, params)
        from nexoclom_b200 import catalogue
        _, files, _, _ = inputs.search()
        sq = np.zeros((16, 16))
        rows = np.zeros((16, 16))
        M = np.asarray(snap.image_rotation())
        for f in files:
            X = catalogue.fetch(f).X
            x, y, z, vy, fr = (np.asarray(X[k], np.float64) for k in ('x', 'y', 'z', 'vy', 'frac'))
            kw = dict(vrplanet=0.0, M=M, dims=[16, 16], xrange=(-4, 4), zrange=(-4, 4),
                      apix=float(snap.Apix), quantity='column')
            s2, cnt, _, _ = imaging.create_image(x, y, z, vy, fr ** 2, **kw)
            sq += s2 / float(snap.Apix)
            live = fr > 0
            rows += imaging.create_image(x[live], y[live], z[live], vy[live], fr[live], **kw)[1]
    finally:
        inputs.delete_files()
    sigma = np.sqrt(sq) * snap.atoms_per_packet
    ok = rows >= 50
    assert ok.sum() >= 20
    z = np.abs(traj.image[ok] - snap.image[ok]) / sigma[ok]
    print('pixels', int(ok.sum()), 'max |z|', z.max(), 'median |z|', np.median(z))
    assert z.max() <= 5.0
    assert traj.totalsource == snap.totalsource and traj.accepted_steps > 0
