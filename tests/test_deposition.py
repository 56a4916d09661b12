"""Surface deposition maps and the loss budget of the adaptive driver (K2 / K2b built with SINK:
nx_integrate_adaptive_deposit, Engine.integrate_adaptive_deposit, ModelDeposition).  The oracle
is oracle/deposition.py: the adaptive drivers with every event recorded and the in-flight loss
summed directly, pinned here to oracle.tracking / oracle.adaptive_bounce bit for bit."""
import ctypes as C
import os

import numpy as np
import pytest

from common import REPO, KERNEL_CELLS, Cell, workload, oracle_constants
from nexoclom_b200._lib import dptr
from nexoclom_b200.runsetup import RunSetup
from oracle import adaptive_bounce, deposition, initial_state, tracking

U32P = C.POINTER(C.c_uint32)
U64P = C.POINTER(C.c_uint64)
NLON, NLAT = 180, 90
EDGE_TOL = 1e-12             # rad: events this close to a cell edge may bin either side
SUM_TOL = 1e-12


def adaptive_inputs(name):
    """A constant-step workload on the adaptive driver (step_size = 0, resolution 1e-4)."""
    inputs = workload(name)
    inputs.options.step_size = 0.
    inputs.options.resolution = 1e-4
    return inputs


def setup_of(name, strict_math=False):
    inputs = adaptive_inputs(name) if name == 'Na.bounce.stick05.input' else workload(name)
    return RunSetup(inputs, strict_math=strict_math)


WORKLOADS = ['Ca.isotropic.flat.input', 'Na.maxwellian.radpres.input', 'Na.bounce.adaptive.input',
             'Na.bounce.stick05.input']


def is_bounce(setup):
    p = setup.params
    return not (p.sticktype == 0 and p.stickcoef == 1.0)


def run_oracle(setup, X0, seed, first_id=0):
    return deposition.integrate_adaptive(X0, oracle_constants(setup),
                                         adaptive_bounce.bounce_uniforms(seed, first_id))


def near_edge(lon, lat, nlon, nlat, tol=EDGE_TOL):
    le, ae = deposition.edges(nlon, nlat)
    dl = np.min(np.abs(lon[:, None] - le[None, :]), axis=1)
    da = np.min(np.abs(lat[:, None] - ae[None, :]), axis=1)
    return (dl < tol) | (da < tol)


def compare_sink(got, ev, nlon, nlat, exact_cells):
    """got = (map, counts, buckets, bucket_counts); ev: the oracle's events."""
    dmap, cnt, sums, counts = got
    omap, ocnt, osums, ocounts = deposition.summarize(ev, nlon, nlat)
    assert np.array_equal(counts, ocounts), (counts, ocounts)
    assert np.allclose(sums, osums, rtol=SUM_TOL, atol=SUM_TOL * max(osums[-1], 1)), (sums, osums)
    ok = np.ones((nlon, nlat), bool)           # cells compared exactly
    if not exact_cells:                        # all but those of events next to an edge
        s = ev['bucket'] == deposition.SURFACE
        edge = near_edge(ev['lon'][s], ev['lat'][s], nlon, nlat)
        touched = np.unique(deposition.cell(ev['lon'][s][edge], ev['lat'][s][edge], nlon, nlat))
        ok.ravel()[touched[touched >= 0]] = False
    assert np.array_equal(cnt[ok], ocnt[ok])
    assert int(cnt.sum()) == int(ocnt.sum())
    assert np.allclose(dmap[ok], omap[ok], rtol=SUM_TOL, atol=SUM_TOL * max(osums[-1], 1))


# ---------------------------------------------------------------------------- host build
@pytest.fixture(scope='module')
def hcd(built):
    return C.CDLL(os.path.join(REPO, 'tests', '_hostcheck', 'libnexo_deposition_hostcheck.so'))


def run_host(hcd, setup, X0, seed, first_id, strict, nlon=NLON, nlat=NLAT):
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
    dmap = np.zeros((nlon, nlat))
    cnt = np.zeros((nlon, nlat), np.uint64)
    sums = np.zeros(6)
    counts = np.zeros(6, np.uint64)
    st = hcd.hc_integrate_adaptive_deposit(
        C.c_long(n), dptr(X), att.ctypes.data_as(U32P), acc.ctypes.data_as(U32P), C.byref(p),
        dptr(rv), dptr(ra), C.c_int(nrp), dptr(tx), C.c_int(len(tx)), dptr(ty), C.c_int(len(ty)),
        dptr(c), C.c_ulonglong(seed), C.c_ulonglong(first_id), C.c_int(strict),
        C.c_int(int(is_bounce(setup))), C.c_int(nlon), C.c_int(nlat), dptr(dmap),
        cnt.ctypes.data_as(U64P), dptr(sums), counts.ctypes.data_as(U64P))
    assert st == 0
    return X, att, acc, (dmap, cnt.astype(np.int64), sums, counts.astype(np.int64))


# ---------------------------------------------------------------------------- CPU
@pytest.mark.parametrize('wl', WORKLOADS)
def test_oracle_states_equal_drivers(wl):
    """The recording driver changes nothing: final states and step counts equal
    tracking.integrate_adaptive (perfect sticking) / adaptive_bounce.integrate_adaptive bit for
    bit; per packet the summed loss plus the events equals the initial frac."""
    setup = setup_of(wl)
    rc = oracle_constants(setup)
    X0 = initial_state.draw_x0(setup, 400, 8)[:, :8]
    seed, first = 13, 500
    X, att, acc, bnc, ev, loss = run_oracle(setup, X0, seed, first)
    if is_bounce(setup):
        Xr, ar, cr, br = adaptive_bounce.integrate_adaptive(
            X0, rc, adaptive_bounce.bounce_uniforms(seed, first))
        assert np.array_equal(bnc, br) and br.sum() > 0
        assert (ev['bucket'] == deposition.SURFACE).sum() == br.sum()
    else:
        Xr, ar, cr = tracking.integrate_adaptive(X0, rc)
    assert np.array_equal(X, Xr) and np.array_equal(att, ar) and np.array_equal(acc, cr)
    per = np.zeros(len(X0))
    mine = ev['bucket'] != deposition.SOURCE
    np.add.at(per, ev['packet'][mine], ev['amount'][mine])
    init = np.where(X0[:, 7] > 0, X0[:, 7], 0.)
    assert np.all(np.abs(per + loss - init) <= 1e-13 * np.maximum(init, 1e-300))


@pytest.mark.parametrize('wl', ['Ca.isotropic.flat.input', 'Na.maxwellian.radpres.input'])
def test_oracle_events_classify_final_state(wl):
    """Perfect sticking: a dead packet inside the planet stuck there, one past outeredge escaped,
    any other dead one vanished; live ones remain."""
    setup = setup_of(wl)
    X0 = initial_state.draw_x0(setup, 600, 9)[:, :8]
    X, _, _, _, ev, _ = run_oracle(setup, X0, 0)
    rc = oracle_constants(setup)
    r2 = (X[:, 1]**2 + X[:, 2]**2) + X[:, 3]**2
    dead = X[:, 7] == 0
    want = np.full(len(X), deposition.REMAINING)
    want[dead & (r2 < 1)] = deposition.SURFACE
    want[dead & (r2 > rc.outeredge)] = deposition.ESCAPED
    want[dead & (r2 >= 1) & (r2 <= rc.outeredge)] = deposition.VANISHED
    fate = ev['bucket'] != deposition.SOURCE
    got = np.full(len(X), -1)
    got[ev['packet'][fate]] = ev['bucket'][fate]
    assert np.bincount(ev['packet'][fate], minlength=len(X)).max() == 1
    assert np.array_equal(got, want)
    assert (want == deposition.SURFACE).sum() > 0


# the workloads, and every force x loss x moon cell of the adaptive driver
@pytest.mark.parametrize('wl', WORKLOADS + [c for c in KERNEL_CELLS if c.driver == 'adaptive'],
                         ids=str)
@pytest.mark.parametrize('strict', [1, 0])
def test_host_build_matches_oracle(hcd, wl, strict):
    from test_hostcheck import host_strict
    if isinstance(wl, Cell):
        setup = wl.setup(strict_math=bool(strict))
        X0 = wl.x0(setup, 300, 21)
    else:
        setup = setup_of(wl, strict_math=bool(strict))
        X0 = initial_state.draw_x0(setup, 300, 21)[:, :8]
    seed, first = 5, 1000
    Xo, a_o, c_o, b_o, ev, _ = run_oracle(setup, X0, seed, first)
    Xh, a_h, c_h, got = run_host(hcd, setup, X0, seed, first,
                                 host_strict(setup, strict, is_bounce(setup)))
    assert np.array_equal(a_h, a_o) and np.array_equal(c_h, c_o)
    compare_sink(got, ev, NLON, NLAT, exact_cells=False)
    # Sigma map == SURFACE, and the host's own sums add up to its source
    dmap, cnt, sums, counts = got
    assert cnt.sum() == counts[deposition.SURFACE]
    assert abs(dmap.sum() - sums[deposition.SURFACE]) <= 1e-12 * max(sums[-1], 1)


def test_bin_helper_matches_histogram2d(hcd):
    """deposit_cell at every edge and one ulp either side, against np.histogram2d's rule."""
    for nlon, nlat in ((180, 90), (7, 5), (1, 1), (360, 181)):
        le, ae = deposition.edges(nlon, nlat)
        lon = np.concatenate([le, np.nextafter(le, -np.inf), np.nextafter(le, np.inf)])
        lat = np.concatenate([ae, np.nextafter(ae, -np.inf), np.nextafter(ae, np.inf)])
        L, A = np.meshgrid(lon, lat[:: max(1, len(lat) // 40)], indexing='ij')
        L2, A2 = np.meshgrid(lon[:: max(1, len(lon) // 40)], lat, indexing='ij')
        L, A = np.concatenate([L.ravel(), L2.ravel()]), np.concatenate([A.ravel(), A2.ravel()])
        want = deposition.cell(L, A, nlon, nlat)
        got = np.array([hcd.hc_deposit_cell(C.c_double(a), C.c_double(b), nlon, nlat)
                        for a, b in zip(L, A)])
        assert np.array_equal(got, want)
        # and deposition.cell is np.histogram2d's rule
        inside = want >= 0
        h, _, _ = np.histogram2d(L, A, bins=(le, ae))
        assert np.array_equal(np.bincount(want[inside], minlength=nlon * nlat).reshape(nlon, nlat),
                              h.astype(np.int64))


def test_validation_before_device_work():
    from nexoclom_b200 import ModelDeposition
    with pytest.raises(ValueError, match='adaptive driver'):
        ModelDeposition(workload('Na.bounce.input'))
    inputs = workload('Na.maxwellian.radpres.input')
    for bad in ({'nlonbins': 0}, {'nlatbins': -3}, {'nlonbins': 2.5}, {'nlatbins': 'x'},
                {'nlonbins': True}):
        with pytest.raises(ValueError, match='positive integer'):
            ModelDeposition(inputs, bad)


def test_validation_bounce_output_without_seed(monkeypatch):
    """A bounce run written by the reference (no seed) cannot be regenerated."""
    from nexoclom_b200 import ModelDeposition, catalogue

    class RefOutput:
        imported_x0 = True
        from_reference = True
        _imported_cols = [np.zeros(3)] * 8
        npackets = 3
        totalsource = 3.
        first_id = 0

    inputs = workload('Na.bounce.adaptive.input')
    monkeypatch.setattr(type(inputs), 'search', lambda self: ([1], ['ref.pkl'], 3, None))
    monkeypatch.setattr(catalogue, 'fetch', lambda f: RefOutput())
    with pytest.raises(ValueError, match='seed'):
        ModelDeposition(inputs)


def test_budget_and_units():
    """The product's host arithmetic: budget fractions, rates, the map in cm^-2 s^-1."""
    from nexoclom_b200.ModelDeposition import ModelDeposition, cell_area
    inputs = workload('Na.maxwellian.radpres.input')
    d = ModelDeposition.__new__(ModelDeposition)
    d.inputs, d.nlon, d.nlat = inputs, 4, 3
    dmap = np.zeros((4, 3))
    dmap[1, 2] = 3.0
    sums = np.array([3.0, 0.5, 1.0, 0.25, 2.0, 10.0])
    d._finish(dmap, np.ones((4, 3), np.int64), sums, np.arange(6), 10.0)
    endtime = float(np.asarray(inputs.options.endtime))
    assert d.atoms_per_packet == pytest.approx(1e23 * endtime / 10.0)
    assert list(d.budget.index) == ['surface', 'moon', 'escaped', 'vanished', 'remaining', 'lost']
    assert d.budget['lost'] == pytest.approx(0.325) and d.budget.sum() == pytest.approx(1.0)
    assert d.rates.sum() == pytest.approx(1e23)
    r_cm = float(np.asarray(inputs.geometry.planet.radius.value)) * 1e5
    area = cell_area(4, 3, r_cm)
    assert area.sum() == pytest.approx(4 * np.pi * r_cm**2)
    assert d.deposition[1, 2] == pytest.approx(3.0 * d.atoms_per_packet / endtime / area[1, 2])
    assert (d.deposition * area).sum() == pytest.approx(d.rates['surface'])


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank),
                      WORLD_SIZE=str(world))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        from nexoclom_b200.sharding import combine_ranks
        dmap = np.full((3, 2), rank + 1.0)
        cnt = np.full((3, 2), rank + 1, np.int64)
        sums = np.arange(6.0) * (rank + 1)
        counts = np.arange(6, dtype=np.int64) * (rank + 1)
        tot, = combine_ranks((dmap, cnt, sums, counts), 10.0 * (rank + 1))
        q.put((rank, dmap.tolist(), cnt.tolist(), sums.tolist(), counts.tolist(), tot))
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
    for _, dmap, cnt, sums, counts, tot in res:
        assert np.all(np.array(dmap) == 3.0) and np.all(np.array(cnt) == 3)
        assert np.array_equal(sums, np.arange(6.0) * 3) and np.array_equal(counts, np.arange(6) * 3)
        assert tot == 30.0


# ---------------------------------------------------------------------------- GPU
def gpu_deposit(engine, setup, X0, seed, first_id=0, nlon=NLON, nlat=NLAT):
    setup.upload(engine)
    engine.import_state(X0)
    engine.deposit_begin(nlon, nlat)
    try:
        att, acc, bnc = engine.integrate_adaptive_deposit(seed, first_id)
        got = engine.deposit_fetch(nlon, nlat)
    finally:
        engine.deposit_end()
    return engine.export_state().T, (att, acc, bnc), engine.export_stats(), got


@pytest.mark.gpu
@pytest.mark.parametrize('wl', WORKLOADS + ['Na.Io.Jupiter.input'])
@pytest.mark.parametrize('strict', [True, False])
def test_kernel_matches_oracle(engine, hcd, wl, strict):
    setup = setup_of(wl, strict_math=strict)
    n, seed, first = 3000, 17, 123
    X0 = initial_state.draw_x0(setup, n, 21)[:, :8]
    Xg, tot, stats, got = gpu_deposit(engine, setup, X0, seed, first)
    _, a_o, c_o, b_o, ev, _ = run_oracle(setup, X0, seed, first)
    assert np.array_equal(stats[0], a_o) and np.array_equal(stats[1], c_o)
    if strict:
        compare_sink(got, ev, NLON, NLAT, exact_cells=True)
    else:
        compare_sink(got, ev, NLON, NLAT, exact_cells=False)
        _, _, _, hgot = run_host(hcd, setup, X0, seed, first, 0)
        assert np.array_equal(got[3], hgot[3]) and np.array_equal(got[1], hgot[1])
        assert np.allclose(got[2], hgot[2], rtol=SUM_TOL, atol=SUM_TOL * n)
    if is_bounce(setup):
        assert got[3][deposition.SURFACE] == tot[2] > 0
    else:
        assert tot[2] == 0
    if wl == 'Na.Io.Jupiter.input':
        assert got[3][deposition.MOON] > 0


@pytest.mark.gpu
@pytest.mark.parametrize('wl', ['Na.maxwellian.radpres.input', 'Na.bounce.adaptive.input'])
def test_sink_leaves_the_run_unchanged(engine, wl):
    """Final state, per-packet and total step counts equal the entry without the sink, bit for
    bit; surface events == bounces for bounce runs."""
    setup = RunSetup(workload(wl))
    X0 = initial_state.draw_x0(setup, 20000, 2)[:, :8]
    seed = 9
    setup.upload(engine)
    engine.import_state(X0)
    if is_bounce(setup):
        att, acc, bnc = engine.integrate_adaptive_bounce(seed, 0)
    else:
        (att, acc), bnc = engine.integrate_adaptive(), 0
    Xa, sa = engine.export_state().T, engine.export_stats()
    Xd, tot, sd, got = gpu_deposit(engine, setup, X0, seed)
    assert np.array_equal(Xa, Xd) and (att, acc, bnc) == tot
    assert np.array_equal(sa[0], sd[0]) and np.array_equal(sa[1], sd[1])
    if is_bounce(setup):
        assert got[3][deposition.SURFACE] == bnc


@pytest.mark.gpu
def test_invariances(engine):
    """Counts do not depend on the packet order, the sharding or a repeated call."""
    setup = RunSetup(workload('Na.bounce.adaptive.input'))
    n, seed = 40000, 77
    X0 = initial_state.draw_x0(setup, n, 3)[:, :8]
    ref = gpu_deposit(engine, setup, X0, seed)
    try:
        engine.set_option('order_packets', 0)
        plain = gpu_deposit(engine, setup, X0, seed)
    finally:
        engine.set_option('order_packets', 3)
    again = gpu_deposit(engine, setup, X0, seed)
    h = 15000
    s0 = gpu_deposit(engine, setup, X0[:h], seed, 0)
    s1 = gpu_deposit(engine, setup, X0[h:], seed, h)
    for run in (plain, again):
        assert np.array_equal(run[3][1], ref[3][1]) and np.array_equal(run[3][3], ref[3][3])
        assert np.allclose(run[3][2], ref[3][2], rtol=1e-12)
    assert np.array_equal(s0[3][1] + s1[3][1], ref[3][1])
    assert np.array_equal(s0[3][3] + s1[3][3], ref[3][3])
    assert np.allclose(s0[3][0] + s1[3][0], ref[3][0], rtol=1e-12, atol=1e-12)


@pytest.mark.gpu
@pytest.mark.parametrize('wl', ['Na.maxwellian.radpres.input', 'Na.bounce.adaptive.input'])
def test_full_size(engine, wl):
    """1e7 packets: the buckets add up, the map sums to SURFACE, REMAINING is the final state's
    frac, and with perfect sticking the fates classify the final state exactly."""
    setup = RunSetup(workload(wl))
    setup.upload(engine)
    n, seed = 10_000_000, 5
    engine.init_state(setup.source_params(engine), seed, 0, n)
    engine.deposit_begin(NLON, NLAT)
    try:
        att, acc, bnc = engine.integrate_adaptive_deposit(seed, 0)
        dmap, cnt, sums, counts = engine.deposit_fetch(NLON, NLAT)
    finally:
        engine.deposit_end()
    X = engine.export_state()
    S = deposition
    assert counts[S.SOURCE] == n and sums[S.SOURCE] == pytest.approx(n, rel=1e-15)
    # SOURCE == the buckets + the in-flight loss, and the loss is >= 0 (to rounding)
    lost = sums[S.SOURCE] - sums[:S.SOURCE].sum()
    assert lost >= -1e-12 * n
    assert cnt.sum() == counts[S.SURFACE]
    assert abs(dmap.sum() - sums[S.SURFACE]) <= 1e-12 * n
    live = X[7] > 0
    assert counts[S.REMAINING] == live.sum()
    assert abs(sums[S.REMAINING] - X[7][live].sum()) <= 1e-12 * n
    if is_bounce(setup):
        assert counts[S.SURFACE] == bnc > n
    else:
        r2 = (X[1]**2 + X[2]**2) + X[3]**2
        dead = ~live
        outer = float(setup.params.outeredge)
        assert counts[S.SURFACE] == (dead & (r2 < 1)).sum()
        assert counts[S.ESCAPED] == (dead & (r2 > outer)).sum()
        assert counts[S.VANISHED] == (dead & (r2 >= 1) & (r2 <= outer)).sum()
        assert counts[S.MOON] == 0
        assert counts[:S.SOURCE].sum() == n


@pytest.mark.gpu
def test_public_api(engine):
    """Over two output files (device-drawn and imported X0): the product's counts are the sum
    of the sink runs of the two.  ModelDeposition leaves what the other products read alone:
    the Outputs' resident tables are bit-identical after it, and so is ModelImage's packet
    image.  The image itself is compared to 1e-12: K4 adds each row's weight to its pixel with
    an f64 atomic, so the order of the additions, and with it the last bits of a pixel, varies
    from one ModelImage to the next whether or not anything ran in between."""
    from nexoclom_b200 import ModelDeposition, ModelImage, Output, catalogue
    inputs = workload('Na.bounce.adaptive.input')
    inputs.delete_files()
    n = 100_000
    try:
        inputs.run(n, seed=41)
        setup = RunSetup(inputs)
        X0b = initial_state.draw_x0(setup, n, 12)[:, :8]
        Output(inputs, n, X0=X0b, seed=42, first_id=n)
        _, files, npk, _ = inputs.search()
        assert npk == 2 * n and len(files) == 2
        outs = [catalogue.fetch(f) for f in files]
        before = [o.X.copy() for o in outs]
        tables = [o.device_table().export() for o in outs]
        params = {'quantity': 'column', 'dims': '80,80', 'width': '8,8', 'center': '0,0',
                  'subobslongitude': '0.7', 'subobslatitude': '0.3'}
        img0 = ModelImage(inputs, params)
        dep = ModelDeposition(inputs, {'nlonbins': 72, 'nlatbins': 36})
        img1 = ModelImage(inputs, params)
        for o, (cols, index) in zip(outs, tables):
            cols1, index1 = o.device_table().export()
            assert np.array_equal(index1, index)
            assert all(np.array_equal(cols1[c], cols[c]) for c in cols)
        for o, b in zip(outs, before):
            assert o.X.equals(b)
        assert np.array_equal(np.asarray(img0.packet_image), np.asarray(img1.packet_image))
        assert np.asarray(img0.packet_image).sum() > 0
        assert np.allclose(np.asarray(img1.image), np.asarray(img0.image), rtol=1e-12, atol=0)
        assert dep.event_counts['source'] == 2 * n
        assert dep.event_counts['surface'] == sum(o.bounces for o in outs)
        assert dep.packet_map.shape == (72, 36) and dep.packet_map.sum() == dep.event_counts['surface']
        assert dep.budget.sum() == pytest.approx(1.0, abs=1e-12)
        assert (dep.budget >= -1e-12).all() and dep.budget['surface'] > 0
        assert dep.budget['lost'] > 0 and dep.budget['remaining'] > 0
        assert dep.totalsource == 2 * n
        # each file on its own through the engine, summed
        tot = np.zeros(6, np.int64)
        for o in outs:
            if o.imported_x0:
                Xs = X0b
            else:
                setup.upload(engine)
                engine.init_state(setup.source_params(engine), o.seed, o.first_id, n)
                Xs = engine.export_x0()[:8].T.copy()
            tot += gpu_deposit(engine, setup, Xs, o.seed, o.first_id, 72, 36)[3][3]
        assert np.array_equal(tot, dep.event_counts.values)
    finally:
        inputs.delete_files()
