"""Doppler line profiles along lines of sight (LOSSpectrum, ``nx_los_spectrum``).

CPU: the oracle against the reference's own compute_iteration output (tests/golden/los.npz),
the host build of the velocity / column helpers against NumPy, input validation and the
sharded reduction.  GPU (``-m gpu``): the kernel against the oracle, the column invariants
against ``nx_los_accumulate`` (directly and through LOSResult), recipe-only runs, a small pair
buffer, K5's kept candidate pairs, edge cases and the full configs[1] size."""
import ctypes as C
import os
import sys

import numpy as np
import pandas as pd
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

from common import REPO, workload
from nexoclom_b200.LOSSpectrum import velocity_bins
from nexoclom_b200.sharding import combine_ranks
from oracle import imaging
from oracle import spectrum as ospec

GOLDEN = os.path.join(REPO, 'tests', 'golden')


def _na_setup():
    from nexoclom_b200.runsetup import RunSetup
    return RunSetup(workload('Na.maxwellian.radpres.input'))


# ---------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------
@pytest.mark.parametrize('tag', ['d1', 'd3'])
@pytest.mark.parametrize('nbins, vmin, vmax', [(1, -5.0, 5.0), (40, -8.0, 8.0), (7, 0.5, 1.5)])
def test_oracle_columns_sum_to_golden(tag, nbins, vmin, vmax):
    """Summed over all columns the oracle spectrum is the reference's own compute_iteration()
    output: hit counts exactly, radiance to 1e-12; the rows with w > 0 are its `used` sets."""
    g = np.load(os.path.join(GOLDEN, 'los.npz'))
    setup = _na_setup()
    X = g['X']
    hits = ospec.los_hits(X[:, 1], X[:, 2], X[:, 3], X[:, 5], X[:, 7], g['los'],
                          vrplanet=setup.vrplanet, dphi=float(g[f'{tag}_dphi']),
                          outeredge=float(g['outeredge']), rp_cm=setup.radius_km * 1e5,
                          gtables=setup.gtables([5891, 5897]))
    spec, cnt = ospec.los_spectrum(X[:, 4], X[:, 5], X[:, 6], g['los'], hits, vmin, vmax, nbins,
                                   setup.radius_km)
    assert np.array_equal(cnt.sum(axis=1), g[f'{tag}_npackets'])
    ref = g[f'{tag}_radiance']
    nz = ref > 0
    assert np.array_equal(spec.sum(axis=1) > 0, nz) and nz.sum() > 10
    assert np.max(np.abs(spec.sum(axis=1)[nz] - ref[nz]) / ref[nz]) < 1e-12
    off, idx = g[f'{tag}_used_off'], g[f'{tag}_used_idx']
    for i, (sel, w) in enumerate(hits):
        assert set(sel[w > 0].tolist()) == set(idx[off[i]:off[i + 1]].tolist())
    if nbins == 7:                    # a narrow range: most of the hits fall outside
        assert cnt[:, [0, -1]].sum() > cnt[:, 1:-1].sum() > 0


@pytest.mark.parametrize('source', ['golden_d1', 'golden_d3', 'cloud'])
def test_oracle_hits_are_los_iteration(source):
    """``los_hits`` is ``imaging.los_iteration`` with its per-line hit sets kept: the same hit
    counts, included mask and `used` sets, and its weights sum to the same radiance bit for bit."""
    setup = _na_setup()
    if source == 'cloud':
        X, los, dphi, edge = _gloo_cloud(), _los(60, 2), np.radians(2.0), 25.0
    else:
        g = np.load(os.path.join(GOLDEN, 'los.npz'))
        tag = source[-2:]
        X, los, dphi, edge = g['X'], g['los'], float(g[f'{tag}_dphi']), float(g['outeredge'])
    kw = dict(vrplanet=setup.vrplanet, dphi=dphi, outeredge=edge, rp_cm=setup.radius_km * 1e5,
              gtables=setup.gtables([5891, 5897]))
    args = (X[:, 1], X[:, 2], X[:, 3], X[:, 5], X[:, 7], los)
    used = []
    rad, npk, inc, _ = imaging.los_iteration(*args, used=used, **kw)
    hits = ospec.los_hits(*args, **kw)
    assert len(hits) == len(los) and npk.sum() > 100
    got_inc = np.zeros(len(X), dtype=bool)
    for i, (sel, w) in enumerate(hits):
        assert len(sel) == npk[i] and len(w) == npk[i]
        assert (w.sum() if len(w) else 0.0) == rad[i]
        assert set(sel[w > 0].tolist()) == used[i]
        got_inc[sel] = True
    assert np.array_equal(got_inc, inc)


@pytest.fixture(scope='module')
def hc(built):
    return C.CDLL(os.path.join(REPO, 'tests', '_hostcheck', 'libnexo_spectrum_hostcheck.so'))


def _host_columns(hc, v, vmin, vmax, nbins):
    v = np.ascontiguousarray(v, dtype=np.float64)
    out = np.zeros(len(v), dtype=np.int32)
    hc.hc_spectrum_column(C.c_long(len(v)), v.ctypes.data_as(C.POINTER(C.c_double)),
                          C.c_double(vmin), C.c_double(vmax), C.c_int(nbins),
                          out.ctypes.data_as(C.POINTER(C.c_int32)))
    return out


def test_host_doppler_matches_numpy(hc):
    g = np.random.default_rng(3)
    n = 100_000
    V = (g.standard_normal((n, 3)) * 3e-3).astype(np.float32)     # R_p/s
    fp = C.POINTER(C.c_float)
    cols = [np.ascontiguousarray(V[:, k]) for k in range(3)]
    for trial in range(5):
        b = g.standard_normal(3)
        b /= np.linalg.norm(b)
        vscale = 2439.7 if trial else 1.0
        got = np.zeros(n)
        hc.hc_los_doppler(C.c_long(n), *[c.ctypes.data_as(fp) for c in cols], *map(C.c_double, b),
                          C.c_double(vscale), got.ctypes.data_as(C.POINTER(C.c_double)))
        W = V.astype(np.float64)
        ref = ospec.doppler(W[:, 0], W[:, 1], W[:, 2], b[0], b[1], b[2], vscale)
        assert np.array_equal(got.view(np.int64), ref.view(np.int64))


@pytest.mark.parametrize('vmin, vmax, nbins', [
    (-10.0, 10.0, 1), (-10.0, 10.0, 64), (-3.3, 7.1, 1000), (0.1, 0.7, 3), (-1e-3, 2.5e-3, 17),
])
def test_host_columns_match_numpy(hc, vmin, vmax, nbins):
    """Every edge exactly, one and two ulps either side of it, vmin / vmax and their
    neighbours, and random values inside and outside the range."""
    edges = np.linspace(vmin, vmax, nbins + 1)
    v = [edges]
    up, dn = edges, edges
    for _ in range(2):
        up, dn = np.nextafter(up, np.inf), np.nextafter(dn, -np.inf)
        v += [up, dn]
    g = np.random.default_rng(nbins)
    span = vmax - vmin
    v.append(g.uniform(vmin - 0.2 * span, vmax + 0.2 * span, 20000))
    v.append(np.array([vmin, vmax, -np.inf, np.inf]))
    v = np.concatenate(v)
    got = _host_columns(hc, v, vmin, vmax, nbins)
    ref = ospec.columns(v, vmin, vmax, nbins)
    assert np.array_equal(got, ref)
    assert got[v == vmax].min() == nbins and got[v == vmin].max() == 1
    assert np.all(got[v < vmin] == 0) and np.all(got[v > vmax] == nbins + 1)


class _SC:
    """Duck type of the spacecraft data LOSResult / LOSSpectrum read."""

    def __init__(self, los, species='Na', index=None):
        self.data = pd.DataFrame(los, columns=['x', 'y', 'z', 'xbore', 'ybore', 'zbore'],
                                 index=index)
        self.data['radiance'] = np.linspace(1.0, 3.0, len(los))
        self.data['sigma'] = 0.1
        self.data['alttan'] = 1.0
        self.species = species
        self.query = 'synthetic'
        self.subslong = self.data.x * 0
        self.frame = None

    def set_frame(self, frame):
        self.frame = frame

    def __len__(self):
        return len(self.data)


def _los(nlos, seed, far=1.5):
    """(nlos, 6) lines of sight from far .. far + 3 R_p towards points within 3 R_p."""
    g = np.random.default_rng(seed)
    x_sc = g.standard_normal((3, nlos))
    x_sc *= (far + 3 * g.random(nlos)) / np.linalg.norm(x_sc, axis=0)
    tgt = g.standard_normal((3, nlos))
    tgt *= (1 + 2 * g.random(nlos)) / np.linalg.norm(tgt, axis=0)
    bore = tgt - x_sc
    bore /= np.linalg.norm(bore, axis=0)
    return np.concatenate([x_sc, bore]).T.copy()


def test_los_spectrum_rejects_bad_input():
    """Bad arguments raise ValueError before anything touches a device."""
    from nexoclom_b200 import LOSSpectrum
    inputs = workload('Na.maxwellian.radpres.input')
    sc = _SC(_los(4, 1))
    for velocity in [(0.0, 1.0), (0.0, 1.0, 4, 5), 'abc', 3.0, None,
                     (np.nan, 1.0, 4), (0.0, np.inf, 4), (1.0, 1.0, 4), (2.0, 1.0, 4),
                     (0.0, 1.0, 0), (0.0, 1.0, -3), (0.0, 1.0, 2.5), (0.0, 1.0, True),
                     (0.0, 1.0, '4'), ('a', 1.0, 4), (0.0, 1.0, 2**31)]:
        with pytest.raises(ValueError):
            LOSSpectrum(sc, inputs, velocity)
    with pytest.raises(ValueError):
        LOSSpectrum(sc, inputs, (0.0, 1.0, 4), params={'quantity': 'column'})
    with pytest.raises(ValueError):
        velocity_bins((0.0, 1.0, 2**20), 2**11)                 # 2**31 + 2**12 cells
    assert velocity_bins((-1, 1, np.int64(3)), 10) == (-1.0, 1.0, 3)


def _gloo_lines():
    return _los(40, 8)


def _gloo_cloud(n=30000):
    g = np.random.default_rng(6)
    X = np.zeros((n, 8))
    u = g.standard_normal((n, 3))
    u /= np.linalg.norm(u, axis=1)[:, None]
    X[:, 1:4] = u * (1 + g.exponential(0.5, n))[:, None]
    X[:, 4:7] = g.standard_normal((n, 3)) * 1e-3
    X[:, 7] = g.random(n) + 0.01
    return X.astype(np.float32).astype(np.float64)


def _oracle_spectrum(X, los, setup, dphi, vmin, vmax, nbins):
    hits = ospec.los_hits(X[:, 1], X[:, 2], X[:, 3], X[:, 5], X[:, 7], los,
                          vrplanet=setup.vrplanet, dphi=dphi, outeredge=25.0,
                          rp_cm=setup.radius_km * 1e5, gtables=setup.gtables([5891, 5897]))
    return ospec.los_spectrum(X[:, 4], X[:, 5], X[:, 6], los, hits, vmin, vmax, nbins,
                              setup.radius_km)


def _gloo_worker(rank, world, port, q):
    sys.path.insert(0, REPO)
    sys.path.insert(0, os.path.join(REPO, 'tests'))
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    from nexoclom_b200.sharding import combine_ranks
    from nexoclom_b200.sharding import shard_range
    X = _gloo_cloud()
    first, n = shard_range(len(X), rank, world)
    spec, cnt = _oracle_spectrum(X[first:first + n], _gloo_lines(), _na_setup(),
                                 np.radians(3.0), -6.0, 6.0, 24)
    tot = combine_ranks((spec, cnt), float(n), n)        # what LOSSpectrum does per product
    if rank == 0:
        q.put((spec, cnt, tot))
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_allreduce_equals_single_rank():
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = 35500 + os.getpid() % 2000
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    spec, cnt, tot = q.get(timeout=300)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    ospec_, ocnt = _oracle_spectrum(_gloo_cloud(), _gloo_lines(), _na_setup(), np.radians(3.0),
                                    -6.0, 6.0, 24)
    assert np.array_equal(cnt, ocnt) and ocnt.sum() > 1000
    assert tot == (30000.0, 30000)
    nz = ospec_ > 0
    assert np.array_equal(spec > 0, nz)
    assert np.max(np.abs(spec[nz] - ospec_[nz]) / ospec_[nz]) < 1e-12
    a, c = ospec_.copy(), ocnt.copy()                    # a single process: left alone
    assert combine_ranks((a, c), 5.0, 5) == (5.0, 5) and np.array_equal(a, ospec_)


# ---------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------
def _lp(setup, dphi_deg, round_f32=1, skip_dead=1):
    from nexoclom_b200._lib import LosParams
    lp = LosParams()
    lp.dphi, lp.outeredge = float(np.radians(dphi_deg)), 25.0
    lp.vrplanet, lp.rp_cm = setup.vrplanet, setup.radius_km * 1e5
    lp.quantity, lp.round_f32, lp.skip_dead = 1, round_f32, skip_dead
    return lp


def _dplan(los):
    x, b = los[:, :3], los[:, 3:]
    d = np.linalg.norm(x, axis=1)
    ang = np.arccos(np.clip(-(x * b).sum(axis=1) / d, -1.0, 1.0))
    return np.where(ang > np.arcsin(1. / d), 1e30, d)


def _assert_spectra(got, ref, tol=1e-12):
    spec, cnt = got
    ospec_, ocnt = ref
    assert np.array_equal(cnt, ocnt), f'counts differ at {np.argwhere(cnt != ocnt)[:10]}'
    nz = ospec_ != 0
    assert np.array_equal(spec != 0, nz)
    if nz.any():
        err = np.abs(spec[nz] - ospec_[nz]) / np.abs(ospec_[nz])
        assert err.max() <= tol, (err.max(), np.argwhere(nz)[int(np.argmax(err))])


def _table_X(table):
    """(n, 8) float64 rows (float32 values) of a packet table, table row order."""
    cols, _ = table.export()
    return np.stack([cols[k].astype(np.float64) for k in
                     ('time', 'x', 'y', 'z', 'vx', 'vy', 'vz', 'frac')], axis=1)


def _run_table(engine, name, n, seed, first_id=0, integrate=True):
    """Saved rows of a run: its final state, or (``integrate=False``) its initial state, where
    every packet is live -- the final state of configs[1] keeps ~1 % of the packets."""
    from nexoclom_b200.runsetup import RunSetup
    setup = RunSetup(workload(name))
    setup.upload(engine)
    engine.init_state(setup.source_params(engine), seed, first_id, n)
    if integrate:
        engine.integrate_adaptive(n)
    return setup, engine.compact_state(skip_dead=True, round_f32=True, n=n)


def _spectrum(engine, table, los, lp, vmin, vmax, nbins, vscale):
    engine.bind_packets(table)
    try:
        return engine.los_spectrum(los.T.copy(), _dplan(los), lp, vmin, vmax, nbins, vscale,
                                   n=table.n)
    finally:
        engine.bind_packets(None)


def _accumulate(engine, table, los, lp):
    engine.bind_packets(table)
    try:
        rad, npk, _ = engine.los_accumulate(los.T.copy(), _dplan(los), lp, n=table.n)
        return rad, npk
    finally:
        engine.bind_packets(None)


def _assert_invariants(got, acc, tol=1e-12):
    spec, cnt = got
    rad, npk = acc
    assert np.array_equal(cnt.sum(axis=1), npk)
    nz = rad > 0
    assert np.array_equal(spec.sum(axis=1) > 0, nz)
    if nz.any():
        assert np.max(np.abs(spec.sum(axis=1)[nz] - rad[nz]) / rad[nz]) <= tol


RANGES = [(-10.0, 10.0, 1), (-10.0, 10.0, 64), (-12.0, 12.0, 1000), (0.2, 0.9, 16)]


@pytest.mark.gpu
def test_kernel_matches_oracle_synthetic(engine):
    setup, table = _run_table(engine, 'Na.maxwellian.radpres.input', 200_000, 11, integrate=False)
    try:
        engine.upload_gtables(setup.gtables([5891, 5897]))
        X = _table_X(table)
        los = _los(150, 12)
        lp = _lp(setup, 2.0)
        acc = _accumulate(engine, table, los, lp)
        hits = ospec.los_hits(X[:, 1], X[:, 2], X[:, 3], X[:, 5], X[:, 7], los,
                              vrplanet=setup.vrplanet, dphi=lp.dphi, outeredge=25.0,
                              rp_cm=lp.rp_cm, gtables=setup.gtables([5891, 5897]))
        for vmin, vmax, nbins in RANGES:
            got = _spectrum(engine, table, los, lp, vmin, vmax, nbins, setup.radius_km)
            assert got[0].shape == (150, nbins + 2)
            ref = ospec.los_spectrum(X[:, 4], X[:, 5], X[:, 6], los, hits, vmin, vmax, nbins,
                                     setup.radius_km)
            _assert_spectra(got, ref)
            _assert_invariants(got, acc)
        assert acc[1].sum() > 10_000
        assert ref[1][:, [0, -1]].sum() > ref[1][:, 1:-1].sum() > 0      # the narrow range
    finally:
        table.free()


@pytest.mark.gpu
@pytest.mark.parametrize('tag', ['d1', 'd3'])
def test_kernel_matches_oracle_golden_packets(engine, tag):
    g = np.load(os.path.join(GOLDEN, 'los.npz'))
    setup = _na_setup()
    engine.upload_gtables(setup.gtables([5891, 5897]))
    X = g['X'][g['X'][:, 7] > 0].astype(np.float32).astype(np.float64)
    los = g['los']
    lp = _lp(setup, np.degrees(float(g[f'{tag}_dphi'])))
    lp.outeredge = float(g['outeredge'])
    table = engine.upload_packets(X)
    try:
        acc = _accumulate(engine, table, los, lp)
        hits = ospec.los_hits(X[:, 1], X[:, 2], X[:, 3], X[:, 5], X[:, 7], los,
                              vrplanet=setup.vrplanet, dphi=lp.dphi, outeredge=lp.outeredge,
                              rp_cm=lp.rp_cm, gtables=setup.gtables([5891, 5897]))
        for vmin, vmax, nbins in RANGES:
            got = _spectrum(engine, table, los, lp, vmin, vmax, nbins, setup.radius_km)
            ref = ospec.los_spectrum(X[:, 4], X[:, 5], X[:, 6], los, hits, vmin, vmax, nbins,
                                     setup.radius_km)
            _assert_spectra(got, ref)
            _assert_invariants(got, acc)
        assert acc[1].sum() > 100
    finally:
        table.free()


@pytest.fixture(scope='module')
def two_files(engine):
    inputs = workload('Na.maxwellian.radpres.input')
    inputs.delete_files()
    inputs.run(200_000, seed=5)
    inputs.run(400_000, seed=6)              # 200 000 more in a second output file
    _, files, npk, _ = inputs.search()
    assert npk == 400_000
    yield inputs, files
    inputs.delete_files()


@pytest.mark.gpu
def test_public_api_matches_losresult(two_files):
    from nexoclom_b200 import LOSResult, LOSSpectrum
    from nexoclom_b200.units import Quantity
    inputs, files = two_files
    assert len(files) == 2
    los = _los(120, 21)
    sc = _SC(los, index=[f's{i}' for i in range(120)])
    res = LOSResult(sc, inputs, dphi=Quantity(3.0, 'deg'))
    res.simulate_data_from_inputs(sc)
    raw = sum(res._iterations[f].radiance.values for f in files) * res.atoms_per_packet / 1e3
    sp = LOSSpectrum(sc, inputs, (-8.0, 8.0, 32), dphi=Quantity(3.0, 'deg'))
    assert sc.frame == 'Model' and list(sp.spectrum.index) == list(sc.data.index)
    assert sp.spectrum.shape == (120, 32) and sp.npackets.shape == (120, 32)
    assert np.array_equal(sp.edges, np.linspace(-8.0, 8.0, 33))
    assert np.allclose(sp.velocity, np.arange(32) * 0.5 - 7.75, rtol=0, atol=1e-12)
    assert sp.atoms_per_packet == res.atoms_per_packet and sp.totalsource == res.totalsource
    assert np.array_equal(sp.npackets_los.values, res.npackets_los.values)
    assert np.array_equal(sp.npackets.values.sum(axis=1) + sp.npackets_outside.values.sum(axis=1),
                          res.npackets_los.values)
    assert res.npackets_los.values.sum() > 500
    nz = raw > 0
    assert np.max(np.abs(sp.radiance.values[nz] - raw[nz]) / raw[nz]) < 1e-12
    # kR per km/s: times the bin width, plus what falls outside, is the radiance
    total = (sp.spectrum.values * 0.5).sum(axis=1) + sp.outside.values.sum(axis=1)
    assert np.max(np.abs(total[nz] - raw[nz]) / raw[nz]) < 1e-12
    # a narrower range: the same radiance, more of it outside
    narrow = LOSSpectrum(sc, inputs, (-1.0, 1.0, 4), dphi=Quantity(3.0, 'deg'))
    assert np.allclose(narrow.radiance.values, sp.radiance.values, rtol=1e-12, atol=0)
    assert narrow.outside.values.sum() > sp.outside.values.sum()
    # one line: what LOSResult gives for that wavelength
    one = LOSSpectrum(sc, inputs, (-8.0, 8.0, 32), dphi=Quantity(3.0, 'deg'),
                      params={'quantity': 'radiance', 'wavelength': '5891'})
    assert np.all(one.radiance.values <= sp.radiance.values) and one.radiance.values.sum() > 0


@pytest.mark.gpu
def test_constant_step_recipe_rows_equal_resident_rows(monkeypatch):
    from nexoclom_b200 import Output, LOSSpectrum
    from nexoclom_b200.units import Quantity
    inputs = workload('Na.bounce.input')
    sc = _SC(_los(100, 31))
    inputs.delete_files()
    kept = Output(inputs, 3000, seed=21, keep_trajectory=True)
    assert kept.trajectory_kept
    dense = LOSSpectrum(sc, inputs, (-5.0, 5.0, 50), dphi=Quantity(3.0, 'deg'))
    inputs.delete_files()
    monkeypatch.setenv('NEXOCLOM_B200_MAX_ROWS', str(1000 * kept.nsteps))      # three chunks
    out = Output(inputs, 3000, seed=21)
    assert not out.trajectory_kept
    chunked = LOSSpectrum(sc, inputs, (-5.0, 5.0, 50), dphi=Quantity(3.0, 'deg'))
    inputs.delete_files()
    assert dense.npackets_los.values.sum() > 1000
    assert np.array_equal(chunked.npackets.values, dense.npackets.values)
    assert np.array_equal(chunked.npackets_outside.values, dense.npackets_outside.values)
    a, b = chunked.spectrum.values, dense.spectrum.values
    nz = b > 0
    assert np.array_equal(a > 0, nz) and np.max(np.abs(a[nz] - b[nz]) / b[nz]) < 1e-12
    assert chunked.totalsource == dense.totalsource


@pytest.mark.gpu
def test_small_pair_buffer_equals_one_batch(engine):
    setup, table = _run_table(engine, 'Na.maxwellian.radpres.input', 300_000, 13, integrate=False)
    try:
        engine.upload_gtables(setup.gtables([5891, 5897]))
        los = _los(4000, 14)
        lp = _lp(setup, 2.0)
        one = _spectrum(engine, table, los, lp, -10.0, 10.0, 100, setup.radius_km)
        engine.set_option('los_pair_cap', table.n + 1024)      # forces many batches
        try:
            many = _spectrum(engine, table, los, lp, -10.0, 10.0, 100, setup.radius_km)
        finally:
            engine.set_option('los_pair_cap', 0)
        assert one[1].sum() > table.n + 1024                   # the pairs did not fit one batch
        _assert_spectra(many, one)
    finally:
        table.free()


@pytest.mark.gpu
def test_spectrum_call_resets_los_candidate_pairs(engine):
    """los_accumulate(count_used) -> los_spectrum -> los_used_fill gives los_used's CSR: the
    spectrum call rebuilt the cell grid the kept pairs point into."""
    setup, table = _run_table(engine, 'Na.maxwellian.radpres.input', 1_000_000, 41)
    engine.upload_gtables(setup.gtables([5891, 5897]))
    los = _los(300, 9)
    lp = _lp(setup, 2.0)
    L, dplan = los.T.copy(), _dplan(los)
    engine.bind_packets(table)
    try:
        _, _, _, cnt = engine.los_accumulate(L, dplan, lp, n=table.n, count_used=True)
        engine.los_spectrum(L, dplan, lp, -5.0, 5.0, 20, setup.radius_km, n=table.n)
        off, idx = engine.los_used_fill(L, dplan, lp, cnt, n=table.n)
        off0, idx0 = engine.los_used(L, dplan, lp, n=table.n)
        assert off0[-1] > 100 and np.array_equal(off, off0)
        for i in range(len(los)):
            assert np.array_equal(np.sort(idx[off[i]:off[i + 1]]), np.sort(idx0[off[i]:off[i + 1]]))
    finally:
        engine.bind_packets(None)
        table.free()


@pytest.mark.gpu
def test_edge_cases(engine):
    setup = _na_setup()
    engine.upload_gtables(setup.gtables([5891, 5897]))
    lp = _lp(setup, 2.0)
    los = _los(20, 3)
    table = engine.upload_packets(np.ones((16, 8)))
    try:
        spec, cnt = _spectrum(engine, table, los, lp, -1.0, 1.0, 4, setup.radius_km)
        assert spec.shape == (20, 6) and cnt.shape == (20, 6)
        _assert_invariants((spec, cnt), _accumulate(engine, table, los, lp))
        engine.bind_packets(table)
        spec, cnt = engine.los_spectrum(los.T.copy(), _dplan(los), lp, -1.0, 1.0, 4,
                                        setup.radius_km, n=0)           # no rows
        engine.bind_packets(None)
        assert cnt.sum() == 0 and not spec.any()
        spec, cnt = _spectrum(engine, table, np.zeros((0, 6)), lp, -1.0, 1.0, 4, setup.radius_km)
        assert spec.shape == (0, 6) and cnt.shape == (0, 6)                 # no lines
        # no hits: the rows sit at (1, 1, 1); the lines look away from them
        away = np.array([[5.0, 0.0, 0.0, 1.0, 0.0, 0.0], [0.0, -5.0, 0.0, 0.0, -1.0, 0.0]])
        spec, cnt = _spectrum(engine, table, away, lp, -1.0, 1.0, 4, setup.radius_km)
        assert cnt.sum() == 0 and not spec.any()
        # one line straight at the rows: every row is a hit, all with v = 3 * vscale
        at = np.array([[3.0, 3.0, 3.0, -1 / np.sqrt(3), -1 / np.sqrt(3), -1 / np.sqrt(3)]])
        spec, cnt = _spectrum(engine, table, at, lp, -1.0, 1.0, 4, 1.0)
        assert cnt[0, -1] == 0 and cnt[0, 0] == 16                          # v = -sqrt(3)
        from nexoclom_b200.engine import NexoclomCudaError
        with pytest.raises(NexoclomCudaError):
            engine.los_spectrum(at.T.copy(), _dplan(at), lp, 1.0, -1.0, 4, 1.0, n=0)
    finally:
        table.free()


@pytest.mark.gpu
def test_full_size_config1(engine):
    """configs[1] at full size: 1e5 lines of sight x 1e7 live packets (the initial state, K5's
    2e8-hit case).  The column invariants against nx_los_accumulate on every line, the oracle
    on 100 of them."""
    setup, table = _run_table(engine, 'Na.maxwellian.radpres.input', 10_000_000, 3, integrate=False)
    try:
        engine.upload_gtables(setup.gtables([5891, 5897]))
        los = _los(100_000, 51)
        lp = _lp(setup, 1.0)
        acc = _accumulate(engine, table, los, lp)
        got = _spectrum(engine, table, los, lp, -10.0, 10.0, 100, setup.radius_km)
        _assert_invariants(got, acc)
        assert acc[1].sum() > 1e8
        sl = slice(0, None, 1000)                                   # 100 lines
        X = _table_X(table)
        ref = _oracle_lines(X, los[sl], setup, lp)
        _assert_spectra((got[0][sl], got[1][sl]), ref)
        assert ref[1].sum() > 5e4
    finally:
        table.free()


def _oracle_lines(X, los, setup, lp):
    hits = ospec.los_hits(X[:, 1], X[:, 2], X[:, 3], X[:, 5], X[:, 7], los,
                          vrplanet=setup.vrplanet, dphi=lp.dphi, outeredge=lp.outeredge,
                          rp_cm=lp.rp_cm, gtables=setup.gtables([5891, 5897]))
    return ospec.los_spectrum(X[:, 4], X[:, 5], X[:, 6], los, hits, -10.0, 10.0, 100,
                              setup.radius_km)
