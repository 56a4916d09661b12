"""Number density at sample points (ModelDensity, K7 ``nx_density_accumulate``).

CPU: the lens volume, the two oracle variants, the host build of the membership predicate,
input validation and the sharded reduction.  GPU (``-m gpu``): the kernel against the oracle,
the public API, constant-step runs, edge cases, the interplay with K5's kept candidate pairs,
and the full configs[1] size."""
import ctypes as C
import os
import sys

import numpy as np
import pandas as pd
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

from common import REPO, workload
from nexoclom_b200.ModelDensity import lens_volume, sample_points
from nexoclom_b200.sharding import combine_ranks
from oracle import density as odens


# ---------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------
def _lens_quad(d, r):
    """Volume outside the unit sphere by integrating, over the shell radius s >= 1, the area
    of the sphere |x| = s that lies inside the ball."""
    from scipy.integrate import quad

    def area(s):
        if d == 0.0:
            return 4 * np.pi * s * s if s <= r else 0.0
        if s <= r - d:
            return 4 * np.pi * s * s
        if abs(d - r) <= s <= d + r:
            return np.pi * s * (r * r - (s - d)**2) / d
        return 0.0
    lo, hi = 1.0, d + r
    if hi <= lo:
        return 0.0
    pts = [p for p in (r - d, abs(d - r)) if lo < p < hi]
    v, _ = quad(area, lo, hi, points=pts or None, epsabs=0.0, epsrel=2e-14, limit=200)
    return v


@pytest.mark.parametrize('d, r', [
    (5.0, 0.5), (3.0, 2.0), (1.5, 0.5),            # d >= r + 1 (the boundary included)
    (0.3, 0.2), (0.0, 0.7), (0.5, 0.5),            # d + r <= 1 (the boundary included)
    (0.0, 2.0), (0.2, 3.0), (0.5, 1.5),            # d + 1 <= r (the boundary included)
    (1.2, 0.3), (1.0, 0.05), (2.0, 1.5), (0.9, 0.4), (0.3, 1.2),       # lens
    (1.5 - 1e-9, 0.5), (0.5 + 1e-9, 0.5), (0.5 - 1e-9, 1.5),           # next to the boundaries
])
def test_lens_volume_matches_integration(d, r):
    ref = _lens_quad(d, r)
    full = 4 / 3 * np.pi * r**3
    # relative to the volume; a sliver next to d + r = 1 (volume ~ (d + r - 1)^2, so one ulp
    # of d or r moves it by ~1e-7 of itself) relative to the ball
    tol = 1e-12 * (ref if ref > 1e-9 * full else full)
    for got in (float(lens_volume(d, r)), float(odens.lens_volume(d, r))):
        assert got >= 0.0 and abs(got - ref) <= tol


def _cloud(n, seed):
    g = np.random.default_rng(seed)
    u = g.standard_normal((n, 3))
    u /= np.linalg.norm(u, axis=1)[:, None]
    X = (u * (1 + g.exponential(0.4, n))[:, None]).astype(np.float32)
    frac = g.random(n).astype(np.float32) + np.float32(0.01)
    return X, frac


def test_oracle_variants_agree_exactly():
    X, frac = _cloud(20000, 1)
    g = np.random.default_rng(2)
    pts = g.uniform(-2.5, 2.5, (300, 3))
    rad = 10 ** g.uniform(-1.5, 0.2, 300)
    a = odens.ball_sums_kdtree(X, frac, pts, rad)
    b = odens.ball_sums_brute(X, frac, pts, rad)
    assert np.array_equal(a[2], b[2]) and a[2].sum() > 10000
    # same members; the sums differ at most by their order
    assert np.allclose(a[0], b[0], rtol=1e-13, atol=0) and np.allclose(a[1], b[1], rtol=1e-13, atol=0)


@pytest.fixture(scope='module')
def hc(built):
    return C.CDLL(os.path.join(REPO, 'tests', '_hostcheck', 'libnexo_density_hostcheck.so'))


def _host_member(hc, P, p, r):
    P = np.ascontiguousarray(P, dtype=np.float32)
    cols = [np.ascontiguousarray(P[:, k]) for k in range(3)]
    out = np.zeros(len(P), dtype=np.uint8)
    fp = C.POINTER(C.c_float)
    hc.hc_density_member(C.c_long(len(P)), *[c.ctypes.data_as(fp) for c in cols],
                         C.c_double(p[0]), C.c_double(p[1]), C.c_double(p[2]), C.c_double(r),
                         out.ctypes.data_as(C.POINTER(C.c_uint8)))
    return out.astype(bool)


def test_host_membership_predicate_matches_numpy(hc):
    """Rows placed on the sphere d = r (rounded to float32) and 1-3 float32 ulps either side of
    it, per coordinate: the predicate decides each exactly as NumPy does."""
    g = np.random.default_rng(7)
    total_in = total_out = 0
    for trial in range(40):
        p = g.uniform(-3, 3, 3) + g.uniform(-1e-7, 1e-7, 3)      # not float32-representable
        r = float(10 ** g.uniform(-2.5, 0.5))
        if trial % 5 == 0:
            p = np.round(p * 8) / 8                                # exactly representable
            r = 0.25
        u = g.standard_normal((4000, 3))
        u /= np.linalg.norm(u, axis=1)[:, None]
        on = (p + r * u).astype(np.float32)
        rows, up, dn = [on], on, on
        for _ in range(3):                                         # 1, 2, 3 ulps out and in
            up = np.nextafter(up, np.float32(np.inf))
            dn = np.nextafter(dn, np.float32(-np.inf))
            rows += [up, dn]
        rows.append(np.nextafter(on, g.choice([-np.inf, np.inf], on.shape).astype(np.float32)))
        P = np.concatenate(rows)
        ref = odens.member_mask(P.astype(np.float64), p, r)
        got = _host_member(hc, P, p, r)
        assert np.array_equal(got, ref)
        total_in += int(ref.sum())
        total_out += int((~ref).sum())
    assert total_in > 10000 and total_out > 10000          # both sides of the sphere exercised


def test_model_density_rejects_bad_input():
    inputs = workload('Na.maxwellian.radpres.input')
    from nexoclom_b200 import ModelDensity
    bad = [
        (np.zeros((4, 2)), 0.1),                       # not (N, 3)
        (np.zeros(3), 0.1),
        (np.array([[0.0, np.nan, 2.0]]), 0.1),         # non-finite point
        (np.array([[0.0, np.inf, 2.0]]), 0.1),
        (np.ones((2, 3)), np.nan),                     # non-finite radius
        (np.ones((2, 3)), 0.0),                        # radius <= 0
        (np.ones((2, 3)), [0.1, -0.1]),
        (np.ones((2, 3)), [0.1, 0.1, 0.1]),            # one radius per point
        (pd.DataFrame({'x': [1.0], 'y': [2.0]}), 0.1),  # no z column
    ]
    for pts, rad in bad:
        with pytest.raises(ValueError):
            ModelDensity(inputs, pts, rad)
    with pytest.raises(ValueError):
        ModelDensity(inputs, np.ones((2, 3)), 0.1, params={'quantity': 'column'})
    p, r, idx = sample_points(pd.DataFrame({'x': [1.0, 2.0], 'y': 0.0, 'z': 3.0},
                                           index=['a', 'b']), 0.5)
    assert p.shape == (2, 3) and np.array_equal(r, [0.5, 0.5]) and list(idx) == ['a', 'b']


def _gloo_worker(rank, world, port, q):
    sys.path.insert(0, REPO)
    sys.path.insert(0, os.path.join(REPO, 'tests'))
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    from nexoclom_b200.sharding import combine_ranks
    from nexoclom_b200.sharding import shard_range
    from oracle import density as od
    X, frac = _cloud(30000, 3)
    pts, rad = _gloo_points()
    first, n = shard_range(len(X), rank, world)
    s1, s2, cnt = od.ball_sums_kdtree(X[first:first + n], frac[first:first + n], pts, rad)
    tot, = combine_ranks((s1, s2, cnt), float(n))       # what ModelDensity does per product
    if rank == 0:
        q.put((s1, s2, cnt, tot))
    dist.barrier()
    dist.destroy_process_group()


def _gloo_points():
    g = np.random.default_rng(4)
    return g.uniform(-2, 2, (200, 3)), 10 ** g.uniform(-1.3, 0.0, 200)


def test_two_rank_allreduce_equals_single_rank():
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = 33500 + os.getpid() % 2000
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    s1, s2, cnt, tot = q.get(timeout=300)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    X, frac = _cloud(30000, 3)
    pts, rad = _gloo_points()
    o1, o2, oc = odens.ball_sums_kdtree(X, frac, pts, rad)
    assert np.array_equal(cnt, oc) and oc.sum() > 1000
    assert tot == 30000.0
    assert np.allclose(s1, o1, rtol=1e-12, atol=0) and np.allclose(s2, o2, rtol=1e-12, atol=0)
    # a single process: the reduction leaves the sums alone
    a, b, c = o1.copy(), o2.copy(), oc.copy()
    assert combine_ranks((a, b, c), 5.0) == (5.0,) and np.array_equal(a, o1) and np.array_equal(c, oc)


# ---------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------
def _assert_sums(got, ref, tol=1e-12):
    s1, s2, cnt = got
    o1, o2, oc = ref
    assert np.array_equal(cnt, oc), f'counts differ at {np.flatnonzero(cnt != oc)[:10]}'
    for what, a, b in (('S1', s1, o1), ('S2', s2, o2)):
        nz = b > 0
        assert np.array_equal(a > 0, nz), what
        if nz.any():
            err = np.abs(a[nz] - b[nz]) / b[nz]
            assert err.max() <= tol, (what, err.max(), int(np.argmax(err)))


def _mixed_points(n, seed, rmin=0.02, rmax=1.0):
    """Sample points from the surface to 6 R_p out, radii log-uniform in [rmin, rmax]."""
    g = np.random.default_rng(seed)
    u = g.standard_normal((n, 3))
    u /= np.linalg.norm(u, axis=1)[:, None]
    alt = 10 ** g.uniform(-2, np.log10(5), n)
    return u * (1 + alt)[:, None], 10 ** g.uniform(np.log10(rmin), np.log10(rmax), n)


def _run_table(engine, name, n, seed, first_id=0, skip_dead=True):
    from nexoclom_b200.runsetup import RunSetup
    setup = RunSetup(workload(name))
    setup.upload(engine)
    engine.init_state(setup.source_params(engine), seed, first_id, n)
    engine.integrate_adaptive(n)
    return engine.compact_state(skip_dead=skip_dead, round_f32=True, n=n)


def _table_rows(table):
    """x, y, z and frac of the rows the density counts (frac > 0)."""
    cols, _ = table.export()
    live = cols['frac'] > 0
    return np.stack([cols['x'], cols['y'], cols['z']], axis=1)[live], cols['frac'][live]


def _density(engine, table, pts, rad):
    s1, s2 = np.zeros(len(pts)), np.zeros(len(pts))
    cnt = np.zeros(len(pts), dtype=np.int64)
    engine.bind_packets(table)
    try:
        engine.density_accumulate(pts, rad, s1, s2, cnt, n=table.n)
    finally:
        engine.bind_packets(None)
    return s1, s2, cnt


@pytest.mark.gpu
def test_kernel_matches_oracle(engine):
    # every packet kept (compress=False): the frac == 0 rows are in the table and must not count
    table = _run_table(engine, 'Na.maxwellian.radpres.input', 200_000, 11, skip_dead=False)
    try:
        X, frac = _table_rows(table)
        assert table.n == 200_000 and len(X) < table.n
        pts, rad = _mixed_points(5000, 12)
        got = _density(engine, table, pts, rad)
        ref = odens.ball_sums_kdtree(X, frac, pts, rad)
        _assert_sums(got, ref)
        assert ref[2].sum() > 50_000 and (ref[2] > 0).sum() > 200
        # the buffers are added to: a second call doubles them exactly
        s1, s2, cnt = got
        engine.bind_packets(table)
        engine.density_accumulate(pts, rad, s1, s2, cnt, n=table.n)
        engine.bind_packets(None)
        assert np.array_equal(cnt, 2 * ref[2])
    finally:
        table.free()


@pytest.fixture(scope='module')
def two_files(engine):
    """Two Input.run calls of configs[1] physics: two output files."""
    inputs = workload('Na.maxwellian.radpres.input')
    inputs.delete_files()
    inputs.run(20_000, seed=5)
    inputs.run(40_000, seed=6)                      # 20 000 more in a second output file
    _, files, npk, _ = inputs.search()
    assert npk == 40_000
    from nexoclom_b200 import catalogue
    X = [catalogue.fetch(f).X for f in files]
    yield inputs, files, X
    inputs.delete_files()


@pytest.mark.gpu
def test_public_api_matches_oracle(two_files):
    from nexoclom_b200 import ModelDensity
    inputs, files, Xs = two_files
    assert len(files) == 2
    pts, rad = _mixed_points(800, 21, 0.05, 1.0)
    frame = pd.DataFrame(pts, columns=['x', 'y', 'z'], index=[f'p{i}' for i in range(800)])
    res = ModelDensity(inputs, frame, rad)
    assert list(res.density.index) == list(frame.index)
    assert res.quantity == 'density' and res.density_unit == 'cm-3'
    parts = [odens.ball_sums_kdtree(X[['x', 'y', 'z']].values, X.frac.values, pts, rad) for X in Xs]
    ref = tuple(sum(p[k] for p in parts) for k in range(3))
    _assert_sums((res.s1.values, res.s2.values, res.npackets.values), ref)
    assert res.totalsource == 40_000.0
    from nexoclom_b200.units import value_of
    apc = 1e23 / (40_000.0 / float(value_of(inputs.options.endtime)))
    assert res.atoms_per_packet == pytest.approx(apc, rel=1e-15)
    r_cm = float(inputs.geometry.planet.radius.value) * 1e5
    vol = odens.lens_volume(np.linalg.norm(pts, axis=1), rad) * r_cm**3
    assert np.all(vol > 0)
    assert np.allclose(res.density.values, apc * ref[0] / vol, rtol=1e-12, atol=0)
    assert np.allclose(res.density_err.values, apc * np.sqrt(ref[1]) / vol, rtol=1e-12, atol=0)


@pytest.mark.gpu
def test_edge_cases(engine, two_files):
    from nexoclom_b200 import ModelDensity
    inputs, files, Xs = two_files
    rows = sum(len(X) for X in Xs)
    fsum = sum(X.frac.values.astype(np.float64).sum() for X in Xs)
    pts = np.array([[0.0, 0.0, 0.0], [0.2, 0.1, 0.0],          # inside the planet
                    [900.0, 0.0, 0.0], [0.0, -400.0, 300.0],    # far outside the packet cube
                    [0.0, 0.0, 0.0]])                          # encloses everything
    rad = np.array([0.5, 0.3, 1.0, 2.0, 1e4])
    res = ModelDensity(inputs, pts, rad)
    assert np.all(np.isnan(res.density.values[:2])) and np.all(res.npackets.values[:2] == 0)
    assert np.all(res.npackets.values[2:4] == 0) and np.all(res.density.values[2:4] == 0)
    assert res.npackets.values[4] == rows
    assert res.s1.values[4] == pytest.approx(fsum, rel=1e-12)
    empty = ModelDensity(inputs, np.zeros((0, 3)), 0.1)
    assert len(empty.density) == 0
    # no packets
    table = engine.upload_packets(np.ones((16, 8)))
    try:
        s1, s2 = np.zeros(len(pts)), np.zeros(len(pts))
        cnt = np.zeros(len(pts), dtype=np.int64)
        engine.bind_packets(table)
        engine.density_accumulate(pts, rad, s1, s2, cnt, n=0)
        engine.bind_packets(None)
        assert not cnt.any() and not s1.any() and not s2.any()
    finally:
        table.free()


@pytest.mark.gpu
def test_constant_step_recipe_rows_equal_resident_rows(monkeypatch):
    """Na.bounce: a resident row table and a recipe-only run (rows regenerated in chunks)
    give the same counts."""
    from nexoclom_b200 import Output, ModelDensity
    inputs = workload('Na.bounce.input')
    pts, rad = _mixed_points(400, 31, 0.05, 1.0)
    inputs.delete_files()
    kept = Output(inputs, 3000, seed=21, keep_trajectory=True)
    assert kept.trajectory_kept
    dense = ModelDensity(inputs, pts, rad)
    inputs.delete_files()
    monkeypatch.setenv('NEXOCLOM_B200_MAX_ROWS', str(1000 * kept.nsteps))      # three chunks
    out = Output(inputs, 3000, seed=21)
    assert not out.trajectory_kept
    chunked = ModelDensity(inputs, pts, rad)
    inputs.delete_files()
    assert dense.npackets.values.sum() > 1e4
    _assert_sums((chunked.s1.values, chunked.s2.values, chunked.npackets.values),
                 (dense.s1.values, dense.s2.values, dense.npackets.values))
    assert chunked.totalsource == dense.totalsource


@pytest.mark.gpu
def test_density_call_resets_los_candidate_pairs(engine):
    """los_accumulate(count_used) -> density_accumulate -> los_used_fill gives the CSR of
    the plain sequence: the density call rebuilds the cell grid the kept pairs point into."""
    from nexoclom_b200._lib import LosParams
    from nexoclom_b200.runsetup import RunSetup
    setup = RunSetup(workload('Na.maxwellian.radpres.input'))
    table = _run_table(engine, 'Na.maxwellian.radpres.input', 1_000_000, 41)
    engine.upload_gtables(setup.gtables([5891, 5897]))
    g = np.random.default_rng(9)
    nlos = 300
    x_sc = g.standard_normal((3, nlos))
    x_sc *= (1.5 + 3 * g.random(nlos)) / np.linalg.norm(x_sc, axis=0)
    tgt = g.standard_normal((3, nlos)) * 0.5
    bore = tgt - x_sc
    bore /= np.linalg.norm(bore, axis=0)
    los = np.ascontiguousarray(np.concatenate([x_sc, bore]))
    dplan = np.full(nlos, 1e30)
    lp = LosParams()
    lp.dphi, lp.outeredge = float(np.radians(2.0)), 25.0
    lp.vrplanet, lp.rp_cm = setup.vrplanet, setup.radius_km * 1e5
    lp.quantity, lp.round_f32, lp.skip_dead = 1, 1, 1
    pts, rad = _mixed_points(500, 42)
    engine.set_option('los_mode', 2)
    engine.bind_packets(table)
    try:
        def csr(with_density):
            _, _, _, cnt = engine.los_accumulate(los, dplan, lp, n=table.n, count_used=True)
            if with_density:
                s1, s2 = np.zeros(len(pts)), np.zeros(len(pts))
                c = np.zeros(len(pts), dtype=np.int64)
                engine.density_accumulate(pts, rad, s1, s2, c, n=table.n)
            off, idx = engine.los_used_fill(los, dplan, lp, cnt, n=table.n)
            return off, np.concatenate([np.sort(idx[off[i]:off[i + 1]]) for i in range(nlos)])
        off0, idx0 = csr(False)
        off1, idx1 = csr(True)
        assert off0[-1] > 100
        assert np.array_equal(off0, off1) and np.array_equal(idx0, idx1)
    finally:
        engine.bind_packets(None)
        engine.set_option('los_mode', 0)
        table.free()


@pytest.mark.gpu
def test_full_size_config1(engine):
    """configs[1] at full size: 1e7 packets x 1e5 points.  Sums are additive over two packet
    shards (each bins its own grid), counts exactly; a slice matches the oracle."""
    name = 'Na.maxwellian.radpres.input'
    n, half = 10_000_000, 5_000_000
    g = np.random.default_rng(51)
    u = g.standard_normal((100_000, 3))
    u /= np.linalg.norm(u, axis=1)[:, None]
    alt = 10 ** g.uniform(np.log10(0.02), np.log10(5), 100_000)
    pts = u * (1 + alt)[:, None]
    rad = np.minimum(0.02 + 0.1 * alt, 0.3)
    whole = _run_table(engine, name, n, 3)
    try:
        full = _density(engine, whole, pts, rad)
        sl = slice(0, None, 50)                                   # 2e3 points
        X, frac = _table_rows(whole)
        ref = odens.ball_sums_kdtree(X, frac, pts[sl], rad[sl])
        _assert_sums(tuple(a[sl] for a in full), ref)
        assert ref[2].sum() > 2000
        del X, frac
    finally:
        whole.free()
    parts = []
    for first in (0, half):
        t = _run_table(engine, name, half, 3, first_id=first)
        try:
            parts.append(_density(engine, t, pts, rad))
        finally:
            t.free()
    summed = tuple(parts[0][k] + parts[1][k] for k in range(3))
    _assert_sums(summed, full)
    assert full[2].sum() > 5e4
