"""Doppler-resolved image cubes (ModelImageCube, ``nx_cube_*``).

CPU: the oracle against the reference's own create_image output (tests/golden/image.npz), its
velocity against the host build of ``los_doppler``, the sign of the velocity, input validation
and the sharded reduction.  GPU (``-m gpu``): the kernel against the oracle, the invariants
against K4 (directly and through ModelImage), recipe-only runs, non-interference with the image
scratch and K5's kept candidate pairs, edge cases and the full configs[1] size."""
import ctypes as C
import os
import sys

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

from common import REPO, workload
from nexoclom_b200.ModelImageCube import cube_bins
from nexoclom_b200.sharding import combine_ranks
from oracle import cube as ocube
from oracle import imaging
from oracle import spectrum as ospec

GOLDEN = os.path.join(REPO, 'tests', 'golden')
TAGS = ['col_pole', 'rad_pole', 'rad_side']


def _na_setup():
    from nexoclom_b200.runsetup import RunSetup
    return RunSetup(workload('Na.maxwellian.radpres.input'))


def _oracle(X, setup, M, dims, apix, quantity, vmin, vmax, nbins, xrange=(-4, 4), zrange=(-4, 4)):
    return ocube.create_cube(X[:, 1], X[:, 2], X[:, 3], X[:, 4], X[:, 5], X[:, 6], X[:, 7],
                             vrplanet=setup.vrplanet, M=M, dims=dims, xrange=xrange,
                             zrange=zrange, apix=apix, quantity=quantity, vmin=vmin, vmax=vmax,
                             nbins=nbins, vscale=setup.radius_km,
                             gtables=setup.gtables([5891, 5897]))


# ---------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------
@pytest.mark.parametrize('tag', TAGS)
@pytest.mark.parametrize('vmin, vmax, nbins', [(-10.0, 10.0, 1), (-2.0, 2.0, 64),
                                               (-3.0, 3.0, 1000), (0.3, 0.9, 7)])
def test_oracle_cube_sums_to_golden(tag, vmin, vmax, nbins):
    """Summed over the velocity axis the oracle cube is the reference's own create_image()
    output: the packet image exactly, the image to 1e-12."""
    g = np.load(os.path.join(GOLDEN, 'image.npz'))
    setup = _na_setup()
    dims = [int(d) for d in g[f'{tag}_dims']]
    M = imaging.image_rotation(*g[f'{tag}_view'])
    cube, cnt = _oracle(g['X'], setup, M, dims, float(g[f'{tag}_apix']),
                        'column' if tag.startswith('col') else 'radiance', vmin, vmax, nbins)
    assert cube.shape == (dims[0], dims[1], nbins + 2) and cnt.dtype == np.int64
    assert np.array_equal(cnt.sum(axis=2), g[f'{tag}_packim'])
    ref = g[f'{tag}_image']
    nz = ref > 0
    assert nz.sum() > 1000 and np.all(cube.sum(axis=2)[~nz] == 0)
    assert np.max(np.abs(cube.sum(axis=2)[nz] - ref[nz]) / ref[nz]) < 1e-12
    if nbins == 7:                    # a narrow range: most rows fall outside
        assert cnt[:, :, [0, -1]].sum() > cnt[:, :, 1:-1].sum() > 0
    else:
        assert cnt[:, :, 1:-1].sum() > 0.9 * cnt.sum()


@pytest.fixture(scope='module')
def hc(built):
    return C.CDLL(os.path.join(REPO, 'tests', '_hostcheck', 'libnexo_spectrum_hostcheck.so'))


VIEWS = [(0.0, np.pi / 2), (0.7, 0.3), (2.5, -0.8), (np.pi, 0.0), (4.0, 1.2)]


@pytest.mark.parametrize('view', VIEWS)
def test_oracle_velocity_is_host_los_doppler(hc, view):
    """The oracle's velocity (NumPy, row 1 of M) equals the kernel's los_doppler, host build,
    bit for bit."""
    g = np.random.default_rng(5)
    n = 100_000
    V = (g.standard_normal((n, 3)) * 3e-3).astype(np.float32)
    cols = [np.ascontiguousarray(V[:, k]) for k in range(3)]
    M = np.asarray(imaging.image_rotation(*view))
    got = np.zeros(n)
    fp = C.POINTER(C.c_float)
    hc.hc_los_doppler(C.c_long(n), *[c.ctypes.data_as(fp) for c in cols],
                      *map(C.c_double, M[1]), C.c_double(2439.7),
                      got.ctypes.data_as(C.POINTER(C.c_double)))
    W = V.astype(np.float64)
    ref = ospec.doppler(W[:, 0], W[:, 1], W[:, 2], M[1, 0], M[1, 1], M[1, 2], 2439.7)
    assert np.array_equal(got.view(np.int64), ref.view(np.int64))


@pytest.mark.parametrize('view', VIEWS)
def test_velocity_sign(view):
    """M takes the observer direction to (0, -1, 0): a row's v is minus its velocity towards
    the observer, so v > 0 recedes.  Over the north pole, rows moving north approach."""
    slong, slat = view
    p_obs = np.array([np.sin(slong) * np.cos(slat), -np.cos(slong) * np.cos(slat), np.sin(slat)])
    M = np.asarray(imaging.image_rotation(slong, slat))
    assert np.allclose(M @ p_obs, [0.0, -1.0, 0.0], rtol=0, atol=1e-14)
    V = np.random.default_rng(2).standard_normal((5000, 3)) * 1e-3
    v = ospec.doppler(V[:, 0], V[:, 1], V[:, 2], M[1, 0], M[1, 1], M[1, 2], 2439.7)
    assert np.allclose(v, -(V @ p_obs) * 2439.7, rtol=0, atol=1e-12)
    if view == (0.0, np.pi / 2):
        assert np.all(v[V[:, 2] > 0] < 0) and np.all(v[V[:, 2] < 0] > 0)


def test_cube_rejects_bad_input():
    """Bad arguments raise ValueError before anything touches a device."""
    from nexoclom_b200 import ModelImageCube
    inputs = workload('Na.maxwellian.radpres.input')
    params = {'quantity': 'column', 'dims': '20,30'}
    for velocity in [(0.0, 1.0), (0.0, 1.0, 4, 5), 'abc', 3.0, None,
                     (np.nan, 1.0, 4), (0.0, np.inf, 4), (1.0, 1.0, 4), (2.0, 1.0, 4),
                     (0.0, 1.0, 0), (0.0, 1.0, -3), (0.0, 1.0, 2.5), (0.0, 1.0, True),
                     (0.0, 1.0, '4'), ('a', 1.0, 4), (0.0, 1.0, 2**31)]:
        with pytest.raises(ValueError):
            ModelImageCube(inputs, params, velocity)
    for quantity in ('density', 'difrad', 'flux', None):
        with pytest.raises(ValueError):
            ModelImageCube(inputs, {'quantity': quantity}, (0.0, 1.0, 4))
    with pytest.raises(ValueError):
        ModelImageCube(inputs, 'params.txt', (0.0, 1.0, 4))
    with pytest.raises(ValueError):                             # 800 x 800 x 3357 cells
        ModelImageCube(inputs, {'quantity': 'radiance'}, (0.0, 1.0, 3355))
    with pytest.raises(ValueError):
        cube_bins((0.0, 1.0, 2**15 - 2), (256, 256))            # exactly 2**31 cells
    assert cube_bins((0.0, 1.0, 2**15 - 3), (256, 256)) == (0.0, 1.0, 2**15 - 3)
    assert cube_bins((-1, 1, np.int64(3)), (800, 800)) == (-1.0, 1.0, 3)


def _gloo_cloud(n=30000):
    g = np.random.default_rng(6)
    X = np.zeros((n, 8))
    u = g.standard_normal((n, 3))
    u /= np.linalg.norm(u, axis=1)[:, None]
    X[:, 1:4] = u * (1 + g.exponential(0.5, n))[:, None]
    X[:, 4:7] = g.standard_normal((n, 3)) * 1e-3
    X[:, 7] = g.random(n) + 0.01
    return X.astype(np.float32).astype(np.float64)


def _gloo_oracle(X):
    M = imaging.image_rotation(0.7, 0.3)
    return _oracle(X, _na_setup(), M, [40, 30], 1e17, 'radiance', -5.0, 5.0, 24)


def _gloo_worker(rank, world, port, q):
    sys.path.insert(0, REPO)
    sys.path.insert(0, os.path.join(REPO, 'tests'))
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    from nexoclom_b200.sharding import combine_ranks
    from nexoclom_b200.sharding import shard_range
    X = _gloo_cloud()
    first, n = shard_range(len(X), rank, world)
    cube, cnt = _gloo_oracle(X[first:first + n])
    tot, = combine_ranks((cube, cnt), float(n))          # what ModelImageCube does off NCCL
    if rank == 0:
        q.put((cube, cnt, tot))
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_allreduce_equals_single_rank():
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = 37500 + os.getpid() % 2000
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    cube, cnt, tot = q.get(timeout=300)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    ocube_, ocnt = _gloo_oracle(_gloo_cloud())
    assert np.array_equal(cnt, ocnt) and ocnt.sum() > 10_000
    assert tot == 30000.0
    nz = ocube_ > 0
    assert np.array_equal(cube > 0, nz)
    assert np.max(np.abs(cube[nz] - ocube_[nz]) / ocube_[nz]) < 1e-12
    a, c = ocube_.copy(), ocnt.copy()                    # a single process: left alone
    assert combine_ranks((a, c), 5.0) == (5.0,) and np.array_equal(a, ocube_)


# ---------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------
def _ip(setup, quantity, view, dims, apix, xrange=(-4.0, 4.0), zrange=(-4.0, 4.0),
        round_f32=0, skip_dead=0):
    from nexoclom_b200._lib import ImageParams
    M = np.asarray(imaging.image_rotation(*view))
    ip = ImageParams()
    for k in range(9):
        ip.M[k] = float(M.flat[k])
    ip.x0, ip.x1 = xrange
    ip.z0, ip.z1 = zrange
    ip.nx, ip.nz = dims
    ip.apix = apix
    ip.vrplanet = setup.vrplanet
    ip.quantity = 0 if quantity == 'column' else 1
    ip.round_f32, ip.skip_dead = round_f32, skip_dead
    return ip, M


def _cube(engine, ip, vmin, vmax, nbins, vscale, n, table=None):
    engine.cube_begin(ip.nx, ip.nz, nbins)
    try:
        engine.bind_packets(table)
        try:
            engine.cube_add(ip, vmin, vmax, nbins, vscale, n=n)
        finally:
            engine.bind_packets(None)
        return engine.cube_fetch(ip.nx, ip.nz, nbins)
    finally:
        engine.cube_end()


def _image(engine, ip, n, table=None):
    engine.image_begin(ip.nx, ip.nz)
    engine.bind_packets(table)
    try:
        engine.image_add(ip, n=n)
    finally:
        engine.bind_packets(None)
    return engine.image_fetch(ip.nx, ip.nz)


def _assert_close(got, ref, tol=1e-12):
    nz = ref != 0
    assert np.array_equal(got != 0, nz)
    if nz.any():
        err = np.abs(got[nz] - ref[nz]) / np.abs(ref[nz])
        assert err.max() <= tol, (err.max(), np.argwhere(nz)[int(np.argmax(err))])


def _assert_cubes(got, ref, tol=1e-12):
    assert np.array_equal(got[1], ref[1]), f'counts differ at {np.argwhere(got[1] != ref[1])[:10]}'
    _assert_close(got[0], ref[0], tol)


def _assert_image(got, img, tol=1e-12):
    """Summed over the velocity axis the cube is K4's image: counts exactly, sums to rounding."""
    assert np.array_equal(got[1].sum(axis=2), img[1])
    _assert_close(got[0].sum(axis=2), img[0], tol)


def _table_X(table):
    cols, _ = table.export()
    return np.stack([cols[k].astype(np.float64) for k in
                     ('time', 'x', 'y', 'z', 'vx', 'vy', 'vz', 'frac')], axis=1)


RANGES = [(-10.0, 10.0, 1), (-3.0, 3.0, 64), (-4.0, 4.0, 1000), (0.3, 0.9, 7)]


@pytest.mark.gpu
@pytest.mark.parametrize('quantity', ['column', 'radiance'])
@pytest.mark.parametrize('view', [(0.0, np.pi / 2), (0.7, 0.3), (2.5, -0.8)])
def test_kernel_matches_oracle_golden_packets(engine, quantity, view):
    g = np.load(os.path.join(GOLDEN, 'image.npz'))
    setup = _na_setup()
    engine.upload_gtables(setup.gtables([5891, 5897]))
    X = g['X'][g['X'][:, 7] > 0].astype(np.float32).astype(np.float64)
    ip, M = _ip(setup, quantity, view, (50, 40), float(g['rad_pole_apix']))
    table = engine.upload_packets(X)
    try:
        img = _image(engine, ip, table.n, table)
        for vmin, vmax, nbins in RANGES:
            got = _cube(engine, ip, vmin, vmax, nbins, setup.radius_km, table.n, table)
            assert got[0].shape == (50, 40, nbins + 2) and got[1].dtype == np.int64
            ref = _oracle(X, setup, M, (50, 40), ip.apix, quantity, vmin, vmax, nbins)
            _assert_cubes(got, ref)
            _assert_image(got, img)
        assert img[1].sum() > 40_000
        assert ref[1][:, :, [0, -1]].sum() > ref[1][:, :, 1:-1].sum() > 0   # the narrow range
    finally:
        table.free()


def _run_slab(engine, name, n, seed, integrate=True):
    from nexoclom_b200.runsetup import RunSetup
    setup = RunSetup(workload(name))
    setup.upload(engine)
    engine.init_state(setup.source_params(engine), seed, 0, n)
    if integrate:
        engine.integrate_adaptive(n)
    return setup


@pytest.mark.gpu
@pytest.mark.parametrize('integrate', [False, True])
def test_kernel_matches_oracle_synthetic(engine, integrate):
    """2e5 packets of configs[1] on the slab, with the slab flags (round_f32; skip_dead or
    dead rows counted with w = 0), and the same rows as a compacted table."""
    setup = _run_slab(engine, 'Na.maxwellian.radpres.input', 200_000, 11, integrate)
    engine.upload_gtables(setup.gtables([5891, 5897]))
    Xs = engine.export_state().T[:, :8].copy()
    X32 = Xs.astype(np.float32).astype(np.float64)
    live = Xs[:, 7] > 0
    if integrate:
        assert 0 < live.sum() < len(Xs) // 2
    for skip_dead in (1, 0):
        rows = X32[live] if skip_dead else X32
        ip, M = _ip(setup, 'radiance', (0.7, 0.3), (64, 48), 1e17, xrange=(-6.0, 6.0),
                    zrange=(-4.5, 4.5), round_f32=1, skip_dead=skip_dead)
        img = _image(engine, ip, 200_000)
        for vmin, vmax, nbins in RANGES:
            got = _cube(engine, ip, vmin, vmax, nbins, setup.radius_km, 200_000)
            ref = _oracle(rows, setup, M, (64, 48), ip.apix, 'radiance', vmin, vmax, nbins,
                          xrange=(-6.0, 6.0), zrange=(-4.5, 4.5))
            _assert_cubes(got, ref)
            _assert_image(got, img)
        assert ref[1].sum() > 1000
    table = engine.compact_state(skip_dead=True, round_f32=True, n=200_000)
    try:
        ip, M = _ip(setup, 'column', (0.0, np.pi / 2), (64, 64), 1e17, xrange=(-6.0, 6.0),
                    zrange=(-6.0, 6.0))
        got = _cube(engine, ip, -3.0, 3.0, 64, setup.radius_km, table.n, table)
        _assert_cubes(got, _oracle(_table_X(table), setup, M, (64, 64), ip.apix, 'column',
                                   -3.0, 3.0, 64, xrange=(-6.0, 6.0), zrange=(-6.0, 6.0)))
    finally:
        table.free()


PARAMS = {'quantity': 'radiance', 'dims': '120,90', 'width': '10,7.5', 'center': '0.5,-0.2',
          'subobslongitude': '0.7', 'subobslatitude': '0.3'}


def _assert_matches_model_image(cube, image):
    assert np.array_equal(cube.packet_image, image.packet_image)
    assert np.array_equal(cube.packet_cube.sum(axis=2) + cube.packet_outside.sum(axis=2),
                          cube.packet_image)
    assert cube.packet_image.sum() > 1000
    _assert_close(cube.image, image.image)
    assert cube.atoms_per_packet == image.atoms_per_packet
    assert cube.totalsource == image.totalsource
    for k in ('xaxis', 'zaxis'):
        assert np.array_equal(np.asarray(getattr(cube, k)), np.asarray(getattr(image, k)))
    assert float(cube.Apix) == float(image.Apix)


@pytest.fixture(scope='module')
def two_files(engine):
    inputs = workload('Na.maxwellian.radpres.input')
    inputs.delete_files()
    inputs.run(200_000, seed=5)
    inputs.run(400_000, seed=6)              # 200 000 more in a second output file
    _, files, npk, _ = inputs.search()
    assert npk == 400_000 and len(files) == 2
    yield inputs
    inputs.delete_files()


@pytest.mark.gpu
@pytest.mark.parametrize('quantity', ['radiance', 'column'])
def test_public_api_matches_model_image(two_files, quantity):
    from nexoclom_b200 import ModelImage, ModelImageCube
    params = dict(PARAMS, quantity=quantity)
    image = ModelImage(two_files, params)
    cube = ModelImageCube(two_files, params, (-6.0, 6.0, 48))
    _assert_matches_model_image(cube, image)
    assert cube.cube.shape == (120, 90, 48) and cube.packet_cube.shape == (120, 90, 48)
    assert cube.outside.shape == (120, 90, 2) and cube.packet_cube.dtype == np.int64
    assert np.array_equal(cube.edges, np.linspace(-6.0, 6.0, 49))
    assert np.allclose(cube.velocity, np.arange(48) * 0.25 - 5.875, rtol=0, atol=1e-12)
    # per km/s: times the bin width, plus what falls outside, is the image
    total = (cube.cube * 0.25).sum(axis=2) + cube.outside.sum(axis=2)
    _assert_close(total, image.image, 1e-11)
    narrow = ModelImageCube(two_files, params, (-0.5, 0.5, 4))
    assert np.array_equal(narrow.packet_image, image.packet_image)
    assert narrow.packet_outside.sum() > cube.packet_outside.sum()


@pytest.mark.gpu
def test_constant_step_recipe_rows_equal_resident_rows(monkeypatch):
    """A constant-step + bounce run, resident and recipe-only (regenerated in three chunks):
    each cube matches ModelImage of the same run, and the two cubes agree."""
    from nexoclom_b200 import ModelImage, ModelImageCube, Output
    inputs = workload('Na.bounce.input')
    params = dict(PARAMS, quantity='column')
    inputs.delete_files()
    kept = Output(inputs, 3000, seed=21, keep_trajectory=True)
    assert kept.trajectory_kept
    dense = ModelImageCube(inputs, params, (-4.0, 4.0, 40))
    _assert_matches_model_image(dense, ModelImage(inputs, params))
    inputs.delete_files()
    monkeypatch.setenv('NEXOCLOM_B200_MAX_ROWS', str(1000 * kept.nsteps))      # three chunks
    out = Output(inputs, 3000, seed=21)
    assert not out.trajectory_kept
    chunked = ModelImageCube(inputs, params, (-4.0, 4.0, 40))
    _assert_matches_model_image(chunked, ModelImage(inputs, params))
    inputs.delete_files()
    assert np.array_equal(chunked.packet_cube, dense.packet_cube)
    assert np.array_equal(chunked.packet_outside, dense.packet_outside)
    _assert_close(chunked.cube, dense.cube)
    assert chunked.totalsource == dense.totalsource


def _lp(setup):
    from nexoclom_b200._lib import LosParams
    lp = LosParams()
    lp.dphi, lp.outeredge = float(np.radians(2.0)), 25.0
    lp.vrplanet, lp.rp_cm = setup.vrplanet, setup.radius_km * 1e5
    lp.quantity, lp.round_f32, lp.skip_dead = 1, 1, 1
    return lp


def _los(nlos, seed):
    g = np.random.default_rng(seed)
    x_sc = g.standard_normal((3, nlos))
    x_sc *= (1.5 + 3 * g.random(nlos)) / np.linalg.norm(x_sc, axis=0)
    tgt = g.standard_normal((3, nlos))
    tgt *= (1 + 2 * g.random(nlos)) / np.linalg.norm(tgt, axis=0)
    bore = tgt - x_sc
    bore /= np.linalg.norm(bore, axis=0)
    d = np.linalg.norm(x_sc, axis=0)
    ang = np.arccos(np.clip(-(x_sc * bore).sum(axis=0) / d, -1.0, 1.0))
    return np.concatenate([x_sc, bore]), np.where(ang > np.arcsin(1. / d), 1e30, d)


@pytest.mark.gpu
def test_cube_calls_leave_image_and_los_pairs_alone(engine):
    """A cube call between two K4 calls into the context-owned image changes nothing there,
    and los_accumulate(count_used) -> cube -> los_used_fill still returns los_used's CSR."""
    setup = _run_slab(engine, 'Na.maxwellian.radpres.input', 1_000_000, 41)
    engine.upload_gtables(setup.gtables([5891, 5897]))
    table = engine.compact_state(skip_dead=True, round_f32=True, n=1_000_000)
    try:
        ip, _ = _ip(setup, 'radiance', (0.7, 0.3), (100, 100), 1e17, xrange=(-6.0, 6.0),
                    zrange=(-6.0, 6.0))
        engine.bind_packets(table)
        engine.image_begin(100, 100)
        engine.image_add(ip, n=table.n)
        engine.cube_begin(100, 100, 20)
        engine.cube_add(ip, -5.0, 5.0, 20, setup.radius_km, n=table.n)
        engine.image_add(ip, n=table.n)
        img, cnt = engine.image_fetch(100, 100)
        engine.image_begin(100, 100)
        engine.image_add(ip, n=table.n)
        one, cnt1 = engine.image_fetch(100, 100)
        assert cnt1.sum() > 1000 and np.array_equal(cnt, 2 * cnt1)
        _assert_close(img, 2 * one)
        cube, ccnt = engine.cube_fetch(100, 100, 20)
        assert np.array_equal(ccnt.sum(axis=2), cnt1)
        engine.cube_end()

        los, dplan = _los(300, 9)
        lp = _lp(setup)
        engine.los_accumulate(los, dplan, lp, n=table.n, count_used=True)     # sizes the buffers
        _, _, _, ucnt = engine.los_accumulate(los, dplan, lp, n=table.n, count_used=True)
        engine.cube_begin(100, 100, 20)
        engine.cube_add(ip, -5.0, 5.0, 20, setup.radius_km, n=table.n)
        engine.cube_fetch(100, 100, 20)
        engine.cube_end()
        launches = engine.kernel_launches()
        off, idx = engine.los_used_fill(los, dplan, lp, ucnt, n=table.n)
        assert engine.kernel_launches() - launches == 1          # the kept pairs, resolved again
        # for contrast, a call that drops the kept pairs: the fill searches again
        engine.los_accumulate(los, dplan, lp, n=table.n, count_used=True)
        engine.los_spectrum(los, dplan, lp, -5.0, 5.0, 20, setup.radius_km, n=table.n)
        launches = engine.kernel_launches()
        off2, _ = engine.los_used_fill(los, dplan, lp, ucnt, n=table.n)
        assert engine.kernel_launches() - launches > 1 and np.array_equal(off2, off)
        off0, idx0 = engine.los_used(los, dplan, lp, n=table.n)
        assert off0[-1] > 100 and np.array_equal(off, off0)
        for i in range(los.shape[1]):
            assert np.array_equal(np.sort(idx[off[i]:off[i + 1]]),
                                  np.sort(idx0[off[i]:off[i + 1]]))
    finally:
        engine.bind_packets(None)
        table.free()


@pytest.mark.gpu
def test_edge_cases(engine, built):
    from nexoclom_b200.engine import Engine, NexoclomCudaError
    setup = _na_setup()
    engine.upload_gtables(setup.gtables([5891, 5897]))
    ip, M = _ip(setup, 'radiance', (0.7, 0.3), (30, 20), 1e17)
    X = np.ones((16, 8))
    X[:, 4:7] = [1e-3, -2e-3, 5e-4]
    table = engine.upload_packets(X)
    try:
        got = _cube(engine, ip, -5.0, 5.0, 4, setup.radius_km, table.n, table)
        _assert_cubes(got, _oracle(X, setup, M, (30, 20), ip.apix, 'radiance', -5.0, 5.0, 4))
        assert got[1].sum() == 16
        got = _cube(engine, ip, -5.0, 5.0, 4, setup.radius_km, 0, table)        # no rows
        assert got[0].shape == (30, 20, 6) and got[1].sum() == 0 and not got[0].any()
        far, _ = _ip(setup, 'radiance', (0.7, 0.3), (30, 20), 1e17, xrange=(10.0, 12.0))
        got = _cube(engine, far, -5.0, 5.0, 4, setup.radius_km, table.n, table)  # all outside
        assert got[1].sum() == 0 and not got[0].any()
        engine.cube_begin(30, 20, 4)
        engine.bind_packets(table)
        try:
            for args, n in [((-5.0, 5.0, 5), table.n), ((5.0, -5.0, 4), table.n),
                            ((-5.0, np.nan, 4), table.n), ((-5.0, 5.0, 4), table.n + 1)]:
                with pytest.raises(NexoclomCudaError):
                    engine.cube_add(ip, *args, setup.radius_km, n=n)
            wrong, _ = _ip(setup, 'radiance', (0.7, 0.3), (20, 30), 1e17)
            with pytest.raises(NexoclomCudaError):
                engine.cube_add(wrong, -5.0, 5.0, 4, setup.radius_km, n=table.n)
        finally:
            engine.bind_packets(None)
            engine.cube_end()
        with pytest.raises(NexoclomCudaError):
            engine.cube_add(ip, -5.0, 5.0, 4, setup.radius_km, n=0)       # no cube
        with pytest.raises(NexoclomCudaError):
            engine.cube_begin(1 << 15, 1 << 15, 1)                       # 3 * 2^30 cells
    finally:
        table.free()
    fresh = Engine(0)                                                     # no g-value tables
    try:
        t2 = fresh.upload_packets(X)
        fresh.cube_begin(30, 20, 4)
        fresh.bind_packets(t2)
        with pytest.raises(NexoclomCudaError, match='g-value'):
            fresh.cube_add(ip, -5.0, 5.0, 4, setup.radius_km, n=t2.n)
        col, _ = _ip(setup, 'column', (0.7, 0.3), (30, 20), 1e17)
        fresh.cube_add(col, -5.0, 5.0, 4, setup.radius_km, n=t2.n)            # column: fine
        fresh.bind_packets(None)
        assert fresh.cube_fetch(30, 20, 4)[1].sum() == 16
        fresh.cube_end()
        t2.free()
    finally:
        fresh.close()


@pytest.mark.gpu
def test_no_output_files(engine):
    """An Input without output files: no rows, and no source to scale by (NaN, as LOSSpectrum
    gives)."""
    from nexoclom_b200 import ModelImageCube
    inputs = workload('Na.maxwellian.radpres.input')
    inputs.delete_files()
    try:
        cube = ModelImageCube(inputs, dict(PARAMS), (-5.0, 5.0, 10))
        assert cube.packet_cube.sum() == 0 and cube.packet_image.sum() == 0
        assert cube.cube.shape == (120, 90, 10) and np.isnan(cube.atoms_per_packet)
        assert np.isnan(cube.cube).all() and cube.totalsource == 0
    finally:
        inputs.delete_files()


@pytest.mark.gpu
def test_full_size_config1(engine):
    """configs[1] at full size: 1e7 live packets (the initial state) into a 200 x 200 x 100
    cube.  The sum over velocity is K4's image; two packet shards add up to the whole."""
    n = 10_000_000
    setup = _run_slab(engine, 'Na.maxwellian.radpres.input', n, 3, integrate=False)
    engine.upload_gtables(setup.gtables([5891, 5897]))
    ip, M = _ip(setup, 'radiance', (0.7, 0.3), (200, 200), 1e17, xrange=(-8.0, 8.0),
                zrange=(-8.0, 8.0), round_f32=1, skip_dead=1)
    img = _image(engine, ip, n)
    whole = _cube(engine, ip, -5.0, 5.0, 100, setup.radius_km, n)
    _assert_image(whole, img)
    assert whole[1].sum() > 0.9 * n and whole[1][:, :, 1:-1].sum() > 0.5 * n
    Xs = engine.export_state().T[:, :8].copy()
    half = n // 2
    engine.init_state(setup.source_params(engine), 3, 0, half)
    a = _cube(engine, ip, -5.0, 5.0, 100, setup.radius_km, half)
    engine.init_state(setup.source_params(engine), 3, half, n - half)
    b = _cube(engine, ip, -5.0, 5.0, 100, setup.radius_km, n - half)
    assert np.array_equal(a[1] + b[1], whole[1])
    _assert_close(a[0] + b[0], whole[0])
    # the compacted table, where K4 privatises its counts (n >= 2^20, all rows live)
    engine.init_state(setup.source_params(engine), 3, 0, n)
    table = engine.compact_state(skip_dead=True, round_f32=True, n=n)
    try:
        ipt, _ = _ip(setup, 'radiance', (0.7, 0.3), (200, 200), 1e17, xrange=(-8.0, 8.0),
                     zrange=(-8.0, 8.0))
        _assert_image(_cube(engine, ipt, -5.0, 5.0, 100, setup.radius_km, table.n, table),
                      _image(engine, ipt, table.n, table))
    finally:
        table.free()
    rows = Xs[::100].astype(np.float32).astype(np.float64)          # 1e5 rows against the oracle
    engine.import_state(rows)
    got = _cube(engine, ip, -5.0, 5.0, 100, setup.radius_km, len(rows))
    _assert_cubes(got, _oracle(rows, setup, M, (200, 200), ip.apix, 'radiance', -5.0, 5.0, 100,
                               xrange=(-8.0, 8.0), zrange=(-8.0, 8.0)))
