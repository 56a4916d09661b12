"""The kernels' shared per-packet physics (nexoclom_b200/csrc/*.cuh), compiled
for the HOST by tests/_hostcheck (test-only), against the oracle.  This pins the
logic of every kernel on machines without a GPU; the GPU parity tests
(test_gpu_parity.py) then only have to show the device build agrees."""
import ctypes as C
import os

import numpy as np
import pytest

from common import (REPO, GOLDEN, KERNEL_CELLS, Cell, adaptive_mode, workload, oracle_constants,
                    state_parity)
from nexoclom_b200._lib import RunParams, SourceParams, ImageParams, dptr
from nexoclom_b200.runsetup import RunSetup
from nexoclom_b200.units import Quantity
from nexoclom_b200.ModelImage import image_rotation
from oracle import tracking, initial_state, imaging


@pytest.fixture(scope='module')
def hc(built):
    lib = C.CDLL(os.path.join(REPO, 'tests', '_hostcheck', 'libnexo_hostcheck.so'))
    return lib


def _rp(setup):
    if setup.radpres_v is None:
        return None, None, 0, np.zeros(1), np.zeros(1)
    rv, ra = np.ascontiguousarray(setup.radpres_v), np.ascontiguousarray(setup.radpres_a)
    return dptr(rv), dptr(ra), len(rv), rv, ra


def run_adaptive(hc, setup, X0, strict):
    p = setup.params
    prv, pra, nrp, _rv, _ra = _rp(setup)
    X = np.ascontiguousarray(X0.copy())
    n = len(X)
    step = np.full(n, 1000.)
    att = np.zeros(n, np.uint32)
    acc = np.zeros(n, np.uint32)
    st = hc.hc_integrate_adaptive(C.c_long(n), dptr(X), dptr(step),
                                  att.ctypes.data_as(C.POINTER(C.c_uint32)),
                                  acc.ctypes.data_as(C.POINTER(C.c_uint32)), C.byref(p), prv, pra,
                                  C.c_int(nrp), C.c_int(strict))
    assert st == 0
    return X, att, acc, step


def host_strict(setup, strict, bounce=False):
    """The host build's flag for the build the device runs: adaptive_attempt_fast_rt has fast
    builds the dispatchers never select (a moon or bounce without gravity), those runs take the
    strict build on the device."""
    return int(bool(strict) or adaptive_mode(setup.params, bounce) < 0)


# the workloads, and every force x loss x moon cell of the perfect-sticking adaptive driver
@pytest.mark.parametrize('wl', ['Na.maxwellian.radpres.input', 'Ca.isotropic.flat.input'] +
                         [c for c in KERNEL_CELLS if c.driver == 'adaptive' and not c.bounce],
                         ids=str)
@pytest.mark.parametrize('strict', [1, 0])
def test_adaptive_attempt_matches_oracle(hc, wl, strict):
    if isinstance(wl, Cell):
        setup = wl.setup()
        X0 = wl.x0(setup, 600, 3)
    else:
        setup = RunSetup(workload(wl))
        X0 = initial_state.draw_x0(setup, 600, 3)[:, :8]
    Xo, a_o, c_o = tracking.integrate_adaptive(X0, oracle_constants(setup))
    Xh, a_h, c_h, _ = run_adaptive(hc, setup, X0, host_strict(setup, strict))
    par = state_parity(Xh, Xo)
    assert par['alive_mismatch'] == 0
    assert np.array_equal(a_h, a_o) and np.array_equal(c_h, c_o)      # same step sequence
    assert max(par['pos'], par['vel'], par['frac']) < 1e-11           # gate is 1e-8


def test_adaptive_against_reference_golden(hc):
    """Import mode on the reference's own driver output (tests/golden)."""
    g = np.load(os.path.join(GOLDEN, 'adaptive_driver.npz'))
    for tag, wl in (('na', 'Na.maxwellian.radpres.input'), ('ca', 'Ca.isotropic.flat.input')):
        setup = RunSetup(workload(wl))
        Xh, _, _, step = run_adaptive(hc, setup, g[f'{tag}_x0'], 0)
        par = state_parity(Xh, g[f'{tag}_final'])
        assert par['alive_mismatch'] == 0
        assert max(par['pos'], par['vel'], par['frac']) < 1e-8


def test_philox_matches_oracle(hc):
    n = 1000
    u0, u1 = np.zeros(n), np.zeros(n)
    for stream, draw, seed, first in ((0, 0, 0, 0), (1, 17, 0x123456789ab, 1 << 33)):
        hc.hc_uniform_pairs(C.c_long(n), C.c_ulonglong(seed), C.c_ulonglong(first),
                            C.c_uint(stream), C.c_uint(draw), dptr(u0), dptr(u1))
        ids = np.arange(first, first + n, dtype=np.uint64)
        o0, o1 = initial_state.uniform_pair(seed, ids, stream, draw)
        assert np.array_equal(u0, o0) and np.array_equal(u1, o1)
        assert 0 <= u0.min() and u0.max() < 1


@pytest.mark.parametrize('wl', ['Na.maxwellian.radpres.input', 'Ca.isotropic.flat.input',
                                'Na.bounce.stick05.input'])
def test_init_state_matches_oracle(hc, wl):
    setup = RunSetup(workload(wl))
    sp = setup.source_params(None)
    n = 5000
    out = np.zeros((n, 14))
    tab = getattr(setup, 'speed_table', None)
    cdf, vt = (np.ascontiguousarray(tab[0]), np.ascontiguousarray(tab[1])) if tab else (None, None)
    hc.hc_init_state(C.c_long(n), C.byref(sp), C.c_ulonglong(42), C.c_ulonglong(1000),
                     None, None, dptr(cdf) if tab else None, dptr(vt) if tab else None,
                     C.c_int(len(cdf) if tab else 0), dptr(out))
    ref = initial_state.draw_x0(setup, n, 42, first_id=1000)
    assert np.max(np.abs(out - ref)) < 1e-13
    r = np.linalg.norm(out[:, 1:4], axis=1)
    assert np.allclose(r, sp.exobase, rtol=1e-14)
    # outward hemisphere
    assert np.all(np.sum(out[:, 1:4] * out[:, 4:7], axis=1) >= -1e-18)


def test_2d_angular_distribution(hc):
    inputs = workload('Ca.isotropic.flat.input')
    from nexoclom_b200.input_classes import AngularDist
    inputs.angulardist = AngularDist({'type': '2d', 'altitude': '0.3, 2.5'})
    setup = RunSetup(inputs)
    sp = setup.source_params(None)
    n = 4000
    out = np.zeros((n, 14))
    hc.hc_init_state(C.c_long(n), C.byref(sp), C.c_ulonglong(1), C.c_ulonglong(0), None, None,
                     None, None, C.c_int(0), dptr(out))
    ref = initial_state.draw_x0(setup, n, 1)
    assert np.max(np.abs(out - ref)) < 1e-13
    assert np.all(out[:, 6] == 0) and np.all(out[:, 13] == 0)          # vz = 0, azimuth = 0
    assert out[:, 12].min() >= 0.3 - 1e-12 and out[:, 12].max() <= 2.5 + 1e-12
    assert np.allclose(np.hypot(out[:, 4], out[:, 5]), out[:, 8], rtol=1e-13)


def test_surface_spot_sampling(hc):
    """surface-spot rejection sampling (source_distribution.py:96-121): device
    logic == oracle transform fed with the same Philox triples."""
    inputs = workload('Na.maxwellian.radpres.input')
    from nexoclom_b200.input_classes import SpatialDist
    inputs.spatialdist = SpatialDist({'type': 'surface spot', 'longitude': '0.5',
                                      'latitude': '0.2', 'sigma': '0.4'})
    setup = RunSetup(inputs)
    sp = setup.source_params(None)
    fmap, lon, lat = setup.sourcemap
    fm = np.ascontiguousarray(fmap)
    axes = np.array([lon[0], lon[-1], lat[0], lat[-1]])
    cdf, vt = (np.ascontiguousarray(a) for a in setup.speed_table)
    n = 3000
    out = np.zeros((n, 14))
    hc.hc_init_state(C.c_long(n), C.byref(sp), C.c_ulonglong(5), C.c_ulonglong(0), dptr(fm),
                     dptr(axes), dptr(cdf), dptr(vt), C.c_int(len(cdf)), dptr(out))
    ref = initial_state.draw_x0(setup, n, 5)
    assert np.max(np.abs(out - ref)) < 1e-12
    # the spot is where it should be (ptsz sign flip, quirk Q19: latitude mirrored)
    assert abs(np.median(out[:, 10]) + 0.2) < 0.1


# the bounce workloads, and every force x loss cell of the constant-step driver with bounce
@pytest.mark.parametrize('tag, wl', [('tdep', 'Na.bounce.input'),
                                     ('c05', 'Na.bounce.stick05.input')] +
                         [pytest.param(c.id, c, id=c.id) for c in KERNEL_CELLS
                          if c.driver == 'constant'])
def test_constant_step_bounce_matches_oracle(hc, tag, wl):
    n, seed, first = 400, 99, 7
    if isinstance(wl, Cell):
        setup = wl.setup()
        X0 = wl.x0(setup, n, 9)
    else:
        inputs = workload(wl)
        inputs.options.endtime = Quantity(1500., 's')
        setup = RunSetup(inputs)
        X0 = initial_state.draw_x0(setup, n, 9)[:, :8]
    rc = oracle_constants(setup)
    p = setup.params
    hits = []
    uniforms = initial_state.bounce_uniforms(seed, first)

    def counted(ct, idx):
        hits.append(len(idx))
        return uniforms(ct, idx)

    ref, nsteps, _ = tracking.integrate_constant(X0, rc, uniforms=counted)
    tx, ty, c = setup.spline_tck
    prv, pra, nrp, _rv, _ra = _rp(setup)
    for strict in (1, 0):
        X = np.ascontiguousarray(X0.copy())
        traj = np.zeros((n, 8, nsteps))
        hc.hc_integrate_constant(C.c_long(n), dptr(X), dptr(traj), C.c_int(nsteps),
                                 C.c_ulonglong(seed), C.c_ulonglong(first), C.byref(p), prv, pra,
                                 C.c_int(nrp), dptr(tx), C.c_int(len(tx)), dptr(ty),
                                 C.c_int(len(ty)), dptr(c), C.c_int(strict))
        assert np.array_equal(traj[:, 7, :] > 0, ref[:, 7, :] > 0)
        assert np.max(np.abs(traj - ref)) < 1e-10
    # packets did bounce (a force brings them back to the surface)
    if p.gravity or p.radpres:
        assert sum(hits) > 0
    if not isinstance(wl, Cell):
        assert (ref[:, 7, -1] < 0.9).any()


def test_spline_matches_scipy(hc):
    setup = RunSetup(workload('Na.bounce.input'))
    tx, ty, c = setup.spline_tck
    rng = np.random.default_rng(0)
    T = rng.uniform(90, 720, 4000)
    pr = rng.random(4000)
    pr[:4] = [0., 1., 0.5, 1e-9]
    out = np.zeros(4000)
    hc.hc_spline_ev(C.c_long(4000), dptr(T), dptr(pr), dptr(out), dptr(tx), C.c_int(len(tx)),
                    dptr(ty), C.c_int(len(ty)), dptr(c))
    ref = setup.surfaceint.v_interp(T, pr)
    assert np.max(np.abs(out - ref)) < 1e-12 * np.abs(ref).max()


@pytest.mark.parametrize('quantity', [0, 1])
@pytest.mark.parametrize('view', [(0.0, np.pi / 2), (0.7, 0.3)])
def test_image_packet_matches_oracle(hc, quantity, view):
    setup = RunSetup(workload('Na.maxwellian.radpres.input'))
    rng = np.random.default_rng(1)
    n = 200000
    X = np.zeros((n, 8))
    X[:, 1:4] = rng.normal(size=(n, 3)) * 1.8
    X[:, 5] = rng.normal(size=n) * 2 / setup.radius_km
    X[:, 7] = rng.random(n)
    X[:50, 1] = 4.0          # right edge belongs to the last bin
    X[50:100, 1] = -4.0
    X = X.astype(np.float32).astype(np.float64)
    M = image_rotation(*view)
    ip = ImageParams()
    for k in range(9):
        ip.M[k] = float(M.flat[k])
    ip.x0, ip.x1, ip.z0, ip.z1 = -4, 4, -4, 4
    ip.nx, ip.nz = 800, 640
    ip.apix = 5.9e11
    ip.vrplanet = setup.vrplanet
    ip.quantity = quantity
    gt = setup.gtables([5891, 5897])
    sizes = (C.c_int * 2)(len(gt[0][0]), len(gt[1][0]))
    v = np.ascontiguousarray(np.concatenate([t[0] for t in gt]))
    g = np.ascontiguousarray(np.concatenate([t[1] for t in gt]))
    img = np.zeros((800, 640))
    cnt = np.zeros((800, 640), dtype=np.int64)
    hc.hc_image(C.c_long(n), dptr(np.ascontiguousarray(X)), C.byref(ip), 2, sizes, dptr(v),
                dptr(g), dptr(img), cnt.ctypes.data_as(C.POINTER(C.c_longlong)))
    oi, oc, _, _ = imaging.create_image(X[:, 1], X[:, 2], X[:, 3], X[:, 5], X[:, 7],
                                        vrplanet=setup.vrplanet, M=imaging.image_rotation(*view),
                                        dims=[800, 640], xrange=(-4, 4), zrange=(-4, 4),
                                        apix=ip.apix, quantity='radiance' if quantity else 'column',
                                        gtables=gt)
    assert np.array_equal(cnt, oc.astype(np.int64))          # pixel indexing bit-exact
    assert np.max(np.abs(img - oi)) <= 1e-12 * oi.max()
