"""The adaptive driver with surface bounce (K2 built with BOUNCE: nx_integrate_adaptive_bounce,
Engine.integrate_adaptive_bounce, Output's adaptive path for surfaces that do not absorb every
packet).  The composition is pinned piecewise: the oracle's adaptive driver and its bounce are
pinned to the reference's own outputs elsewhere; here the oracle with bounce deviates reduces
to the reference's driver for perfect sticking, conserves energy across bounces, and the host
build of the attempt functions, then the kernel, reproduce it.  The oracle is
oracle/adaptive_bounce.py: oracle.tracking's driver with the bounce branch added."""
import ctypes as C
import os

import numpy as np
import pytest

from common import REPO, KERNEL_CELLS, Cell, workload, oracle_constants, state_parity
from nexoclom_b200._lib import dptr
from nexoclom_b200.runsetup import RunSetup
from nexoclom_b200.units import Quantity
from oracle import adaptive_bounce, tracking, initial_state

STATE_TOL = 1e-8
BOUNCE_WORKLOADS = ['Na.bounce.input', 'Na.bounce.stick05.input']
U32P = C.POINTER(C.c_uint32)


def adaptive_inputs(name):
    """A constant-step workload on the adaptive driver (step_size = 0, resolution 1e-4)."""
    inputs = workload(name)
    inputs.options.step_size = 0.
    inputs.options.resolution = 1e-4
    return inputs


def run_oracle(setup, X0, seed, first_id=0):
    return adaptive_bounce.integrate_adaptive(X0, oracle_constants(setup),
                                              adaptive_bounce.bounce_uniforms(seed, first_id))


@pytest.fixture(scope='module')
def hcb(built):
    return C.CDLL(os.path.join(REPO, 'tests', '_hostcheck', 'libnexo_adaptive_bounce_hostcheck.so'))


def run_host(hcb, setup, X0, seed, first_id, strict):
    p = setup.params
    n = len(X0)
    X = np.ascontiguousarray(X0, dtype=np.float64).copy()
    att, acc, bnc = (np.zeros(n, np.uint32) for _ in range(3))
    rv = ra = np.zeros(1)
    nrp = 0
    if setup.radpres_v is not None:
        rv, ra = np.ascontiguousarray(setup.radpres_v), np.ascontiguousarray(setup.radpres_a)
        nrp = len(rv)
    tck = setup.spline_tck or (np.zeros(8), np.zeros(8), np.zeros(16))
    tx, ty, c = (np.ascontiguousarray(a, dtype=np.float64) for a in tck)
    st = hcb.hc_integrate_adaptive_bounce(
        C.c_long(n), dptr(X), att.ctypes.data_as(U32P), acc.ctypes.data_as(U32P),
        bnc.ctypes.data_as(U32P), C.byref(p), dptr(rv), dptr(ra), C.c_int(nrp), dptr(tx),
        C.c_int(len(tx)), dptr(ty), C.c_int(len(ty)), dptr(c), C.c_ulonglong(seed),
        C.c_ulonglong(first_id), C.c_int(strict))
    assert st == 0
    return X, att, acc, bnc


# ---------------------------------------------------------------------------- CPU
@pytest.mark.parametrize('wl', ['Na.maxwellian.radpres.input', 'Ca.isotropic.flat.input'])
def test_oracle_perfect_sticking_unchanged_by_uniforms(wl):
    """With stickcoef == 1 the bounce deviates are never drawn: bit for bit the reference's
    driver (tracking.integrate_adaptive, pinned to the reference), which pins the restatement."""
    setup = RunSetup(workload(wl))
    X0 = initial_state.draw_x0(setup, 500, 4)[:, :8]
    Xq, aq, cq = tracking.integrate_adaptive(X0, oracle_constants(setup))
    Xb, ab, cb, bn = run_oracle(setup, X0, seed=11)
    assert np.array_equal(Xq, Xb) and np.array_equal(aq, ab) and np.array_equal(cq, cb)
    assert bn.sum() == 0


def test_energy_conserved_across_bounces(hcb):
    """Gravity only, stickcoef = 0, no accommodation: a bounce keeps the speed the packet has
    at r = 1, so the orbital energy E = v^2/2 + GM/r only changes by the integration error.
    Per accepted step the error control bounds the position error by res (1 + |x|) and the
    velocity error by 0.1 res (1 + |v|) per component, so |dE| <= sqrt(3) res (0.1 (1 + v) v +
    |GM| (1 + r) / r^2) per step; summed over a packet's accepted steps at r >= 1 and v <= its
    speed at the surface that is the bound checked here."""
    inputs = adaptive_inputs('Na.bounce.stick05.input')
    inputs.surfaceinteraction.stickcoef = 0.
    inputs.surfaceinteraction.accomfactor = None
    inputs.forces.radpres = False
    setup = RunSetup(inputs)
    p = setup.params
    assert p.accomfactor == 0.0 and p.stickcoef == 0.0 and not p.radpres
    X0 = initial_state.draw_x0(setup, 300, 6)[:, :8]

    def energy(X):
        r = np.sqrt((X[:, 1:4] ** 2).sum(axis=1))
        return 0.5 * (X[:, 4:7] ** 2).sum(axis=1) + p.GM / r, r

    E0, r0 = energy(X0)
    vsurf = np.sqrt(np.maximum(2 * (E0 - p.GM), 0.0))            # speed at r = 1
    res, gm = p.resolution, abs(p.GM)
    per_step = np.sqrt(3) * res * (0.1 * (1 + vsurf) * vsurf + 2 * gm)
    for strict in (1, 0):
        X, att, acc, bnc = run_host(hcb, setup, X0, seed=3, first_id=0, strict=strict)
        assert bnc.sum() > 300                                   # packets hop many times
        E1, _ = energy(X)
        dE = np.abs(E1 - E0)
        assert np.all(dE <= acc * per_step), np.max(dE / (acc * per_step))
        # and in practice far inside it: fifth-order steps under a fourth-order error estimate
        assert np.median(dE / np.abs(E0)) < 1e-6


# the workloads, and every force x loss x moon cell of the adaptive driver with bounce
@pytest.mark.parametrize('wl', BOUNCE_WORKLOADS +
                         [c for c in KERNEL_CELLS if c.driver == 'adaptive' and c.bounce], ids=str)
@pytest.mark.parametrize('strict', [1, 0])
def test_host_build_matches_oracle(hcb, wl, strict):
    from test_hostcheck import host_strict
    if isinstance(wl, Cell):
        setup = wl.setup()
        X0 = wl.x0(setup, 300, 21)
    else:
        setup = RunSetup(adaptive_inputs(wl))
        X0 = initial_state.draw_x0(setup, 300, 21)[:, :8]
    seed, first = 5, 1000
    Xo, a_o, c_o, b_o = run_oracle(setup, X0, seed, first)
    Xh, a_h, c_h, b_h = run_host(hcb, setup, X0, seed, first, host_strict(setup, strict, True))
    par = state_parity(Xh, Xo)
    assert par['alive_mismatch'] == 0, par
    assert np.array_equal(a_h, a_o) and np.array_equal(c_h, c_o)
    # without gravity only radiation pressure brings a few packets back
    assert np.array_equal(b_h, b_o) and b_o.sum() > (300 if setup.params.gravity else 0)
    assert max(par['pos'], par['vel'], par['frac']) < STATE_TOL, par


def test_adaptive_workload_is_the_bounce_workload_without_step():
    a, b = workload('Na.bounce.adaptive.input'), workload('Na.bounce.input')
    assert a.options.step_size == 0 and float(a.options.resolution) == 1e-4
    assert a.surfaceinteraction == b.surfaceinteraction and a.geometry == b.geometry
    assert a.speeddist == b.speeddist and a.forces == b.forces
    assert float(np.asarray(a.options.endtime)) == float(np.asarray(b.options.endtime))


# ---------------------------------------------------------------------------- GPU
def gpu_run(engine, setup, X0, seed, first_id=0):
    setup.upload(engine)
    engine.import_state(X0)
    att, acc, bnc = engine.integrate_adaptive_bounce(seed, first_id)
    a, c = engine.export_stats()
    return engine.export_state().T, att, acc, bnc, a, c


@pytest.mark.gpu
@pytest.mark.parametrize('wl', BOUNCE_WORKLOADS)
@pytest.mark.parametrize('strict', [True, False])
def test_kernel_matches_oracle(engine, wl, strict):
    setup = RunSetup(adaptive_inputs(wl), strict_math=strict)
    n, seed, first = 3000, 17, 123
    X0 = initial_state.draw_x0(setup, n, 21)[:, :8]
    Xg, att, acc, bnc, a_g, c_g = gpu_run(engine, setup, X0, seed, first)
    Xo, a_o, c_o, b_o = run_oracle(setup, X0, seed, first)
    par = state_parity(Xg, Xo)
    assert par['alive_mismatch'] == 0, par
    assert max(par['pos'], par['vel'], par['frac']) < STATE_TOL, par
    assert np.array_equal(a_g, a_o) and np.array_equal(c_g, c_o)
    assert att == int(a_o.sum()) and acc == int(c_o.sum())
    assert bnc == int(b_o.sum()) and bnc > n
    assert np.all(Xg[Xo[:, 7] == 0, 0] == 0)                      # dead => time = 0


@pytest.mark.gpu
def test_perfect_sticking_equals_adaptive_entry(engine):
    setup = RunSetup(workload('Na.maxwellian.radpres.input'))
    setup.upload(engine)
    X0 = initial_state.draw_x0(setup, 20000, 2)[:, :8]
    engine.import_state(X0)
    att, acc = engine.integrate_adaptive()
    Xa, sa = engine.export_state(), engine.export_stats()
    Xb, att_b, acc_b, bnc, a_b, c_b = gpu_run(engine, setup, X0, seed=9)
    assert np.array_equal(Xa.T, Xb) and (att, acc) == (att_b, acc_b) and bnc == 0
    assert np.array_equal(sa[0], a_b) and np.array_equal(sa[1], c_b)


@pytest.mark.gpu
def test_bit_for_bit_invariances(engine):
    """Packet order, sharding (first_id) and the seed: only the seed changes results."""
    setup = RunSetup(workload('Na.bounce.adaptive.input'))
    n, seed = 40000, 77
    X0 = initial_state.draw_x0(setup, n, 3)[:, :8]
    ref = gpu_run(engine, setup, X0, seed)
    assert ref[3] > n
    try:
        engine.set_option('order_packets', 0)
        plain = gpu_run(engine, setup, X0, seed)
    finally:
        engine.set_option('order_packets', 3)
    again = gpu_run(engine, setup, X0, seed)
    h = 15000
    s0 = gpu_run(engine, setup, X0[:h], seed, 0)
    s1 = gpu_run(engine, setup, X0[h:], seed, h)
    other = gpu_run(engine, setup, X0, seed + 1)
    for run in (plain, again):
        assert np.array_equal(run[0], ref[0]) and run[1:4] == ref[1:4]
        assert np.array_equal(run[4], ref[4]) and np.array_equal(run[5], ref[5])
    assert np.array_equal(np.concatenate([s0[0], s1[0]]), ref[0])
    assert np.array_equal(np.concatenate([s0[4], s1[4]]), ref[4])
    assert s0[3] + s1[3] == ref[3] and s0[1] + s1[1] == ref[1]
    assert not np.array_equal(other[0], ref[0])


def _shell_profile(x, y, z, f, edges):
    r = np.sqrt((x * x + y * y) + z * z)
    return np.histogram(r, bins=edges, weights=f)[0]


@pytest.mark.gpu
def test_steady_state_profile_matches_constant_step(engine):
    """Both drivers sample packet ages uniformly over endtime, so Sigma frac per packet in radial
    shells (1-5 R_p) estimates the same exosphere.  Gate, fixed before looking at the data:
    5 standard errors (per-packet sums, both runs) plus 3% of the shell's value, for K3's
    30 s step: a bounce is only seen after up to one step inside the planet and the lost
    time is not given back (Q17), ~15 s of a ~500 s hop on average."""
    edges = np.array([1.0, 1.05, 1.1, 1.2, 1.4, 1.7, 2.2, 3.0, 5.0])
    na = 1_000_000
    setup_a = RunSetup(workload('Na.bounce.adaptive.input'))
    setup_a.upload(engine)
    engine.init_state(setup_a.source_params(engine), 31, 0, na)
    engine.integrate_adaptive_bounce(31, 0)
    Xa = engine.export_state()
    contrib = np.zeros((na, len(edges) - 1))
    r = np.sqrt((Xa[1] ** 2 + Xa[2] ** 2) + Xa[3] ** 2)
    k = np.searchsorted(edges, r, side='right') - 1
    ok = (k >= 0) & (k < len(edges) - 1)
    contrib[np.nonzero(ok)[0], k[ok]] = Xa[7][ok]
    prof_a, err_a = contrib.mean(axis=0), contrib.std(axis=0) / np.sqrt(na)

    nc = 200_000
    setup_c = RunSetup(workload('Na.bounce.input'))
    setup_c.upload(engine)
    engine.init_state(setup_c.source_params(engine), 32, 0, nc)
    table, nsteps, _ = engine.integrate_constant_rows(seed=32, skip_dead=True, round_f32=False)
    cols, index, _ = table.export(with_step=True)
    table.free()
    rr = np.sqrt((cols['x'].astype(np.float64) ** 2 + cols['y'].astype(np.float64) ** 2)
                 + cols['z'].astype(np.float64) ** 2)
    kc = np.searchsorted(edges, rr, side='right') - 1
    okc = (kc >= 0) & (kc < len(edges) - 1)
    per_packet = np.zeros((nc, len(edges) - 1))
    np.add.at(per_packet, (index[okc].astype(np.int64), kc[okc]), cols['frac'][okc].astype(np.float64))
    per_packet /= nsteps
    prof_c, err_c = per_packet.mean(axis=0), per_packet.std(axis=0) / np.sqrt(nc)

    gate = 5 * np.hypot(err_a, err_c) + 0.03 * prof_c
    print('adaptive', prof_a, '\nconstant', prof_c, '\ngate', gate)
    assert np.all(prof_a[:5] > 0) and np.all(prof_c[:5] > 0)   # the populated shells
    assert np.all(np.abs(prof_a - prof_c) <= gate), (prof_a, prof_c, gate)


@pytest.mark.gpu
def test_public_api_products(engine):
    """Input.run on the adaptive bounce workload feeds ModelImage, LOSResult and ModelDensity;
    an Output on imported X0 with the same seed and ids equals the device-drawn run."""
    from nexoclom_b200 import LOSResult, ModelDensity, ModelImage, Output, catalogue
    from test_spectrum import _SC, _los
    inputs = workload('Na.bounce.adaptive.input')
    inputs.delete_files()
    n = 200_000
    try:
        inputs.run(n, seed=41)
        _, files, npk, _ = inputs.search()
        assert npk == n and len(files) == 1
        out = catalogue.fetch(files[0])
        assert out.bounces > n and out.attempted_steps > out.accepted_steps > 0
        X = out.X
        assert len(X) > 0 and np.all(X['frac'].values > 0)

        params = {'quantity': 'column', 'dims': '100,100', 'width': '8,8', 'center': '0,0',
                  'subobslongitude': '0.7', 'subobslatitude': '0.3'}
        img = ModelImage(inputs, params)
        assert 0 < np.asarray(img.packet_image).sum() <= len(X)
        sc = _SC(_los(60, 3), index=[f's{i}' for i in range(60)])
        res = LOSResult(sc, inputs, dphi=Quantity(3.0, 'deg'))
        res.simulate_data_from_inputs(sc)
        assert res.npackets_los.values.sum() > 0
        pts = np.array([[1.05, 0.0, 0.0], [0.0, -1.2, 0.0]])
        dens = ModelDensity(inputs, pts, 0.2)
        assert np.all(dens.npackets.values > 0)

        # the same packets in full precision (Output.X0 holds them rounded to float32, as saved)
        setup = RunSetup(inputs)
        setup.upload(engine)
        engine.init_state(setup.source_params(engine), 41, 0, n)
        cols = engine.export_x0()[:8].T.copy()
        imp = Output(inputs, n, X0=cols, seed=41, first_id=0)
        assert imp.bounces == out.bounces and imp.attempted_steps == out.attempted_steps
        Xi = imp.X
        for c in ('x', 'y', 'z', 'vx', 'vy', 'vz', 'frac', 'time'):
            assert np.array_equal(Xi[c].values, X[c].values), c
    finally:
        inputs.delete_files()


@pytest.mark.gpu
def test_full_size(engine):
    """1e7 packets: no status bits, two shards equal one run, oracle parity on a slice."""
    setup = RunSetup(workload('Na.bounce.adaptive.input'))
    setup.upload(engine)
    n, seed = 10_000_000, 5
    engine.init_state(setup.source_params(engine), seed, 0, n)
    X0 = engine.export_x0()[:8].T.copy()
    att, acc, bnc = engine.integrate_adaptive_bounce(seed, 0)
    X = engine.export_state()
    a, _ = engine.export_stats()
    assert bnc > n and att == int(a.astype(np.int64).sum())
    h = 4_000_000
    engine.import_state(X0[h:])
    att1, acc1, bnc1 = engine.integrate_adaptive_bounce(seed, h)
    X1 = engine.export_state()
    engine.import_state(X0[:h])
    att0, acc0, bnc0 = engine.integrate_adaptive_bounce(seed, 0)
    X0s = engine.export_state()
    assert np.array_equal(np.concatenate([X0s, X1], axis=1), X)
    assert (att0 + att1, acc0 + acc1, bnc0 + bnc1) == (att, acc, bnc)
    sl = slice(5_000_000, 5_001_500)
    Xo, a_o, _, _ = run_oracle(setup, X0[sl], seed, sl.start)
    par = state_parity(X.T[sl], Xo)
    assert par['alive_mismatch'] == 0 and np.array_equal(a[sl], a_o)
    assert max(par['pos'], par['vel'], par['frac']) < STATE_TOL, par
