"""K5's line-of-sight membership on the host build (tests/_hostcheck/los_hostcheck.cpp: the
ladder and constants of nx_los.h, los_hit and los_weight of nx_image.cuh, compiled with g++)
against the reference's rule (oracle.imaging.los_iteration, compute_iteration.py:151-222):

  ladder      the KD-ball ladder of a call is the reference's `t` list bit for bit, however
              many entries the aperture and the distance need, and every line's ball count is
              the length of its own list (NaN and short boresight distances included);
  membership  hit sets, `included`, `used` sets and radiance over the geometry families of
              los_cases (far observers, observers inside the cloud, members past the outer
              edge, wide cones, shadow, limb, axis boresights, observers outside the edge);
  shortcuts   the `cover` and `cos_accept2` shortcuts decide as the full test on packets a few
              ulp either side of the cone surface and of the ball boundaries;
  validation  a bad cone half-angle, or a ladder above the budget, is refused (C ABI and the
              public classes)."""
import ctypes as C
import os

import numpy as np
import pytest

import los_cases
from common import REPO, workload
from oracle import imaging

LADDER_MAX = 1 << 25
ARCSEC = los_cases.ARCSEC
VRPLANET = los_cases.VRPLANET
gtables = los_cases.gtables


@pytest.fixture(scope='module')
def hc(built):
    return C.CDLL(os.path.join(REPO, 'tests', '_hostcheck', 'libnexo_los_hostcheck.so'))


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def prepare(hc, los, dphi, outeredge):
    """Host per-line preparation of (nlos, 6) lines: (nball, constants, ladder, wid2); raises
    ValueError with the library's reason when the call is refused."""
    L = np.ascontiguousarray(los.T, dtype=np.float64)
    nlos = los.shape[0]
    nball = np.zeros(nlos, dtype=np.int32)
    consts = np.zeros(9)
    nl = C.c_longlong()
    err = C.create_string_buffer(512)
    rc = hc.hc_los_prepare(_dp(L), C.c_longlong(nlos), C.c_double(dphi), C.c_double(outeredge),
                           nball.ctypes.data_as(C.POINTER(C.c_int)), _dp(consts), C.byref(nl),
                           err, C.c_int(512))
    if rc != 0:
        raise ValueError(err.value.decode())
    ladder, wid2 = np.zeros(nl.value), np.zeros(nl.value)
    hc.hc_los_ladder(_dp(ladder), _dp(wid2))
    return nball, consts, ladder, wid2


def members(hc, los, dist, nball, X, dphi, gt, cover=-1, accept_off=0):
    """(hit, weight), each (nlos, n), of every (line, packet) pair by the host los_hit /
    los_weight, over the ladder of the last ``prepare``."""
    L = np.ascontiguousarray(los.T, dtype=np.float64)
    nlos, n = los.shape[0], X.shape[0]
    cols = [np.ascontiguousarray(X[:, k]) for k in (1, 2, 3, 5, 7)]
    sizes = np.array([len(v) for v, _ in gt], dtype=np.int32)
    gv = np.ascontiguousarray(np.concatenate([v for v, _ in gt]))
    gg = np.ascontiguousarray(np.concatenate([g for _, g in gt]))
    hit = np.zeros((nlos, n), dtype=np.uint8)
    w = np.zeros((nlos, n))
    dist = np.ascontiguousarray(dist, dtype=np.float64)
    rc = hc.hc_los_members(_dp(L), C.c_longlong(nlos), _dp(dist),
                           np.ascontiguousarray(nball).ctypes.data_as(C.POINTER(C.c_int)),
                           C.c_longlong(n), *[_dp(c) for c in cols], C.c_double(dphi),
                           C.c_double(VRPLANET), C.c_double(los_cases.RP_CM), C.c_int(len(gt)),
                           sizes.ctypes.data_as(C.POINTER(C.c_int)), _dp(gv), _dp(gg),
                           C.c_int(cover), C.c_int(accept_off),
                           hit.ctypes.data_as(C.POINTER(C.c_uint8)), _dp(w))
    assert rc == 0
    return hit.astype(bool), w


def oracle_ladder(dphi, dd):
    """The reference's ladder (compute_iteration.py:158-160, oracle.imaging.los_iteration):
    t = [sin(dphi)]; while t[-1] < dd: t.append(t[-1] + t[-1] * sin(dphi)).  The sine is taken
    once (the same float64 each time) and the sums are Python floats, the same IEEE float64
    operations as NumPy's scalars."""
    s = float(np.sin(dphi))
    t = [s]
    last = s
    while last < dd:
        last = last + last * s
        t.append(last)
    return np.array(t)


def oracle_dd(row, outeredge):
    """The boresight distance to the outer edge, statement by statement as the oracle."""
    x_sc, bore = row[0:3].astype(float), row[3:6].astype(float)
    b = 2 * np.sum(x_sc * bore)
    c = np.linalg.norm(x_sc)**2 - outeredge**2
    return (-b + np.sqrt(b**2 - 4 * 1 * c)) / 2


# ---- ladder -----------------------------------------------------------------------------------
DPHIS = [(45.0, 'deg'), (28.0, 'deg'), (26.0, 'deg'), (1.0, 'deg'), (0.1, 'deg'),
         (10.0, 'arcsec'), (4.0, 'arcsec'), (2.0, 'arcsec'), (1.0, 'arcsec')]
DDS = [0.5, 30.0, 1.5e4, 5e4]


def _rad(v, unit):
    return np.radians(v) if unit == 'deg' else v * ARCSEC


@pytest.mark.parametrize('dphi', DPHIS, ids=[f'{v:g}{u}' for v, u in DPHIS])
def test_ladder_is_the_references(hc, dphi):
    """For every distance: the ladder of a call whose longest boresight distance is dd is the
    reference's `t` list for dd, length and values bit for bit; wid2 is its squared ball
    radius (t sin 2 dphi)^2."""
    dphi = _rad(*dphi)
    full = oracle_ladder(dphi, max(DDS))     # every shorter ladder is a prefix of this one
    s2 = np.sin(dphi * 2)
    for dd in DDS:
        n = int(np.searchsorted(full, dd, 'left')) + 1 if full[0] < dd else 1
        ref = full[:n]
        assert ref[-1] >= dd and (n == 1 or ref[-2] < dd)
        los = np.array([[0.0, 0.0, 0.0, 1.0, 0.0, 0.0]])
        assert oracle_dd(los[0], dd) == dd
        nball, consts, ladder, wid2 = prepare(hc, los, dphi, dd)
        assert len(ladder) == n, (dd, len(ladder), n)
        assert np.array_equal(ladder.view(np.int64), ref.view(np.int64)), dd
        assert np.array_equal(wid2.view(np.int64), ((ref * s2) ** 2).view(np.int64)), dd
        assert nball[0] == n and consts[8] == n


@pytest.mark.parametrize('dphi', [np.radians(1.0), 2 * ARCSEC, np.radians(28.0)])
def test_ball_counts_are_the_references(hc, dphi):
    """Per line: the ball count is the length of the reference's own ladder for that line --
    observers inside and outside the edge, boresights that miss it (dd NaN), point away from
    it (dd < 0) or leave it closer than the first ball centre (dd < t_0)."""
    rng = np.random.default_rng(5)
    oe = 25.0
    rows = []
    for r in (0.3, 1.5, 6.0, 24.9999, 25.0, 40.0, 1e4):
        for _ in range(4):
            x = r * los_cases.unit(rng.normal(size=3))
            rows.append(los_cases.line(x, bore=los_cases.unit(rng.normal(size=3))))
            rows.append(los_cases.line(x, [0.0, 0.0, 0.0]))
    x = np.array([0.0, 0.0, oe - 0.25 * np.sin(dphi)])
    rows.append(los_cases.line(x, bore=[0.0, 0.0, 1.0]))              # dd < t_0
    rows.append(los_cases.line([30.0, 0.0, 0.0], bore=[0.0, 1.0, 0.0]))   # misses: NaN
    rows.append(los_cases.line([30.0, 0.0, 0.0], bore=[1.0, 0.0, 0.0]))   # points away: dd < 0
    los = np.array(rows)
    with np.errstate(invalid='ignore'):
        dd = np.array([oracle_dd(r, oe) for r in los])
        assert np.isnan(dd).any() and (dd < 0).any() and ((dd > 0) & (dd < np.sin(dphi))).any()
    nball, consts, ladder, _ = prepare(hc, los, dphi, oe)
    full = oracle_ladder(dphi, np.nanmax(dd))
    assert np.array_equal(ladder, full)
    for i, d in enumerate(dd):
        assert nball[i] == len(oracle_ladder(dphi, d)), (i, d)


# ---- membership -------------------------------------------------------------------------------
def _groups(name):
    rng = np.random.default_rng(sum(map(ord, name)))
    fam = los_cases.FAMILIES[name]
    if name == 'far':
        return fam(400, rng, arcsec=(10.0,))
    if name == 'inside':
        return fam(600, rng, arcsec=2.0)
    return fam(600, rng)


def _check_group(hc, g, gt):
    los, X, dphi, oe = g['los'], g['X'], g['dphi'], g['outeredge']
    used_o = []
    rad_o, np_o, inc_o, dist = imaging.los_iteration(
        X[:, 1], X[:, 2], X[:, 3], X[:, 5], X[:, 7], los, vrplanet=VRPLANET, dphi=dphi,
        outeredge=oe, rp_cm=los_cases.RP_CM, gtables=gt, used=used_o)
    nball, _, _, _ = prepare(hc, los, dphi, oe)
    hit, w = members(hc, los, dist, nball, X, dphi, gt)
    assert np.array_equal(hit.sum(axis=1), np_o), (g['name'], hit.sum(axis=1), np_o)
    assert np.array_equal(hit.any(axis=0), inc_o), g['name']
    for i in range(len(los)):
        assert set(np.flatnonzero(hit[i] & (w[i] > 0)).tolist()) == used_o[i], (g['name'], i)
    rad = w.sum(axis=1)
    assert np.array_equal(rad == 0, rad_o == 0), g['name']
    nz = rad_o > 0
    assert np.all(np.abs(rad[nz] - rad_o[nz]) <= 1e-12 * rad_o[nz]), g['name']
    return np_o


@pytest.mark.parametrize('family', sorted(los_cases.FAMILIES))
def test_membership_matches_oracle(hc, family):
    gt = gtables()
    for g in _groups(family):
        np_o = _check_group(hc, g, gt)
        assert np_o.sum() > 0, g['name']


def test_arcsecond_line_from_3_rp_keeps_every_member(hc):
    """The line of the ladder-cap report: observer at 3 R_p, dphi = 2", packets inside the
    cone from 0.05 to 6 R_p.  A ladder truncated at 2^20 entries ends 0.25 R_p from the
    observer and loses every member past it."""
    rng = np.random.default_rng(2)
    x = 3.0 * los_cases.unit([0.3, -0.8, 0.5])
    row = los_cases.line(x, bore=los_cases.unit(los_cases.unit(x) + 0.2 * los_cases.unit([1., 1., 0.])))
    dphi = 2 * ARCSEC
    P = los_cases.cone_points(row, dphi, rng.uniform(0.05, 6.0, 4000), rng, spread=0.9)
    X = los_cases.packets(P, rng)
    los = row[None, :]
    nball, _, ladder, _ = prepare(hc, los, dphi, 25.0)
    assert len(ladder) > 1 << 20
    hit, _ = members(hc, los, los_cases.dist_from_plan(los), nball, X, dphi, gtables())
    ang = np.arccos(np.clip(((P - x) @ row[3:]) / np.linalg.norm(P - x, axis=1), -1, 1))
    inside = ang <= dphi * (1 - 1e-6)
    assert inside.sum() > 3000 and hit[0][inside].all()


# ---- shortcuts --------------------------------------------------------------------------------
def _edge_packets(row, dphi, ladder, wid2, nball, rng, n=3000):
    """Packets a few ulp either side of the cone surface and of the ball boundaries of one
    line."""
    x, b = row[:3], row[3:]
    e1, e2 = los_cases._basis(b)
    out = []
    # on the cone surface at random axial distances, nudged by -4..4 ulp per coordinate
    t = los_cases.log_uniform(rng, ladder[0] * 0.5, ladder[nball - 1] * 1.2, n)
    phi = rng.uniform(0, 2 * np.pi, n)
    d = np.cos(dphi) * b + np.sin(dphi) * (np.cos(phi)[:, None] * e1 + np.sin(phi)[:, None] * e2)
    out.append(x + (t / np.cos(dphi))[:, None] * d)
    # on the surface of ball k (random k, random direction in the plane across the boresight
    # and along it), at the cone-ball intersections
    k = rng.integers(0, nball, n)
    r = np.sqrt(wid2[k])
    u = rng.normal(size=(n, 3))
    u /= np.linalg.norm(u, axis=1)[:, None]
    out.append(x + ladder[k][:, None] * b + r[:, None] * u)
    P = np.concatenate(out)
    steps = rng.integers(-4, 5, P.shape)
    for _ in range(4):
        up = steps > 0
        P = np.where(up, np.nextafter(P, np.inf), np.where(steps < 0, np.nextafter(P, -np.inf), P))
        steps = steps - np.sign(steps)
    return P


@pytest.mark.parametrize('deg', [26.0, 28.0, 10.0])
def test_shortcuts_decide_as_the_full_test(hc, deg):
    """`cover` forced off and `cos_accept2` forced to +inf (every candidate through acos and
    the ball-window search) decide every packet as the default test, on packets crowded at the
    cone surface and the ball boundaries; 26 and 28 deg sit either side of the `cover` flip."""
    dphi = np.radians(deg)
    rng = np.random.default_rng(int(deg))
    gt = gtables()
    rows = [los_cases.line(r * los_cases.unit(rng.normal(size=3)), 0.3 * los_cases.unit(rng.normal(size=3)))
            for r in (1.5, 4.0, 9.0)]
    los = np.array(rows)
    dist = los_cases.dist_from_plan(los)
    nball, consts, ladder, wid2 = prepare(hc, los, dphi, 25.0)
    assert consts[4] == (1 if deg < 27 else 0)
    for i, row in enumerate(rows):
        P = _edge_packets(row, dphi, ladder, wid2, nball[i], rng)
        X = los_cases.packets(P, rng, dead=0.0)
        X[:, 1:4] = P                               # the ulp-nudged positions, not rounded
        one = los[i:i + 1]
        ref, wref = members(hc, one, dist[i:i + 1], nball[i:i + 1], X, dphi, gt, cover=0, accept_off=1)
        for cover, acc in ((-1, 0), (0, 0), (-1, 1)):
            h, w = members(hc, one, dist[i:i + 1], nball[i:i + 1], X, dphi, gt, cover=cover, accept_off=acc)
            assert np.array_equal(h, ref), (deg, i, cover, acc, int((h != ref).sum()))
            assert np.array_equal(w, wref)
        assert 0 < ref.sum() < ref.size


# ---- validation -------------------------------------------------------------------------------
BAD_DPHI = [0.0, -1e-6, np.nan, np.inf, -np.inf, np.pi / 2, 2.0]


@pytest.mark.parametrize('dphi', BAD_DPHI)
def test_bad_cone_half_angle_is_refused(hc, dphi):
    los = np.array([[0.0, -3.0, 0.0, 0.0, 1.0, 0.0]])
    with pytest.raises(ValueError, match='dphi'):
        prepare(hc, los, dphi, 25.0)


def test_ladder_above_the_budget_is_refused(hc):
    """0.1" from 5e4 R_p needs ~4.8e7 entries, more than the 2^25 budget: refused with the
    angle and the entry count, never truncated."""
    dphi = 0.1 * ARCSEC
    need = np.log(5e4 / np.sin(dphi)) / np.log1p(np.sin(dphi))
    assert need > LADDER_MAX
    los = np.array([[5e4, 0.0, 0.0, -1.0, 0.0, 0.0]])
    with pytest.raises(ValueError, match=r'dphi = .*arcsec.*ladder entries.*33554432'):
        prepare(hc, los, dphi, 25.0)
    # 1" from 5e4 R_p (4.8e6 entries) fits
    nball, _, ladder, _ = prepare(hc, los, ARCSEC, 25.0)
    assert len(ladder) > 4_000_000 and nball[0] == len(ladder)


@pytest.mark.parametrize('dphi', [0.0, -1.0, np.nan, np.inf, 90.0, 120.0])
def test_public_classes_refuse_bad_dphi(dphi):
    """LOSResult, LOSResultFitted and LOSSpectrum raise ValueError before any device work."""
    from nexoclom_b200 import LOSResult, LOSSpectrum
    from nexoclom_b200.LOSResultFitted import LOSResultFitted
    from nexoclom_b200.units import Quantity
    from test_spectrum import _SC, _los
    inputs = workload('Na.maxwellian.radpres.input')
    sc = _SC(_los(4, 1))
    for q in (Quantity(dphi, 'deg'), dphi):
        with pytest.raises(ValueError, match='dphi'):
            LOSResult(sc, inputs, dphi=q)
        with pytest.raises(ValueError, match='dphi'):
            LOSSpectrum(sc, inputs, (-5.0, 5.0, 10), dphi=q)
    sc.model_result = {'unfit': type('R', (), {'inputs': inputs})()}
    with pytest.raises(ValueError, match='dphi'):
        LOSResultFitted(sc, 'unfit', dphi=Quantity(dphi, 'deg'))
