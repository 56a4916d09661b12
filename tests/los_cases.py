"""Line-of-sight geometry families for the K5 membership tests (test_los_membership.py on the
host build, test_los_geometry.py on the GPU).  Each family is a list of groups: lines of sight
that share one cone half-angle and outer edge, and a synthetic cloud that puts packets inside
and just outside every cone (and, where the family is about them, at the edges the test
should decide: the last KD ball, the planet cut, the shadow).

Clouds are float32-representable, so the F64 and F32 record builds see the same packets, and
about 20 % of their rows are dead (frac = 0)."""
import numpy as np

ARCSEC = np.pi / (180.0 * 3600.0)
RP_CM = 2439.7e5
VRPLANET = 1e-3


def gtables():
    """Two synthetic g-value tables (velocity [R_p/s], g [1/s]) that vary across the packets'
    velocities, so a weight error shows."""
    v = np.linspace(-0.02, 0.02, 41)
    return [(v, 1.0 + 0.5 * np.sin(60 * v) + 40 * v), (v, 0.7 + 0.2 * np.cos(90 * v))]


def unit(v):
    v = np.asarray(v, dtype=np.float64)
    return v / np.linalg.norm(v)


def dist_from_plan(los):
    """The planet cut of every line: |x_sc| if the boresight hits the planet, else 1e30
    (reference compute_iteration.py:105-115, as oracle.imaging.los_iteration computes it)."""
    sx, sy, sz, bx, by, bz = (los[:, k] for k in range(6))
    d = np.sqrt(sx**2 + sy**2 + sz**2)
    ang = np.arccos((-sx * bx - sy * by - sz * bz) / d)
    d = d.copy()
    d[ang > np.arcsin(1. / d)] = 1e30
    return d


def line(x_sc, target=None, bore=None):
    x_sc = np.asarray(x_sc, dtype=np.float64)
    b = unit(np.asarray(target, dtype=np.float64) - x_sc) if bore is None else np.asarray(bore, np.float64)
    return np.concatenate([x_sc, b])


def _basis(b):
    a = np.array([1., 0., 0.]) if abs(b[0]) < 0.9 else np.array([0., 1., 0.])
    e1 = unit(np.cross(b, a))
    return e1, np.cross(b, e1)


def cone_points(row, dphi, t, rng, spread=1.3):
    """Points at axial distances t from the observer of ``row``, at angles up to spread * dphi
    from its boresight (uniform over the disc: 1 / spread^2 of them inside the cone)."""
    x, b = row[:3], row[3:]
    e1, e2 = _basis(b)
    n = len(t)
    ang = spread * dphi * np.sqrt(rng.random(n))
    phi = rng.uniform(0.0, 2 * np.pi, n)
    d = (np.cos(ang)[:, None] * b + np.sin(ang)[:, None] *
         (np.cos(phi)[:, None] * e1 + np.sin(phi)[:, None] * e2))
    return x + (t / np.cos(ang))[:, None] * d


def log_uniform(rng, lo, hi, n):
    return np.exp(rng.uniform(np.log(lo), np.log(hi), n))


def packets(P, rng, dead=0.2):
    """(n, 8) state rows time, x, y, z, vx, vy, vz, frac at positions P, float32 values."""
    n = len(P)
    X = np.zeros((n, 8))
    X[:, 0] = 1.0
    X[:, 1:4] = P
    X[:, 4:7] = rng.normal(size=(n, 3)) * 3.0 / 2439.7
    X[:, 7] = rng.random(n)
    X[rng.random(n) < dead, 7] = 0.0
    return X.astype(np.float32).astype(np.float64)


def _group(name, dphi, outeredge, rows, parts, rng):
    los = np.array(rows, dtype=np.float64)
    return {'name': name, 'dphi': float(dphi), 'outeredge': float(outeredge), 'los': los,
            'X': packets(np.concatenate(parts), rng)}


def _cone_group(name, dphi, outeredge, rows, tfun, per, rng, spread=1.3):
    parts = [cone_points(r, dphi, tfun(r, per), rng, spread) for r in rows]
    return _group(name, dphi, outeredge, rows, parts, rng)


def _near_planet(r, per, rng, half=8.0):
    """Axial distances of the part of a line within `half` R_p of the planet's centre."""
    tc = -float(np.dot(r[:3], r[3:]))                 # closest approach
    return rng.uniform(max(tc - half, 1e-3), tc + half, per)


def fam_far(per, rng, arcsec=(2.0, 10.0)):
    """Observers at 1e4 and 5e4 R_p (ground-based geometry) through the disk, the limb and
    the tail, at arcsecond apertures and at 1 deg."""
    groups = []
    for a in arcsec:
        d1, d2 = unit(rng.normal(size=3)), unit(rng.normal(size=3))
        rows = [line(1e4 * d1, [0.2, -0.3, 0.1]),                      # the disk
                line(5e4 * d2, 1.0005 * unit(np.cross(d2, [0., 0., 1.])))]   # just off the limb
        groups.append(_cone_group(f'far{a:g}"', a * ARCSEC, 25.0, rows,
                                  lambda r, n: _near_planet(r, n, rng, 6.0), per, rng))
    rows = []
    for dist in (1e4, 5e4):
        d = unit(rng.normal(size=3))
        rows += [line(dist * d, [0.1, 0.2, -0.3]), line(dist * d, [0.0, 3.0, 0.5]),        # disk, tail
                 line(dist * d, 1.01 * unit(np.cross(d, [1., 0., 0.])))]                  # limb
    groups.append(_cone_group('far1deg', np.radians(1.0), 25.0, rows,
                              lambda r, n: _near_planet(r, n, rng, 10.0), per, rng))
    return groups


def fam_inside(per, rng, arcsec=None):
    """Observers at 1.2-3 R_p inside the cloud, looking outward (no planet cut); packets from
    1e-3 R_p (closer than the first ball centre) to 10 R_p."""
    rows = []
    for r in (1.2, 2.0, 3.0):
        x = r * unit(rng.normal(size=3))
        rows.append(line(x, bore=unit(unit(x) + 0.4 * unit(rng.normal(size=3)))))
    groups = [_cone_group('inside1deg', np.radians(1.0), 25.0, rows,
                          lambda r, n: log_uniform(rng, 1e-3, 10.0, n), per, rng)]
    if arcsec:
        # one line at an arcsecond aperture from 3 R_p: 1.5e6 ladder entries to the outer edge
        x = 3.0 * unit([0.3, -0.8, 0.5])
        rows = [line(x, bore=unit(unit(x) + 0.2 * unit([1., 1., 0.])))]
        groups.append(_cone_group(f'inside{arcsec:g}"', arcsec * ARCSEC, 25.0, rows,
                                  lambda r, n: rng.uniform(0.05, 6.0, n), per, rng, spread=0.9))
    return groups


def fam_beyond(per, rng):
    """Outer edge 4 R_p inside a 10 R_p cloud: members in the last ball, past the boresight's
    exit from the outer edge, and packets beyond it."""
    groups = []
    for deg in (1.0, 5.0):
        rows = []
        for r in (2.0, 3.0):
            x = r * unit(rng.normal(size=3))
            rows.append(line(x, bore=unit(unit(x) + 0.3 * unit(rng.normal(size=3)))))
        rows.append(line([0.5, -6.0, 1.0], [0.0, 0.5, 2.0]))          # from outside the edge, across

        def tfun(r, n, deg=deg):
            x, b = r[:3], r[3:]
            c = x @ x - 16.0
            dd = (-2 * (x @ b) + np.sqrt(4 * (x @ b) ** 2 - 4 * c)) / 2
            # half the packets in (dd, dd (1 + sin 2 dphi)^2): the last ball and past it
            s2 = np.sin(2 * np.radians(deg))
            return np.concatenate([rng.uniform(0.01, dd, n - n // 2),
                                   rng.uniform(dd, dd * (1 + s2) ** 2, n // 2)])
        groups.append(_cone_group(f'beyond{deg:g}deg', np.radians(deg), 4.0, rows, tfun, per, rng))
    return groups


def fam_wide(per, rng):
    """Wide cones either side of the `cover` flip near 27 deg: the ball-window search."""
    groups = []
    for deg in (10.0, 26.0, 28.0):
        rows = []
        for r in (1.5, 3.0, 6.0):
            x = r * unit(rng.normal(size=3))
            rows.append(line(x, 0.5 * unit(rng.normal(size=3))))
        groups.append(_cone_group(f'wide{deg:g}deg', np.radians(deg), 25.0, rows,
                                  lambda r, n: log_uniform(rng, 1e-2, 12.0, n), per, rng, spread=1.1))
    return groups


def fam_shadow(per, rng):
    """Lines whose foot-points cross the planet's shadow (y > 0, x^2 + z^2 < 1): hits of
    weight 0, counted but not `used`."""
    rows = [line([-6.0, 2.0, 0.3], bore=[1.0, 0.0, 0.0]),
            line([0.2, 1.5, -6.0], bore=[0.0, 0.0, 1.0]),
            line([-4.0, 6.0, 3.0], [0.3, 1.2, -0.2])]
    return [_cone_group('shadow', np.radians(2.0), 25.0, rows,
                        lambda r, n: rng.uniform(0.5, 12.0, n), per, rng)]


def fam_limb(per, rng):
    """Boresights at asin(1 / |x_sc|) +- 1e-9 rad from the planet's centre: the planet cut on
    and off, packets either side of losrad = |x_sc|."""
    rows = []
    for r, delta in ((2.0, -1e-9), (2.0, 1e-9), (5.0, -1e-9), (5.0, 1e-9), (1e4, -1e-9), (1e4, 1e-9)):
        d = unit(rng.normal(size=3))
        e1, _ = _basis(-d)
        a = np.arcsin(1.0 / r) + delta
        rows.append(line(r * d, bore=unit(np.cos(a) * -d + np.sin(a) * e1)))
    assert np.array_equal(dist_from_plan(np.array(rows)) < 1e30, [True, False] * 3)

    def tfun(r, n):
        d = np.linalg.norm(r[:3])
        return np.concatenate([rng.uniform(max(d - 2.0, 1e-3), d + 3.0, n - n // 4),
                               d + rng.uniform(-1e-6, 1e-6, n // 4) * max(d, 1.0)])
    return [_cone_group('limb', np.radians(1.0), 25.0, rows, tfun, per, rng)]


def fam_axis(per, rng):
    """Observers on the axes, boresights exactly +-x, +-y, +-z (components 0.0 and -0.0)."""
    rows = []
    for a in range(3):
        for sgn in (1.0, -1.0):
            x = np.zeros(3)
            x[a] = 5.0 * sgn
            rows.append(np.concatenate([x, -x / 5.0]))                 # at the centre: -0.0 parts
    rows.append(np.array([1.5, 0.0, 0.0, 1.0, 0.0, 0.0]))            # outward along +x
    rows.append(np.array([0.0, -3.0, 0.0, 0.0, 1.0, -0.0]))          # into the planet along +y
    assert any(np.signbit(r[3:]).any() and (r[3:] == 0).any() for r in rows)
    return [_cone_group('axis', np.radians(1.0), 25.0, rows,
                        lambda r, n: log_uniform(rng, 1e-2, 12.0, n), per, rng)]


def fam_outside(per, rng):
    """Observers beyond the outer edge (4 R_p) whose boresight misses the sphere (dd NaN) or
    points away from it (dd < 0): one ball, around the observer."""
    rows = [line([6.0, 0.0, 1.0], bore=unit([0.0, 1.0, 0.1])),       # misses: dd NaN
            line([0.0, -7.0, 2.0], bore=unit([1.0, 0.05, 0.0])),      # misses
            line([5.0, 3.0, 0.0], bore=unit([1.0, 0.5, 0.2])),        # points away: dd < 0
            line([0.0, 0.0, 4.5], [0.0, 0.0, 0.0])]                   # enters the sphere
    return [_cone_group('outside', np.radians(10.0), 4.0, rows,
                        lambda r, n: log_uniform(rng, 1e-3, 0.6, n), per, rng)]


FAMILIES = {'far': fam_far, 'inside': fam_inside, 'beyond': fam_beyond, 'wide': fam_wide,
            'shadow': fam_shadow, 'limb': fam_limb, 'axis': fam_axis, 'outside': fam_outside}
