"""Oracle: where the frac of the adaptive driver's packets goes (ModelDeposition, an extension:
the reference records neither the deposit nor the loss budget).

TEST INFRASTRUCTURE -- see oracle/__init__.py for who may import this.

``integrate_adaptive`` is ``adaptive_bounce.integrate_adaptive`` (which is
``tracking.integrate_adaptive`` for perfect sticking) statement for statement, with every event
of an accepted step recorded as ``Events`` rows: SURFACE (the deposited frac, at the post-step
point for perfect sticking, the bounce point otherwise), then MOON / ESCAPED / VANISHED for the
first of those tests that zeroes a frac that is not already 0.  REMAINING is the final frac of
the packets still > 0, SOURCE the initial frac > 0.  The frac lost in flight is summed directly,
``frac before - frac after the Runge-Kutta step`` of every accepted step, so that the buckets
plus the loss equal the source as an independent check.
"""
import numpy as np

from .tracking import bounce, dp_step, moon_xy

SURFACE, MOON, ESCAPED, VANISHED, REMAINING, SOURCE = range(6)
BUCKETS = ('surface', 'moon', 'escaped', 'vanished', 'remaining', 'source')


def lonlat(pos):
    """Surface longitude / latitude of event points (K, 3): the bounce's convention."""
    x, y, z = pos[:, 0], pos[:, 1], pos[:, 2]
    lon = np.fmod(np.arctan2(x, -y) + 2 * np.pi, 2 * np.pi)
    lat = np.arctan2(z, np.sqrt(x * x + y * y))
    return lon, lat


def edges(nlon, nlat):
    """The map's axes: those of make_source_map."""
    return np.linspace(0, 2 * np.pi, nlon + 1), np.linspace(-np.pi / 2, np.pi / 2, nlat + 1)


def cell(lon, lat, nlon, nlat):
    """Cell index ilon * nlat + ilat of each point by np.histogram2d's rule (searchsorted
    'right', the last edge inclusive), -1 outside."""
    out = []
    for v, e in zip((np.asarray(lon, float), np.asarray(lat, float)), edges(nlon, nlat)):
        k = np.searchsorted(e, v, side='right') - 1
        k[v == e[-1]] = len(e) - 2
        k[(v < e[0]) | (v > e[-1]) | np.isnan(v)] = -1
        out.append(k)
    i, j = out
    return np.where((i >= 0) & (j >= 0), i * nlat + j, -1)


class Events:
    def __init__(self):
        self.parts = []

    def add(self, packet, bucket, amount, pos=None):
        k = len(packet)
        if k == 0:
            return
        lon = lat = np.full(k, np.nan)
        if pos is not None:
            lon, lat = lonlat(pos)
        self.parts.append((np.asarray(packet, np.int64), np.full(k, bucket, np.int64),
                           np.asarray(amount, np.float64), lon, lat))

    def arrays(self):
        """dict of packet, bucket, amount, lon, lat (NaN unless SURFACE), in event order."""
        names = ('packet', 'bucket', 'amount', 'lon', 'lat')
        if not self.parts:
            return {n: np.zeros(0, np.int64 if n in ('packet', 'bucket') else np.float64)
                    for n in names}
        return {n: np.concatenate([p[i] for p in self.parts]) for i, n in enumerate(names)}


def integrate_adaptive(X0, rc, uniforms=None, step0=1000.):
    """Adaptive driver with the events recorded.  ``uniforms``: as in
    ``adaptive_bounce.integrate_adaptive`` (unused for perfect sticking).
    Returns (X, attempted, accepted, bounces, events dict, loss (N,))."""
    simple_stick = rc.sticktype == 'constant' and rc.stickcoef == 1.
    safety, shrink = 0.95, -0.25
    res = rc.resolution
    resx, resv, resf = res, 0.1 * res, res

    X = np.array(X0, dtype=np.float64, copy=True)
    n = X.shape[0]
    step = np.zeros(n) + step0
    attempted = np.zeros(n, dtype=np.int64)
    accepted = np.zeros(n, dtype=np.int64)
    bounces = np.zeros(n, dtype=np.int64)
    loss = np.zeros(n)
    ev = Events()
    src = np.nonzero(X[:, 7] > 0)[0]
    ev.add(src, SOURCE, X[src, 7])
    live = (X[:, 0] > res) & (X[:, 7] > 0.)
    while live.any():
        idx = np.nonzero(live)[0]
        cur = X[idx]
        h = np.minimum(cur[:, 0], step[idx])
        assert np.all(h > 0), 'Bad step size'
        nxt, delta = dp_step(cur, h, rc, want_error=True)

        scale = np.empty((len(idx), 8))
        scale[:, 0] = 1.0
        scale[:, 1:4] = resx + np.abs(nxt[:, 1:4]) * resx
        scale[:, 4:7] = resv + np.abs(nxt[:, 4:7]) * resv
        scale[:, 7] = resf + np.abs(nxt[:, 7]) * resf
        ratio = delta / scale
        ratio[:, 0] = delta[:, 0]
        errmax = ratio.max(axis=1)
        assert np.all(np.isfinite(errmax)), '\n\tInfinite values of emax'
        assert not np.any((nxt[:, 7] < 0) & (errmax < 1)), (
            'Found new values of frac that are negative')

        errmax[(nxt[:, 7] - cur[:, 7] > scale[:, 7]) & (errmax > 1)] = 1.1   # Q9
        noerr = errmax < 1e-7
        errmax[noerr] = 1
        htried = h.copy()
        htried[noerr] *= 10
        good = errmax < 1.0
        bad = ~good
        attempted[idx] += 1

        if good.any():
            gidx = idx[good]
            gn = nxt[good]
            loss[gidx] += cur[good, 7] - gn[:, 7]          # in-flight loss of the step
            r2 = (gn[:, 1]**2 + gn[:, 2]**2) + gn[:, 3]**2
            hit = r2 < 1
            f_before = gn[hit, 7].copy()
            if simple_stick:
                gn[hit, 7] = 0
            elif hit.any():
                ids = gidx[hit]
                u_alt, u_az, u_prob = uniforms(accepted[ids] + 1, ids)
                gn[hit] = bounce(rc, gn[hit], np.sqrt(r2[hit]), u_alt, u_az, u_prob)
                bounces[ids] += 1
            ev.add(gidx[hit], SURFACE, f_before - gn[hit, 7], gn[hit, 1:4])
            for mo in rc.moons:
                mx, my = moon_xy(mo, gn[:, 0])
                dx, dy = gn[:, 1] - mx, gn[:, 2] - my
                m = dx * dx + dy * dy + gn[:, 3] * gn[:, 3] < mo['radius']**2
                first = m & (gn[:, 7] != 0)
                ev.add(gidx[first], MOON, gn[first, 7])
                gn[m, 7] = 0
            esc = r2 > rc.outeredge
            first = esc & (gn[:, 7] != 0)
            ev.add(gidx[first], ESCAPED, gn[first, 7])
            gn[esc, 7] = 0
            van = gn[:, 7] < 1e-10
            first = van & (gn[:, 7] != 0)
            ev.add(gidx[first], VANISHED, gn[first, 7])
            gn[van, 7] = 0.
            gn[gn[:, 7] == 0, 0] = 0
            X[gidx] = gn
            accepted[gidx] += 1
        if bad.any():
            old = htried[bad]
            new = safety * old * errmax[bad]**shrink
            assert not np.any(np.isclose(new, old))
            assert np.all(np.isfinite(new)), '\n\tInfinite values of step_size'
            step[idx[bad]] = np.maximum(new, 0.1 * old)

        live = (X[:, 0] > res) & (X[:, 7] > 0.)
    rem = np.nonzero(X[:, 7] > 0)[0]
    ev.add(rem, REMAINING, X[rem, 7])
    return X, attempted, accepted, bounces, ev.arrays(), loss


def summarize(events, nlon, nlat):
    """(map (nlon, nlat), map counts, bucket sums (6,), bucket counts (6,)) of an events dict;
    the map by np.histogram2d itself."""
    b = events['bucket']
    sums = np.array([events['amount'][b == k].sum() for k in range(6)])
    counts = np.array([(b == k).sum() for k in range(6)], dtype=np.int64)
    s = b == SURFACE
    le, ae = edges(nlon, nlat)
    dmap, _, _ = np.histogram2d(events['lon'][s], events['lat'][s], bins=(le, ae),
                                weights=events['amount'][s])
    cnt, _, _ = np.histogram2d(events['lon'][s], events['lat'][s], bins=(le, ae))
    return dmap, cnt.astype(np.int64), sums, counts
