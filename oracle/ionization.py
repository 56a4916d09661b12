"""Oracle: where the adaptive driver's packets lose their frac in flight (ModelIonization, an
extension: the reference has no ion production map).

TEST INFRASTRUCTURE -- see oracle/__init__.py for who may import this.

``integrate_adaptive`` is ``deposition.integrate_adaptive`` statement for statement, with one
addition: an optional ``recorder`` receives every accepted step's loss (``frac before - frac of
the Runge-Kutta step``, the subtraction that sums the deposition oracle's ``loss``) and the
midpoint of its chord.  With the recorder on or off it returns what ``deposition`` returns, bit
for bit (tests/test_ionization.py).  ``Recorder`` keeps what it receives; ``bin_steps`` puts the
steps on the grid by ``np.histogramdd``'s rule (the last right edge in the last cell),
everything else (outside the box, NaN) in OUTSIDE.  ``exterior_fraction_reference`` is the
product's exterior-fraction rule with a brute-force 64^3 sub-sampling, used only to bound the
error of the product's 16^3.
"""
import numpy as np

from .deposition import (ESCAPED, MOON, REMAINING, SOURCE, SURFACE, VANISHED, Events)
from .tracking import bounce, dp_step, moon_xy


def integrate_adaptive(X0, rc, uniforms=None, step0=1000., recorder=None):
    """``deposition.integrate_adaptive`` with a recorder.  ``recorder``: None, or called as
    ``recorder(packet, loss, mid)`` for the accepted steps of each pass with a loss != 0: the
    packets (K,), ``frac before - frac of the Runge-Kutta step`` (K,) and the chord midpoints
    ``(x + x_rk) * 0.5`` (K, 3), before any surface handling.
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
            step_loss = cur[good, 7] - gn[:, 7]           # in-flight loss of the step
            loss[gidx] += step_loss
            if recorder is not None:
                rec = step_loss != 0
                recorder(gidx[rec], step_loss[rec], (cur[good][rec, 1:4] + gn[rec, 1:4]) * 0.5)
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


class Recorder:
    """A ``recorder`` for ``integrate_adaptive`` that keeps the steps it receives."""

    def __init__(self):
        self.parts = []

    def __call__(self, packet, loss, mid):
        self.parts.append((np.asarray(packet, np.int64), np.asarray(loss, np.float64),
                           np.asarray(mid, np.float64).reshape(-1, 3)))

    def arrays(self):
        """(packet (K,), loss (K,), mid (K, 3)) in the order the steps were recorded."""
        if not self.parts:
            return np.zeros(0, np.int64), np.zeros(0), np.zeros((0, 3))
        return tuple(np.concatenate([p[i] for p in self.parts]) for i in range(3))

    def per_packet(self, n):
        """(n,) sum of the recorded loss of each packet, added in step order."""
        out = np.zeros(n)
        for packet, loss, _ in self.parts:
            np.add.at(out, packet, loss)
        return out


def edges(lo, hi, dims):
    return tuple(np.linspace(a, b, n + 1) for a, b, n in zip(lo, hi, dims))


def cell(mid, lo, hi, dims):
    """Row-major cell index (ix * ny + iy) * nz + iz of each point (K, 3) by np.histogramdd's
    rule per axis, -1 outside the box or NaN."""
    mid = np.asarray(mid, np.float64).reshape(-1, 3)
    idx = []
    for k, e in enumerate(edges(lo, hi, dims)):
        v = mid[:, k]
        i = np.searchsorted(e, v, side='right') - 1
        i[v == e[-1]] = len(e) - 2
        i[(v < e[0]) | (v > e[-1]) | np.isnan(v)] = -1
        idx.append(i)
    i, j, k = idx
    ok = (i >= 0) & (j >= 0) & (k >= 0)
    return np.where(ok, (i * dims[1] + j) * dims[2] + k, -1)


def bin_steps(loss, mid, lo, hi, dims):
    """(sums (nx, ny, nz), counts (nx, ny, nz) int64, outside sum, outside count) of recorded
    steps; the grid by np.histogramdd itself."""
    loss = np.asarray(loss, np.float64)
    mid = np.asarray(mid, np.float64).reshape(-1, 3)
    inside = cell(mid, lo, hi, dims) >= 0
    e = edges(lo, hi, dims)
    sums, _ = np.histogramdd(mid[inside], bins=e, weights=loss[inside])
    cnt, _ = np.histogramdd(mid[inside], bins=e)
    return sums, cnt.astype(np.int64), float(loss[~inside].sum()), int((~inside).sum())


def exterior_fraction_reference(edges_xyz, sub=64):
    """The exterior-fraction rule of ModelIonization with sub**3 sub-cell midpoints: 1 when a
    cell's nearest point is at r >= 1, 0 when its farthest corner is at r <= 1, else the
    fraction of the sub-cell midpoints at r >= 1."""
    ex, ey, ez = (np.asarray(e, np.float64) for e in edges_xyz)
    out = np.empty((len(ex) - 1, len(ey) - 1, len(ez) - 1))
    t = (np.arange(sub) + 0.5) / sub
    for i in range(len(ex) - 1):
        for j in range(len(ey) - 1):
            for k in range(len(ez) - 1):
                box = [(ex[i], ex[i + 1]), (ey[j], ey[j + 1]), (ez[k], ez[k + 1])]
                near = sum(0.0 if a <= 0 <= b else min(abs(a), abs(b)) ** 2 for a, b in box)
                far = sum(max(abs(a), abs(b)) ** 2 for a, b in box)
                if near >= 1.0:
                    out[i, j, k] = 1.0
                elif far <= 1.0:
                    out[i, j, k] = 0.0
                else:
                    x, y, z = (a + t * (b - a) for a, b in box)
                    r2 = (x * x)[:, None, None] + (y * y)[None, :, None] + (z * z)[None, None, :]
                    out[i, j, k] = (r2 >= 1.0).mean()
    return out
