"""Oracle: images and density grids from every accepted step of the adaptive driver
(ModelTrajectoryImage / ModelTrajectoryDensity, an extension: the reference has no such
product).

TEST INFRASTRUCTURE -- see oracle/__init__.py for who may import this.

``integrate_adaptive`` is ``ionization.integrate_adaptive`` statement for statement, with the
recorder receiving every accepted step (packet, h, the state before it, the Runge-Kutta state)
instead of the loss of the steps that have one.  With the recorder on or off it returns what
``ionization`` returns, bit for bit (tests/test_trace.py).  ``Recorder`` keeps the steps;
``steps`` turns them into midpoints and age-weighted dwells with the product's arithmetic:

    m = (s + s_rk) * 0.5                          per component
    a = (h * T) / ((T - t0) + (t - 0.5 * h))      T = endtime, t0 = X0 time, t = s's time

``bin_image`` puts the midpoints through ``imaging.create_image`` (ModelImage's rules) with the
frac scaled by ``a`` (so the weight is w * a), ``bin_grid`` bins ``frac(m) * a`` by
``ionization.bin_steps`` (np.histogramdd's rule, OUTSIDE beyond the box).
"""
import numpy as np

from . import imaging, ionization
from .deposition import ESCAPED, MOON, REMAINING, SOURCE, SURFACE, VANISHED, Events
from .tracking import bounce, dp_step, moon_xy


def integrate_adaptive(X0, rc, uniforms=None, step0=1000., recorder=None):
    """``ionization.integrate_adaptive`` with a recorder of every accepted step.  ``recorder``:
    None, or called as ``recorder(packet, h, s, s_rk)`` for the accepted steps of each pass: the
    packets (K,), their steps (K,), the states before the steps (K, 8) and the Runge-Kutta
    states (K, 8), before any surface, moon, escape or vanish handling.
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
                recorder(gidx, h[good], cur[good], gn.copy())
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
    """A ``recorder`` for ``integrate_adaptive`` that keeps every accepted step."""

    def __init__(self):
        self.parts = []

    def __call__(self, packet, h, s, s_rk):
        self.parts.append((np.asarray(packet, np.int64), np.asarray(h, np.float64),
                           np.asarray(s, np.float64).reshape(-1, 8),
                           np.asarray(s_rk, np.float64).reshape(-1, 8)))

    def arrays(self):
        """(packet (K,), h (K,), s (K, 8), s_rk (K, 8)) in the order the steps were recorded."""
        if not self.parts:
            return np.zeros(0, np.int64), np.zeros(0), np.zeros((0, 8)), np.zeros((0, 8))
        return tuple(np.concatenate([p[i] for p in self.parts]) for i in range(4))


def steps(rec, t0, endtime):
    """(mid (K, 8), a (K,)) of the recorded steps: the midpoints (s + s_rk) * 0.5 (column 0 is
    the time, unused) and the age-weighted dwells; ``t0`` (N,) the packets' initial times."""
    packet, h, s, s_rk = rec.arrays()
    mid = (s + s_rk) * 0.5
    age0 = endtime - np.asarray(t0, np.float64)[packet]
    a = (h * endtime) / (age0 + (s[:, 0] - 0.5 * h))
    return mid, a


def bin_image(mid, a, **image_kw):
    """(sums (nx, nz), counts (nx, nz)) of the midpoints by ``imaging.create_image`` with the
    frac scaled by the dwell; ``image_kw`` as ``create_image`` takes them."""
    img, cnt, _, _ = imaging.create_image(mid[:, 1], mid[:, 2], mid[:, 3], mid[:, 5],
                                          mid[:, 7] * a, **image_kw)
    return img, cnt.astype(np.int64)


def bin_grid(mid, a, lo, hi, dims):
    """(sums (nx, ny, nz), counts, outside sum, outside count) of ``frac(m) * a``."""
    return ionization.bin_steps(mid[:, 7] * a, mid[:, 1:4], lo, hi, dims)
