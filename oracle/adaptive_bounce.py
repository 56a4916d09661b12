"""Oracle: the adaptive driver with surface bounce (an extension: the reference's driver asserts
'Not set up' unless stickcoef == 1, Output.py:309-315, quirk Q6).

TEST INFRASTRUCTURE -- see oracle/__init__.py for who may import this.

``integrate_adaptive`` is ``tracking.integrate_adaptive`` statement for statement, with one
branch added to the accepted steps: a step that ends inside the planet (r2 < 1) goes through
``tracking.bounce`` with r = sqrt(r2) unless the sticking is perfect, and the moon, escape and
vanish tests then see the bounced state, as in ``tracking.integrate_constant``.  For perfect
sticking it equals ``tracking.integrate_adaptive`` bit for bit (tests/test_adaptive_bounce.py),
which pins the restatement to the reference's driver.
"""
import numpy as np

from .initial_state import STREAM_BOUNCE, uniform_pair
from .tracking import bounce, dp_step, moon_xy


def bounce_uniforms(seed, first_id=0):
    """``uniforms(k, packet_indices)`` for ``integrate_adaptive``, reproducing the kernel's
    bounce stream: draws 2k and 2k + 1 of packet first_id + i, k (per packet) = its accepted
    steps counting the one that hit."""
    def fn(k, idx):
        ids = np.asarray(idx, dtype=np.uint64) + np.uint64(first_id)
        k = np.asarray(k, dtype=np.uint64)
        u_alt, u_az = uniform_pair(seed, ids, STREAM_BOUNCE, 2 * k)
        u_prob, _ = uniform_pair(seed, ids, STREAM_BOUNCE, 2 * k + 1)
        return u_alt, u_az, u_prob
    return fn


def integrate_adaptive(X0, rc, uniforms, step0=1000.):
    """Adaptive driver with bounce.  ``uniforms(k, packet_indices) -> (u_alt, u_az, u_prob)``.
    Returns (X (N,8) final, attempted, accepted, bounces (N,) int64)."""
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
            gn = nxt[good]
            r2 = (gn[:, 1]**2 + gn[:, 2]**2) + gn[:, 3]**2
            hit = r2 < 1
            if simple_stick:
                gn[hit, 7] = 0
            elif hit.any():                           # the added branch
                ids = idx[good][hit]
                u_alt, u_az, u_prob = uniforms(accepted[ids] + 1, ids)
                gn[hit] = bounce(rc, gn[hit], np.sqrt(r2[hit]), u_alt, u_az, u_prob)
                bounces[ids] += 1
            for mo in rc.moons:
                mx, my = moon_xy(mo, gn[:, 0])
                dx, dy = gn[:, 1] - mx, gn[:, 2] - my
                gn[dx * dx + dy * dy + gn[:, 3] * gn[:, 3] < mo['radius']**2, 7] = 0
            gn[r2 > rc.outeredge, 7] = 0
            gn[gn[:, 7] < 1e-10, 7] = 0.
            gn[gn[:, 7] == 0, 0] = 0
            X[idx[good]] = gn
            accepted[idx[good]] += 1
        if bad.any():
            old = htried[bad]
            new = safety * old * errmax[bad]**shrink
            assert not np.any(np.isclose(new, old))
            assert np.all(np.isfinite(new)), '\n\tInfinite values of step_size'
            step[idx[bad]] = np.maximum(new, 0.1 * old)

        live = (X[:, 0] > res) & (X[:, 7] > 0.)
    return X, attempted, accepted, bounces
