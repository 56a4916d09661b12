#!/usr/bin/env python
"""LOSSpectrum timing: a Doppler-spectrum call (``nx_los_spectrum``) against the radiance-only
K5 call (``nx_los_accumulate``, grid path) on the same rows and lines of sight.

  (a) 1e5 lines of sight of the MESSENGER-like sweep bench.py times (dphi 1 deg) over 1e7
      Na packets (configs[1] physics), twice: the initial state (every packet live at the
      surface: the dense extreme) and the final state of the adaptive run.  Spectra with 100
      and 1000 bins over -15 .. 15 km/s; the calls alternate with the radiance-only call.
  (b) a 1e4-line track: one orbit of lines of sight that look at the planet's limb, over
      the final state.

Per call: the median of 5 warmed-up CUDA-event times (grid build + candidates + exact test;
``last_kernel_ms``) and of the wall times including the host preparation and copies.  Every
spectrum's columns are checked against the radiance-only call (counts exactly, sums to
1e-12).  Prints the GPU's name, power limit and max SM clock with the numbers; writes them as
JSON too when a path is given.

    python tools/diag_spectrum.py [npackets] [report.json]
"""
import json
import os
import subprocess
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, 'tests'))
import numpy as np                                                       # noqa: E402

from bench import synthetic_los                                          # noqa: E402
from common import workload                                              # noqa: E402
from nexoclom_b200._lib import LosParams                                 # noqa: E402
from nexoclom_b200.engine import Engine                                  # noqa: E402
from nexoclom_b200.runsetup import RunSetup                              # noqa: E402

REPS = 5


def gpu_identity():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm',
                              '--format=csv,noheader'], capture_output=True, text=True, timeout=30)
        return out.stdout.strip().splitlines()[0]
    except Exception as e:                                              # noqa: BLE001
        return f'nvidia-smi unavailable ({e})'


def limb_track(nlos):
    """One polar orbit (1.2 - 4 R_p) whose boresight grazes the limb at 1.05 - 1.5 R_p."""
    th = np.linspace(0, 2 * np.pi, nlos, endpoint=False)
    rr = 1.2 + 2.8 * (0.5 + 0.5 * np.cos(th))
    x_sc = np.stack([0.2 * rr * np.cos(th), -0.3 * rr, rr * np.sin(th)])
    x_sc *= rr / np.linalg.norm(x_sc, axis=0)
    up = np.array([1.0, 0.0, 0.0])[:, None] * np.ones(nlos)
    side = np.cross(x_sc.T, up.T).T
    side /= np.linalg.norm(side, axis=0)
    tgt = side * (1.05 + 0.45 * (0.5 + 0.5 * np.sin(7 * th)))
    bore = tgt - x_sc
    bore /= np.linalg.norm(bore, axis=0)
    dplan = np.linalg.norm(x_sc, axis=0)
    ang = np.arccos(-(x_sc * bore).sum(axis=0) / dplan)
    dplan = np.where(ang > np.arcsin(1. / dplan), 1e30, dplan)
    return np.ascontiguousarray(np.concatenate([x_sc, bore])), np.ascontiguousarray(dplan)


def timed(fn, eng):
    t0 = time.perf_counter()
    out = fn()
    return out, eng.last_kernel_ms(), (time.perf_counter() - t0) * 1e3


def compare(eng, table, los, dplan, lp, vscale, bins):
    """Alternating calls: radiance-only, then each spectrum; medians of REPS after a warm-up."""
    eng.bind_packets(table)
    try:
        calls = {'radiance': lambda: eng.los_accumulate(los, dplan, lp, n=table.n)}
        for nb in bins:
            calls[f'spectrum_{nb}'] = (lambda nb=nb: eng.los_spectrum(los, dplan, lp, -15.0, 15.0, nb,
                                                                      vscale, n=table.n))
        times = {k: ([], []) for k in calls}
        out = {}
        for rep in range(REPS + 1):
            for k, fn in calls.items():
                out[k], kern, wall = timed(fn, eng)
                if rep:
                    times[k][0].append(kern)
                    times[k][1].append(wall)
    finally:
        eng.bind_packets(None)
    rad, npk, _ = out['radiance']
    res = {'hits': int(npk.sum())}
    nz = rad > 0
    for k, (kern, wall) in times.items():
        res[k] = dict(kernel_ms=float(np.median(kern)), wall_ms=float(np.median(wall)),
                      kernel_ms_all=[round(v, 3) for v in kern])
        if k != 'radiance':
            spec, cnt = out[k]
            assert np.array_equal(cnt.sum(axis=1), npk), f'{k}: counts differ from the radiance call'
            err = np.abs(spec.sum(axis=1)[nz] - rad[nz]) / rad[nz]
            assert err.max(initial=0.0) <= 1e-12, f'{k}: sums differ ({err.max()})'
            res[k]['inside'] = int(cnt[:, 1:-1].sum())
            res[k]['ratio_kernel'] = res[k]['kernel_ms'] / res['radiance']['kernel_ms']
            res[k]['ratio_wall'] = res[k]['wall_ms'] / res['radiance']['wall_ms']
    return res


def show(label, res):
    r = res['radiance']
    print(f'  {label}: {res["hits"]:.4g} hits; radiance-only {r["kernel_ms"]:.2f} ms kernel, '
          f'{r["wall_ms"]:.2f} ms wall')
    for k, v in res.items():
        if k.startswith('spectrum_'):
            print(f'    {k}: {v["kernel_ms"]:.2f} ms kernel ({v["ratio_kernel"]:.3f}x), '
                  f'{v["wall_ms"]:.2f} ms wall ({v["ratio_wall"]:.3f}x), {v["inside"]:.4g} hits in range')


def main():
    n = int(float(sys.argv[1])) if len(sys.argv) > 1 else 10_000_000
    ident = gpu_identity()
    print('GPU (name, power limit, max SM clock):', ident)
    eng = Engine(0)
    setup = RunSetup(workload('Na.maxwellian.radpres.input'))
    setup.upload(eng)
    eng.upload_gtables(setup.gtables([5891, 5897]))
    sp = setup.source_params(eng)
    lp = LosParams()
    lp.dphi, lp.outeredge = float(np.radians(1.0)), 25.0
    lp.vrplanet, lp.rp_cm = setup.vrplanet, setup.radius_km * 1e5
    lp.quantity, lp.round_f32, lp.skip_dead = 1, 1, 1
    eng.set_option('los_mode', 2)                 # the radiance-only call on the same grid path
    report = {'gpu': ident, 'npackets': n, 'reps': REPS, 'cases': {}}
    los, dplan = synthetic_los(100_000)
    track, tplan = limb_track(10_000)
    for label, integrate in (('initial_state_all_live', False), ('final_state', True)):
        eng.init_state(sp, 1, 0, n)
        if integrate:
            eng.integrate_adaptive(n)
        table = eng.compact_state(skip_dead=True, round_f32=True, n=n)
        print(f'{label}: {n} packets, {table.n} saved rows')
        res = compare(eng, table, los, dplan, lp, setup.radius_km, (100, 1000))
        res['rows'] = table.n
        report['cases'][f'a_1e5_lines_{label}'] = res
        show('(a) 1e5 lines', res)
        if integrate:
            res = compare(eng, table, track, tplan, lp, setup.radius_km, (100, 1000))
            res['rows'] = table.n
            report['cases']['b_1e4_track_final_state'] = res
            show('(b) 1e4-line limb track', res)
        table.free()
    eng.set_option('los_mode', 0)
    eng.close()
    if len(sys.argv) > 2:
        with open(sys.argv[2], 'w') as f:
            json.dump(report, f, indent=1)


if __name__ == '__main__':
    main()
