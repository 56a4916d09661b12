#!/usr/bin/env python
"""Cost and noise of the adaptive driver's trajectory sink (K2t: k_trace_adaptive).

Cost: alternating in one process, `reps` times each, on the same device-drawn packets:
  (a) configs[1] (Na.maxwellian.radpres.input, perfect sticking): nx_integrate_adaptive against
      nx_integrate_adaptive_trace with an 800 x 800 radiance image, and with a 100^3 grid over
      8 R_p;
  (b) Na.bounce.adaptive.input: nx_integrate_adaptive_bounce against the same two traces.
Kernel ms are the CUDA events the C ABI records around its launches (the longest-first order
included); medians are reported.  Also prints the accepted steps per packet and the GPU's name
and power limit, read in the same process.

Noise: per-pixel relative standard deviation over `nseed` seeds of `npix_packets` packets of
configs[1], on a 40 x 40 column image over 8 R_p: the snapshot (ModelImage's estimator, the
final rows binned by K4) against the trajectory image (ModelTrajectoryImage's estimator), both
scaled to the same units.  Reported as the median over pixels that every seed of the snapshot
hits, and per radial band.

Caveats of the midpoint rule, from the oracle on the host (`nsample` packets of each workload):
the share of the age-weighted dwell, sum of frac(m) a, from steps whose chord starts and ends
in different cells of the 100^3 grid (or leaves the box), which the product puts wholly in the
midpoint's cell; and the share from steps that end inside the planet, which count their full h.

    python tools/diag_trace.py [npackets] [reps] [report.json] [nseed] [npix_packets] [nsample]
"""
import json
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, 'tests'))
import numpy as np                                                       # noqa: E402

from common import workload                                              # noqa: E402
from nexoclom_b200._lib import ImageParams                               # noqa: E402
from nexoclom_b200.engine import Engine                                  # noqa: E402
from nexoclom_b200.ModelImage import image_rotation                      # noqa: E402
from nexoclom_b200.runsetup import RunSetup                              # noqa: E402

GRID = ((-4.0,) * 3, (4.0,) * 3, (100,) * 3)


def gpu_identity():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm',
                              '--format=csv,noheader'], capture_output=True, text=True, timeout=30)
        return out.stdout.strip().splitlines()[0]
    except Exception as e:                                              # noqa: BLE001
        return f'nvidia-smi unavailable ({e})'


def image_params(setup, quantity, dims, half=4.0):
    M = np.asarray(image_rotation(0.0, np.pi / 2))
    ip = ImageParams()
    for k in range(9):
        ip.M[k] = float(M.flat[k])
    ip.x0, ip.x1, ip.z0, ip.z1 = -half, half, -half, half
    ip.nx = ip.nz = dims
    rcm = setup.radius_km * 1e5
    ip.apix = (2 * half / dims * rcm) ** 2
    ip.vrplanet = setup.vrplanet
    ip.quantity = 1 if quantity == 'radiance' else 0
    ip.round_f32 = ip.skip_dead = 0
    return ip


def cost(eng, wl, n, reps):
    setup = RunSetup(workload(wl))
    setup.upload(eng)
    eng.upload_gtables(setup.gtables([5891, 5897]))
    bounce = not (setup.params.sticktype == 0 and setup.params.stickcoef == 1.0)
    eng.init_state(setup.source_params(eng), 3, 0, n)
    X0 = eng.export_x0()[:8].T.copy()
    ip = image_params(setup, 'radiance', 800)
    runs = {
        'plain': lambda: (eng.integrate_adaptive_bounce(1, 0) if bounce
                          else eng.integrate_adaptive()),
        'image800': None, 'grid100': None}

    def traced(ipar, grid):
        eng.trace_begin(ipar, grid)
        try:
            return eng.integrate_adaptive_trace(1, 0)
        finally:
            eng.trace_end()
    runs['image800'] = lambda: traced(ip, None)
    runs['grid100'] = lambda: traced(None, GRID)
    ms = {k: [] for k in runs}
    steps = {}
    for r in range(reps + 1):                      # the first round warms every path up
        for k, f in runs.items():
            eng.import_state(X0)
            tot = f()
            if r:
                ms[k].append(eng.last_kernel_ms())
            steps[k] = tot
    med = {k: float(np.median(v)) for k, v in ms.items()}
    assert steps['image800'][:2] == steps['grid100'][:2] == tuple(steps['plain'][:2])
    return {'workload': wl, 'packets': n, 'median_ms': med, 'all_ms': ms,
            'accepted_per_packet': steps['plain'][1] / n,
            'ratio_image800': med['image800'] / med['plain'],
            'ratio_grid100': med['grid100'] / med['plain']}


def noise(eng, nseed, n):
    """Per-pixel RSD over seeds: snapshot against trajectory, same units (sum of w over the
    seeds' packets, the trajectory's divided by T)."""
    setup = RunSetup(workload('Na.maxwellian.radpres.input'))
    setup.upload(eng)
    T = float(setup.params.endtime)
    ip = image_params(setup, 'column', 40)
    snap, traj = [], []
    for seed in range(nseed):
        eng.init_state(setup.source_params(eng), 100 + seed, 0, n)
        X0 = eng.export_x0()[:8].T.copy()
        eng.integrate_adaptive()
        table = eng.compact_state(skip_dead=True, round_f32=True)
        eng.bind_packets(table)
        img, _ = eng.image_accumulate(ip, n=table.n)
        eng.bind_packets(None)
        table.free()
        snap.append(np.array(img))
        eng.import_state(X0)
        eng.trace_begin(ip, None)
        try:
            eng.integrate_adaptive_trace(0, 0)
            timg = eng.trace_fetch()[0]
        finally:
            eng.trace_end()
        traj.append(np.array(timg) / T)
    snap, traj = np.array(snap), np.array(traj)
    hit = np.all(snap > 0, axis=0)
    rs = snap.std(axis=0, ddof=1) / snap.mean(axis=0)
    rt = traj.std(axis=0, ddof=1) / traj.mean(axis=0)
    c = (np.arange(40) + 0.5) * 0.2 - 4.0
    b = np.sqrt(c[:, None] ** 2 + c[None, :] ** 2)
    bands = {}
    for lo, hi in ((1.0, 1.5), (1.5, 2.5), (2.5, 4.0)):
        m = hit & (b >= lo) & (b < hi)
        if m.any():
            bands[f'[{lo}, {hi})'] = {'pixels': int(m.sum()),
                                      'snapshot_rsd': float(np.median(rs[m])),
                                      'trajectory_rsd': float(np.median(rt[m]))}
    mean_ratio = float(np.median(traj.mean(axis=0)[hit] / snap.mean(axis=0)[hit]))
    return {'seeds': nseed, 'packets': n, 'pixels_hit_by_every_seed': int(hit.sum()),
            'snapshot_rsd_median': float(np.median(rs[hit])),
            'trajectory_rsd_median': float(np.median(rt[hit])),
            'trajectory_over_snapshot_median': mean_ratio, 'bands': bands}


def midpoint_caveats(wl, nsample, seed=7):
    from common import oracle_constants
    from oracle import adaptive_bounce, initial_state, ionization, trace
    setup = RunSetup(workload(wl))
    X0 = initial_state.draw_x0(setup, nsample, seed)[:, :8]
    rec = trace.Recorder()
    trace.integrate_adaptive(X0, oracle_constants(setup), adaptive_bounce.bounce_uniforms(1, 0),
                             recorder=rec)
    _, _, s, s_rk = rec.arrays()
    mid, a = trace.steps(rec, X0[:, 0], float(setup.params.endtime))
    d = mid[:, 7] * a
    c0 = ionization.cell(s[:, 1:4], *GRID)
    c1 = ionization.cell(s_rk[:, 1:4], *GRID)
    inside = (s_rk[:, 1:4] ** 2).sum(axis=1) < 1.0
    return {'workload': wl, 'packets': nsample, 'steps': int(len(d)),
            'dwell_share_chord_crosses_cells': float(d[(c0 != c1) | (c0 < 0)].sum() / d.sum()),
            'dwell_share_step_ends_inside_planet': float(d[inside].sum() / d.sum())}


def main():
    n = int(float(sys.argv[1])) if len(sys.argv) > 1 else 10_000_000
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 5
    dest = sys.argv[3] if len(sys.argv) > 3 else None
    nseed = int(sys.argv[4]) if len(sys.argv) > 4 else 8
    npix = int(float(sys.argv[5])) if len(sys.argv) > 5 else 1_000_000
    nsample = int(float(sys.argv[6])) if len(sys.argv) > 6 else 2000
    if n == 0:                       # the oracle part alone, no device
        print(json.dumps([midpoint_caveats(wl, nsample) for wl in
                          ('Na.maxwellian.radpres.input', 'Na.bounce.adaptive.input')], indent=1))
        return
    eng = Engine(0)
    report = {'gpu': gpu_identity()}
    report['cost'] = [cost(eng, wl, n, reps) for wl in ('Na.maxwellian.radpres.input',
                                                         'Na.bounce.adaptive.input')]
    report['noise'] = noise(eng, nseed, npix)
    report['gpu_after'] = gpu_identity()
    eng.close()
    text = json.dumps(report, indent=1)
    print(text)
    if dest:
        os.makedirs(os.path.dirname(os.path.abspath(dest)), exist_ok=True)
        with open(dest, 'w') as f:
            f.write(text)


if __name__ == '__main__':
    main()
