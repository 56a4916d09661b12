#!/usr/bin/env python
"""Cost of the adaptive driver's ion-production sink (K2i: k_ionize_adaptive).

Alternating in one process, `reps` times each, on the same device-drawn packets:
  (a) configs[1] (Na.maxwellian.radpres.input, perfect sticking): nx_integrate_adaptive against
      nx_integrate_adaptive_ionize;
  (b) Na.bounce.adaptive.input: nx_integrate_adaptive_bounce against
      nx_integrate_adaptive_ionize.
The grid is ModelIonization's default (100^3 cells over 8 R_p).  Kernel ms are the CUDA events
the C ABI records around its launches (the longest-first order included).  Also prints the
recorded steps per packet, the share of the loss that falls OUTSIDE the grid, and the GPU's name
and power limit.

The midpoint rule puts a step's whole loss in the cell of its chord's midpoint.  To show whether
that is adequate at the default grid, the oracle re-runs `nsample` packets of each workload on
the host and reports the share of the recorded loss whose step starts and ends in different
cells (or leaves the box).  Writes the numbers as JSON when a path is given.

    python tools/diag_ionization.py [npackets] [reps] [report.json] [nsample]
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

from common import oracle_constants, workload                            # noqa: E402
from nexoclom_b200.engine import Engine                                  # noqa: E402
from nexoclom_b200.runsetup import RunSetup                              # noqa: E402

LO, HI, DIMS = (-4.0,) * 3, (4.0,) * 3, (100,) * 3


def gpu_identity():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm',
                              '--format=csv,noheader'], capture_output=True, text=True, timeout=30)
        return out.stdout.strip().splitlines()[0]
    except Exception as e:                                              # noqa: BLE001
        return f'nvidia-smi unavailable ({e})'


def chord_share(setup, nsample, seed=7):
    """Share of the oracle's recorded loss (sum of |loss|) from steps whose chord starts and
    ends in different cells of the default grid, over `nsample` packets.  The chord's ends
    come from the Runge-Kutta step itself: the oracle driver's dp_step is wrapped, and each
    recorded step is found among the pass's rows by its (loss, midpoint), which the oracle
    computes from the same two rows."""
    from oracle import adaptive_bounce, initial_state, ionization
    X0 = initial_state.draw_x0(setup, nsample, seed)[:, :8]
    rows = {}
    inner = ionization.dp_step

    def dp_step(cur, h, rc, want_error=False):
        nxt, delta = inner(cur, h, rc, want_error=want_error)
        rows['a'], rows['b'] = cur[:, 1:4].copy(), nxt[:, 1:4].copy()
        rows['loss'] = cur[:, 7] - nxt[:, 7]
        return nxt, delta

    spans = {'all': 0.0, 'multi': 0.0}

    def recorder(packet, loss, mid):
        a, b, dl = rows['a'], rows['b'], rows['loss']
        m_all = (a + b) * 0.5
        j = 0
        ends = []
        for k in range(len(loss)):                  # recorded steps: an ordered subsequence
            while not (dl[j] == loss[k] and np.array_equal(m_all[j], mid[k])):
                j += 1
            ends.append(j)
            j += 1
        ends = np.array(ends, np.int64)
        ca = ionization.cell(a[ends], LO, HI, DIMS)
        cb = ionization.cell(b[ends], LO, HI, DIMS)
        w = np.abs(loss)
        spans['all'] += w.sum()
        spans['multi'] += w[(ca != cb) | (ca < 0)].sum()

    ionization.dp_step = dp_step
    try:
        ionization.integrate_adaptive(X0, oracle_constants(setup),
                                      adaptive_bounce.bounce_uniforms(seed, 0), recorder=recorder)
    finally:
        ionization.dp_step = inner
    return spans['multi'] / spans['all'] if spans['all'] > 0 else float('nan')


def main():
    n = int(float(sys.argv[1])) if len(sys.argv) > 1 else 10_000_000
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 5
    dest = sys.argv[3] if len(sys.argv) > 3 else None
    nsample = int(float(sys.argv[4])) if len(sys.argv) > 4 else 2000
    ident = gpu_identity()
    print('GPU (name, power limit, max SM clock):', ident)
    eng = Engine(0)
    setups = {'configs[1]': RunSetup(workload('Na.maxwellian.radpres.input')),
              'bounce': RunSetup(workload('Na.bounce.adaptive.input'))}

    def run(case, sink):
        setup = setups[case]
        setup.upload(eng)
        eng.init_state(setup.source_params(eng), 7, 0, n)
        got = None
        if sink:
            eng.ionize_begin(LO, HI, DIMS)
            try:
                att, acc, bnc = eng.integrate_adaptive_ionize(7, 0)
                got = eng.ionize_fetch(DIMS)
            finally:
                eng.ionize_end()
        elif case == 'configs[1]':
            (att, acc), bnc = eng.integrate_adaptive(), 0
        else:
            att, acc, bnc = eng.integrate_adaptive_bounce(7, 0)
        return eng.last_kernel_ms(), att, acc, got

    for case in setups:                                   # warm-up: modules, tables
        run(case, False)
        run(case, True)
    res = {c: {'plain': [], 'ion': []} for c in setups}
    info = {}
    for _ in range(reps):
        for case in setups:
            for sink in (False, True):
                ms, att, acc, got = run(case, sink)
                res[case]['ion' if sink else 'plain'].append(ms)
                if sink:
                    grid, cnt, out, out_n = got
                    steps = int(cnt.sum()) + out_n
                    total = float(grid.sum()) + out
                    info[case] = {'attempted': att, 'accepted': acc, 'recorded_steps': steps,
                                  'recorded_steps_per_packet': steps / n,
                                  'recorded_per_accepted_step': steps / acc,
                                  'lost_frac_per_packet': total / n,
                                  'outside_share': out / total if total else float('nan'),
                                  'outside_steps': out_n}
    report = {'gpu': ident, 'npackets': n, 'reps': reps, 'grid': [LO, HI, DIMS]}
    for case in setups:
        p, s = np.array(res[case]['plain']), np.array(res[case]['ion'])
        d = {'plain_ms': p.tolist(), 'ion_ms': s.tolist(),
             'plain_median_ms': float(np.median(p)), 'ion_median_ms': float(np.median(s)),
             'overhead': float(np.median(s) / np.median(p) - 1), **info[case]}
        report[case] = d
        print(f"{case}: plain {d['plain_median_ms']:.2f} ms  ion {d['ion_median_ms']:.2f} ms  "
              f"overhead {100 * d['overhead']:+.1f}%  (plain {np.round(p, 2).tolist()}, "
              f"ion {np.round(s, 2).tolist()})  recorded steps/packet "
              f"{d['recorded_steps_per_packet']:.1f}  outside share {d['outside_share']:.4f}")
    for case, setup in setups.items():
        share = chord_share(setup, nsample)
        report[case]['multi_cell_loss_share'] = share
        report[case]['multi_cell_sample'] = nsample
        print(f'{case}: share of the loss from steps whose chord spans > 1 cell '
              f'({nsample} oracle packets): {share:.4f}')
    if dest:
        os.makedirs(os.path.dirname(os.path.abspath(dest)), exist_ok=True)
        with open(dest, 'w') as f:
            json.dump(report, f, indent=1)


if __name__ == '__main__':
    main()
