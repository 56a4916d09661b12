#!/usr/bin/env python
"""Cost of the adaptive driver's deposition sink (K2 / K2b built with SINK).

Alternating in one process, `reps` times each:
  (a) K2 on configs[1] (Na.maxwellian.radpres.input, perfect sticking): nx_integrate_adaptive
      against nx_integrate_adaptive_deposit on the same device-drawn packets;
  (b) K2b on Na.bounce.adaptive.input: nx_integrate_adaptive_bounce against
      nx_integrate_adaptive_deposit.
Kernel ms are the CUDA events the C ABI records around its launches (the longest-first order
included).  Also prints the events per packet and per attempted step, the GPU's name and power
limit; writes the numbers as JSON when a path is given.

    python tools/diag_deposition.py [npackets] [reps] [report.json]
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
from nexoclom_b200.engine import Engine                                  # noqa: E402
from nexoclom_b200.runsetup import RunSetup                              # noqa: E402


def gpu_identity():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm',
                              '--format=csv,noheader'], capture_output=True, text=True, timeout=30)
        return out.stdout.strip().splitlines()[0]
    except Exception as e:                                              # noqa: BLE001
        return f'nvidia-smi unavailable ({e})'


def main():
    n = int(float(sys.argv[1])) if len(sys.argv) > 1 else 10_000_000
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 5
    dest = sys.argv[3] if len(sys.argv) > 3 else None
    ident = gpu_identity()
    print('GPU (name, power limit, max SM clock):', ident)
    eng = Engine(0)
    setups = {'k2': RunSetup(workload('Na.maxwellian.radpres.input')),
              'k2b': RunSetup(workload('Na.bounce.adaptive.input'))}

    def run(case, sink):
        setup = setups[case]
        setup.upload(eng)
        eng.init_state(setup.source_params(eng), 7, 0, n)
        events = None
        if sink:
            eng.deposit_begin(180, 90)
            try:
                att, acc, bnc = eng.integrate_adaptive_deposit(7, 0)
                events = eng.deposit_fetch(180, 90)[3]
            finally:
                eng.deposit_end()
        elif case == 'k2':
            (att, acc), bnc = eng.integrate_adaptive(), 0
        else:
            att, acc, bnc = eng.integrate_adaptive_bounce(7, 0)
        return eng.last_kernel_ms(), att, bnc, events

    for case in setups:                                   # warm-up: modules, tables
        run(case, False)
        run(case, True)
    res = {c: {'plain': [], 'sink': []} for c in setups}
    info = {}
    for _ in range(reps):
        for case in setups:
            for sink in (False, True):
                ms, att, bnc, ev = run(case, sink)
                res[case]['sink' if sink else 'plain'].append(ms)
                if sink:
                    fates = int(ev[:4].sum())
                    info[case] = {'attempted': att, 'bounces': bnc,
                                  'events': fates, 'events_per_packet': fates / n,
                                  'events_per_attempted_step': fates / att}
    report = {'gpu': ident, 'npackets': n, 'reps': reps}
    for case in setups:
        p, s = np.array(res[case]['plain']), np.array(res[case]['sink'])
        d = {'plain_ms': p.tolist(), 'sink_ms': s.tolist(),
             'plain_median_ms': float(np.median(p)), 'sink_median_ms': float(np.median(s)),
             'overhead': float(np.median(s) / np.median(p) - 1), **info[case]}
        report[case] = d
        print(f"{case}: plain {d['plain_median_ms']:.2f} ms  sink {d['sink_median_ms']:.2f} ms  "
              f"overhead {100 * d['overhead']:+.1f}%  (plain {np.round(p, 2).tolist()}, "
              f"sink {np.round(s, 2).tolist()})  events/packet {d['events_per_packet']:.3f}  "
              f"events/attempted step {d['events_per_attempted_step']:.4f}")
    if dest:
        os.makedirs(os.path.dirname(os.path.abspath(dest)), exist_ok=True)
        with open(dest, 'w') as f:
            json.dump(report, f, indent=1)


if __name__ == '__main__':
    main()
