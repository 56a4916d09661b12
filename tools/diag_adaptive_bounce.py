#!/usr/bin/env python
"""Timing of the adaptive driver with surface bounce (K2 built with BOUNCE) against K2 and K3.

  (a) Na.bounce.adaptive.input, device-drawn packets, nx_integrate_adaptive_bounce with the
      longest-first order (option order_packets = 3, the default) and without it (0);
  (b) K2 on configs[1] (Na.maxwellian.radpres.input, perfect sticking), nx_integrate_adaptive;
  (c) K3 on Na.bounce.input (30 s step, the same physics as (a)), nx_integrate_constant.

Per case, `reps` repetitions alternating the cases: kernel ms from the CUDA events the C ABI
records around its launches (the cost-order kernels included when ordering is on),
attempted steps, packet-steps/s (attempted / kernel time), bounces per attempted step and the
longest packet's attempted steps, which bounds the tail: its steps run one after another on
one lane.  Prints the GPU's name and power limit with the numbers; writes them as JSON too
when a path is given.

    python tools/diag_adaptive_bounce.py [npackets] [reps] [report.json]
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
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
    dest = sys.argv[3] if len(sys.argv) > 3 else None
    ident = gpu_identity()
    print('GPU (name, power limit, max SM clock):', ident)
    eng = Engine(0)
    setups = {'bounce': RunSetup(workload('Na.bounce.adaptive.input')),
              'k2': RunSetup(workload('Na.maxwellian.radpres.input')),
              'k3': RunSetup(workload('Na.bounce.input'))}

    def run(case, order=3):
        setup = setups[case]
        setup.upload(eng)
        eng.init_state(setup.source_params(eng), 7, 0, n)
        eng.set_option('order_packets', order)
        try:
            if case == 'k3':
                _, nsteps, steps = eng.integrate_constant(seed=7)
                return dict(ms=eng.last_kernel_ms(), attempted=steps, bounces=None, longest=nsteps - 1)
            if case == 'k2':
                att, acc = eng.integrate_adaptive()
                bnc = None
            else:
                att, acc, bnc = eng.integrate_adaptive_bounce(7, 0)
            ms = eng.last_kernel_ms()
            a, _ = eng.export_stats()
            return dict(ms=ms, attempted=att, accepted=acc, bounces=bnc, longest=int(a.max()),
                        p99=float(np.percentile(a, 99)), median=float(np.median(a)))
        finally:
            eng.set_option('order_packets', 3)

    cases = [('bounce', 3), ('bounce', 0), ('k2', 3), ('k3', 3)]
    for case, order in cases:                                          # warm-up (module load)
        setups[case].upload(eng)
    results = {f'{c}/order{o}': [] for c, o in cases}
    for r in range(reps + 1):
        for case, order in cases:
            res = run(case, order)
            if r > 0:                                                  # the first pass warms up
                results[f'{case}/order{order}'].append(res)
    report = {'gpu': ident, 'npackets': n, 'reps': reps, 'cases': {}}
    for key, runs in results.items():
        ms = np.array([x['ms'] for x in runs])
        att = runs[0]['attempted']
        rate = att / (np.median(ms) * 1e-3)
        row = dict(ms_median=float(np.median(ms)), ms_min=float(ms.min()), ms_max=float(ms.max()),
                   attempted=int(att), packet_steps_per_s=float(rate),
                   longest_packet_steps=runs[0]['longest'])
        if runs[0].get('bounces') is not None:
            row['bounces'] = int(runs[0]['bounces'])
            row['bounces_per_attempted_step'] = runs[0]['bounces'] / att
        for k in ('median', 'p99', 'accepted'):
            if k in runs[0]:
                row[k] = runs[0][k]
        report['cases'][key] = row
        print(f'{key:16s} kernel {row["ms_median"]:9.2f} ms (min {row["ms_min"]:.2f}, max '
              f'{row["ms_max"]:.2f})  attempted {att:.4g}  {rate:.3g} packet-steps/s  '
              f'longest {row["longest_packet_steps"]}'
              + (f'  bounces/attempted {row["bounces_per_attempted_step"]:.4f}'
                 if 'bounces' in row else ''))
    eng.close()
    if dest:
        with open(dest, 'w') as f:
            json.dump(report, f, indent=1)


if __name__ == '__main__':
    main()
