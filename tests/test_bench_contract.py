"""bench.py contract: the reference arm runs anywhere (it is the CPU leg) and prints one JSON
line with the keys the driver reads; the GPU arm refuses to run without a CUDA device."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(REPO, 'bench.py'), '--impl', 'reference',
                          '--steps', '1', '--warmup', '0', '--ref-packets', '150'],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    assert len(out.stdout.splitlines()) == 1          # stdout carries the JSON line, nothing else
    line = json.loads(out.stdout)
    assert line['impl'] == 'reference' and line['metric'] == 'packet-steps/s (FP64)'
    assert line['unit'] == 'packet-steps/s' and line['higher_is_better'] is True
    assert line['value'] > 0 and line['e2e']['value'] == line['value']
    assert line['e2e']['h2d_bytes_per_step'] == 0 and line['e2e']['d2h_bytes_per_step'] == 0
    cb = line['cpu_baseline']
    assert cb['kind'] == 'port' and cb['cores'] >= 1 and 'packets' in cb['sample']
    assert 'workload' in line['config']


def test_reference_arm_is_silent_on_other_ranks():
    env = dict(os.environ, RANK='1', WORLD_SIZE='2')
    out = subprocess.run([sys.executable, os.path.join(REPO, 'bench.py'), '--impl', 'reference',
                          '--steps', '1', '--warmup', '0'], capture_output=True, text=True,
                         timeout=120, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ''


def test_stdout_is_kept_for_the_json_line():
    """Whatever a library prints to fd 1 while the bench runs (NCCL's version banner does) must
    not end up on stdout."""
    code = ("import os, sys; sys.path.insert(0, %r); import bench; bench.claim_stdout(); "
            "os.write(1, b'library banner\\n'); print('python print'); bench.emit({'a': 1})" % REPO)
    out = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr[-1000:]
    assert out.stdout == '{"a": 1}\n'
    assert 'library banner' in out.stderr and 'python print' in out.stderr


@pytest.mark.gpu
def test_dump_outputs_is_the_last_step_and_repeatable(tmp_path):
    """--dump-outputs: the products of the last timed step, the same whatever the number of
    timed steps (every step integrates the same resident initial state)."""
    small = ['--packets', '20000', '--no-e2e', '--no-los', '--no-k3', '--no-k14', '--no-cpu']
    dumps = []
    for steps in (1, 3):
        dest = tmp_path / f'steps{steps}'
        out = subprocess.run([sys.executable, os.path.join(REPO, 'bench.py'), '--steps', str(steps),
                              '--warmup', '1', '--dump-outputs', str(dest)] + small,
                             capture_output=True, text=True, timeout=900)
        assert out.returncode == 0, out.stderr[-2000:]
        assert json.loads(out.stdout)['steps'] == steps
        names = sorted(p.name for p in dest.iterdir())
        assert names == sorted(n + '.npy' for n in (
            'image', 'packet_counts', 'step_totals', 'packet_ids', 'final_state',
            'attempted_steps', 'accepted_steps'))
        dumps.append({p.stem: np.load(p) for p in dest.iterdir()})
    one, three = dumps
    for name, a in one.items():
        assert a.dtype == np.float64, name
    assert one['final_state'].shape == (20000, 8) and one['packet_counts'].sum() > 0
    for name in ('packet_counts', 'step_totals', 'packet_ids', 'final_state', 'attempted_steps',
                 'accepted_steps'):
        assert np.array_equal(one[name], three[name]), name
    assert one['step_totals'][0] == one['attempted_steps'].sum()
    nz = one['image'] > 0
    assert np.array_equal(nz, three['image'] > 0)
    assert np.max(np.abs(three['image'][nz] - one['image'][nz]) / one['image'][nz]) < 1e-12


def test_gpu_arm_needs_a_gpu():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES='')           # no device, on any host
    out = subprocess.run([sys.executable, os.path.join(REPO, 'bench.py'), '--steps', '1',
                          '--warmup', '0'], capture_output=True, text=True, timeout=300, env=env)
    assert out.returncode != 0 and 'no CPU fallback' in (out.stderr + out.stdout)
