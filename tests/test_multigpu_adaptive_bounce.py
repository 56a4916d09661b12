"""Sharded adaptive runs with surface bounce on real GPUs: N ranks under torchrun, each
integrating its slice of the global packet ids, give the single-process run exactly (the bounce
deviates are keyed by the global packet id).  Needs >= 2 GPUs."""
import os
import subprocess
import sys

import numpy as np
import pytest

from common import REPO

WORKER = os.path.join(REPO, 'tests', '_multigpu', 'adaptive_bounce_worker.py')


def _gpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


def _run(world, npackets, seed, dest):
    env = dict(os.environ)
    env.pop('NEXOCLOM_B200_SAVEPATH', None)
    args = [str(npackets), str(seed), dest]
    if world == 1:
        cmd = [sys.executable, WORKER] + args
    else:
        port = 29900 + os.getpid() % 300
        cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1',
               f'--nproc-per-node={world}', '--master-addr', '127.0.0.1', '--master-port',
               str(port), WORKER] + args
    res = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stderr[-4000:]
    return np.load(dest)


@pytest.mark.gpu
def test_sharded_adaptive_bounce_equals_single_process(tmp_path):
    world = min(_gpus(), 8)
    if world < 2:
        pytest.skip('needs at least 2 GPUs')
    npackets = 400_000
    one = _run(1, npackets, 4, str(tmp_path / 'one.npz'))
    many = _run(world, npackets, 4, str(tmp_path / 'many.npz'))
    assert int(many['world']) == world and int(one['world']) == 1
    assert int(many['mine']) < npackets                    # rank 0 ran only its share
    assert np.array_equal(many['totals'], one['totals']) and one['totals'][0] > npackets
    assert np.array_equal(many['npackets'], one['npackets'])
    a, b = many['density'], one['density']
    nz = b > 0
    assert np.array_equal(nz, a > 0) and nz.sum() > 1000
    assert np.max(np.abs(a[nz] - b[nz]) / b[nz]) < 1e-12
