"""Sharded ion production on real GPUs: N ranks under torchrun, each regenerating its slice of
the global packet ids through the ion-production sink, give the single-process grid (the bounce
deviates are keyed by the global packet id; the ranks are combined with one all-reduce).  Needs
>= 2 GPUs."""
import os
import subprocess
import sys

import numpy as np
import pytest

from common import REPO

WORKER = os.path.join(REPO, 'tests', '_multigpu', 'ionization_worker.py')


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
        port = 29600 + os.getpid() % 300
        cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1',
               f'--nproc-per-node={world}', '--master-addr', '127.0.0.1', '--master-port',
               str(port), WORKER] + args
    res = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stderr[-4000:]
    return np.load(dest)


@pytest.mark.gpu
def test_sharded_ionization_equals_single_process(tmp_path):
    world = min(_gpus(), 8)
    if world < 2:
        pytest.skip('needs at least 2 GPUs')
    npackets = 400_000
    one = _run(1, npackets, 4, str(tmp_path / 'one.npz'))
    many = _run(world, npackets, 4, str(tmp_path / 'many.npz'))
    assert int(many['world']) == world and int(one['world']) == 1
    assert int(many['mine']) < npackets                    # rank 0 ran only its share
    assert np.array_equal(many['packet_grid'], one['packet_grid']) and one['packet_grid'].sum() > 0
    assert int(many['outside_count']) == int(one['outside_count'])
    assert float(many['totalsource']) == float(one['totalsource']) == npackets
    assert abs(float(many['outside']) - float(one['outside'])) <= 1e-12 * npackets
    assert np.allclose(many['ionized'], one['ionized'], rtol=1e-12, atol=1e-12 * npackets)
    assert int(one['bounces']) > 0                         # the bounce build ran
