"""Sharded ModelImageCube on real GPUs: N ranks under torchrun, each integrating its slice of
the global packet ids and binning its own rows, combined with one all-reduce == the
single-process product.  Needs >= 2 GPUs."""
import os
import subprocess
import sys

import numpy as np
import pytest

from common import REPO

WORKER = os.path.join(REPO, 'tests', '_multigpu', 'cube_worker.py')


def _gpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


def _run(world, name, npackets, seed, dest):
    env = dict(os.environ)
    env.pop('NEXOCLOM_B200_SAVEPATH', None)
    args = [name, str(npackets), str(seed), dest]
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
def test_sharded_cube_equals_single_process(tmp_path):
    world = min(_gpus(), 8)
    if world < 2:
        pytest.skip('needs at least 2 GPUs')
    name, npackets = 'Na.maxwellian.radpres.input', 400_000
    one = _run(1, name, npackets, 4, str(tmp_path / 'one.npz'))
    many = _run(world, name, npackets, 4, str(tmp_path / 'many.npz'))
    assert int(many['world']) == world and int(one['world']) == 1
    assert int(many['mine']) < npackets                    # rank 0 ran only its share
    assert float(many['totalsource']) == float(one['totalsource'])
    assert float(many['atoms_per_packet']) == float(one['atoms_per_packet'])
    for key in ('packet_cube', 'packet_outside'):                         # counts: exact
        assert np.array_equal(many[key], one[key])
    assert one['packet_cube'].sum() > 1e5
    for key in ('cube', 'outside'):
        a, b = many[key], one[key]
        nz = b > 0
        assert np.array_equal(nz, a > 0)
        assert np.max(np.abs(a[nz] - b[nz]) / b[nz]) < 1e-12
