"""One rank of a sharded ModelDensity run (launched by torchrun from
tests/test_multigpu_density.py, or with WORLD_SIZE unset for the single-process answer).

    density_worker.py <workload> <npackets> <seed> <out.npz>

Input.run -> ModelDensity; rank 0 writes the products to <out.npz>."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, 'tests'))


def sample_points(n=3000):
    g = np.random.default_rng(8)
    u = g.standard_normal((n, 3))
    u /= np.linalg.norm(u, axis=1)[:, None]
    alt = 10 ** g.uniform(-2, np.log10(5), n)
    return u * (1 + alt)[:, None], 0.02 + 0.2 * alt


def main():
    name, npackets, seed, dest = sys.argv[1], int(float(sys.argv[2])), int(sys.argv[3]), sys.argv[4]
    from common import workload
    from nexoclom_b200 import ModelDensity, sharding
    rank, world = sharding.init()
    inputs = workload(name)
    inputs.delete_files()
    inputs.run(npackets, seed=seed)
    _, files, mine, _ = inputs.search()
    pts, rad = sample_points()
    res = ModelDensity(inputs, pts, rad)
    if rank == 0:
        np.savez(dest, density=res.density.values, density_err=res.density_err.values,
                 npackets=res.npackets.values, totalsource=res.totalsource,
                 atoms_per_packet=res.atoms_per_packet, world=world, mine=mine)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
