"""One rank of a sharded ModelImageCube run (launched by torchrun from
tests/test_multigpu_cube.py, or with WORLD_SIZE unset for the single-process answer).

    cube_worker.py <workload> <npackets> <seed> <out.npz>

Input.run -> ModelImageCube; rank 0 writes the products to <out.npz>."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, REPO)
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(REPO, 'tests'))


def main():
    name, npackets, seed, dest = sys.argv[1], int(float(sys.argv[2])), int(sys.argv[3]), sys.argv[4]
    from common import workload
    from nexoclom_b200 import ModelImageCube, sharding
    rank, world = sharding.init()
    inputs = workload(name)
    inputs.delete_files()
    inputs.run(npackets, seed=seed)
    _, files, mine, _ = inputs.search()
    params = {'quantity': 'radiance', 'dims': '160,120', 'width': '10,7.5',
              'subobslongitude': '0.7', 'subobslatitude': '0.3'}
    res = ModelImageCube(inputs, params, (-6.0, 6.0, 60))
    if rank == 0:
        np.savez(dest, cube=res.cube, packet_cube=res.packet_cube, outside=res.outside,
                 packet_outside=res.packet_outside, totalsource=res.totalsource,
                 atoms_per_packet=res.atoms_per_packet, world=world, mine=mine)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
