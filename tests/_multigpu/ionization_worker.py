"""One rank of a sharded ion production map (launched by torchrun from
tests/test_multigpu_ionization.py, or with WORLD_SIZE unset for the single-process answer).

    ionization_worker.py <npackets> <seed> <out.npz>

Input.run on Na.bounce.adaptive.input -> ModelIonization; rank 0 writes the product to
<out.npz>."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, 'tests'))


def main():
    npackets, seed, dest = int(float(sys.argv[1])), int(sys.argv[2]), sys.argv[3]
    from common import workload
    from nexoclom_b200 import ModelIonization, sharding
    rank, world = sharding.init()
    inputs = workload('Na.bounce.adaptive.input')
    inputs.delete_files()
    inputs.run(npackets, seed=seed)
    _, _, mine, _ = inputs.search()
    res = ModelIonization(inputs, {'dims': '60,50,40', 'width': '10,10,8'})
    if rank == 0:
        np.savez(dest, packet_grid=res.packet_grid, ionized=res.ionized, outside=res.outside,
                 outside_count=res.outside_count, totalsource=res.totalsource,
                 bounces=res.bounces, world=world, mine=mine)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
