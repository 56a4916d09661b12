"""One rank of a sharded deposition (launched by torchrun from tests/test_multigpu_deposition.py,
or with WORLD_SIZE unset for the single-process answer).

    deposition_worker.py <npackets> <seed> <out.npz>

Input.run on Na.bounce.adaptive.input -> ModelDeposition; rank 0 writes the product to
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
    from nexoclom_b200 import ModelDeposition, sharding
    rank, world = sharding.init()
    inputs = workload('Na.bounce.adaptive.input')
    inputs.delete_files()
    inputs.run(npackets, seed=seed)
    _, _, mine, _ = inputs.search()
    res = ModelDeposition(inputs, {'nlonbins': 72, 'nlatbins': 36})
    if rank == 0:
        np.savez(dest, packet_map=res.packet_map, deposited=res.deposited,
                 counts=res.event_counts.values, buckets=res.buckets.values,
                 totalsource=res.totalsource, world=world, mine=mine)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
