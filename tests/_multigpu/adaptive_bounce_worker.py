"""One rank of a sharded adaptive run with surface bounce (launched by torchrun from
tests/test_multigpu_adaptive_bounce.py, or with WORLD_SIZE unset for the single-process answer).

    adaptive_bounce_worker.py <npackets> <seed> <out.npz>

Input.run on Na.bounce.adaptive.input -> ModelDensity; rank 0 writes the products and the
run's bounce and step totals (summed over ranks) to <out.npz>."""
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
    from density_worker import sample_points
    from nexoclom_b200 import ModelDensity, catalogue, sharding
    rank, world = sharding.init()
    inputs = workload('Na.bounce.adaptive.input')
    inputs.delete_files()
    inputs.run(npackets, seed=seed)
    _, files, mine, _ = inputs.search()
    outs = [catalogue.fetch(f) for f in files]
    tot = np.array([sum(o.bounces for o in outs), sum(o.attempted_steps for o in outs),
                    sum(o.accepted_steps for o in outs)], dtype=np.int64)
    if world > 1:
        sharding.allreduce_sum(tot)
    pts, rad = sample_points()
    res = ModelDensity(inputs, pts, rad)
    if rank == 0:
        np.savez(dest, density=res.density.values, npackets=res.npackets.values,
                 totals=tot, world=world, mine=mine)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
