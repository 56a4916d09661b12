"""One rank of a sharded trajectory density grid and image (launched by torchrun from
tests/test_multigpu_trace.py, or with WORLD_SIZE unset for the single-process answer).

    trace_worker.py <npackets> <seed> <out.npz>

Input.run on Na.bounce.adaptive.input -> ModelTrajectoryDensity and ModelTrajectoryImage; rank 0
writes the products to <out.npz>."""
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
    from nexoclom_b200 import ModelTrajectoryDensity, ModelTrajectoryImage, sharding
    rank, world = sharding.init()
    inputs = workload('Na.bounce.adaptive.input')
    inputs.delete_files()
    inputs.run(npackets, seed=seed)
    _, _, mine, _ = inputs.search()
    res = ModelTrajectoryDensity(inputs, {'dims': '60,50,40', 'width': '10,10,8'})
    img = ModelTrajectoryImage(inputs, {'quantity': 'radiance', 'dims': '60,50', 'width': '10,8'})
    if rank == 0:
        np.savez(dest, step_grid=res.step_grid, dwell=res.dwell, outside=res.outside,
                 outside_count=res.outside_count, totalsource=res.totalsource,
                 bounces=res.bounces, world=world, mine=mine, image=img.image,
                 step_image=img.step_image, image_totalsource=img.totalsource)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
