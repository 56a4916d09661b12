"""One rank of a sharded LOSSpectrum run (launched by torchrun from
tests/test_multigpu_spectrum.py, or with WORLD_SIZE unset for the single-process answer).

    spectrum_worker.py <workload> <npackets> <seed> <out.npz>

Input.run -> LOSSpectrum; rank 0 writes the products to <out.npz>."""
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
    from worker import synthetic_scdata
    from nexoclom_b200 import LOSSpectrum, sharding
    from nexoclom_b200.units import Quantity
    rank, world = sharding.init()
    inputs = workload(name)
    inputs.delete_files()
    inputs.run(npackets, seed=seed)
    _, files, mine, _ = inputs.search()
    sc = synthetic_scdata(300, inputs.options.species)
    res = LOSSpectrum(sc, inputs, (-10.0, 10.0, 80), dphi=Quantity(2.0, 'deg'))
    if rank == 0:
        np.savez(dest, spectrum=res.spectrum.values, npackets=res.npackets.values,
                 outside=res.outside.values, npackets_outside=res.npackets_outside.values,
                 totalsource=res.totalsource, atoms_per_packet=res.atoms_per_packet,
                 world=world, mine=mine)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
