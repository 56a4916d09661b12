"""``ModelImageCube``: Doppler-resolved image cubes of the modelled exosphere.

The reference has no such product; this one adds a velocity axis to ``ModelImage``.  The rows,
the pixel and the weight of a row are exactly ``ModelImage``'s (the saved rows, float32, frac ==
0 dropped; the same rotation, occultation, sunlight mask and weighting; an occulted or shadowed
row counts with weight 0).  A row's Doppler velocity is

    v = ((vx*M[1,0] + vy*M[1,1]) + vz*M[1,2]) * R_p[km]      [km/s], every op float64 rounded

with ``M = image_rotation()``, which takes the observer direction to (0, -1, 0): v is the
velocity along the line of sight, positive away from the observer (a red shift), in the
planet's rest frame.  The observer's own velocity relative to the planet is left to the user:
shift ``velocity`` by it.  Bins are ``edges = np.linspace(vmin, vmax, nbins + 1)`` with
``np.histogram``'s rule (vmax belongs to the last bin); rows below vmin and above vmax are
kept in ``outside``.  So, per pixel, the sum over the velocity axis plus ``outside`` is
``ModelImage``'s image (to rounding) and packet image (exactly).

The cube is summed on the GPU (``nx_cube_add``) over every output file and, under
torch.distributed, over the ranks with one all-reduce.  As in ``ModelImage`` the source rate is
1e23 atoms/s (``atoms_per_packet = 1e23 / (totalsource / endtime)``).

Attributes: ``edges`` and ``velocity`` (bin centres), km/s; ``cube`` (nx, nz, nbins): R per
km/s (radiance) or atoms cm^-2 per km/s (column); ``packet_cube`` (int64 rows per cell);
``outside`` / ``packet_outside`` (nx, nz, 2): below / above the range, not divided by a width;
``image`` / ``packet_image``: summed over all columns; ``xaxis``, ``zaxis``, ``Apix``,
``atoms_per_packet``, ``sourcerate``, ``totalsource``.
"""
import numpy as np

from . import catalogue
from .engine import get_engine
from .LOSSpectrum import velocity_bins
from .ModelImage import ModelImage
from .ModelResult import ModelResult
from .runsetup import get_setup
from .sharding import combine_ranks, nccl_comm
from .units import Quantity

MAX_CELLS = 2**31          # nx * nz * (nbins + 2) must stay below (32-bit cell index)


def cube_bins(velocity, dims):
    """(vmin, vmax, nbins) from ``velocity = (vmin, vmax, nbins)`` in km/s for an image of
    ``dims = (nx, nz)`` pixels; raises ValueError unless the triple is valid (see
    ``LOSSpectrum.velocity_bins``) and nx * nz * (nbins + 2) < 2**31."""
    vmin, vmax, nbins = velocity_bins(velocity, 0)
    nx, nz = (int(d) for d in dims)
    if nx < 1 or nz < 1:
        raise ValueError(f'image dims must be >= 1, got {nx} x {nz}')
    if nx * nz * (nbins + 2) >= MAX_CELLS:
        raise ValueError(f'{nx} x {nz} pixels x {nbins + 2} columns is more than 2**31 cells')
    return vmin, vmax, nbins


class ModelImageCube(ModelImage):
    def __init__(self, inputs, params, velocity, device=None):
        if not isinstance(params, dict):
            raise ValueError('params must be a dict')
        if params.get('quantity', None) not in ('column', 'radiance'):
            raise ValueError("ModelImageCube computes quantity = 'column' or 'radiance'")
        ModelResult.__init__(self, inputs, params)
        self.type = 'image cube'
        self._image_geometry(inputs, device)
        vmin, vmax, nbins = cube_bins(velocity, self.dims)
        self.edges = np.linspace(vmin, vmax, nbins + 1)
        self.velocity = 0.5 * (self.edges[:-1] + self.edges[1:])
        self.velocity_unit = 'km/s'
        nx, nz = self.dims

        self.outid, self.outputfiles, _, _ = self.inputs.search()
        comm = nccl_comm()
        sums = np.zeros((nx, nz, nbins + 2))
        counts = np.zeros((nx, nz, nbins + 2), dtype=np.int64)
        totalsource = 0.
        self.kernel_ms = 0.0
        if self.outputfiles or comm is not None:
            eng = get_engine(self._device)
            eng.cube_begin(nx, nz, nbins)
            try:
                for fname in self.outputfiles:
                    output = catalogue.fetch(fname)
                    totalsource += self._accumulate_cube(output, eng, vmin, vmax, nbins)
                if comm is not None:          # one collective; totalsource rides with the sums
                    totalsource = eng.cube_allreduce_total(comm[1], totalsource)
                sums, counts = eng.cube_fetch(nx, nz, nbins)
            finally:
                eng.cube_end()
        if comm is None:
            totalsource, = combine_ranks((sums, counts), totalsource)
        self.totalsource = totalsource

        endtime = float(self.inputs.options.endtime.value)
        self.atoms_per_packet = (1e23 / (self.totalsource / endtime) if self.totalsource > 0
                                 else np.nan)
        self.sourcerate = Quantity(1e23, '1/s')
        scaled = sums * self.atoms_per_packet
        self.cube = scaled[:, :, 1:-1] / np.diff(self.edges)
        self.packet_cube = counts[:, :, 1:-1]
        self.outside = scaled[:, :, [0, -1]]
        self.packet_outside = counts[:, :, [0, -1]]
        self.image = scaled.sum(axis=2)
        self.packet_image = counts.sum(axis=2).astype(np.float64)

    def _accumulate_cube(self, output, eng, vmin, vmax, nbins):
        """One Output into the context-owned cube: its resident rows, or -- recipe-only
        constant-step runs -- the same rows regenerated chunk by chunk.  Returns its
        totalsource."""
        if self.origin != self.inputs.geometry.planet:
            raise NotImplementedError('transform_reference_frame')   # ModelResult base stub
        setup = get_setup(self.inputs, strict_math=getattr(output, 'strict_math', False))
        ip = self.image_params(setup)
        for table, _ in output.tables():
            self._upload_weighting_tables(eng, setup)
            eng.bind_packets(table)
            try:
                eng.cube_add(ip, vmin, vmax, nbins, setup.radius_km, n=table.n)
                self.kernel_ms += eng.last_kernel_ms()
            finally:
                eng.bind_packets(None)
        return output.totalsource

    def __repr__(self):
        return self.__str__()

    def __str__(self):
        return f'''Image cube
quantity = {self.quantity}
dims = {self.dims[0]} x {self.dims[1]}
velocity = {self.edges[0]} .. {self.edges[-1]} km/s in {len(self.velocity)} bins
totalsource = {self.totalsource}
atoms per packet = {self.atoms_per_packet}'''
