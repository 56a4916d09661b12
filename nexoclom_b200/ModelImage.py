"""``ModelImage``: column-density / radiance images of the modelled exosphere.

Drop-in for the reference ``data_simulation/ModelImage.py:26-105, 229-274,
367-395`` (``display`` / SQL ``save`` / ``restore`` are out of scope).  The body
of ``create_image`` -- rotation to the observer frame, planet occultation,
sunlight mask, packet weighting and the two ``np.histogram2d`` calls -- is one
CUDA kernel (K4, ``nx_image_accumulate``).
"""
import json

import numpy as np

from . import catalogue
from .engine import get_engine
from .ModelResult import ModelResult
from .Output import Output
from .runsetup import get_setup
from ._lib import ImageParams
from .units import Quantity, def_unit


def rotation_matrix(theta, axis):
    """Rotation of ``theta`` about ``axis`` (reference math/rotation_matrix.py:5-14)."""
    unit_vec = axis / np.linalg.norm(axis)
    lx, ly, lz = unit_vec[0], unit_vec[1], unit_vec[2]
    c, s = np.cos(theta), np.sin(theta)
    return np.array(
        [[lx**2 + (1 - lx**2) * c, lx * ly * (1 - c) + lz * s, lx * lz * (1 - c) - ly * s],
         [lx * ly * (1 - c) - lz * s, ly**2 + (1 - ly**2) * c, ly * lz * (1 - c) + lx * s],
         [lx * lz * (1 - c) + ly * s, ly * lz * (1 - c) - lx * s, lz**2 + (1 - lz**2) * c]])


def image_rotation(subobslongitude, subobslatitude):
    """Matrix taking the Sun direction (0,-1,0) to the observer direction
    (reference ModelImage.py:367-384)."""
    slong, slat = float(subobslongitude), float(subobslatitude)
    pSun = np.array([0., -1., 0.])
    pObs = np.array([np.sin(slong) * np.cos(slat), -np.cos(slong) * np.cos(slat),
                     np.sin(slat)])
    if np.array_equal(pSun, pObs):
        return np.eye(3)
    costh = np.dot(pSun, pObs) / np.linalg.norm(pSun) / np.linalg.norm(pObs)
    theta = np.arccos(np.clip(costh, -1, 1))
    return rotation_matrix(theta, np.cross(pSun, pObs))


class _Hist2d:
    """Same attributes as the reference's ``Histogram2d`` (math/histogram.py:28-39)."""

    def __init__(self, histogram, xrange, zrange, dims):
        self.histogram = histogram
        x = np.linspace(xrange[0], xrange[1], dims[0] + 1)
        y = np.linspace(zrange[0], zrange[1], dims[1] + 1)
        self.dx, self.dy = x[1] - x[0], y[1] - y[0]
        self.x = x[:-1] + self.dx / 2
        self.y = y[:-1] + self.dy / 2


class ModelImage(ModelResult):
    def __init__(self, inputs, params, overwrite=False, distribute=None, device=None):
        from .sharding import allreduce_sum, combine_ranks, nccl_comm
        super().__init__(inputs, params)
        self.type = 'image'
        self._image_geometry(inputs, device)
        self.image = np.zeros(self.dims)
        self.packet_image = np.zeros(self.dims)

        # Every output file of this rank is binned into ONE image that stays on the device
        # (the reference adds the per-file histograms on the host, ModelImage.py:92-99) ...
        self.outid, self.outputfiles, _, _ = self.inputs.search()
        comm = nccl_comm()
        eng = None
        if self.outputfiles or comm is not None:
            eng = get_engine(self._device)
            eng.image_begin(*self.dims)
            for fname in self.outputfiles:
                print(f'Output filename: {fname}')
                self.totalsource += self._accumulate(catalogue.fetch(fname), eng)
        # ... and the ranks of a sharded run are combined with ONE all-reduce per product: on
        # the device over NCCL / NVLink (before the image crosses PCIe once), through
        # torch.distributed for the gloo backend of the CPU tests
        if comm is not None:                       # (totalsource rides with the image)
            self.totalsource = eng.image_allreduce_total(comm[1], float(self.totalsource))
        else:
            self.totalsource, = combine_ranks((), self.totalsource)

        mod_rate = self.totalsource / self.inputs.options.endtime.value
        self.atoms_per_packet = 1e23 / mod_rate
        self.sourcerate = Quantity(1e23, '1/s')
        if eng is not None:
            # `image *= atoms_per_packet` and the float packet image (ModelImage.py:92-105)
            # are formed on the device; the two planes arrive in page-locked arrays
            self.image, self.packet_image = eng.image_fetch_scaled(
                *self.dims, self.atoms_per_packet)
        if comm is None:
            allreduce_sum(self.image, self.packet_image)       # gloo (CPU tests of the host logic)

    def _image_geometry(self, inputs, device):
        """The image plane from ``params`` (host only; ModelImageCube shares it): origin, unit,
        dims, center, width, sub-observer point, xrange / zrange, Apix, xaxis / zaxis and the
        device."""
        from .sharding import local_device
        self.origin = self.params.get('origin', inputs.geometry.planet)
        self.unit = def_unit('R_' + self.origin.object, 'length',
                             float(self.origin.radius.value) * 1e3)
        R = lambda v: Quantity(v, self.unit)      # noqa: E731

        dimtemp = self.params.get('dims', '800,800').split(',')
        self.dims = [int(dimtemp[0]), int(dimtemp[1])]
        centtemp = self.params.get('center', '0,0').split(',')
        self.center = [R(float(centtemp[0])), R(float(centtemp[1]))]
        widtemp = self.params.get('width', '8,8').split(',')
        self.width = [R(float(widtemp[0])), R(float(widtemp[1]))]
        self.subobslongitude = Quantity(float(self.params.get('subobslongitude', '0')), 'rad')
        self.subobslatitude = Quantity(float(self.params.get('subobslatitude', np.pi / 2)),
                                       'rad')

        self.blimits = None
        immin = tuple(float(c) - float(w) / 2 for c, w in zip(self.center, self.width))
        immax = tuple(float(c) + float(w) / 2 for c, w in zip(self.center, self.width))
        self.xrange = [R(immin[0]), R(immax[0])]
        self.zrange = [R(immin[1]), R(immax[1])]
        scale = tuple(float(w) / d for w, d in zip(self.width, self.dims))
        r_cm = float(self.origin.radius.value) * 1e5
        self.Apix = Quantity((scale[0] * r_cm) * (scale[1] * r_cm), 'cm2')
        self._device = local_device() if device is None else device
        xr = [float(x) for x in self.xrange]
        zr = [float(z) for z in self.zrange]
        axes = _Hist2d(None, xr, zr, self.dims)
        self.xaxis = R(axes.x)
        self.zaxis = R(axes.y)

    def image_rotation(self):
        return image_rotation(self.subobslongitude, self.subobslatitude)

    def image_params(self, setup):
        ip = ImageParams()
        M = self.image_rotation()
        for k in range(9):
            ip.M[k] = float(M.flat[k])
        ip.x0, ip.x1 = float(self.xrange[0]), float(self.xrange[1])
        ip.z0, ip.z1 = float(self.zrange[0]), float(self.zrange[1])
        ip.nx, ip.nz = self.dims
        ip.apix = float(self.Apix)
        ip.vrplanet = setup.vrplanet
        ip.quantity = 0 if self.quantity in ('column', 'density') else 1
        ip.round_f32 = 0
        ip.skip_dead = 0
        return ip

    def _accumulate(self, output, eng):
        """K4 of one Output into the context-owned device image; returns its totalsource.
        The packet table holds exactly what the reference would read from disk (f32-rounded,
        frac == 0 rows removed when ``compress``)."""
        if self.origin != self.inputs.geometry.planet:
            raise NotImplementedError('transform_reference_frame')   # ModelResult base stub
        setup = get_setup(self.inputs, strict_math=getattr(output, 'strict_math', False))
        self._upload_weighting_tables(eng, setup)
        ip = self.image_params(setup)
        if getattr(output, 'trajectory_kept', True):
            table = output.device_table()
            eng.bind_packets(table)
            try:
                eng.image_add(ip, n=table.n)
            finally:
                eng.bind_packets(None)
        else:
            self._accumulate_fused(output, eng, setup, ip)
        return output.totalsource

    def _accumulate_fused(self, output, eng, setup, ip):
        """Recipe-only constant-step output (its rows were too many to keep): run K1 + K3
        again with this image fused into the integrator.  The packets (Philox keyed by seed
        and packet id) and every bounce (keyed by packet id and step) are reproduced exactly,
        the rows are binned as the reference would bin the saved ones: rounded to float32
        (Output.save, quirk Q14) and without the frac == 0 rows that `compress` drops."""
        setup.upload(eng)
        self._upload_weighting_tables(eng, setup)
        eng.init_state(setup.source_params(eng), output.seed, output.first_id, output.npackets)
        ip.round_f32, ip.skip_dead = 1, 1
        img_dev, cnt_dev = eng.image_device_ptrs()
        eng.integrate_constant(seed=output.seed, first_id=output.first_id, image_params=ip,
                               image_dev=img_dev, counts_dev=cnt_dev, n=output.npackets)

    def create_image(self, fname):
        """reference ModelImage.py:229-274 for ONE output file: (image, packet image) as
        ``Histogram2d``-like objects."""
        output = fname if isinstance(fname, Output) else catalogue.fetch(fname)
        eng = get_engine(self._device)
        eng.image_begin(*self.dims)
        self._accumulate(output, eng)
        img, cnt = eng.image_fetch(*self.dims)
        xr = [float(x) for x in self.xrange]
        zr = [float(z) for z in self.zrange]
        return (_Hist2d(img, xr, zr, self.dims),
                _Hist2d(cnt.astype(float), xr, zr, self.dims))

    def export(self, filename='image.json'):
        if filename.endswith('.json'):
            saveimage = {'image': self.image.tolist(),
                         'xaxis': np.asarray(self.xaxis).tolist(),
                         'zaxis': np.asarray(self.zaxis).tolist()}
            with open(filename, 'w') as f:
                json.dump(saveimage, f)
        else:
            raise TypeError('Not an valid file format')
