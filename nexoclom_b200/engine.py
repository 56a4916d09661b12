"""Thin object wrapper over the C ABI (one ``Engine`` == one ``nx_ctx`` == one GPU).

All arrays crossing this layer are plain NumPy float64 / int64 host buffers
(or raw device pointers for the ``*_dev`` calls); there is no CPU fallback --
construction raises if the library or a CUDA device is missing.
"""
import ctypes as C
import weakref

import numpy as np

from . import _lib
from ._lib import (RunParams, SourceParams, ImageParams, LosParams, SpectrumParams, as_f64,
                   dptr, c_double_p, NX_PRODUCT_IMAGE, NX_PRODUCT_CUBE, NX_PRODUCT_DEPOSIT,
                   NX_PRODUCT_IONIZE)

STATE_COLS = ('time', 'x', 'y', 'z', 'vx', 'vy', 'vz', 'frac')
X0_COLS = ('time', 'x', 'y', 'z', 'vx', 'vy', 'vz', 'frac', 'v', 'longitude', 'latitude',
           'local_time', 'altitude', 'azimuth')


class NexoclomCudaError(RuntimeError):
    pass


class _PinnedPool:
    """Page-locked result buffers (``nx_host_alloc``), handed out as NumPy arrays and recycled
    once every array that views them has been garbage-collected: a device -> host copy into
    fresh pageable memory pays a page fault per 4 KB and a staging copy (2.6 ms for the two
    800 x 800 planes of an image against 0.2 ms of DMA).  Capacities are rounded up to eighths
    of an octave so that results of slightly different sizes share buffers; idle buffers are
    kept up to ``IDLE_BYTES`` in total, the rest goes back to the driver."""
    IDLE_BYTES = 1 << 30

    def __init__(self, lib):
        self.lib = lib
        self.idle = {}                           # capacity -> [pointers]
        self.idle_bytes = 0

    @staticmethod
    def _capacity(nbytes):
        if nbytes <= 4096:
            return 4096
        step = 1 << max(12, nbytes.bit_length() - 4)
        return (nbytes + step - 1) // step * step

    def array(self, shape, dtype=np.float64):
        dtype = np.dtype(dtype)
        count = int(np.prod(shape))
        nbytes = count * dtype.itemsize
        if nbytes == 0:
            return np.empty(shape, dtype=dtype)
        cap = self._capacity(nbytes)
        idle = self.idle.get(cap)
        if idle:
            ptr = idle.pop()
            self.idle_bytes -= cap
        else:
            p = C.c_void_p()
            if self.lib.nx_host_alloc(cap, C.byref(p)) != 0 or not p.value:
                return np.empty(shape, dtype=dtype)            # pageable: staged by the library
            ptr = p.value
        buf = (C.c_char * cap).from_address(ptr)
        weakref.finalize(buf, self._release, cap, ptr)
        return np.frombuffer(buf, dtype=dtype, count=count).reshape(shape)

    def _release(self, cap, ptr):
        if self.idle_bytes + cap <= self.IDLE_BYTES:
            self.idle.setdefault(cap, []).append(ptr)
            self.idle_bytes += cap
        else:
            self.lib.nx_host_free(ptr)


_POOL = None


def _pinned_pool(lib):
    global _POOL
    if _POOL is None:
        _POOL = _PinnedPool(lib)
    return _POOL


class Engine:
    def __init__(self, device=0):
        self.lib = _lib.load()
        self.ctx = C.c_void_p()
        rc = self.lib.nx_ctx_create(int(device), C.byref(self.ctx))
        if rc != 0 or not self.ctx:
            raise NexoclomCudaError(
                f'nx_ctx_create(device={device}) failed with code {rc}: nexoclom_b200 needs a '
                'CUDA device (sm_100a); there is no CPU fallback')
        self.device = int(device)
        self.n = 0
        self.params = None

    # -- plumbing -------------------------------------------------------------
    def close(self):
        if getattr(self, 'ctx', None):
            self.lib.nx_ctx_destroy(self.ctx)
            self.ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc < 0:
            msg = self.lib.nx_last_error(self.ctx)
            raise NexoclomCudaError(f'{what} failed ({rc}): {msg.decode() if msg else ""}')
        if rc > 0:
            # device-side numerical invariants == the reference's bare asserts
            msgs = []
            if rc & 4:
                msgs.append('\n\tInfinite values of emax')                  # Output.py:284
            if rc & 8:
                msgs.append('Found new values of frac that are negative')   # Output.py:287
            if rc & 16:
                msgs.append('\n\tInfinite values of step_size')             # Output.py:338
            if rc & 32:
                msgs.append('non-finite packet state')                      # Output.py:389
            if rc & 64:
                msgs.append('a packet segment never arrived on the device')
            if rc & 128:
                msgs.append('a packet made no progress in 2**22 attempted steps '
                            '(the reference loop, Output.py:248-353, would not end)')
            raise AssertionError('; '.join(msgs) or f'invariant bits {rc}')
        return rc

    def set_stream(self, cuda_stream_ptr):
        self._check(self.lib.nx_ctx_set_stream(self.ctx, C.c_void_p(int(cuda_stream_ptr))),
                    'nx_ctx_set_stream')

    def set_option(self, name, value):
        self._check(self.lib.nx_ctx_set_option(self.ctx, name.encode(), int(value)),
                    'nx_ctx_set_option')

    def sync(self):
        self._check(self.lib.nx_ctx_sync(self.ctx), 'nx_ctx_sync')

    def last_kernel_ms(self):
        ms = C.c_float()
        self._check(self.lib.nx_last_kernel_ms(self.ctx, C.byref(ms)), 'nx_last_kernel_ms')
        return float(ms.value)

    def kernel_launches(self):
        v = C.c_ulonglong()
        self.lib.nx_kernel_launches(self.ctx, C.byref(v))
        return int(v.value)

    def measure_fp64_peak(self):
        v = C.c_double()
        self._check(self.lib.nx_measure_fp64_peak(self.ctx, C.byref(v)), 'nx_measure_fp64_peak')
        return float(v.value)

    def measure_copy_bw(self, nbytes=1 << 30):
        v = C.c_double()
        self._check(self.lib.nx_measure_copy_bw(self.ctx, int(nbytes), C.byref(v)),
                    'nx_measure_copy_bw')
        return float(v.value)

    # -- tables ---------------------------------------------------------------
    def upload_tables(self, params, radpres_v=None, radpres_a=None, spline_tck=None):
        """params: RunParams; radpres_* in R_p/s, R_p/s^2; spline_tck = (tx, ty, c)."""
        self.params = params
        self._uploaded_setup = self._uploaded_gtables = None     # caches of RunSetup.upload
        if radpres_v is not None:
            rv, ra = as_f64(radpres_v), as_f64(radpres_a)
            nrp = len(rv)
            prv, pra = dptr(rv), dptr(ra)
        else:
            nrp, prv, pra = 0, None, None
        if spline_tck is not None:
            tx, ty, c = (as_f64(a) for a in spline_tck)
            args = (dptr(tx), len(tx), dptr(ty), len(ty), dptr(c))
        else:
            args = (None, 0, None, 0, None)
        self._check(self.lib.nx_tables_upload(self.ctx, C.byref(params), prv, pra, nrp, *args),
                    'nx_tables_upload')

    def upload_gtables(self, tables):
        """tables: list of (velocity [R_p/s], g [1/s]) arrays, one per emission line."""
        self._uploaded_gtables = None
        sizes = (C.c_int * len(tables))(*[len(v) for v, _ in tables])
        v = as_f64(np.concatenate([t[0] for t in tables])) if tables else np.zeros(1)
        g = as_f64(np.concatenate([t[1] for t in tables])) if tables else np.zeros(1)
        self._check(self.lib.nx_gtables_upload(self.ctx, len(tables), sizes, dptr(v), dptr(g)),
                    'nx_gtables_upload')

    def upload_sourcemap(self, fmap, xaxis, yaxis):
        f = as_f64(fmap)
        xa, ya = as_f64(xaxis), as_f64(yaxis)
        self._check(self.lib.nx_sourcemap_upload(self.ctx, dptr(f), f.shape[0], f.shape[1],
                                                 dptr(xa), dptr(ya)), 'nx_sourcemap_upload')

    def upload_speedtable(self, cdf, v):
        c, vv = as_f64(cdf), as_f64(v)
        self._check(self.lib.nx_speedtable_upload(self.ctx, dptr(c), dptr(vv), len(c)),
                    'nx_speedtable_upload')

    def upload_lontable(self, cdf, lon):
        """Inverse CDF of a longitude-only source map (random_deviates_1d)."""
        c, ll = as_f64(cdf), as_f64(lon)
        self._check(self.lib.nx_lontable_upload(self.ctx, dptr(c), dptr(ll), len(c)),
                    'nx_lontable_upload')

    # -- packets --------------------------------------------------------------
    def import_state(self, cols):
        """cols: sequence of 8 arrays (time,x,y,z,vx,vy,vz,frac) or an (N,8) array."""
        if isinstance(cols, np.ndarray) and cols.ndim == 2:
            cols = [cols[:, k] for k in range(8)]
        arrs = [as_f64(c) for c in cols]
        n = len(arrs[0])
        ptrs = (c_double_p * 8)(*[dptr(a) for a in arrs])
        self._check(self.lib.nx_import_state(self.ctx, n, ptrs), 'nx_import_state')
        self.n = n

    def export_state(self):
        out = np.empty((8, self.n))
        ptrs = (c_double_p * 8)(*[dptr(out[k]) for k in range(8)])
        self._check(self.lib.nx_export_state(self.ctx, self.n, ptrs), 'nx_export_state')
        return out

    def export_x0(self):
        out = np.empty((14, self.n))
        ptrs = (c_double_p * 14)(*[dptr(out[k]) for k in range(14)])
        self._check(self.lib.nx_export_x0(self.ctx, self.n, ptrs), 'nx_export_x0')
        return out

    def export_stats(self):
        a = np.empty(self.n, dtype=np.uint32)
        b = np.empty(self.n, dtype=np.uint32)
        self._check(self.lib.nx_export_stats(self.ctx, self.n,
                                             a.ctypes.data_as(_lib.c_u32_p),
                                             b.ctypes.data_as(_lib.c_u32_p)), 'nx_export_stats')
        return a, b

    def export_step(self):
        s = np.empty(self.n)
        self._check(self.lib.nx_export_step(self.ctx, self.n, dptr(s)), 'nx_export_step')
        return s

    def state_device_ptr(self, column):
        p = C.c_void_p()
        self._check(self.lib.nx_state_device_ptr(self.ctx, int(column), C.byref(p)),
                    'nx_state_device_ptr')
        return p.value

    def init_state(self, source_params, seed, first_id, n):
        self._check(self.lib.nx_init_state(self.ctx, C.byref(source_params), int(seed),
                                           int(first_id), int(n)), 'nx_init_state')
        self.n = int(n)

    def init_state_deviates(self, source_params, n, u_time=None, u_sinlat=None, u_lon=None,
                            lon=None, lat=None, u_speed=None, z_normal=None, u_alt=None,
                            u_az=None):
        """K1's deviate -> state transform on caller-supplied deviates (host arrays of
        length n; ``lon`` / ``lat``: surface points sampled elsewhere)."""
        arrs = [None if a is None else as_f64(a)
                for a in (u_time, u_sinlat, u_lon, lon, lat, u_speed, z_normal, u_alt, u_az)]
        ptrs = [None if a is None else dptr(a) for a in arrs]
        self._check(self.lib.nx_init_state_deviates(self.ctx, C.byref(source_params), int(n),
                                                    *ptrs), 'nx_init_state_deviates')
        self.n = int(n)

    def rewind_state(self):
        """The resident initial state becomes the current state again (no copy)."""
        self._check(self.lib.nx_rewind_state(self.ctx), 'nx_rewind_state')

    # -- resident packet tables (device-side Output.save) -----------------------
    def compact_state(self, skip_dead=True, round_f32=True, n=None):
        """Copy the current state into a packet table that stays on the GPU: frac == 0 rows
        dropped when ``skip_dead``, columns rounded to float32 when ``round_f32``
        (reference Output.save, Output.py:522-543).  Returns a ``PacketTable``."""
        n = self.n if n is None else n
        h, cnt = C.c_void_p(), C.c_longlong()
        self._check(self.lib.nx_compact_state(self.ctx, int(n), int(bool(skip_dead)),
                                              int(bool(round_f32)), C.byref(h), C.byref(cnt)),
                    'nx_compact_state')
        return PacketTable(self, h, int(cnt.value))

    def upload_packets(self, cols, index=None):
        """Host columns (8 arrays time..frac, or (N, 8)) -> resident ``PacketTable``."""
        if isinstance(cols, np.ndarray) and cols.ndim == 2:
            cols = [cols[:, k] for k in range(8)]
        arrs = [as_f64(c) for c in cols]
        n = len(arrs[0])
        idx = (np.arange(n, dtype=np.uint32) if index is None
               else np.ascontiguousarray(index, dtype=np.uint32))
        ptrs = (c_double_p * 8)(*[dptr(a) for a in arrs])
        h = C.c_void_p()
        self._check(self.lib.nx_packets_upload(self.ctx, n, ptrs, idx.ctypes.data_as(_lib.c_u32_p),
                                               C.byref(h)), 'nx_packets_upload')
        return PacketTable(self, h, n)

    def bind_packets(self, table):
        """K4 / K5 read ``table`` (None: the context's own slab) until the next bind."""
        self._check(self.lib.nx_packets_bind(self.ctx, table.handle if table is not None else None),
                    'nx_packets_bind')

    # -- hot kernels ----------------------------------------------------------
    def integrate_adaptive(self, n=None):
        att, acc = C.c_ulonglong(), C.c_ulonglong()
        n = self.n if n is None else n
        self._check(self.lib.nx_integrate_adaptive(self.ctx, n, C.byref(att), C.byref(acc)),
                    'nx_integrate_adaptive')
        return int(att.value), int(acc.value)

    def integrate_adaptive_bounce(self, seed, first_id=0, n=None):
        """K2 with surface bounce on the resident packets: deviates keyed by (seed, first_id +
        packet index).  Returns (attempted, accepted, bounces)."""
        att, acc, bnc = C.c_ulonglong(), C.c_ulonglong(), C.c_ulonglong()
        n = self.n if n is None else n
        self._check(self.lib.nx_integrate_adaptive_bounce(self.ctx, int(n), int(seed), int(first_id),
                                                          C.byref(att), C.byref(acc), C.byref(bnc)),
                    'nx_integrate_adaptive_bounce')
        return int(att.value), int(acc.value), int(bnc.value)

    def integrate_adaptive_host(self, cols, nchunks=8):
        """import_state + integrate_adaptive with the H2D copy pipelined against
        the integration (host columns should be pinned for real overlap)."""
        if isinstance(cols, np.ndarray) and cols.ndim == 2:
            cols = [cols[:, k] for k in range(8)]
        arrs = [as_f64(c) for c in cols]
        n = len(arrs[0])
        ptrs = (c_double_p * 8)(*[dptr(a) for a in arrs])
        att, acc = C.c_ulonglong(), C.c_ulonglong()
        self._check(self.lib.nx_integrate_adaptive_host(self.ctx, n, ptrs, int(nchunks),
                                                        C.byref(att), C.byref(acc)),
                    'nx_integrate_adaptive_host')
        self.n = n
        return int(att.value), int(acc.value)

    def integrate_constant(self, seed=0, first_id=0, image_params=None, image_dev=None,
                           counts_dev=None, trajectory=False, n=None):
        n = self.n if n is None else n
        p = self.params
        nsteps = int(np.ceil(p.endtime / p.step_size + 1))
        traj = np.zeros((n, 8, nsteps)) if trajectory else None
        steps = C.c_ulonglong()
        self._check(self.lib.nx_integrate_constant(
            self.ctx, n, int(seed), int(first_id),
            C.byref(image_params) if image_params is not None else None,
            C.c_void_p(image_dev) if image_dev else None,
            C.c_void_p(counts_dev) if counts_dev else None,
            dptr(traj) if traj is not None else None, C.byref(steps)), 'nx_integrate_constant')
        return traj, nsteps, int(steps.value)

    def integrate_constant_rows(self, seed=0, first_id=0, skip_dead=True, round_f32=True, n=None):
        """K3 with the row sink: returns (PacketTable of the kept rows, nsteps, packet-steps)."""
        n = self.n if n is None else n
        p = self.params
        nsteps = int(np.ceil(p.endtime / p.step_size + 1))
        h, nrows, steps = C.c_void_p(), C.c_longlong(), C.c_ulonglong()
        self._check(self.lib.nx_integrate_constant_rows(
            self.ctx, int(n), int(seed), int(first_id), int(bool(skip_dead)), int(bool(round_f32)),
            C.byref(h), C.byref(nrows), C.byref(steps)), 'nx_integrate_constant_rows')
        return PacketTable(self, h, int(nrows.value)), nsteps, int(steps.value)

    def image_accumulate(self, image_params, n=None):
        n = self.n if n is None else n
        img = np.zeros((image_params.nx, image_params.nz))
        cnt = np.zeros((image_params.nx, image_params.nz), dtype=np.int64)
        self._check(self.lib.nx_image_accumulate(self.ctx, n, C.byref(image_params), dptr(img),
                                                 cnt.ctypes.data_as(_lib.c_i64_p)),
                    'nx_image_accumulate')
        return img, cnt

    def image_begin(self, nx, nz):
        """Zero the context-owned device image (nx x nz, f64 + u64 counts)."""
        self._check(self.lib.nx_image_begin(self.ctx, int(nx), int(nz)), 'nx_image_begin')

    def image_add(self, image_params, n=None):
        """K4 of the bound packet table (or the slab) into the context-owned image."""
        n = self.n if n is None else n
        self._check(self.lib.nx_image_add(self.ctx, int(n), C.byref(image_params)),
                    'nx_image_add')

    def image_fetch(self, nx, nz):
        return self._product_fetch(NX_PRODUCT_IMAGE, (nx, nz))

    def image_fetch_scaled(self, nx, nz, scale):
        """(image * scale, packet counts as float64): what ``ModelImage`` keeps
        (ModelImage.py:92-105), converted on the device and copied ONCE into page-locked
        result arrays (no staging copy, no host passes)."""
        img = _pinned_pool(self.lib).array((nx, nz))
        cnt = _pinned_pool(self.lib).array((nx, nz))
        self._check(self.lib.nx_image_fetch_scaled(self.ctx, float(scale), dptr(img), dptr(cnt)),
                    'nx_image_fetch_scaled')
        return img, cnt

    def image_allreduce(self, comm):
        """Sum the context-owned image + counts over the ranks of ``comm`` (an ``nx_comm``
        handle), in place on the device: the one collective of an image product."""
        self._product_allreduce(NX_PRODUCT_IMAGE, comm)

    def image_allreduce_total(self, comm, total):
        """``image_allreduce`` with one scalar riding along; returns the summed scalar."""
        return self._product_allreduce(NX_PRODUCT_IMAGE, comm, total)

    def stream_ptr(self):
        p = C.c_void_p()
        self._check(self.lib.nx_ctx_stream(self.ctx, C.byref(p)), 'nx_ctx_stream')
        return p.value

    def image_device_ptrs(self):
        a, b = C.c_void_p(), C.c_void_p()
        self._check(self.lib.nx_product_device_ptrs(self.ctx, NX_PRODUCT_IMAGE, C.byref(a),
                                                    C.byref(b)), 'nx_product_device_ptrs')
        return a.value, b.value

    def image_accumulate_dev(self, image_params, image_dev, counts_dev, n=None):
        n = self.n if n is None else n
        self._check(self.lib.nx_image_accumulate_dev(self.ctx, n, C.byref(image_params),
                                                     C.c_void_p(image_dev),
                                                     C.c_void_p(counts_dev)),
                    'nx_image_accumulate_dev')

    def los_accumulate(self, los, dist_from_plan, los_params, n=None, count_used=False):
        """los: (6, nlos) array x,y,z,xbore,ybore,zbore.  Returns (radiance, hit counts,
        included mask); with ``count_used`` also the number of `used` packets (weight > 0) per
        line of sight, counted in the same pass -- ``los_used_fill`` then delivers their
        indices from the candidate pairs this call left on the device."""
        n = self.n if n is None else n
        los = as_f64(los)
        nlos = los.shape[1]
        dist = as_f64(dist_from_plan)
        # results land in page-locked arrays (direct DMA; the `included` mask is one byte per
        # packet: 10 MB per 1e7 packets) and the mask is viewed, not converted
        pool = _pinned_pool(self.lib)
        rad = pool.array((nlos,))
        npk = pool.array((nlos,), dtype=np.int64)
        inc = pool.array((max(n, 1),), dtype=np.uint8)
        if count_used:
            cnt = np.zeros(nlos, dtype=np.int64)
            self._check(self.lib.nx_los_accumulate_counted(
                self.ctx, n, nlos, dptr(los), dptr(dist), C.byref(los_params), dptr(rad),
                npk.ctypes.data_as(_lib.c_i64_p), inc.ctypes.data_as(_lib.c_u8_p),
                cnt.ctypes.data_as(_lib.c_i64_p)), 'nx_los_accumulate_counted')
            return rad, npk, inc[:n].view(np.bool_), cnt
        self._check(self.lib.nx_los_accumulate(self.ctx, n, nlos, dptr(los), dptr(dist),
                                               C.byref(los_params), dptr(rad),
                                               npk.ctypes.data_as(_lib.c_i64_p),
                                               inc.ctypes.data_as(_lib.c_u8_p)),
                    'nx_los_accumulate')
        return rad, npk, inc[:n].view(np.bool_)

    def los_used_fill(self, los, dist_from_plan, los_params, used_count, n=None):
        """CSR (offsets[nlos+1], packet indices) of the `used` packets, given the counts
        ``los_accumulate(..., count_used=True)`` returned for the same arguments."""
        n = self.n if n is None else n
        los = as_f64(los)
        nlos = los.shape[1]
        dist = as_f64(dist_from_plan)
        off = np.zeros(nlos + 1, dtype=np.int64)
        np.cumsum(used_count, out=off[1:])
        idx = np.zeros(max(int(off[-1]), 1), dtype=np.uint32)
        if off[-1] > 0:
            self._check(self.lib.nx_los_used_fill(
                self.ctx, n, nlos, dptr(los), dptr(dist), C.byref(los_params),
                off.ctypes.data_as(_lib.c_i64_p), idx.ctypes.data_as(_lib.c_u32_p)),
                'nx_los_used_fill')
        return off, idx[:int(off[-1])]

    def los_used(self, los, dist_from_plan, los_params, n=None):
        """CSR of the `used` packets (weight > 0) per line of sight:
        (offsets[nlos+1], packet indices)."""
        n = self.n if n is None else n
        los = as_f64(los)
        nlos = los.shape[1]
        dist = as_f64(dist_from_plan)
        cnt = np.zeros(nlos, dtype=np.int64)
        self._check(self.lib.nx_los_used(self.ctx, n, nlos, dptr(los), dptr(dist),
                                         C.byref(los_params), None,
                                         cnt.ctypes.data_as(_lib.c_i64_p), None), 'nx_los_used')
        off = np.zeros(nlos + 1, dtype=np.int64)
        np.cumsum(cnt, out=off[1:])
        idx = np.zeros(max(int(off[-1]), 1), dtype=np.uint32)
        if off[-1] > 0:
            self._check(self.lib.nx_los_used(self.ctx, n, nlos, dptr(los), dptr(dist),
                                             C.byref(los_params),
                                             off.ctypes.data_as(_lib.c_i64_p),
                                             cnt.ctypes.data_as(_lib.c_i64_p),
                                             idx.ctypes.data_as(_lib.c_u32_p)), 'nx_los_used')
        return off, idx[:int(off[-1])]

    def los_accumulate_dev(self, nlos, los_dev, dist_dev, los_params, rad_dev, npk_dev, inc_dev,
                           n=None):
        n = self.n if n is None else n
        self._check(self.lib.nx_los_accumulate_dev(
            self.ctx, n, int(nlos), C.c_void_p(los_dev), C.c_void_p(dist_dev),
            C.byref(los_params), C.c_void_p(rad_dev), C.c_void_p(npk_dev),
            C.c_void_p(inc_dev)), 'nx_los_accumulate_dev')

    def los_spectrum(self, los, dist_from_plan, los_params, vmin, vmax, nbins, vscale, n=None):
        """Doppler line profiles of the hits of ``los_accumulate``: los (6, nlos) as there;
        velocities along the boresight in km/s (``vscale`` km/s per R_p/s), binned on
        ``np.linspace(vmin, vmax, nbins + 1)``.  Returns (spectrum, counts), both
        (nlos, nbins + 2): column 0 holds v < vmin, 1..nbins the bins, nbins + 1 v > vmax;
        the sum of the hits' weights (float64) and their number (int64)."""
        n = self.n if n is None else n
        los = as_f64(los)
        nlos = los.shape[1]
        dist = as_f64(dist_from_plan)
        sp = SpectrumParams()
        sp.vmin, sp.vmax, sp.vscale, sp.nbins = float(vmin), float(vmax), float(vscale), int(nbins)
        # page-locked results (16 B per line and column: 160 MB for 1e5 lines x 100 bins)
        pool = _pinned_pool(self.lib)
        spec = pool.array((nlos, int(nbins) + 2))
        cnt = pool.array((nlos, int(nbins) + 2), dtype=np.int64)
        self._check(self.lib.nx_los_spectrum(self.ctx, int(n), nlos, dptr(los), dptr(dist),
                                             C.byref(los_params), C.byref(sp), dptr(spec),
                                             cnt.ctypes.data_as(_lib.c_i64_p)), 'nx_los_spectrum')
        return spec, cnt

    def cube_begin(self, nx, nz, nbins):
        """Allocate and zero the context-owned image cube: (nx, nz, nbins + 2) f64 sums and
        int64 counts (16 B per cell) until ``cube_end``."""
        self._check(self.lib.nx_cube_begin(self.ctx, int(nx), int(nz), int(nbins)),
                    'nx_cube_begin')

    def cube_add(self, image_params, vmin, vmax, nbins, vscale, n=None):
        """K4's rows, pixels and weights of the bound packet table (or the slab) binned into the
        cube by their velocity along the observer's line of sight (``vscale`` km/s per R_p/s),
        on ``np.linspace(vmin, vmax, nbins + 1)``; column 0 holds v < vmin, nbins + 1 v > vmax."""
        n = self.n if n is None else n
        sp = SpectrumParams()
        sp.vmin, sp.vmax, sp.vscale, sp.nbins = float(vmin), float(vmax), float(vscale), int(nbins)
        self._check(self.lib.nx_cube_add(self.ctx, int(n), C.byref(image_params), C.byref(sp)),
                    'nx_cube_add')

    def cube_fetch(self, nx, nz, nbins):
        """(sums, counts), both (nx, nz, nbins + 2), float64 and int64, in page-locked arrays."""
        return self._product_fetch(NX_PRODUCT_CUBE, (int(nx), int(nz), int(nbins) + 2))

    def cube_allreduce_total(self, comm, total):
        """Sum the cube's sums and counts over the ranks of ``comm`` in place, with one scalar
        riding along; returns the summed scalar."""
        return self._product_allreduce(NX_PRODUCT_CUBE, comm, total)

    def cube_end(self):
        """Release the cube's device memory."""
        self._product_end(NX_PRODUCT_CUBE)

    # bucket order of the deposition sink (nx_deposit_bucket)
    DEPOSIT_BUCKETS = ('surface', 'moon', 'escaped', 'vanished', 'remaining', 'source')

    def deposit_begin(self, nlon, nlat):
        """Allocate and zero the context-owned deposition sink: an (nlon, nlat) map of f64
        sums and int64 counts plus the bucket sums and counts, until ``deposit_end``."""
        self._check(self.lib.nx_deposit_begin(self.ctx, int(nlon), int(nlat)), 'nx_deposit_begin')

    def integrate_adaptive_deposit(self, seed, first_id=0, n=None):
        """K2 on the resident packets through its deposition sink: the run
        ``integrate_adaptive`` (perfect sticking) or ``integrate_adaptive_bounce`` (deviates
        keyed by (seed, first_id + packet index)) would make, its events added to the sink.
        Returns (attempted, accepted, bounces)."""
        att, acc, bnc = C.c_ulonglong(), C.c_ulonglong(), C.c_ulonglong()
        n = self.n if n is None else n
        self._check(self.lib.nx_integrate_adaptive_deposit(self.ctx, int(n), int(seed),
                                                           int(first_id), C.byref(att),
                                                           C.byref(acc), C.byref(bnc)),
                    'nx_integrate_adaptive_deposit')
        return int(att.value), int(acc.value), int(bnc.value)

    def deposit_fetch(self, nlon, nlat):
        """(map, counts, buckets, bucket_counts): (nlon, nlat) float64 and int64, then the
        six buckets in ``DEPOSIT_BUCKETS`` order, float64 and int64."""
        ncell = int(nlon) * int(nlat)
        sums, cnt = self._product_fetch(NX_PRODUCT_DEPOSIT, (ncell + len(self.DEPOSIT_BUCKETS),))
        shape = (int(nlon), int(nlat))
        return sums[:ncell].reshape(shape), cnt[:ncell].reshape(shape), sums[ncell:], cnt[ncell:]

    def deposit_allreduce(self, comm, total):
        """Sum the deposition sink over the ranks of ``comm`` in place, with one scalar riding
        along; returns the summed scalar."""
        return self._product_allreduce(NX_PRODUCT_DEPOSIT, comm, total)

    def deposit_end(self):
        """Release the deposition sink's device memory."""
        self._product_end(NX_PRODUCT_DEPOSIT)

    def ionize_begin(self, lo, hi, dims):
        """Allocate and zero the context-owned ion-production grid: the box ``lo``..``hi``
        (x, y, z in R_p) in ``dims`` = (nx, ny, nz) cells of f64 loss sums and int64 step
        counts, plus OUTSIDE, until ``ionize_end``."""
        g = _lib.IonGrid()
        for k in range(3):
            g.lo[k], g.hi[k], g.n[k] = float(lo[k]), float(hi[k]), int(dims[k])
        self._check(self.lib.nx_ionize_begin(self.ctx, C.byref(g)), 'nx_ionize_begin')

    def integrate_adaptive_ionize(self, seed, first_id=0, n=None):
        """K2 on the resident packets through its ion-production sink: the run
        ``integrate_adaptive_deposit`` would make, the frac each accepted step loses in flight
        added to the grid at the step's chord midpoint.  Returns (attempted, accepted,
        bounces)."""
        att, acc, bnc = C.c_ulonglong(), C.c_ulonglong(), C.c_ulonglong()
        n = self.n if n is None else n
        self._check(self.lib.nx_integrate_adaptive_ionize(self.ctx, int(n), int(seed),
                                                          int(first_id), C.byref(att),
                                                          C.byref(acc), C.byref(bnc)),
                    'nx_integrate_adaptive_ionize')
        return int(att.value), int(acc.value), int(bnc.value)

    def ionize_fetch(self, dims):
        """(sums, counts, outside, outside_count): the (nx, ny, nz) grid's loss sums (float64)
        and recorded steps (int64), then OUTSIDE's sum and count."""
        shape = tuple(int(d) for d in dims)
        ncell = shape[0] * shape[1] * shape[2]
        sums, cnt = self._product_fetch(NX_PRODUCT_IONIZE, (ncell + 1,))
        return (sums[:ncell].reshape(shape), cnt[:ncell].reshape(shape), float(sums[ncell]),
                int(cnt[ncell]))

    def ionize_allreduce(self, comm, total):
        """Sum the ion-production grid over the ranks of ``comm`` in place, with one scalar
        riding along; returns the summed scalar."""
        return self._product_allreduce(NX_PRODUCT_IONIZE, comm, total)

    def ionize_end(self):
        """Release the ion-production grid's device memory."""
        self._product_end(NX_PRODUCT_IONIZE)

    # -- context-owned accumulators (nx_product) --------------------------------
    def _product_fetch(self, which, shape):
        """(sums, counts) of an accumulator, both ``shape``, float64 and int64, in page-locked
        arrays (a direct DMA)."""
        pool = _pinned_pool(self.lib)
        sums, cnt = pool.array(shape), pool.array(shape, dtype=np.int64)
        self._check(self.lib.nx_product_fetch(self.ctx, which, dptr(sums),
                                              cnt.ctypes.data_as(_lib.c_i64_p)), 'nx_product_fetch')
        return sums, cnt

    def _product_allreduce(self, which, comm, total=None):
        """The accumulator summed over the ranks of ``comm`` in place; with ``total``, that
        scalar rides along and the sum over the ranks is returned."""
        v = None if total is None else C.c_double(float(total))
        self._check(self.lib.nx_product_allreduce(self.ctx, which, comm,
                                                  None if v is None else C.byref(v)),
                    'nx_product_allreduce')
        return None if v is None else v.value

    def _product_end(self, which):
        self._check(self.lib.nx_product_end(self.ctx, which), 'nx_product_end')

    def density_accumulate(self, points, radius, s1, s2, count, n=None):
        """K7 of the bound packet table (or the slab): ADDS to ``s1`` (sum of frac), ``s2``
        (sum of frac**2) and ``count`` (member rows) of every ball.  ``points``: (npts, 3) in
        R_p; ``radius``: (npts,) in R_p; ``s1`` / ``s2`` float64 and ``count`` int64 arrays of
        length npts, C-contiguous (updated in place)."""
        n = self.n if n is None else n
        pts = np.ascontiguousarray(np.asarray(points, dtype=np.float64).T)
        rad = as_f64(radius)
        npts = len(rad)
        if pts.shape != (3, npts):
            raise ValueError('points must be (npts, 3) with one radius per point')
        for a, dt in ((s1, np.float64), (s2, np.float64), (count, np.int64)):
            if not (isinstance(a, np.ndarray) and a.dtype == dt and a.flags.c_contiguous and
                    a.shape == (npts,)):
                raise TypeError('s1 / s2 must be float64 and count int64 arrays of length npts')
        self._check(self.lib.nx_density_accumulate(
            self.ctx, int(n), npts, dptr(pts), dptr(rad), dptr(s1), dptr(s2),
            count.ctypes.data_as(C.POINTER(C.c_ulonglong))), 'nx_density_accumulate')
        return s1, s2, count

    def source_map(self, params, longitude, latitude, speed_kms, altitude, azimuth, frac,
                   point_lon, point_lat, point_radius):
        """K6 (reference make_source_map.py:67-160).  Returns a dict of ndarrays; per-point
        arrays are shaped (nlon, nlat[, nbins])."""
        cols = [as_f64(a) for a in (longitude, latitude, speed_kms, altitude, azimuth, frac)]
        n = len(cols[0])
        plon, plat, prad = as_f64(point_lon), as_f64(point_lat), as_f64(point_radius)
        nlon, nlat = params.nlon, params.nlat
        npts = nlon * nlat
        out = {
            'abundance_hist': np.zeros((nlon, nlat)),
            'speed_dist': np.zeros(params.nvel), 'altitude_dist': np.zeros(params.nalt),
            'azimuth_dist': np.zeros(params.naz),
            'n_included': np.zeros((nlon, nlat), dtype=np.int64),
            'n_total': np.zeros((nlon, nlat), dtype=np.int64),
            'abundance': np.zeros((nlon, nlat)),
            'speed_map': np.zeros((nlon, nlat, params.nvel)),
            'altitude_map': np.zeros((nlon, nlat, params.nalt)),
            'azimuth_map': np.zeros((nlon, nlat, params.naz)),
        }
        assert npts == out['abundance'].size
        i64p = lambda a: a.ctypes.data_as(_lib.c_i64_p)     # noqa: E731
        self._check(self.lib.nx_source_map(
            self.ctx, n, C.byref(params), *[dptr(c) for c in cols], dptr(plon), dptr(plat),
            dptr(prad), dptr(out['abundance_hist']), dptr(out['speed_dist']),
            dptr(out['altitude_dist']), dptr(out['azimuth_dist']), i64p(out['n_included']),
            i64p(out['n_total']), dptr(out['abundance']), dptr(out['speed_map']),
            dptr(out['altitude_map']), dptr(out['azimuth_map'])), 'nx_source_map')
        return out


class PacketTable:
    """A compacted packet table resident on one GPU (``nx_packets``): what a saved Output
    holds -- float32-rounded time, x, y, z, vx, vy, vz, frac of the rows that survive
    ``compress`` plus their packet index -- without having left the device."""

    def __init__(self, engine, handle, n):
        self.engine, self.handle, self.n = engine, handle, int(n)

    def export(self, with_step=False):
        """(dict of float32 columns, int32 packet index[, uint16 step]): the D2H copy of a
        save."""
        cols = np.full((9, self.n), 1000.0, dtype=np.float32)
        index = np.empty(self.n, dtype=np.int32)
        step = np.zeros(self.n, dtype=np.uint16)
        if self.n:
            fp = C.POINTER(C.c_float)
            ptrs = (fp * 9)(*[cols[k].ctypes.data_as(fp) for k in range(9)])
            eng = self.engine
            eng._check(eng.lib.nx_packets_export(
                eng.ctx, self.handle, ptrs, index.ctypes.data_as(C.POINTER(C.c_int32)),
                step.ctypes.data_as(C.POINTER(C.c_uint16)) if with_step else None),
                'nx_packets_export')
        out = {c: cols[k] for k, c in enumerate(STATE_COLS + ('step_size',))}
        return (out, index, step) if with_step else (out, index)

    def index_host(self):
        """int64 packet index of every row (cached; 4 B per row over PCIe)."""
        if getattr(self, '_index', None) is None:
            self._index = self.export_index()
        return self._index

    def export_index(self):
        index = np.empty(self.n, dtype=np.int32)
        if self.n:
            eng = self.engine
            fp = C.POINTER(C.c_float)
            ptrs = (fp * 9)(*([None] * 9))
            eng._check(eng.lib.nx_packets_export(eng.ctx, self.handle, ptrs,
                                                 index.ctypes.data_as(C.POINTER(C.c_int32)), None),
                       'nx_packets_export')
        return index.astype(np.int64)

    def export_steps(self):
        step = np.zeros(self.n, dtype=np.uint16)
        if self.n:
            eng = self.engine
            fp = C.POINTER(C.c_float)
            ptrs = (fp * 9)(*([None] * 9))
            eng._check(eng.lib.nx_packets_export(eng.ctx, self.handle, ptrs, None,
                                                 step.ctypes.data_as(C.POINTER(C.c_uint16))),
                       'nx_packets_export')
        return step

    def free(self):
        if self.handle is not None and getattr(self.engine, 'ctx', None):
            self.engine.lib.nx_packets_free(self.engine.ctx, self.handle)
        self.handle = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


_engines = {}


def get_engine(device=0):
    """Process-wide engine per device (the reference is single-threaded too)."""
    if device not in _engines:
        _engines[device] = Engine(device)
    return _engines[device]
