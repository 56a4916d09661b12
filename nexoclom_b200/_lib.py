"""ctypes binding of ``libnexo_b200.so`` (the C ABI declared in
``include/nexoclom_b200.h``).

There is NO CPU fallback: importing this module without the built library, or
creating a context without a CUDA device, raises.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('NEXOCLOM_B200_LIB', os.path.join(_HERE, 'libnexo_b200.so'))

c_double_p = C.POINTER(C.c_double)
c_i64_p = C.POINTER(C.c_longlong)
c_u32_p = C.POINTER(C.c_uint32)
c_u8_p = C.POINTER(C.c_uint8)

# nx_product: the context-owned accumulators
NX_PRODUCT_IMAGE, NX_PRODUCT_CUBE, NX_PRODUCT_DEPOSIT, NX_PRODUCT_IONIZE = 0, 1, 2, 3


class RunParams(C.Structure):
    """Mirror of ``nx_run_params`` (include/nexoclom_b200.h)."""
    _fields_ = [
        ('GM', C.c_double), ('vrplanet', C.c_double), ('loss_rate', C.c_double),
        ('outeredge', C.c_double), ('resolution', C.c_double), ('step_size', C.c_double),
        ('endtime', C.c_double), ('stickcoef', C.c_double), ('accomfactor', C.c_double),
        ('stick_A', C.c_double * 3), ('surf_t1', C.c_double), ('planet_radius_km', C.c_double),
        ('radpres_amax', C.c_double),
        ('gravity', C.c_int32), ('radpres', C.c_int32), ('loss_mode', C.c_int32),
        ('sticktype', C.c_int32), ('strict_math', C.c_int32), ('nmoons', C.c_int32),
        ('moon_GM', C.c_double * 4), ('moon_a', C.c_double * 4), ('moon_omega', C.c_double * 4),
        ('moon_phi', C.c_double * 4), ('moon_r2', C.c_double * 4),
    ]


class IonGrid(C.Structure):
    """Mirror of ``nx_ion_grid``: the ion-production grid's box and cells per axis."""
    _fields_ = [('lo', C.c_double * 3), ('hi', C.c_double * 3), ('n', C.c_int32 * 3),
                ('reserved', C.c_int32)]


class SourceParams(C.Structure):
    """Mirror of ``nx_source_params``."""
    _fields_ = [
        ('spatial_type', C.c_int32), ('speed_type', C.c_int32), ('angular_type', C.c_int32),
        ('is_planet', C.c_int32),
        ('exobase', C.c_double),
        ('sinlat0', C.c_double), ('sinlat1', C.c_double),
        ('lon0', C.c_double), ('lon1', C.c_double),
        ('vprob', C.c_double), ('vsigma', C.c_double), ('delv', C.c_double),
        ('v_scale', C.c_double),
        ('sinalt0', C.c_double), ('sinalt1', C.c_double),
        ('az0', C.c_double), ('az1', C.c_double),
        ('endtime', C.c_double), ('random_time', C.c_int32), ('map_nx', C.c_int32),
        ('map_ny', C.c_int32), ('map_lat_is_sin', C.c_int32),
        ('map_fmax', C.c_double),
        ('start_is_moon', C.c_int32), ('reserved', C.c_int32),
        ('moon_a', C.c_double), ('moon_omega', C.c_double), ('moon_phi', C.c_double),
        ('moon_radius', C.c_double),
    ]


class ImageParams(C.Structure):
    """Mirror of ``nx_image_params``."""
    _fields_ = [
        ('M', C.c_double * 9),
        ('x0', C.c_double), ('x1', C.c_double), ('z0', C.c_double), ('z1', C.c_double),
        ('apix', C.c_double),               # pixel area [cm^2]
        ('vrplanet', C.c_double),
        ('nx', C.c_int32), ('nz', C.c_int32),
        ('quantity', C.c_int32),            # 0 column, 1 radiance
        ('round_f32', C.c_int32),
        ('skip_dead', C.c_int32), ('reserved', C.c_int32),
    ]


class LosParams(C.Structure):
    """Mirror of ``nx_los_params``."""
    _fields_ = [
        ('dphi', C.c_double), ('outeredge', C.c_double), ('vrplanet', C.c_double),
        ('rp_cm', C.c_double),
        ('quantity', C.c_int32), ('round_f32', C.c_int32),
        ('skip_dead', C.c_int32), ('reserved', C.c_int32),
    ]


class SpectrumParams(C.Structure):
    """Mirror of ``nx_spectrum_params``."""
    _fields_ = [
        ('vmin', C.c_double), ('vmax', C.c_double), ('vscale', C.c_double),
        ('nbins', C.c_int32), ('reserved', C.c_int32),
    ]


class SourceMapParams(C.Structure):
    """Mirror of ``nx_source_map_params``."""
    _fields_ = [
        ('smear_radius', C.c_double), ('vmax', C.c_double),
        ('nlon', C.c_int32), ('nlat', C.c_int32), ('nvel', C.c_int32), ('nalt', C.c_int32),
        ('naz', C.c_int32), ('weight_is_frac', C.c_int32),
    ]


_lib = None


def load():
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f'{LIB_PATH} not found: build it with `python -c "import __graft_entry__ as g; '
            'g.build()"` (nvcc, sm_100a).  nexoclom_b200 has no CPU fallback.')
    lib = C.CDLL(LIB_PATH)
    vp = C.c_void_p
    i64 = C.c_longlong
    u64 = C.c_ulonglong
    sig = {
        'nx_ctx_create': [C.c_int, C.POINTER(vp)],
        'nx_ctx_destroy': [vp],
        'nx_ctx_set_stream': [vp, vp],
        'nx_ctx_stream': [vp, C.POINTER(vp)],
        'nx_ctx_sync': [vp],
        'nx_ctx_set_option': [vp, C.c_char_p, C.c_int],
        'nx_last_error': [vp],
        'nx_status': [vp, C.POINTER(C.c_int)],
        'nx_tables_upload': [vp, C.POINTER(RunParams), c_double_p, c_double_p, C.c_int,
                             c_double_p, C.c_int, c_double_p, C.c_int, c_double_p],
        'nx_gtables_upload': [vp, C.c_int, C.POINTER(C.c_int), c_double_p, c_double_p],
        'nx_packets_resize': [vp, i64],
        'nx_import_state': [vp, i64, C.POINTER(c_double_p)],
        'nx_export_state': [vp, i64, C.POINTER(c_double_p)],
        'nx_export_x0': [vp, i64, C.POINTER(c_double_p)],
        'nx_export_stats': [vp, i64, c_u32_p, c_u32_p],
        'nx_export_step': [vp, i64, c_double_p],
        'nx_sourcemap_upload': [vp, c_double_p, C.c_int, C.c_int, c_double_p, c_double_p],
        'nx_speedtable_upload': [vp, c_double_p, c_double_p, C.c_int],
        'nx_init_state': [vp, C.POINTER(SourceParams), u64, u64, i64],
        'nx_lontable_upload': [vp, c_double_p, c_double_p, C.c_int],
        'nx_init_state_deviates': [vp, C.POINTER(SourceParams), i64] + [c_double_p] * 9,
        'nx_rewind_state': [vp],
        'nx_integrate_adaptive': [vp, i64, C.POINTER(u64), C.POINTER(u64)],
        'nx_integrate_adaptive_host': [vp, i64, C.POINTER(c_double_p), C.c_int, C.POINTER(u64),
                                       C.POINTER(u64)],
        'nx_integrate_adaptive_bounce': [vp, i64, u64, u64, C.POINTER(u64), C.POINTER(u64),
                                         C.POINTER(u64)],
        'nx_integrate_constant': [vp, i64, u64, u64, C.POINTER(ImageParams), vp, vp,
                                  c_double_p, C.POINTER(u64)],
        'nx_image_accumulate': [vp, i64, C.POINTER(ImageParams), c_double_p, c_i64_p],
        'nx_image_accumulate_dev': [vp, i64, C.POINTER(ImageParams), vp, vp],
        'nx_image_begin': [vp, C.c_int, C.c_int],
        'nx_image_add': [vp, i64, C.POINTER(ImageParams)],
        'nx_image_fetch_scaled': [vp, C.c_double, c_double_p, c_double_p],
        'nx_host_alloc': [i64, C.POINTER(vp)],
        'nx_host_free': [vp],
        'nx_los_accumulate': [vp, i64, i64, c_double_p, c_double_p, C.POINTER(LosParams),
                              c_double_p, c_i64_p, c_u8_p],
        'nx_los_accumulate_dev': [vp, i64, i64, vp, vp, C.POINTER(LosParams), vp, vp, vp],
        'nx_los_accumulate_counted': [vp, i64, i64, c_double_p, c_double_p, C.POINTER(LosParams),
                                      c_double_p, c_i64_p, c_u8_p, c_i64_p],
        'nx_los_used_fill': [vp, i64, i64, c_double_p, c_double_p, C.POINTER(LosParams), c_i64_p,
                             c_u32_p],
        'nx_los_used': [vp, i64, i64, c_double_p, c_double_p, C.POINTER(LosParams), c_i64_p,
                        c_i64_p, c_u32_p],
        'nx_los_spectrum': [vp, i64, i64, c_double_p, c_double_p, C.POINTER(LosParams),
                            C.POINTER(SpectrumParams), c_double_p, c_i64_p],
        'nx_cube_begin': [vp, C.c_int, C.c_int, C.c_int],
        'nx_cube_add': [vp, i64, C.POINTER(ImageParams), C.POINTER(SpectrumParams)],
        'nx_deposit_begin': [vp, C.c_int, C.c_int],
        'nx_integrate_adaptive_deposit': [vp, i64, u64, u64, C.POINTER(u64), C.POINTER(u64),
                                          C.POINTER(u64)],
        'nx_ionize_begin': [vp, C.POINTER(IonGrid)],
        'nx_integrate_adaptive_ionize': [vp, i64, u64, u64, C.POINTER(u64), C.POINTER(u64),
                                         C.POINTER(u64)],
        'nx_product_fetch': [vp, C.c_int, c_double_p, c_i64_p],
        'nx_product_device_ptrs': [vp, C.c_int, C.POINTER(vp), C.POINTER(vp)],
        'nx_product_allreduce': [vp, C.c_int, vp, C.POINTER(C.c_double)],
        'nx_product_end': [vp, C.c_int],
        'nx_density_accumulate': [vp, i64, i64, c_double_p, c_double_p, c_double_p, c_double_p,
                                  C.POINTER(u64)],
        'nx_source_map': [vp, i64, C.POINTER(SourceMapParams)] + [c_double_p] * 9 +
                         [c_double_p] * 4 + [c_i64_p] * 2 + [c_double_p] * 4,
        'nx_state_device_ptr': [vp, C.c_int, C.POINTER(vp)],
        'nx_compact_state': [vp, i64, C.c_int, C.c_int, C.POINTER(vp), C.POINTER(i64)],
        'nx_packets_upload': [vp, i64, C.POINTER(c_double_p), c_u32_p, C.POINTER(vp)],
        'nx_packets_bind': [vp, vp],
        'nx_packets_count': [vp, vp, C.POINTER(i64)],
        'nx_packets_export': [vp, vp, C.POINTER(C.POINTER(C.c_float)), C.POINTER(C.c_int32),
                              C.POINTER(C.c_uint16)],
        'nx_integrate_constant_rows': [vp, i64, u64, u64, C.c_int, C.c_int, C.POINTER(vp),
                                       C.POINTER(i64), C.POINTER(u64)],
        'nx_packets_free': [vp, vp],
        'nx_comm_unique_id': [vp],
        'nx_comm_create': [C.c_int, vp, C.c_int, C.c_int, C.POINTER(vp)],
        'nx_allreduce': [vp, vp, i64, C.c_int, vp],
        'nx_allreduce_host': [vp, vp, i64, C.c_int],
        'nx_comm_rank': [vp, C.POINTER(C.c_int), C.POINTER(C.c_int)],
        'nx_comm_destroy': [vp],
        'nx_comm_last_error': [],
        'nx_last_kernel_ms': [vp, C.POINTER(C.c_float)],
        'nx_kernel_launches': [vp, C.POINTER(u64)],
        'nx_measure_fp64_peak': [vp, C.POINTER(C.c_double)],
        'nx_measure_copy_bw': [vp, i64, C.POINTER(C.c_double)],
    }
    for name, args in sig.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = (C.c_char_p if name in ('nx_last_error', 'nx_comm_last_error')
                      else C.c_int)
    _lib = lib
    return lib


def as_f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def dptr(a):
    return a.ctypes.data_as(c_double_p)
