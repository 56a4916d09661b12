#!/usr/bin/env python
"""ModelImageCube timing: a cube call (``nx_cube_add``) against the radiance K4 call
(``nx_image_add``) on the same rows and view.

Rows: configs[1] physics (Na, Maxwellian source, radiation pressure), N packets, twice: the
initial state (every packet live at the surface, the dense extreme; K4 takes its privatised
path there) and the final state of the adaptive run (~1 % of the packets survive).  Both are
compacted tables, as ModelImage / ModelImageCube bin them.  Cubes: 200 x 200 x {20, 100} and
800 x 800 x 100 bins over -5 .. 5 km/s, radiance, sub-observer point (0.7, 0.3) rad; the image
is the same view at the same dims.

Per case: the median of REPS warmed-up calls of the add alone -- device time (CUDA events,
``last_kernel_ms``) and call time (host clock around the add and a device synchronise) --,
alternating cube and image calls; and the whole product call begin + add + fetch + end, whose
fetch moves nx * nz * (nbins + 2) * 16 bytes to the host.  Every cube is checked against the
image (counts exactly, sums to 1e-12).  Prints the GPU's name, power limit and max SM clock with
the numbers; writes them as JSON too when a path is given.

    python tools/diag_cube.py [npackets] [report.json]
"""
import json
import os
import subprocess
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, 'tests'))
import numpy as np                                                       # noqa: E402

from common import workload                                              # noqa: E402
from nexoclom_b200._lib import ImageParams                               # noqa: E402
from nexoclom_b200.engine import Engine                                  # noqa: E402
from nexoclom_b200.ModelImage import image_rotation                      # noqa: E402
from nexoclom_b200.runsetup import RunSetup                              # noqa: E402

REPS = 7
VMIN, VMAX = -5.0, 5.0


def gpu_identity():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm',
                              '--format=csv,noheader'], capture_output=True, text=True, timeout=30)
        return out.stdout.strip().splitlines()[0]
    except Exception as e:                                              # noqa: BLE001
        return f'nvidia-smi unavailable ({e})'


def image_params(setup, dims):
    M = np.asarray(image_rotation(0.7, 0.3))
    ip = ImageParams()
    for k in range(9):
        ip.M[k] = float(M.flat[k])
    ip.x0, ip.x1, ip.z0, ip.z1 = -4.0, 4.0, -4.0, 4.0
    ip.nx, ip.nz = dims
    ip.apix = (8.0 / dims[0] * setup.radius_km * 1e5) * (8.0 / dims[1] * setup.radius_km * 1e5)
    ip.vrplanet = setup.vrplanet
    ip.quantity, ip.round_f32, ip.skip_dead = 1, 0, 0
    return ip


def add_ms(eng, fn):
    eng.sync()
    t0 = time.perf_counter()
    fn()
    eng.sync()
    return eng.last_kernel_ms(), (time.perf_counter() - t0) * 1e3


def case(eng, setup, table, dims, nbins):
    ip = image_params(setup, dims)
    nx, nz = dims
    eng.image_begin(nx, nz)
    eng.cube_begin(nx, nz, nbins)
    img_dev, img_call, cube_dev, cube_call = [], [], [], []
    for rep in range(REPS + 1):                                   # the first pair warms up
        d, c = add_ms(eng, lambda: eng.image_add(ip, n=table.n))
        if rep:
            img_dev.append(d)
            img_call.append(c)
        d, c = add_ms(eng, lambda: eng.cube_add(ip, VMIN, VMAX, nbins, setup.radius_km,
                                                n=table.n))
        if rep:
            cube_dev.append(d)
            cube_call.append(c)
    img, cnt = eng.image_fetch(nx, nz)
    cube, ccnt = eng.cube_fetch(nx, nz, nbins)
    eng.cube_end()
    reps = REPS + 1                                               # both hold reps adds
    assert np.array_equal(ccnt.sum(axis=2), cnt), 'cube counts differ from K4'
    nzm = img != 0
    err = float(np.max(np.abs(cube.sum(axis=2)[nzm] - img[nzm]) / np.abs(img[nzm])))
    assert err < 1e-12, err
    # the whole product call, as ModelImageCube makes it for one table
    prod = []
    for rep in range(3):
        eng.sync()
        t0 = time.perf_counter()
        eng.cube_begin(nx, nz, nbins)
        eng.cube_add(ip, VMIN, VMAX, nbins, setup.radius_km, n=table.n)
        eng.cube_fetch(nx, nz, nbins)
        eng.cube_end()
        prod.append((time.perf_counter() - t0) * 1e3)
    del cube, ccnt
    med = lambda v: float(np.median(v))                         # noqa: E731
    return {'dims': list(dims), 'nbins': nbins, 'rows': int(table.n),
            'rows_in_image': int(cnt.sum() // reps),
            'inside_velocity_range': float(ccnt_inside(eng, ip, nbins, table, setup)),
            'image_add_device_ms': med(img_dev), 'image_add_call_ms': med(img_call),
            'cube_add_device_ms': med(cube_dev), 'cube_add_call_ms': med(cube_call),
            'cube_over_image_device': med(cube_dev) / med(img_dev),
            'cube_product_call_ms': med(prod),
            'result_bytes': nx * nz * (nbins + 2) * 16, 'max_rel_err_vs_image': err}


def ccnt_inside(eng, ip, nbins, table, setup):
    """Fraction of the binned rows inside vmin .. vmax (one extra call, not timed)."""
    eng.cube_begin(ip.nx, ip.nz, nbins)
    eng.cube_add(ip, VMIN, VMAX, nbins, setup.radius_km, n=table.n)
    _, c = eng.cube_fetch(ip.nx, ip.nz, nbins)
    eng.cube_end()
    tot = c.sum()
    return c[:, :, 1:-1].sum() / tot if tot else 0.0


def main():
    npackets = int(float(sys.argv[1])) if len(sys.argv) > 1 else 10_000_000
    dest = sys.argv[2] if len(sys.argv) > 2 else None
    ident = gpu_identity()
    print(f'GPU: {ident}')
    eng = Engine(0)
    setup = RunSetup(workload('Na.maxwellian.radpres.input'))
    setup.upload(eng)
    eng.upload_gtables(setup.gtables([5891, 5897]))
    report = {'gpu': ident, 'npackets': npackets, 'vmin': VMIN, 'vmax': VMAX, 'cases': {}}
    for state in ('initial', 'final'):
        eng.init_state(setup.source_params(eng), 3, 0, npackets)
        if state == 'final':
            eng.integrate_adaptive(npackets)
        table = eng.compact_state(skip_dead=True, round_f32=True, n=npackets)
        eng.bind_packets(table)
        try:
            for dims, nbins in (((200, 200), 20), ((200, 200), 100), ((800, 800), 100)):
                r = case(eng, setup, table, dims, nbins)
                key = f'{state}_{dims[0]}x{dims[1]}x{nbins}'
                report['cases'][key] = r
                print(f"{key:>24}: rows {r['rows']:>9} ({r['inside_velocity_range']:.3f} in range)"
                      f"  image add {r['image_add_device_ms']:.3f} ms dev / "
                      f"{r['image_add_call_ms']:.3f} ms call   cube add "
                      f"{r['cube_add_device_ms']:.3f} ms dev / {r['cube_add_call_ms']:.3f} ms call"
                      f"  ({r['cube_over_image_device']:.2f}x)   product call "
                      f"{r['cube_product_call_ms']:.1f} ms for {r['result_bytes'] / 1e6:.0f} MB",
                      flush=True)
        finally:
            eng.bind_packets(None)
            table.free()
    eng.close()
    if dest:
        with open(dest, 'w') as f:
            json.dump(report, f, indent=1)


if __name__ == '__main__':
    main()
