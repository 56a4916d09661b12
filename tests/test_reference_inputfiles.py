"""The reference's own boundary regression (tests/unit_tests/Initial_state/
test_input_classes.py:17-143), restated against THIS package's Input class.  The per-group
cases read tests/golden/inputfiles/*.input, which carry the settings that test's inputfiles
(tests/test_data/inputfiles/) are asserted to hold; the reference's whole inputfile directory
and its surface map are read where the reference source tree is present (refimport.REF, as
for the other cross-checks against the reference).  Also test_SSObject.py:6-34."""
import os

import numpy as np
import pytest

import refimport
from nexoclom_b200 import Input, SSObject
from nexoclom_b200.units import Quantity

INPUTS = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'inputfiles')
REF_INPUTS = os.path.join(refimport.REF, 'tests', 'test_data', 'inputfiles')
needs_reference = pytest.mark.skipif(not os.path.isdir(REF_INPUTS),
                                     reason='reference tree not present')


def rad(v):
    return Quantity(v, 'rad')


def same(d, expected):
    assert set(d) == set(expected), (sorted(d), sorted(expected))
    for k, v in expected.items():
        got = d[k]
        if isinstance(v, tuple):
            assert len(got) == len(v) and all(float(a) == pytest.approx(float(b)) for a, b in zip(got, v)), k
        elif isinstance(v, (float, Quantity)) and not isinstance(v, bool):
            assert float(got) == pytest.approx(float(v)), k
        else:
            assert got == v, (k, got, v)


def test_geometry():
    g1 = Input(os.path.join(INPUTS, 'Geometry.01.input')).geometry
    same(g1.__dict__, {'planet': SSObject('Jupiter'), 'startpoint': 'Io',
                       'objects': {SSObject('Jupiter'), SSObject('Io'), SSObject('Europa')},
                       'type': 'geometry without starttime', 'phi': (rad(1), rad(2)),
                       'subsolarpoint': (rad(3.14), rad(0)), 'taa': rad(1.57)})
    g2 = Input(os.path.join(INPUTS, 'Geometry.02.input')).geometry
    assert g2.planet == SSObject('Jupiter') and g2.startpoint == 'Io'
    assert g2.objects == {SSObject('Jupiter'), SSObject('Io')}
    assert g2.type == 'geometry with starttime' and '2022-03-08T19:53:21' in str(g2.time)
    g3 = Input(os.path.join(INPUTS, 'Geometry.03.input')).geometry
    same(g3.__dict__, {'planet': SSObject('Mercury'), 'startpoint': 'Mercury',
                       'objects': {SSObject('Mercury')}, 'type': 'geometry without starttime',
                       'subsolarpoint': (rad(0), rad(0)), 'phi': None, 'taa': rad(3.14)})
    assert g1 == g1 and g1 != g2 and g1 != g3


def test_surface_interaction():
    def si(k):
        return Input(os.path.join(INPUTS, f'SurfaceInteraction.0{k}.input')).surfaceinteraction
    same(si(1).__dict__, {'sticktype': 'constant', 'stickcoef': 1., 'accomfactor': None})
    same(si(2).__dict__, {'sticktype': 'constant', 'stickcoef': 0.5, 'accomfactor': 0.2})
    assert si(1) == si(1) and si(1) != si(2)
    same(si(3).__dict__, {'sticktype': 'temperature dependent', 'accomfactor': 0.2,
                          'A': (1.57014, -0.006262, 0.1614157)})
    same(si(4).__dict__, {'sticktype': 'temperature dependent', 'accomfactor': 0.5,
                          'A': (1., 0.001, 0.2)})
    # The reference's test expects a 'coordinate_system' key here, but its code
    # (input_classes.py:277-295, v3.7.4) sets 'stick_map' instead -- the test is stale and
    # fails on the reference itself; the code is the specification.
    same(si(5).__dict__, {'sticktype': 'surface map', 'stick_mapfile': 'default',
                          'stick_map': None, 'subsolarlon': None, 'accomfactor': 0.5})
    same(si(6).__dict__, {'sticktype': 'surface map', 'stick_mapfile': 'Orbit3576.Ca.pkl',
                          'stick_map': None, 'subsolarlon': None, 'accomfactor': 0.5})


def test_forces():
    for k, (g, r) in enumerate([(True, True), (False, True), (True, False)], start=1):
        f = Input(os.path.join(INPUTS, f'Forces.0{k}.input')).forces
        assert f.__dict__ == {'gravity': g, 'radpres': r}


def test_spatial_dist():
    s1 = Input(os.path.join(INPUTS, 'Spatial.01.input')).spatialdist
    same(s1.__dict__, {'type': 'uniform', 'longitude': (rad(0), rad(2 * np.pi)),
                       'latitude': (rad(-np.pi / 2), rad(np.pi / 2)), 'exobase': 1.})
    s2 = Input(os.path.join(INPUTS, 'Spatial.02.input')).spatialdist
    same(s2.__dict__, {'type': 'uniform', 'longitude': (rad(0), rad(3.14)),
                       'latitude': (rad(0), rad(0.79)), 'exobase': 2.1})


@needs_reference
def test_every_reference_inputfile_parses():
    for fn in sorted(os.listdir(REF_INPUTS)):
        if fn.endswith('.input'):
            inp = Input(os.path.join(REF_INPUTS, fn))
            assert inp.geometry.planet.object is not None, fn


def test_ssobject():
    """reference tests/unit_tests/solarsystem/test_SSObject.py:6-34."""
    m = SSObject('Mercury')
    assert m.object == 'Mercury' and m.moons is None and m.type == 'Planet' and len(m) == 1
    j = SSObject('Jupiter')
    assert j.moons is not None and len(j) == len(j.moons) + 1
    assert {x.object for x in j.moons} >= {'Io', 'Europa', 'Ganymede', 'Callisto'}
    io = SSObject('Io')
    assert io.type == 'Moon' and io.orbits == 'Jupiter' and io.GM.value < 0


MAPFILE = os.path.join(os.path.dirname(REF_INPUTS), 'surface_maps', 'Orbit3576.Ca.pkl')


@pytest.mark.skipif(not os.path.exists(MAPFILE), reason='reference surface map not present')
def test_surface_map_source_with_the_references_own_map(tmp_path):
    """`SpatialDist.type = surface map` driven by a map file the reference ships
    (tests/test_data/surface_maps/Orbit3576.Ca.pkl, written with astropy Quantities inside):
    it loads without astropy, the kernel's sampler (host build) follows the oracle draw for
    draw, and the sampled surface density follows the map (source_distribution.py:63-95,
    randomdeviates.py:41-83)."""
    import ctypes as C
    from nexoclom_b200._lib import as_f64, dptr
    from nexoclom_b200.runsetup import RunSetup
    from nexoclom_b200.sourcemap import SourceMap
    from oracle import initial_state
    src = open(os.path.join(REF_INPUTS, 'Ca.surfacemap.maxwellian.input')).read()
    f = tmp_path / 'map.input'
    f.write_text(src + f'\nSpatialDist.mapfile = {MAPFILE}\n')
    setup = RunSetup(Input(str(f)))
    sp = setup.source_params(None)
    smap = SourceMap(MAPFILE)
    assert sp.spatial_type == 1 and sp.map_lat_is_sin == 1 and (sp.map_nx, sp.map_ny) == (72, 36)
    n = 60000
    ref = initial_state.draw_x0(setup, n, 5)
    hc_path = os.path.join(os.path.dirname(os.path.abspath(__file__)), '_hostcheck',
                           'libnexo_hostcheck.so')
    if not os.path.exists(hc_path):
        import subprocess
        subprocess.run(['sh', os.path.join(os.path.dirname(hc_path), 'build.sh')], check=True)
    hc = C.CDLL(hc_path)
    fmap, xa, ya = setup.sourcemap if hasattr(setup, 'sourcemap') and setup.sourcemap else (None,) * 3
    if fmap is None:
        fmap = np.asarray(smap.abundance, dtype=float)
        xa = np.linspace(np.min(smap.longitude), np.max(smap.longitude), fmap.shape[0])
        ya = np.linspace(np.sin(np.min(smap.latitude)), np.sin(np.max(smap.latitude)), fmap.shape[1])
    fm = as_f64(fmap)
    axes = as_f64(np.array([xa.min(), xa.max(), ya.min(), ya.max()]))
    cdf, vt = (as_f64(a) for a in setup.speed_table)
    out = np.zeros((n, 14))
    hc.hc_init_state(C.c_long(n), C.byref(sp), C.c_ulonglong(5), C.c_ulonglong(0), dptr(fm),
                     dptr(axes), dptr(cdf), dptr(vt), C.c_int(len(cdf)), dptr(out))
    assert np.max(np.abs(out - ref) / np.maximum(np.abs(ref), 1e-3)) < 1e-12
    # the sampled (lon, sin lat) density follows the map
    H, _, _ = np.histogram2d(ref[:, 9], np.sin(ref[:, 10]), bins=(18, 9),
                             range=[[0, 2 * np.pi], [-1, 1]])
    coarse = fmap.reshape(18, 4, 9, 4).sum(axis=(1, 3))
    expect = coarse / coarse.sum() * n
    big = expect > 200
    assert big.sum() > 20
    assert np.max(np.abs(H[big] - expect[big]) / np.sqrt(expect[big])) < 6.0
