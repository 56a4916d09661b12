"""K5 across observing geometries: brute force (los_mode 1) and the cell grid (los_mode 2, at
32 and NX_LOS_GRID_MAX cells per axis and sized from the packet count) against the oracle on
the geometry families of los_cases -- far observers at arcsecond apertures, observers inside
the cloud, members past the outer edge, wide cones either side of the `cover` flip, shadowed
foot-points, limb-grazing boresights, axis boresights, observers outside the edge -- with the
F64 and F32 record builds (round_f32 0 / 1) and with the dead rows kept or skipped.

Per case: hit counts, `included` and the `used` sets (from nx_los_used and from
nx_los_accumulate_counted + nx_los_used_fill) exact, radiance to 1e-12, and the Doppler spectra
of nx_los_spectrum summed over their columns equal to the counts and the radiance.  The oracle
is oracle.spectrum.los_hits, imaging.los_iteration statement by statement with the per-line hit
sets kept (test_spectrum.py pins the two together), so one oracle pass serves both dead-row
settings."""
import re
import time

import numpy as np
import pytest

import los_cases
from common import workload
from nexoclom_b200._lib import LosParams
from oracle import imaging
from oracle import spectrum as ospec

pytestmark = pytest.mark.gpu
GRID_MAX = 160                    # NX_LOS_GRID_MAX (nx_kernels.h)
PER = {'far': 3000}               # packets per line; the arcsecond oracle lines are the slow part
VSCALE = 2439.7                   # km per R_p
VBINS = (-6.0, 6.0, 24)


def _groups(name):
    rng = np.random.default_rng(1000 + sum(map(ord, name)))
    return los_cases.FAMILIES[name](PER.get(name, 4000), rng)


def _lp(g, round_f32, skip_dead):
    lp = LosParams()
    lp.dphi, lp.outeredge = g['dphi'], g['outeredge']
    lp.vrplanet, lp.rp_cm = los_cases.VRPLANET, los_cases.RP_CM
    lp.quantity, lp.round_f32, lp.skip_dead = 1, round_f32, skip_dead
    return lp


def _expected(hits, n, live):
    """(hit counts, radiance, included, used sets) of the oracle's per-line hits, the dead
    rows dropped when ``live`` is given."""
    npk, rad = np.zeros(len(hits), dtype=np.int64), np.zeros(len(hits))
    inc = np.zeros(n, dtype=bool)
    used = []
    for i, (sel, w) in enumerate(hits):
        if live is not None:
            keep = live[sel]
            sel, w = sel[keep], w[keep]
        npk[i], rad[i] = len(sel), w.sum() if len(w) else 0.0
        inc[sel] = True
        used.append(set(sel[w > 0].tolist()))
    return npk, rad, inc, used


def _close(got, ref, what):
    assert np.array_equal(got == 0, ref == 0), what
    nz = ref != 0
    assert np.all(np.abs(got[nz] - ref[nz]) <= 1e-12 * np.abs(ref[nz])), what


def _same_sets(off, idx, used, what):
    assert np.array_equal(np.diff(off), [len(u) for u in used]), what
    for i, u in enumerate(used):
        assert set(idx[off[i]:off[i + 1]].tolist()) == u, (what, i)


def _run_group(engine, g, gt):
    los, X = g['los'], g['X']
    los6 = los.T.copy()
    n = len(X)
    hits = ospec.los_hits(X[:, 1], X[:, 2], X[:, 3], X[:, 5], X[:, 7], los,
                          vrplanet=los_cases.VRPLANET, dphi=g['dphi'], outeredge=g['outeredge'],
                          rp_cm=los_cases.RP_CM, gtables=gt)
    dist = los_cases.dist_from_plan(los)
    engine.import_state(X)
    live = X[:, 7] > 0
    vmin, vmax, nbins = VBINS
    checked = 0
    for skip_dead in (0, 1):
        npk_o, rad_o, inc_o, used_o = _expected(hits, n, live if skip_dead else None)
        for round_f32 in (0, 1):
            lp = _lp(g, round_f32, skip_dead)
            tag = f"{g['name']} round_f32={round_f32} skip_dead={skip_dead}"
            for mode, grids in ((1, (0,)), (2, (32, GRID_MAX, 0))):
                engine.set_option('los_mode', mode)
                for G in grids:
                    engine.set_option('los_grid', G)
                    what = f'{tag} los_mode={mode} los_grid={G}'
                    rad, npk, inc = engine.los_accumulate(los6, dist, lp)
                    assert np.array_equal(npk, npk_o), (what, npk, npk_o)
                    assert np.array_equal(inc, inc_o), what
                    _close(rad, rad_o, what)
                    if mode == 2:
                        rad, npk, inc, cnt = engine.los_accumulate(los6, dist, lp, count_used=True)
                        assert np.array_equal(npk, npk_o) and np.array_equal(inc, inc_o), what
                        _close(rad, rad_o, what)
                        _same_sets(*engine.los_used_fill(los6, dist, lp, cnt), used_o, what + ' fill')
                        _same_sets(*engine.los_used(los6, dist, lp), used_o, what + ' used')
                        spec, scnt = engine.los_spectrum(los6, dist, lp, vmin, vmax, nbins, VSCALE)
                        assert np.array_equal(scnt.sum(axis=1), npk_o), what + ' spectrum'
                        _close(spec.sum(axis=1), rad_o, what + ' spectrum')
                    checked += 1
            engine.set_option('los_grid', 0)
            engine.set_option('los_mode', 0)
    return hits, checked


@pytest.mark.parametrize('family', sorted(los_cases.FAMILIES))
def test_family_matches_oracle(engine, family):
    gt = los_cases.gtables()
    engine.upload_gtables(gt)
    t0 = time.perf_counter()
    try:
        for g in _groups(family):
            hits, checked = _run_group(engine, g, gt)
            inside = [len(sel) for sel, _ in hits]
            print(f"{g['name']}: {len(g['los'])} lines, hits per line {inside}, {checked} runs")
            assert min(inside) > 0, (g['name'], inside)
    finally:
        engine.set_option('los_grid', 0)
        engine.set_option('los_mode', 0)
    print(f'{family}: {time.perf_counter() - t0:.1f} s')


def test_far_arcsecond_lines_brute_vs_grid(engine):
    """2048 lines from 1e4-5e4 R_p at 4" through a 2e5-packet cloud (enough lines for the
    Morton-ordered march): brute force and the cell grid agree line by line, F64 and F32."""
    rng = np.random.default_rng(77)
    nlos = 2048
    dirs = rng.normal(size=(nlos, 3))
    dirs /= np.linalg.norm(dirs, axis=1)[:, None]
    x_sc = dirs * rng.uniform(1e4, 5e4, nlos)[:, None]
    tgt = rng.uniform(-2.5, 2.5, (nlos, 3))
    bore = tgt - x_sc
    bore /= np.linalg.norm(bore, axis=1)[:, None]
    los = np.concatenate([x_sc, bore], axis=1)
    n = 200_000
    P = rng.normal(size=(n, 3))
    P *= (1.0 + 3.0 * rng.random(n) ** 2 / np.linalg.norm(P, axis=1))[:, None]
    X = los_cases.packets(P, rng)
    engine.upload_gtables(los_cases.gtables())
    engine.import_state(X)
    dist = los_cases.dist_from_plan(los)
    g = {'dphi': 4 * los_cases.ARCSEC, 'outeredge': 25.0}
    try:
        for round_f32 in (0, 1):
            lp = _lp(g, round_f32, 1)
            engine.set_option('los_mode', 1)
            ref = engine.los_accumulate(los.T.copy(), dist, lp)
            ref = [a.copy() for a in ref]
            engine.set_option('los_mode', 2)
            got = engine.los_accumulate(los.T.copy(), dist, lp)
            assert np.array_equal(got[1], ref[1]) and np.array_equal(got[2], ref[2])
            _close(got[0], ref[0], f'round_f32={round_f32}')
            assert ref[1].sum() > 10 * nlos
    finally:
        engine.set_option('los_mode', 0)


def test_far_arcsecond_line_hits_every_member(engine):
    """The ground-based case at 2": one line from 1.5e4 R_p and one from 3 R_p, packets inside
    their cones near the planet.  Every packet well inside a cone is a hit (a ladder that
    stopped short of the planet would drop them) and the counts are the oracle's."""
    rng = np.random.default_rng(12)
    dphi = 2 * los_cases.ARCSEC
    rows = [los_cases.line(1.5e4 * los_cases.unit([0.6, -0.7, 0.4]), [0.0, 3.0, 0.5]),     # the tail
            los_cases.line(3.0 * los_cases.unit([0.3, -0.8, 0.5]),
                           bore=los_cases.unit(los_cases.unit([0.3, -0.8, 0.5]) + 0.2 * los_cases.unit([1., 1., 0.])))]
    parts = [los_cases.cone_points(rows[0], dphi, los_cases._near_planet(rows[0], 5000, rng, 4.0), rng),
             los_cases.cone_points(rows[1], dphi, rng.uniform(0.05, 6.0, 5000), rng)]
    P = np.concatenate(parts)
    X = los_cases.packets(P, rng, dead=0.0)
    los = np.array(rows)
    gt = los_cases.gtables()
    engine.upload_gtables(gt)
    engine.import_state(X)
    dist = los_cases.dist_from_plan(los)
    rad_o, np_o, inc_o, _ = imaging.los_iteration(
        X[:, 1], X[:, 2], X[:, 3], X[:, 5], X[:, 7], los, vrplanet=los_cases.VRPLANET, dphi=dphi,
        outeredge=25.0, rp_cm=los_cases.RP_CM, gtables=gt)
    inside = []
    for i, row in enumerate(rows):
        Q = X[5000 * i:5000 * (i + 1), 1:4] - row[:3]
        ang = np.arccos(np.clip((Q @ row[3:]) / np.linalg.norm(Q, axis=1), -1, 1))
        inside.append(int((ang <= dphi * (1 - 1e-6)).sum()))
    try:
        for mode in (1, 2):
            engine.set_option('los_mode', mode)
            rad, npk, inc = engine.los_accumulate(los.T.copy(), dist, _lp({'dphi': dphi, 'outeredge': 25.0}, 1, 0))
            print(f'los_mode {mode}: hits {npk.tolist()}, oracle {np_o.tolist()}, well inside the cones {inside}')
            assert np.array_equal(npk, np_o) and np.array_equal(inc, inc_o)
            _close(rad, rad_o, f'los_mode {mode}')
    finally:
        engine.set_option('los_mode', 0)
    assert np.all(np_o >= inside) and min(inside) > 2500


def test_losresult_at_two_arcseconds(engine):
    """A 2" LOSResult through the public API against the oracle, on a small output."""
    from nexoclom_b200 import Output, LOSResult
    from nexoclom_b200.runsetup import RunSetup
    from nexoclom_b200.units import Quantity
    from test_gpu_parity import _FakeSCData
    inputs = workload('Ca.isotropic.flat.input')
    inputs.delete_files()
    out = Output(inputs, 100_000, seed=4)
    rows = []
    for k, alt in enumerate((0.3, 0.7, 1.05, 1.3)):         # two through the disk, two off the limb
        d = los_cases.unit([np.cos(k), np.sin(k), 0.3])
        rows.append(los_cases.line(1.5e4 * d, alt * los_cases.unit(np.cross(d, [0.0, 0.0, 1.0]))))
    los = np.array(rows)
    sc = _FakeSCData(los, np.array([1.0, 2.0, 3.0, 4.0]))
    res = LOSResult(sc, inputs, dphi=Quantity(2.0 / 3600, 'deg'))
    res.simulate_data_from_inputs(sc)
    P = Output.restore(out.filename).X
    setup = RunSetup(inputs)
    rad_o, np_o, _, _ = imaging.los_iteration(
        P.x.values, P.y.values, P.z.values, P.vy.values, P.frac.values, los,
        vrplanet=setup.vrplanet, dphi=float(np.radians(2.0 / 3600)),
        outeredge=float(inputs.options.outeredge), rp_cm=setup.radius_km * 1e5,
        gtables=setup.gtables([4227]))
    print('2" LOSResult hits', res.npackets_los.values.tolist(), 'oracle', np_o.tolist())
    assert np.array_equal(res.npackets_los.values, np_o) and np_o.sum() > 0
    kR = rad_o * res.atoms_per_packet / 1e3 * float(res.sourcerate)
    _close(res.radiance.values, kR, 'LOSResult 2"')
    inputs.delete_files()


def _k_los_builds(names):
    """{'k_los_resolve<1,0>', 'k_los_prepare', ...} from profiler kernel names."""
    out = set()
    for name in names:
        m = re.search(r'(k_los_\w+)(<([^>]*)>)?', name)
        if not m:
            continue
        if m.group(3) is None:
            out.add(m.group(1))
            continue
        args = [a.strip().replace('(bool)', '') for a in m.group(3).split(',')]
        args = ['1' if a in ('true', '1') else '0' for a in args]
        out.add(f"{m.group(1)}<{','.join(args)}>")
    return out


def test_profiler_sees_every_los_build(engine):
    """Brute force, the grid with both record builds, the spectrum resolve and the
    Morton-ordered march once under torch.profiler: the k_los_* kernels that ran are exactly
    the predicted set."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    assert _k_los_builds(['void nx::k_los_resolve<true, false>(nx::LosSorted)',
                          'void nx::k_los_candidates<(bool)0>(x)', 'nx::k_los_prepare(double)']) == \
        {'k_los_resolve<1,0>', 'k_los_candidates<0>', 'k_los_prepare'}
    gt = los_cases.gtables()
    engine.upload_gtables(gt)
    rng = np.random.default_rng(4)
    g = los_cases.fam_wide(500, rng)[0]
    many = np.repeat(g['los'], 400, axis=0)           # 1200 lines: the Morton order runs
    dist = los_cases.dist_from_plan(many)
    engine.import_state(g['X'])
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        try:
            for round_f32 in (0, 1):
                lp = _lp(g, round_f32, 1)
                for mode in (1, 2):
                    engine.set_option('los_mode', mode)
                    engine.los_accumulate(many.T.copy(), dist, lp)
                engine.los_spectrum(many.T.copy(), dist, lp, *VBINS, VSCALE)
        finally:
            engine.set_option('los_mode', 0)
        engine.sync()
    seen = _k_los_builds(e.name for e in prof.events())
    print('k_los kernels seen:', sorted(seen))
    assert seen == {'k_los_accumulate', 'k_los_prepare', 'k_los_key_scan', 'k_los_finish',
                    'k_los_extent', 'k_los_cell_count', 'k_los_cell_scatter<0>',
                    'k_los_cell_scatter<1>', 'k_los_candidates<0>', 'k_los_candidates<1>',
                    'k_los_resolve<0,0>', 'k_los_resolve<1,0>', 'k_los_resolve<0,1>',
                    'k_los_resolve<1,1>'}
