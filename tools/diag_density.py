#!/usr/bin/env python
"""K7 timing: number density at sample points over the configs[1] final state (1e7 packets,
adaptive Na with radiation pressure), three kinds of sample sets:

  (a) a 1e4-point orbit-like track, altitudes 0.05-5 R_p, r = 0.05 R_p;
  (b) a 64^3 grid over +-4 R_p, r = the grid spacing;
  (c) a 200-point altitude profile above the subsolar point, r = 0.2 altitude + 0.02 R_p.

The same cases run on the initial state of the same packets too (every packet live, at the
surface): the final state keeps only the rows that were neither ionised nor stuck.

Per case: CUDA-event times of the cell-grid build (a call with one empty ball) and of the
query (a full call minus the build), the records the query streams (the grid is replayed on
the host: same cell rule, NumPy's asinh), the member rows, and the byte floor: 16 B per
streamed record over the measured device copy bandwidth.  Then the same track on 1e6 packets
against scipy's cKDTree on the CPU.  Prints the GPU's name and power limit with the numbers;
writes them as JSON too when a path is given.

    python tools/diag_density.py [npackets] [report.json]
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
from nexoclom_b200.engine import Engine                                  # noqa: E402
from nexoclom_b200.runsetup import RunSetup                              # noqa: E402
from oracle import density as odens                                      # noqa: E402


def gpu_identity():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm',
                              '--format=csv,noheader'], capture_output=True, text=True, timeout=30)
        return out.stdout.strip().splitlines()[0]
    except Exception as e:                                              # noqa: BLE001
        return f'nvidia-smi unavailable ({e})'


def orbit_track(n):
    th = np.linspace(0, 2 * np.pi, n, endpoint=False)
    rp, ra = 1.05, 6.0
    a, e = (rp + ra) / 2, (ra - rp) / (ra + rp)
    rr = a * (1 - e * e) / (1 + e * np.cos(th))
    inc = np.radians(80.0)
    u = np.stack([np.cos(th), np.sin(th) * np.cos(inc), np.sin(th) * np.sin(inc)], axis=1)
    return u * rr[:, None], np.full(n, 0.05)


def grid_cube():
    ax = np.linspace(-4, 4, 64)
    X, Y, Z = np.meshgrid(ax, ax, ax, indexing='ij')
    return np.stack([X.ravel(), Y.ravel(), Z.ravel()], axis=1), np.full(64**3, ax[1] - ax[0])


def profile():
    alt = np.geomspace(0.005, 5.0, 200)
    pts = np.zeros((200, 3))
    pts[:, 1] = -(1 + alt)                                   # Sun at -y
    return pts, 0.2 * alt + 0.02


class HostGrid:
    """launch_los_grid_build's cell rule, replayed on the host to count streamed records."""

    def __init__(self, P):
        ext = float(np.abs(P).max()) if len(P) else 1.0
        G = int(0.55 * np.cbrt(max(len(P), 1)) / 32.0 + 0.5) * 32
        self.G = G = min(max(G, 32), 160)
        self.half = ext * (1 + 1e-9) + 1e-9
        self.scale = min(self.half, 1.0)
        self.k = 0.5 * G / np.arcsinh(self.half / self.scale)
        c = [self.cell(P[:, a]) for a in range(3)]
        cnt = np.bincount((c[0] * G + c[1]) * G + c[2], minlength=G**3).reshape(G, G, G)
        self.cum = np.zeros((G + 1, G + 1, G + 1), dtype=np.int64)
        self.cum[1:, 1:, 1:] = cnt.cumsum(0).cumsum(1).cumsum(2)

    def cell(self, v):
        c = np.floor(self.k * np.arcsinh(v / self.scale) + 0.5 * self.G).astype(np.int64)
        return np.clip(c, 0, self.G - 1)

    def streamed(self, pts, rad):
        rr = rad * (1 + 1e-9) + 1e-12
        lo = [self.cell(pts[:, a] - rr) for a in range(3)]
        hi = [self.cell(pts[:, a] + rr) + 1 for a in range(3)]
        out = np.abs(pts) - rr[:, None] > self.half
        C = self.cum
        tot = (C[hi[0], hi[1], hi[2]] - C[lo[0], hi[1], hi[2]] - C[hi[0], lo[1], hi[2]]
               - C[hi[0], hi[1], lo[2]] + C[lo[0], lo[1], hi[2]] + C[lo[0], hi[1], lo[2]]
               + C[hi[0], lo[1], lo[2]] - C[lo[0], lo[1], lo[2]])
        return int(np.where(out.any(axis=1), 0, tot).sum())


def timed(eng, table, pts, rad, reps):
    ms = []
    for _ in range(reps):
        s1, s2 = np.zeros(len(pts)), np.zeros(len(pts))
        c = np.zeros(len(pts), dtype=np.int64)
        eng.bind_packets(table)
        eng.density_accumulate(pts, rad, s1, s2, c, n=table.n)
        eng.bind_packets(None)
        ms.append(eng.last_kernel_ms())
    return float(np.median(ms)), (s1, s2, c)


def main():
    n = int(float(sys.argv[1])) if len(sys.argv) > 1 else 10_000_000
    ident = gpu_identity()
    print('GPU (name, power limit, max SM clock):', ident)
    eng = Engine(0)
    bw = eng.measure_copy_bw(1 << 31) * 1e9            # read + write bytes per second
    print(f'device copy bandwidth {bw / 1e12:.2f} TB/s')
    setup = RunSetup(workload('Na.maxwellian.radpres.input'))
    setup.upload(eng)
    sp = setup.source_params(eng)
    report = {'gpu': ident, 'copy_bw_TBs': bw / 1e12, 'npackets': n, 'sets': {}}
    empty = (np.array([[1e6, 0.0, 0.0]]), np.array([1e-3]))
    # the final state keeps the ~1 % of the packets that are neither ionised nor stuck; the
    # initial state (every packet live, all at the surface) is the dense near-planet extreme
    for label, integrate in (('final_state', True), ('initial_state_all_live', False)):
        eng.init_state(sp, 1, 0, n)
        if integrate:
            eng.integrate_adaptive(n)
        table = eng.compact_state(skip_dead=True, round_f32=True, n=n)
        cols, _ = table.export()
        P = np.stack([cols['x'], cols['y'], cols['z']], axis=1).astype(np.float64)
        frac = cols['frac']
        hg = HostGrid(P)
        timed(eng, table, *empty, 2)                   # warm-up
        build_ms, _ = timed(eng, table, *empty, 5)
        rep = report['sets'][label] = {'rows': table.n, 'grid_G': hg.G, 'build_ms': build_ms,
                                       'cases': {}}
        print(f'{label}: {n} packets, {table.n} saved rows, grid G = {hg.G}, '
              f'build (a call with one empty ball) {build_ms:.3f} ms')
        for name, (pts, rad) in (('a_track_1e4', orbit_track(10_000)),
                                 ('b_grid_64cube', grid_cube()), ('c_profile_200', profile())):
            timed(eng, table, pts, rad, 1)
            total_ms, (s1, s2, c) = timed(eng, table, pts, rad, 5)
            query_ms = total_ms - build_ms
            streamed = hg.streamed(pts, rad)
            floor_ms = streamed * 16 / bw * 1e3
            rep['cases'][name] = dict(points=len(pts), total_ms=total_ms, query_ms=query_ms,
                                      streamed=streamed, members=int(c.sum()),
                                      max_members=int(c.max()), floor_ms=floor_ms,
                                      query_over_floor=query_ms / max(floor_ms, 1e-12))
            print(f'  {name}: {len(pts)} points, call {total_ms:.3f} ms, query {query_ms:.3f} ms, '
                  f'streamed {streamed:.4g} records, members {c.sum():.4g} (max {c.max()}), '
                  f'byte floor {floor_ms:.4f} ms, query / floor {query_ms / max(floor_ms, 1e-12):.1f}')
        table.free()

    # 1e6 rows of the initial state: the GPU against cKDTree (build + query + the exact
    # rule) on the CPU
    m = 1_000_000
    small = eng.upload_packets([np.zeros(m)] + [P[:m, a] for a in range(3)] +
                               [np.zeros(m)] * 3 + [frac[:m].astype(np.float64)])
    pts, rad = orbit_track(10_000)
    timed(eng, small, pts, rad, 1)
    g_ms, (s1, s2, c) = timed(eng, small, pts, rad, 5)
    t0 = time.perf_counter()
    o1, o2, oc = odens.ball_sums_kdtree(P[:m], frac[:m], pts, rad)
    cpu_ms = (time.perf_counter() - t0) * 1e3
    assert np.array_equal(c, oc), 'GPU counts differ from the oracle'
    small.free()
    report['kdtree_1e6'] = dict(points=len(pts), gpu_call_ms=g_ms, cpu_kdtree_ms=cpu_ms,
                                members=int(oc.sum()), cpu_threads=os.cpu_count())
    print(f'1e6 initial-state rows, track (a): GPU call {g_ms:.3f} ms, cKDTree on the CPU {cpu_ms:.1f} ms '
          f'(tree build + query + exact rule, {os.cpu_count()} CPUs), counts equal')
    eng.close()
    if len(sys.argv) > 2:
        with open(sys.argv[2], 'w') as f:
            json.dump(report, f, indent=1)


if __name__ == '__main__':
    main()
