#!/usr/bin/env python
"""Benchmark of the nexoclom hot path on B200 (see DESIGN.md section 6).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--packets P] [--impl reference]
                    [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic packets: rewind the
resident initial state, K2 adaptive integration, K4 radiance image (800x800) --
BASELINE.json configs[1] (Na at Mercury, Maxwellian surface source, radiation pressure +
photoionisation, 1e7 packets per GPU).  Metric: packet-steps/s = attempted Dormand-Prince
steps / time, whole job over all GPUs.  Packets are sharded over ranks by global id (weak
scaling, no data-path collective); the per-GPU images are combined with ONE NCCL all-reduce
per run (inside the timed region).  `e2e` is the same work through the public API with host
buffers: Output(inputs, n, X0=<pinned host columns>) -> ModelImage.  The other kernels of the
path ride along as flat `config` keys: K1 (warm), K4 on an all-live state, K3 on configs[2],
K5 for 1e5 lines of sight incl. its host preparation, and -- at N > 1 -- an assertion that
the all-reduced product of two shards equals the single-rank product.

`--dump-outputs DIR` writes what the last timed step computed, so that two builds can be
compared output for output (the inputs depend only on the arguments): `image.npy` and
`packet_counts.npy` (the 800x800 radiance image and packet counts of one step, all ranks),
`step_totals.npy` (attempted, accepted steps of rank 0's K2) and, for a fixed seeded sample of
at most 2^18 of rank 0's packets, `packet_ids.npy`, `final_state.npy` (time, x, y, z, vx, vy,
vz, frac) and the per-packet `attempted_steps.npy` / `accepted_steps.npy`.  All float64,
under 34 MB in all.  `image` is the image accumulated over the K timed steps divided by K, and
K4 adds with atomics in no fixed order: it matches between runs and builds only to rounding,
not bit for bit (compare it with a relative tolerance); the other arrays of a build repeat
exactly.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
# the bench leaves the source tree untouched (it may be read-only): no bytecode caches there,
# in this process or in the worker processes it spawns
sys.dont_write_bytecode = True
os.environ['PYTHONDONTWRITEBYTECODE'] = '1'
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, 'tests'))

WORKLOAD = 'Na.maxwellian.radpres.input'
FLOP_PER_STEP = 764          # SURVEY section 8(d): algorithmic flop per attempted step
METRIC = 'packet-steps/s (FP64)'


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
         'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', f'--id={self.gpu}', f'--query-gpu={self.Q}',
                 '--format=csv,noheader,nounits', '-lms', '100'],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smmax, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for ln in self.lines:
            f = [x.strip() for x in ln.split(',')]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smmax.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': float(np.median(sm)) if sm else None,
                'sm_max_mhz': float(max(smmax)) if smmax else None,
                'samples': len(sm), 'reasons': sorted(reasons)}


def measured_peaks():
    path = os.path.join(REPO, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f), 'measured'
    return {'hbm_gbs': 6650.0}, 'fallback'


# ---------------------------------------------------------------------------
# CPU arms (oracle port of the reference's NumPy path)
# ---------------------------------------------------------------------------
def _cpu_chunk(args):
    name, X0 = args
    from common import workload, oracle_constants
    from nexoclom_b200.runsetup import RunSetup
    from oracle import tracking
    rc = oracle_constants(RunSetup(workload(name)))
    t0 = time.time()
    _, att, _ = tracking.integrate_adaptive(X0, rc)
    return int(att.sum()), time.time() - t0


def cpu_steps_per_s(X0, procs):
    """Oracle adaptive driver over X0 split into `procs` chunks; packet-steps/s."""
    import multiprocessing as mp
    chunks = np.array_split(X0, procs)
    t0 = time.time()
    if procs == 1:
        res = [_cpu_chunk((WORKLOAD, chunks[0]))]
    else:
        with mp.get_context('spawn').Pool(procs) as pool:
            res = pool.map(_cpu_chunk, [(WORKLOAD, c) for c in chunks])
    wall = time.time() - t0
    steps = sum(r[0] for r in res)
    return steps / wall, steps, wall


def synth_x0_host(n, seed=0):
    """Host-side synthetic initial state of the bench workload for the CPU arm
    (NumPy draws through the oracle's restatement of the reference's samplers)."""
    from common import workload
    from nexoclom_b200.runsetup import RunSetup
    from oracle import initial_state
    setup = RunSetup(workload(WORKLOAD))
    return initial_state.draw_x0(setup, n, seed)[:, :8]


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    procs = max(1, min(cores, 64))
    n = args.ref_packets * procs
    X0 = synth_x0_host(n)
    vals = []
    for it in range(args.warmup + args.steps):
        sps, steps, wall = cpu_steps_per_s(X0, procs)
        if it >= args.warmup:
            vals.append((sps, steps, wall))
    sps = float(np.mean([v[0] for v in vals]))
    ms = float(np.mean([v[2] for v in vals])) * 1e3
    sample = f'{n} packets of {WORKLOAD} per step ({procs} processes x {args.ref_packets})'
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': sps, 'unit': 'packet-steps/s',
        'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64',
        'data': 'synthetic',
        'config': {'workload': 'Na at Mercury, Maxwellian 1200 K surface source, radiation '
                               'pressure + photoionisation, adaptive RK5(4) (configs[1]); '
                               'bounded CPU sample', 'inputfile': WORKLOAD, 'packets': n},
        'cpu_baseline': {'value': sps, 'unit': 'packet-steps/s', 'cores': procs, 'kind': 'port',
                         'sample': sample},
        'e2e': {'value': sps, 'unit': 'packet-steps/s', 'h2d_bytes_per_step': 0,
                'd2h_bytes_per_step': 0},
    }
    emit(line)
    return 0


# ---------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------
FP64_LANES_PER_SM = 64       # DFMA per clock per SM on B200


def image_params(setup, quantity=1, round_f32=1, skip_dead=1, dims=800, width=8.0):
    """ImageParams of the default ModelImage view (ModelImage.py:53-68: from the north pole,
    800 x 800 pixels over 8 x 8 R_p)."""
    from nexoclom_b200._lib import ImageParams
    from nexoclom_b200.ModelImage import image_rotation
    M = np.asarray(image_rotation(0.0, np.pi / 2))
    ip = ImageParams()
    for k in range(9):
        ip.M[k] = float(M.flat[k])
    ip.x0, ip.x1, ip.z0, ip.z1 = -width / 2, width / 2, -width / 2, width / 2
    ip.nx = ip.nz = dims
    rcm = setup.radius_km * 1e5
    ip.apix = (width / dims * rcm) * (width / dims * rcm)
    ip.vrplanet = setup.vrplanet
    ip.quantity, ip.round_f32, ip.skip_dead = quantity, round_f32, skip_dead
    return ip, M


def synthetic_los(nlos, seed=1):
    """MESSENGER-UVVS-like sweep (BASELINE configs[4]): spacecraft on an eccentric polar
    ellipse 1.1 - 6 R_p, boresights towards points 1 - 4 R_p from the planet centre."""
    g = np.random.default_rng(seed)
    th = g.random(nlos) * 2 * np.pi
    rr = 1.1 + 4.9 * g.random(nlos)
    x_sc = np.stack([0.3 * rr * np.cos(th), 0.2 * rr * np.cos(th) - 0.5, rr * np.sin(th)])
    nrm = np.linalg.norm(x_sc, axis=0)
    x_sc *= np.maximum(nrm, 1.1) / nrm
    tgt = g.standard_normal((3, nlos))
    tgt *= (1 + 3 * g.random(nlos)) / np.linalg.norm(tgt, axis=0)
    bore = tgt - x_sc
    bore /= np.linalg.norm(bore, axis=0)
    dplan = np.linalg.norm(x_sc, axis=0)
    ang = np.arccos(-(x_sc * bore).sum(axis=0) / dplan)
    dplan = np.where(ang > np.arcsin(1. / dplan), 1e30, dplan)      # compute_iteration.py:105-115
    return np.ascontiguousarray(np.concatenate([x_sc, bore])), np.ascontiguousarray(dplan)


DUMP_SAMPLE = 1 << 18        # packets of the final state written by --dump-outputs
DUMP_SEED = 12345


def dump_outputs(dest, eng, img, cnt, steps, first_id):
    """What the last of `steps` timed steps computed, as float64 .npy files in `dest` (see the
    module docstring).  The engine still holds that step's final state and step counts; the
    context-owned image summed the same packets once per step."""
    n = eng.n
    idx = np.sort(np.random.default_rng(DUMP_SEED).choice(n, min(n, DUMP_SAMPLE), replace=False))
    state = eng.export_state()
    att, acc = eng.export_stats()
    out = {'image': img / steps, 'packet_counts': cnt // steps,
           'step_totals': [int(att.sum(dtype=np.int64)), int(acc.sum(dtype=np.int64))],
           'packet_ids': first_id + idx, 'final_state': state[:, idx].T,
           'attempted_steps': att[idx], 'accepted_steps': acc[idx]}
    os.makedirs(dest, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(dest, name + '.npy'), np.ascontiguousarray(a, dtype=np.float64))


def run_gpu(args):
    import torch
    import torch.distributed as dist
    from common import workload
    from nexoclom_b200 import Output, ModelImage, sharding
    from nexoclom_b200._lib import LosParams
    from nexoclom_b200.engine import get_engine
    from nexoclom_b200.runsetup import get_setup

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise RuntimeError('bench.py needs a CUDA device: nexoclom_b200 has no CPU fallback')
    torch.cuda.set_device(local)
    try:
        # run this rank (and first-touch its pinned buffers) on the CPUs next to its GPU
        if os.environ.get('NX_BENCH_NO_AFFINITY'):
            raise RuntimeError('affinity disabled')
        import pynvml
        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(local))
    except Exception:
        pass
    sharding.init()                                   # NCCL process group under torchrun
    comm = sharding.nccl_comm()                       # (lib, nx_comm) or None

    eng = get_engine(local)                           # the engine the product classes use
    stream = torch.cuda.current_stream()
    eng.set_stream(stream.cuda_stream)

    n = args.packets
    inputs = workload(WORKLOAD)
    setup = get_setup(inputs)
    setup.upload(eng)
    gt = setup.gtables([5891, 5897])
    eng.upload_gtables(gt)
    sp = setup.source_params(eng)
    first_id = rank * n
    ip, M = image_params(setup)
    extras = {}

    def fence():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def best_ms(fn, reps=3):
        b = 1e30
        for _ in range(reps):
            fn()
            eng.sync()
            b = min(b, eng.last_kernel_ms())
        return b

    peaks, peak_kind = measured_peaks()

    eng.init_state(sp, args.seed, first_id, n)        # resident inputs of the step
    eng.sync()
    extras['k1_first_launch_ms'] = eng.last_kernel_ms()

    # ---- the step: rewind the resident X0 -> K2 -> K4 into the context-owned image -----
    k2_ms, k4_ms, steps_total = [], [], []

    def one_step(record):
        eng.rewind_state()                          # the resident X0 is the input again
        att, _ = eng.integrate_adaptive(n)
        if record:
            k2_ms.append(eng.last_kernel_ms())
        eng.image_add(ip, n)
        if record:
            eng.sync()
            k4_ms.append(eng.last_kernel_ms())
            steps_total.append(att)

    eng.image_begin(800, 800)
    for _ in range(args.warmup):
        one_step(False)
    if comm is not None:
        eng.image_allreduce(comm[1])                # NCCL sets its channels up on first use
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()                             # (spawns nvidia-smi: before the fence, so
    eng.image_begin(800, 800)                       #  that every rank starts at the same time)
    fence()
    launches0 = eng.kernel_launches()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(args.steps):
        one_step(True)
    ev_pre = torch.cuda.Event(enable_timing=True)
    ev_pre.record(stream)
    if comm is not None:
        eng.image_allreduce(comm[1])                # ONE all-reduce per product (image + counts)
    ev1.record(stream)
    fence()
    launches = eng.kernel_launches() - launches0
    clocks = sampler.stop() if rank == 0 else None
    if comm is not None:                            # the collective on its own
        ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ar = []
        for _ in range(3):
            fence()
            ea.record(stream)
            eng.image_allreduce(comm[1])
            eb.record(stream)
            torch.cuda.synchronize()
            ar.append(ea.elapsed_time(eb))
        extras['allreduce_image_counts_ms'] = float(min(ar))
    elapsed_ms = ev0.elapsed_time(ev1)
    img_run, cnt_run = eng.image_fetch(800, 800)
    t = torch.tensor([elapsed_ms, float(sum(steps_total))], dtype=torch.float64, device='cuda')
    if world > 1:
        tmax = t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone()
        dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        tmin = t.clone()
        dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
        extras['rank_ms_per_step_min'] = float(tmin[0]) / args.steps
        extras['rank_ms_per_step_max'] = float(tmax[0]) / args.steps
        # per rank, without the collective: own steps, mean K2 and the host gap between kernels
        mine = torch.tensor([ev0.elapsed_time(ev_pre) / args.steps, float(np.mean(k2_ms)),
                             float(np.mean(k4_ms)), float(np.max(k2_ms))],
                            dtype=torch.float64, device='cuda')
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        extras['rank_own_ms_per_step'] = [round(float(v[0]), 3) for v in allr]
        extras['rank_k2_ms'] = [round(float(v[1]), 3) for v in allr]
        extras['rank_k2_max_ms'] = [round(float(v[3]), 3) for v in allr]
        elapsed_ms, all_steps = float(tmax[0]), float(tsum[1])
    else:
        all_steps = float(t[1])
    value = all_steps / (elapsed_ms * 1e-3)
    # the image accumulated over K steps of the same packets is K x one run's image
    live_hits = int(cnt_run.sum())
    extras['image_hits_per_step_all_ranks'] = live_hits // args.steps
    x0_dev_cols = None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, eng, img_run, cnt_run, args.steps, first_id)

    # ---- multi-rank product check: all-reduced == recomputed on rank 0 ------------------
    if world > 1:
        m = args.check_packets
        ipc, _ = image_params(setup, dims=200)
        img = np.zeros((200, 200))
        cnt = np.zeros((200, 200), dtype=np.int64)
        if rank < 2:
            eng.init_state(sp, args.seed + 7, rank * m, m)
            eng.integrate_adaptive(m)
            img, cnt = eng.image_accumulate(ipc, m)
        sharding.allreduce_sum(img, cnt)
        if rank == 0:
            eng.init_state(sp, args.seed + 7, 0, 2 * m)        # both shards as ONE run
            eng.integrate_adaptive(2 * m)
            img1, cnt1 = eng.image_accumulate(ipc, 2 * m)
            if not np.array_equal(cnt, cnt1):
                raise AssertionError('all-reduced packet counts differ from the single-rank run')
            nz = img1 > 0
            err = float(np.max(np.abs(img[nz] - img1[nz]) / img1[nz]))
            if not (np.array_equal(nz, img > 0) and err < 1e-12):
                raise AssertionError(f'all-reduced image differs from the single-rank run: {err}')
            extras['multirank_check'] = (f'2 shards x {m} packets: counts exact '
                                         f'({int(cnt.sum())} hits), image max rel diff {err:.1e}')
        eng.init_state(sp, args.seed, first_id, n)             # the bench state again

    # ---- end to end through the public API, HOST buffers (import mode) ------------------
    # Output(inputs, n, X0=<host columns>) -> ModelImage(inputs, params): pinned H2D of the
    # initial state (64 B/packet) streamed behind K2, device-side Output.save (compaction +
    # float32), K4 over the resident table, one all-reduce, D2H of image + packet image.
    e2e = None
    params = {'quantity': 'radiance'}
    if not args.no_e2e:
        host_in = torch.empty((8, n), dtype=torch.float64).pin_memory()
        x0h = eng.export_x0()[:8]
        host_in.copy_(torch.from_numpy(x0h))
        del x0h
        host_np = host_in.numpy()
        cols = {c: host_np[k] for k, c in enumerate(
            ('time', 'x', 'y', 'z', 'vx', 'vy', 'vz', 'frac'))}
        reps = max(1, min(args.steps, 5))
        rep_ms, rep_steps = [], []
        warm = 2           # (the page-locked result arrays of two generations of ModelImage)
        for it in range(warm + reps):
            inputs.delete_files()
            fence()
            t0 = time.perf_counter()
            out = Output(inputs, n, X0=cols, first_id=first_id)
            t1 = time.perf_counter()
            im = ModelImage(inputs, params)
            checksum = float(im.image.sum())                   # the result is on the host
            t2 = time.perf_counter()
            fence()
            if it >= warm:
                rep_ms.append((time.perf_counter() - t0) * 1e3)
                rep_steps.append(float(out.attempted_steps))
                print(f'e2e rep {it - warm + 1}: Output {1e3 * (t1 - t0):.2f} ms (kernels {out.kernel_ms:.2f}), '
                      f'ModelImage {1e3 * (t2 - t1):.2f} ms', file=sys.stderr)
        inputs.delete_files()
        # per repetition: the slowest rank's time and the steps of all ranks; the line quotes
        # the MEDIAN repetition (a single host hiccup on one of N ranks otherwise decides a
        # 3-5 sample mean), the mean is reported next to it
        tm = torch.tensor(rep_ms, dtype=torch.float64, device='cuda')
        ts = torch.tensor(rep_steps, dtype=torch.float64, device='cuda')
        if world > 1:
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
            dist.all_reduce(ts, op=dist.ReduceOp.SUM)
        e2e_ms = float(tm.median())
        e2e_steps = float(ts[0])
        e2e = {'value': e2e_steps / (e2e_ms * 1e-3), 'unit': 'packet-steps/s',
               'h2d_bytes_per_step': 64 * n, 'd2h_bytes_per_step': 2 * 8 * 800 * 800,
               'ms_per_step': e2e_ms, 'ms_per_step_mean': float(tm.mean()),
               'ms_per_step_all': [round(float(v), 3) for v in tm],
               'stat': f'median of {reps} repetitions, each = max over ranks',
               'call': 'Output(inputs, n, X0=<pinned host columns>, first_id) -> '
                       'ModelImage(inputs, {quantity: radiance}) -> image on the host',
               'image_checksum': checksum}

        # the product's normal path draws the packets on the device (K1): Input.run -> ModelImage
        api_ms, api_steps = [], []
        for it in range(1 + reps):
            inputs.delete_files()
            fence()
            t0 = time.perf_counter()
            inputs.run(n * world, seed=args.seed, overwrite=True)
            im = ModelImage(inputs, params)
            float(im.image.sum())
            fence()
            if it > 0:
                api_ms.append((time.perf_counter() - t0) * 1e3)
                _, files, _, _ = inputs.search()
                from nexoclom_b200 import catalogue
                api_steps.append(float(sum(catalogue.fetch(f).attempted_steps for f in files)))
        inputs.delete_files()
        tm = torch.tensor(api_ms, dtype=torch.float64, device='cuda')
        ts = torch.tensor(api_steps, dtype=torch.float64, device='cuda')
        if world > 1:                                  # per repetition: slowest rank, all steps
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
            dist.all_reduce(ts, op=dist.ReduceOp.SUM)
        api_med = float(tm.median())
        extras['api_device_drawn_steps_per_s'] = float(ts[0]) / (api_med * 1e-3)
        extras['api_device_drawn_ms_per_step'] = api_med
        extras['api_device_drawn_ms_per_step_all'] = [round(float(v), 3) for v in tm]
        extras['api_device_drawn_call'] = 'Input.run(n) -> ModelImage(inputs, params)'
        del host_in, host_np, cols

    # ---- K5: line-of-sight sweep over the resident final state (configs[4]) -------------
    if not args.no_los:
        setup.upload(eng)
        eng.upload_gtables(gt)
        eng.init_state(sp, args.seed, first_id, n)
        eng.integrate_adaptive(n)                              # the final state of the run
        nlos = args.los
        los, dplan = synthetic_los(nlos)
        lp = LosParams()
        lp.dphi, lp.outeredge = float(np.radians(1.0)), 25.0
        lp.vrplanet, lp.rp_cm = setup.vrplanet, setup.radius_km * 1e5
        lp.quantity, lp.round_f32, lp.skip_dead = 1, 1, 0
        wall, kern = [], []
        for it in range(3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            rad, npk, inc = eng.los_accumulate(los, dplan, lp, n=n)   # host prep + kernels + D2H
            wall.append((time.perf_counter() - t0) * 1e3)
            kern.append(eng.last_kernel_ms())
        hits = np.array([float(npk.sum())])
        if world > 1:
            sharding.allreduce_sum(rad, npk)
        extras.update(k5_lines_of_sight=nlos, k5_packets_per_gpu=n, k5_dphi_deg=1.0,
                      k5_ms_incl_host_prep=float(min(wall)), k5_kernel_ms=float(min(kern)),
                      k5_ms_per_1e8_packets=float(min(wall)) * 1e8 / n,
                      k5_hits=int(hits[0]),
                      k5_effective_pairs_per_s=float(nlos) * n / (min(wall) * 1e-3))

    # ---- K3: configs[2] physics (bounce, T-dependent sticking), image fused -------------
    if not args.no_k3:
        n3 = args.k3_packets
        setup3 = get_setup(workload('Na.bounce.input'))
        setup3.upload(eng)
        eng.upload_gtables(setup3.gtables([5891, 5897]))
        sp3 = setup3.source_params(eng)
        ip3, _ = image_params(setup3)
        res3 = {}
        for fused in (False, True):
            ms = []
            for it in range(2):
                eng.init_state(sp3, args.seed, rank * n3, n3)
                if fused:
                    eng.image_begin(800, 800)
                    a, b = eng.image_device_ptrs()
                    _, nsteps, psteps = eng.integrate_constant(
                        seed=args.seed + 1, first_id=rank * n3, image_params=ip3, image_dev=a,
                        counts_dev=b, n=n3)
                else:
                    _, nsteps, psteps = eng.integrate_constant(seed=args.seed + 1,
                                                               first_id=rank * n3, n=n3)
                eng.sync()
                ms.append(eng.last_kernel_ms())
            res3[fused] = (min(ms), psteps, nsteps)
        sm_mhz = (clocks or {}).get('sm_mhz') or peaks.get('sm_max_mhz', 1965.0)
        nominal = 148 * FP64_LANES_PER_SM * 2 * sm_mhz * 1e6 / 1e12
        for fused, tag in ((False, 'k3'), (True, 'k3_fused_image')):
            ms, psteps, nsteps = res3[fused]
            sps = psteps / (ms * 1e-3)
            extras[f'{tag}_steps_per_s'] = sps
            extras[f'{tag}_ms'] = ms
            extras[f'{tag}_fp64_frac'] = sps * 626 / 1e12 / nominal
        extras.update(k3_packets_per_gpu=n3, k3_nsteps=int(res3[False][2]),
                      k3_flop_per_packet_step=626,
                      k3_workload='Na.bounce.input (BASELINE configs[2])')
        setup.upload(eng)                                      # back to the configs[1] tables
        eng.upload_gtables(gt)
        sp = setup.source_params(eng)

    # ---- K1 (warm) and K4 on an ALL-LIVE state, at the size the metric is quoted on -------
    if not args.no_k14:
        nk = args.k14_packets
        eng.init_state(sp, args.seed, rank * nk, nk)
        k1 = best_ms(lambda: eng.init_state(sp, args.seed, rank * nk, nk))
        extras.update(k14_packets_per_gpu=nk, k1_ms=k1, k1_bytes_per_packet=112,
                      k1_hbm_gbs=112.0 * nk / k1 / 1e6,
                      k1_hbm_frac=112.0 * nk / k1 / 1e6 / peaks['hbm_gbs'])
        eng.image_begin(800, 800)
        for name, quantity in (('column', 0), ('radiance', 1)):
            ipa, _ = image_params(setup, quantity=quantity, skip_dead=0)
            t = best_ms(lambda: eng.image_add(ipa, nk))
            extras[f'k4_alllive_{name}_ms_per_1e8'] = t * 1e8 / nk
            extras[f'k4_alllive_{name}_hbm_frac'] = 40.0 * nk / t / 1e6 / peaks['hbm_gbs']
        extras['k4_alllive_state'] = ('the initial state: every packet live, all of them on the '
                                      'planet disk of the image (worst case for the atomics)')

    if rank == 0:
        fp64_micro = eng.measure_fp64_peak()
        sm_mhz = (clocks or {}).get('sm_mhz') or peaks.get('sm_max_mhz', 1965.0)
        nominal = 148 * FP64_LANES_PER_SM * 2 * sm_mhz * 1e6 / 1e12
        k2 = float(np.mean(k2_ms))
        k4 = float(np.mean(k4_ms))
        steps_per_launch = float(np.mean(steps_total))
        achieved = steps_per_launch * FLOP_PER_STEP / (k2 * 1e-3) / 1e12
        traffic = None
        tpath = os.path.join(REPO, 'profiles', 'k2_traffic_bytes.json')
        if os.path.exists(tpath):
            with open(tpath) as f:
                traffic = json.load(f).get('dram_bytes_per_launch')
        config = {
            'workload': 'BASELINE configs[1]: Na at Mercury, Maxwellian 1200 K surface source, '
                        'radiation pressure + photoionisation, adaptive RK5(4), 800x800 '
                        'radiance image',
            'inputfile': WORKLOAD, 'packets_per_gpu': n, 'packets_total': n * world,
            'attempted_steps_per_packet': steps_per_launch / n,
            'l2': 'inputs (640 MB state per 1e7 packets) exceed the 126 MB L2; no flush',
            'step': 'rewind resident X0 -> K2 adaptive integrate -> K4 image'
                    + ('; ONE NCCL all-reduce(image, counts) per run' if world > 1 else ''),
            'k2_integrate_ms': k2, 'k4_image_ms': k4,
            'k4_benchstate_ms_per_1e8_packets': k4 * 1e8 / n,
            'fp64_peak_microbenchmark_tflops': fp64_micro,
        }
        config.update(extras)
        line = {
            'metric': METRIC, 'value': value, 'unit': 'packet-steps/s', 'n_gpus': world,
            'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': elapsed_ms / args.steps, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
            'config': config,
            'roofline': {
                'bound': 'fp64', 'kernel': 'k_integrate_adaptive', 'achieved': achieved,
                'peak': nominal, 'unit': 'TFLOP/s', 'frac': achieved / nominal,
                'traffic': traffic,
                'peak_source': f'nominal 148 SM x 64 DFMA/clk x 2 at the SM clock observed '
                               f'during the timed region ({sm_mhz:.0f} MHz); MEASURED_PEAKS.json '
                               f'has no FP64 entry; live DFMA microbenchmark reads '
                               f'{fp64_micro:.1f}',
                'flop_per_packet_step': FLOP_PER_STEP,
            },
            'e2e': e2e,
            'gpu_launches': int(launches),
            'clocks': clocks,
        }
        if world == 1 and not args.no_cpu:
            eng.init_state(sp, args.seed, first_id, args.cpu_packets)
            X0h = np.ascontiguousarray(eng.export_x0()[:8].T)
            sps, steps, wall = cpu_steps_per_s(X0h, 1)
            line['cpu_baseline'] = {
                'value': sps, 'unit': 'packet-steps/s', 'cores': 1, 'kind': 'port',
                'sample': f'first {args.cpu_packets} packets of the same X0, '
                          f'{steps} steps in {wall:.1f} s, NumPy oracle port of the '
                          'reference driver, 1 process (host has '
                          f'{os.cpu_count()} cores)'}
            m = min(n, args.cpu_product_packets)
            eng.init_state(sp, args.seed, first_id, m)
            eng.integrate_adaptive(m)
            fin = eng.export_state()[[1, 2, 3, 5, 7]]
            cp = cpu_products(fin, setup, gt, M, ip.apix,
                              synthetic_los(args.cpu_product_los)[0].T.copy()
                              if not args.no_los else None)
            config['cpu_image_ms_per_1e8_packets'] = cp['image']['ms_per_1e8_packets']
            if 'los' in cp:
                config['cpu_los_ms_per_line_of_sight_1e6_packets'] = cp['los']['ms_per_line_of_sight']
        emit(line)
    fence()
    if world > 1:
        dist.destroy_process_group()
    return 0


def cpu_products(fin, setup, gtables, M, apix, los):
    """CPU timings of the two products of the path on a bounded sample of the bench's final
    state: the NumPy oracle port of create_image (two np.histogram2d passes) and of the
    compute_iteration loop (sklearn KDTree), one process each."""
    from oracle import imaging
    x, y, z, vy, frac = (np.ascontiguousarray(fin[k].astype(np.float32).astype(np.float64))
                         for k in range(5))
    m = len(x)
    t0 = time.time()
    imaging.create_image(x, y, z, vy, frac, vrplanet=setup.vrplanet, M=M, dims=[800, 800],
                         xrange=(-4., 4.), zrange=(-4., 4.), apix=apix, quantity='radiance',
                         gtables=gtables)
    t_img = time.time() - t0
    out = {'image': {'packets': m, 'ms': t_img * 1e3, 'ms_per_1e8_packets': t_img * 1e3 * 1e8 / m,
                     'kind': 'port', 'cores': 1}}
    if los is not None and len(los):
        t0 = time.time()
        _, npk, _, _ = imaging.los_iteration(
            x, y, z, vy, frac, los, vrplanet=setup.vrplanet, dphi=float(np.radians(1.0)),
            outeredge=25.0, rp_cm=setup.radius_km * 1e5, gtables=gtables)
        t_los = time.time() - t0
        out['los'] = {'packets': m, 'lines_of_sight': int(len(los)), 's': t_los,
                      'ms_per_line_of_sight': t_los * 1e3 / len(los), 'hits': int(npk.sum()),
                      'kind': 'port', 'cores': 1}
    return out


_OUT = None


def claim_stdout():
    """Keep stdout for the ONE JSON line: whatever libraries print there while the bench runs
    (NCCL writes its version banner to stdout) is sent to stderr instead."""
    global _OUT
    if _OUT is None:
        sys.stdout.flush()
        _OUT = os.fdopen(os.dup(1), 'w')
        os.dup2(2, 1)


def emit(line):
    out = _OUT if _OUT is not None else sys.stdout
    out.write(json.dumps(line) + '\n')
    out.flush()


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--packets', type=int, default=10_000_000, help='packets per GPU')
    ap.add_argument('--cpu-packets', type=int, default=100000,
                    help='packets of the bounded CPU sample (about 15 s on one core)')
    ap.add_argument('--cpu-product-packets', type=int, default=1_000_000,
                    help='packets of the CPU image / line-of-sight timing sample')
    ap.add_argument('--cpu-product-los', type=int, default=200,
                    help='lines of sight of the CPU line-of-sight timing sample')
    ap.add_argument('--ref-packets', type=int, default=20000,
                    help='packets per host process and step of the --impl reference arm')
    ap.add_argument('--seed', type=int, default=0)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--no-los', action='store_true')
    ap.add_argument('--no-e2e', action='store_true',
                    help='skip the end-to-end leg (its streaming kernel waits for concurrent '
                         'copies, which a serialising profiler never runs)')
    ap.add_argument('--los', type=int, default=100_000, help='lines of sight of the K5 sweep')
    ap.add_argument('--no-k3', action='store_true', help='skip the configs[2] (K3) leg')
    ap.add_argument('--no-k14', action='store_true', help='skip the K1 / all-live K4 leg')
    ap.add_argument('--k14-packets', type=int, default=100_000_000,
                    help='packets per GPU of the K1 / all-live K4 leg (18 GB of slabs at 1e8)')
    ap.add_argument('--k3-packets', type=int, default=12_500_000,
                    help='packets per GPU of the configs[2] leg (361 steps each; 1e8 / 8 GPUs)')
    ap.add_argument('--check-packets', type=int, default=200_000,
                    help='packets per shard of the multi-rank product check')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write what the last timed step computed to DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be at least 1 and --warmup at least 0')
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs writes the products of the GPU path (--impl b200)')
    if args.impl == 'reference':
        return run_reference(args)
    return run_gpu(args)


if __name__ == '__main__':
    sys.exit(main())
