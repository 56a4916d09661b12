"""``Output``: initial state + packet tracking on the GPU.

Drop-in for the reference ``particle_tracking/Output.py:23-202`` -- same
constructor, same attributes (``X0, X, npackets, totalsource, unit, GM, aplanet,
vrplanet, radpres, loss_info, compress, filename, idnum``) -- with the bodies of
``surface/speed/angular_distribution`` (:160-170), ``variable_step_size_driver``
(:221-366), ``constant_step_size_driver`` (:368-455) and the frac > 0 / float32 part of
``save`` (:522-543) replaced by calls through the C ABI (``nx_init_state``,
``nx_integrate_adaptive``, ``nx_integrate_constant[_rows]``, ``nx_compact_state``).

What differs from the reference is WHERE the packets live, not what they are: after the run
the rows the reference would pickle (frac > 0 when ``compress``, float32) stay on the GPU as
a compacted ``PacketTable``; ``ModelImage`` / ``LOSResult`` of the same process read it
there.  ``X`` and ``X0`` are built on first access (``X0`` by re-running K1: the packets are
a pure function of (seed, global packet id)), and only when the run is written to disk
(``NEXOCLOM_B200_SAVEPATH``) do the surviving rows cross PCIe, as float32.

Extensions: ``X0=`` accepts a reference-generated initial state (import mode);
``first_id=`` is the global id of the first packet (sharded runs: the Philox counter of
packet i is ``first_id + i``, so products do not depend on the number of GPUs).
"""
import copy
import os

import numpy as np
import pandas as pd

from . import catalogue
from .engine import get_engine, STATE_COLS, X0_COLS
from .runsetup import get_setup
from .units import Quantity, def_unit


class RadPres:
    """Radiation-pressure table the reference attaches as ``output.radpres``
    (velocity [R_p/s], accel [R_p/s^2]; reference Output.py:113-121).  Module level: saved
    Outputs are pickles."""
    velocity = None
    accel = None


def _max_rows():
    """Rows of a constant-step run that are kept resident as one table (about 70 B each)."""
    return int(float(os.environ.get('NEXOCLOM_B200_MAX_ROWS', '4e8')))


class Output:
    def __init__(self, inputs, npackets, compress=True, run_model=True, seed=None,
                 X0=None, device=None, strict_math=False, keep_trajectory=None, first_id=0):
        from .sharding import local_device
        self.inputs = inputs
        self.planet = inputs.geometry.planet
        npackets = int(npackets)
        self._X = self._X0 = None
        self._table = None           # resident PacketTable (what save() would pickle)
        self._host = None            # the same rows as float32 host arrays (evicted / unpickled)
        self._upcast = False
        self.first_id = int(first_id)
        self.strict_math = bool(strict_math)
        self.device = local_device() if device is None else int(device)
        if run_model:
            # the reference seeds numpy's PCG64 (Output.py:92); here the seed keys the
            # per-packet Philox streams.  seed=None -> fresh entropy, like default_rng(None)
            if seed is None:
                seed = int(np.random.SeedSequence().entropy & ((1 << 63) - 1))
            self.seed = int(seed)

            assert self.inputs.geometry.type != 'geometry with time', (
                'Initialization with time stamp not implemented yet.')
            self.compress = compress
            self.unit = def_unit('R_' + self.planet.object, 'length',
                                 float(self.planet.radius.value) * 1e3)

            setup = get_setup(inputs, strict_math=strict_math)
            self.GM = setup.GM
            self.aplanet = setup.aplanet
            self.vrplanet = setup.vrplanet
            self.loss_info = setup.loss_info
            self.radpres = None
            if inputs.forces.radpres:
                self.radpres = RadPres()
                self.radpres.velocity = setup.radpres_v
                self.radpres.accel = setup.radpres_a
            if setup.surfaceint is not None:
                self.surfaceint = setup.surfaceint

            self.npackets = npackets
            self.totalsource = float(npackets)        # sum of frac == 1 (Output.py:150)

            # The reference stops here for planets with moons (`assert False, 'Not set up'`,
            # Output.py:153-155) and for StartPoint != planet (:173-175).  Extension: moons
            # listed in geometry.objects act on the packets from circular orbits at the
            # phases geometry.phi, and a moon can be the start point (DESIGN.md section 8).
            if setup.moons:
                print('Including the gravity of ' + ', '.join(m['name'] for m in setup.moons))

            eng = get_engine(self.device)
            setup.upload(eng)

            self.imported_x0 = X0 is not None
            host_cols = None
            if X0 is not None:
                cols = self._coerce_x0(X0, npackets)
                if self.inputs.options.step_size == 0:
                    # adaptive run on imported packets: the copy is streamed behind the
                    # integrator (nx_integrate_adaptive_host), see variable_step_size_driver
                    host_cols = cols
                else:
                    eng.import_state(cols)
                self._imported_cols = cols           # X0 (a 64 B/packet frame) is built on access
            else:
                if self.inputs.spatialdist.type not in ('uniform', 'surface map',
                                                        'surface spot'):
                    assert 0, 'Not a valid spatial distribution type'
                eng.init_state(setup.source_params(eng), self.seed, self.first_id, npackets)

            if self.inputs.options.step_size == 0:
                print('Running variable step size integrator.')
                self.variable_step_size_driver(eng, host_cols)
            else:
                print('Running constant step size integrator.')
                self.constant_step_size_driver(eng, setup, keep_trajectory)
            self._finish_units()
        else:
            print('Not running anything')
            self.compress = False
            self._X0 = pd.DataFrame()
            self._X = pd.DataFrame()
            self.npackets = npackets
            self.totalsource = npackets

        self.save()

    @staticmethod
    def _coerce_x0(X0, npackets):
        if isinstance(X0, pd.DataFrame):
            cols = [np.ascontiguousarray(X0[c].values, dtype=np.float64) for c in STATE_COLS]
        elif isinstance(X0, dict):
            cols = [np.ascontiguousarray(X0[c], dtype=np.float64) for c in STATE_COLS]
        else:
            a = np.asarray(X0, dtype=np.float64)
            assert a.ndim == 2 and a.shape[1] == 8, 'X0 must be (N, 8)'
            cols = [np.ascontiguousarray(a[:, k]) for k in range(8)]
        assert len(cols[0]) == npackets, 'X0 length != npackets'
        return cols

    def __len__(self):
        return self.npackets

    def __getitem__(self, keys):
        self.X = self.X.iloc[keys]

    # ------------------------------------------------------------------
    def variable_step_size_driver(self, eng, host_cols=None):
        """Adaptive driver on the GPU (K2).  Semantics of reference
        Output.py:221-366, including quirks Q1-Q9 (see DESIGN.md).  Extension: a surface that
        does not absorb every packet (stickcoef < 1, temperature-dependent sticking) makes the
        packets bounce (K3's surface interaction, deviates keyed by ``seed`` and the packet
        id); ``bounces`` counts the surface interactions of the run."""
        p = eng.params
        self.bounces = 0
        if not (p.sticktype == 0 and p.stickcoef == 1.0):
            if host_cols is not None:
                eng.import_state(host_cols)
            self.attempted_steps, self.accepted_steps, self.bounces = eng.integrate_adaptive_bounce(
                self.seed, self.first_id, self.npackets)
        elif host_cols is not None:
            self.attempted_steps, self.accepted_steps = eng.integrate_adaptive_host(
                host_cols, nchunks=16)
        else:
            self.attempted_steps, self.accepted_steps = eng.integrate_adaptive(self.npackets)
        self.kernel_ms = eng.last_kernel_ms()
        # Output.save on the device: frac > 0 rows (if compress), float32, packet index
        self._table = eng.compact_state(skip_dead=self.compress, round_f32=True,
                                        n=self.npackets)
        self.trajectory_kept = True

    def constant_step_size_driver(self, eng, setup, keep_trajectory=None):
        """Constant-step driver + bounce on the GPU (K3).  Semantics of reference
        Output.py:368-455: every step of every packet is a row of ``X``
        (``totalsource *= nsteps``).  The dense (N, 8, nsteps) tensor never exists: the rows
        ``save`` would keep are appended to a resident table inside the integrator.  A run
        whose rows exceed ``NEXOCLOM_B200_MAX_ROWS`` keeps only its recipe (seed, first
        packet id, count): packets and bounce deviates are pure functions of (seed, packet
        id, step), so ``tables()`` regenerates the same rows chunk by chunk for
        ``ModelImage`` / ``LOSResult``."""
        p = setup.params
        self.nsteps = int(np.ceil(p.endtime / p.step_size + 1))
        if keep_trajectory is None:
            keep_trajectory = self.npackets * self.nsteps <= _max_rows()
        if keep_trajectory:
            self._table, _, self.attempted_steps = eng.integrate_constant_rows(
                seed=self.seed, first_id=self.first_id, skip_dead=self.compress, round_f32=True,
                n=self.npackets)
        else:
            if self.imported_x0 or not self.compress:
                raise NotImplementedError(
                    'a constant-step run that is too large to keep its rows resident needs '
                    'device-drawn packets and compress=True (raise NEXOCLOM_B200_MAX_ROWS or '
                    'run fewer packets per Output)')
            _, _, self.attempted_steps = eng.integrate_constant(
                seed=self.seed, first_id=self.first_id, n=self.npackets)
        self.kernel_ms = eng.last_kernel_ms()
        self.totalsource *= self.nsteps
        self.trajectory_kept = bool(keep_trajectory)

    def _finish_units(self):
        # "Add units back in" (Output.py:361-366, 451-455)
        self.aplanet = Quantity(self.aplanet, 'au')
        self.vrplanet = Quantity(self.vrplanet * float(self.planet.radius.value), 'km/s')
        self.GM = Quantity(self.GM, '')

    # ---- packets on the device -------------------------------------------------------
    def _engine(self):
        return get_engine(self.device)

    def _device_bytes(self):
        t = self._table
        return 0 if t is None or t.handle is None else t.n * 84

    def _release_device(self):
        if self._table is not None:
            self._table.free()
            self._table = None

    def _evict_to_host(self):
        """Residency budget exceeded: keep the rows as float32 host arrays instead."""
        if self._table is not None and self._table.handle is not None:
            self._host = self._table.export(with_step=True)
            self._release_device()

    def _rows_host(self):
        """(float32 columns, int32 packet index, uint16 step) of the saved rows."""
        if self._host is not None:
            return self._host
        if self._table is not None:
            return self._table.export(with_step=True)
        if self._X is not None:                  # unpickled: rebuild from the frame
            X = self._X
            cols = {c: np.ascontiguousarray(X[c].values, dtype=np.float32)
                    for c in STATE_COLS}
            cols['step_size'] = (np.ascontiguousarray(X['step_size'].values, dtype=np.float32)
                                 if 'step_size' in X else np.full(len(X), 1000., np.float32))
            index = (X['Index'].values if 'Index' in X else np.asarray(X.index)).astype(np.int32)
            step = np.zeros(len(X), dtype=np.uint16)
            nsteps = getattr(self, 'nsteps', None)
            if nsteps:
                step = (np.asarray(X.index) - index.astype(np.int64) * nsteps).astype(np.uint16)
            return cols, index, step
        raise RuntimeError('this Output holds no packets')

    def device_table(self):
        """The saved rows as a resident ``PacketTable`` (uploaded again if they were evicted
        or came from a file).  Not available for recipe-only constant-step runs: iterate
        ``tables()`` instead."""
        live = getattr(self, '_live', None)
        if live is not None:                      # a restore()d copy: the registered object
            return live.device_table()            # owns the table
        if self._table is None or self._table.handle is None:
            if not getattr(self, 'trajectory_kept', True):
                raise RuntimeError('recipe-only Output: use tables()')
            cols, index, _ = self._rows_host()
            eng = self._engine()
            self._table = eng.upload_packets([cols[c].astype(np.float64) for c in STATE_COLS],
                                             index.astype(np.uint32))
            self._host = (cols, index, _)
        catalogue.touch(self)
        return self._table

    def row_labels(self):
        """Row label of every row of the resident table, as ``X.index`` has them: the packet
        index (adaptive), packet * nsteps + step (constant step)."""
        table = self.device_table()
        index = table.index_host()
        if self.inputs.options.step_size != 0:
            return index * self.nsteps + table.export_steps().astype(np.int64)
        return index

    def tables(self, max_rows=None):
        """Iterate ``(PacketTable, packet offset)`` over the saved rows: one resident table, or
        -- recipe-only constant-step runs -- tables regenerated chunk by chunk (K1 + K3 with
        the row sink; freed after use).  ``table.index + offset`` is the 'Index' column."""
        if getattr(self, 'trajectory_kept', True):
            yield self.device_table(), 0
            return
        eng = self._engine()
        setup = get_setup(self.inputs, strict_math=self.strict_math)
        setup.upload(eng)
        sp = setup.source_params(eng)
        max_rows = max_rows or _max_rows()
        chunk = max(1, int(max_rows // self.nsteps))
        for first in range(0, self.npackets, chunk):
            m = min(chunk, self.npackets - first)
            eng.init_state(sp, self.seed, self.first_id + first, m)
            table, _, _ = eng.integrate_constant_rows(
                seed=self.seed, first_id=self.first_id + first, skip_dead=True, round_f32=True,
                n=m)
            try:
                yield table, first
            finally:
                table.free()

    # ---- X0 / X as DataFrames (built on access) -----------------------------------------
    def _cast(self, frame):
        """float32 / int32 as saved (Output.py:528-543), or 64 bit for a restore()d copy
        (:555-570)."""
        f_t, i_t = (np.float64, np.int64) if self._upcast else (np.float32, np.int32)
        for column in frame:
            kind = frame[column].dtype.kind
            if kind == 'f' and frame[column].dtype != f_t:
                frame[column] = frame[column].astype(f_t)
            elif kind in 'iu' and frame[column].dtype != i_t:
                frame[column] = frame[column].astype(i_t)
        return frame

    def _build_X0(self):
        if getattr(self, 'imported_x0', False):
            cols = self._imported_cols
            return pd.DataFrame({c: cols[k] for k, c in enumerate(STATE_COLS)})
        eng = self._engine()
        setup = get_setup(self.inputs, strict_math=self.strict_math)
        setup.upload(eng)
        eng.init_state(setup.source_params(eng), self.seed, self.first_id, self.npackets)
        x0 = eng.export_x0()
        return pd.DataFrame({c: x0[k] for k, c in enumerate(X0_COLS)})

    @property
    def X0(self):
        if self._X0 is None:
            self._X0 = self._build_X0()
        return self._cast(self._X0)

    @X0.setter
    def X0(self, frame):
        self._X0 = frame

    def _build_X(self):
        constant = self.inputs.options.step_size != 0
        if constant and not getattr(self, 'trajectory_kept', True):
            parts = []
            for table, first in self.tables():
                cols, index, step = table.export(with_step=True)
                parts.append((cols, index + first, step))
            cols = {c: np.concatenate([p[0][c] for p in parts]) for c in parts[0][0]}
            index = np.concatenate([p[1] for p in parts])
            step = np.concatenate([p[2] for p in parts])
        else:
            cols, index, step = self._rows_host()
        if constant:
            order = np.lexsort((step, index))
            X = pd.DataFrame({'Index': index[order]})
            for c in STATE_COLS:
                X[c] = cols[c][order]
            # running loss of each packet (Output.py:420-421 summed from 0, quirk Q13):
            # sum_{j<k} (frac_j - frac_{j+1}) = frac_0 - frac_k with frac_0 = 1
            X['lossfrac'] = (1.0 - X['frac'].values.astype(np.float64)).astype(np.float32)
            X.index = index[order].astype(np.int64) * self.nsteps + step[order]
        else:
            X = pd.DataFrame({c: cols[c] for c in STATE_COLS})
            if not getattr(self, 'imported_x0', False):
                X0 = self.X0
                for c in ('v', 'altitude', 'azimuth'):
                    X[c] = X0[c].values[index]
            X['lossfrac'] = np.zeros(len(index), dtype=np.float32)
            X['step_size'] = cols['step_size']
            X['Index'] = index
            X.index = index.astype(np.int64)
        return X

    @property
    def X(self):
        if self._X is None:
            self._X = self._build_X()
        return self._cast(self._X)

    @X.setter
    def X(self, frame):
        self._X = frame

    def _drop_host_frames(self):
        """After the run was pickled: the frames can be rebuilt from the device table."""
        if self._table is not None or self._host is not None:
            self._X = None
        if not getattr(self, 'imported_x0', False) and hasattr(self, 'seed'):
            self._X0 = None

    # ------------------------------------------------------------------
    def save(self):
        """Register in the local catalogue.  The reference's save (Output.py:522-543) drops
        the frac == 0 rows if ``compress`` and down-casts every column to float32 (quirk
        Q14) -- both already happened on the device (``nx_compact_state`` /
        ``nx_integrate_constant_rows``); the pickle is only written when
        ``NEXOCLOM_B200_SAVEPATH`` is set."""
        catalogue.register(self.inputs, self)

    def __getstate__(self):
        """The pickle holds what the reference's holds: X0 / X as float32 DataFrames."""
        d = dict(self.__dict__)
        for k in ('_table', '_host', '_X', '_X0', '_imported_cols', '_upcast', '_live'):
            d.pop(k, None)
        up, self._upcast = self._upcast, False
        try:
            d['X0'] = self.X0
            d['X'] = self.X
        finally:
            self._upcast = up
        return d

    def __setstate__(self, d):
        """Also the entry point for files written by the REFERENCE (``refpickle.load`` maps its
        ``Output`` class here): whatever this package's own pickles carry beyond the
        reference's attributes gets its default."""
        d = dict(d)
        self._X0 = d.pop('X0', None)
        self._X = d.pop('X', None)
        self._table = self._host = None
        self._upcast = False
        self.__dict__.update(d)
        from .sharding import local_device
        unit = self.__dict__.get('unit')
        if unit is not None and not isinstance(unit, str) and hasattr(unit, 'name'):
            name, dim, scale = unit.name()            # astropy unit of a reference file
            self.unit = def_unit(name, dim, scale)
        self.__dict__.setdefault('device', local_device())
        self.__dict__.setdefault('first_id', 0)
        self.__dict__.setdefault('strict_math', False)
        self.__dict__.setdefault('trajectory_kept', True)
        if 'imported_x0' not in self.__dict__:
            # a reference file: its X0 was drawn from NumPy streams, it cannot be re-drawn here
            self.imported_x0 = True
            self.from_reference = True
        opts = getattr(getattr(self, 'inputs', None), 'options', None)
        if 'nsteps' not in self.__dict__ and opts is not None and getattr(opts, 'step_size', 0):
            self.nsteps = int(np.ceil(float(np.asarray(opts.endtime)) / opts.step_size + 1))
        if getattr(self, 'imported_x0', False) and self._X0 is not None and \
                all(c in self._X0 for c in STATE_COLS):
            self._imported_cols = [np.ascontiguousarray(self._X0[c].values, dtype=np.float64)
                                   for c in STATE_COLS]

    @classmethod
    def restore(cls, filename):
        """Fetch a saved Output; its X0 / X read as 64 bit (Output.py:550-572).  The copy
        shares the resident packet table with the registered object."""
        live = catalogue.fetch(filename)
        output = copy.copy(live)
        output._upcast = True
        output._X0 = None if live._X0 is None else live._X0.copy()
        output._X = None if live._X is None else live._X.copy()
        output._live = live
        return output
