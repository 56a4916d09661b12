"""Sharded runs: one process per GPU, packets split by global id, one all-reduce per product.

Packets are independent (reference rk5 is row-wise; the reference's own ``Input.run`` loops
chunks serially, ``initial_state/Input.py:243-249``), so a run of N packets is sharded into
contiguous GLOBAL packet-id ranges, one per rank.  The Philox counter of a packet is its
global id, hence every product is independent of the number of GPUs.  There is no data-path
collective; the only exchange is ONE sum all-reduce per product -- image f64 + packet counts,
LOS radiance f64 + hit counts (SURVEY section 8e) -- over NCCL/NVLink through the C ABI
(``nx_comm_create`` / ``nx_allreduce_host``; the communicator id travels through the
``torch.distributed`` store the launcher set up).  With the ``gloo`` backend (CPU tests of
the host logic) the same sum goes through ``torch.distributed`` itself.

Usage under ``torchrun``::

    from nexoclom_b200 import Input, ModelImage, sharding
    sharding.init()                       # NCCL on the GPU box; picks cuda:LOCAL_RANK
    inputs = Input('Na.input')
    inputs.run(1e8, seed=0)               # each rank integrates its 1/world of the ids
    image = ModelImage(inputs, params)    # identical, complete image on every rank
"""
import ctypes as C
import os

import numpy as np

_comm = {'handle': None, 'lib': None, 'world': None}


def _dist():
    try:
        import torch.distributed as dist
    except ImportError:
        return None
    return dist if dist.is_available() and dist.is_initialized() else None


def rank_world():
    """(rank, world) of this process: ``torch.distributed`` if initialised, else (0, 1)."""
    dist = _dist()
    if dist is None:
        return 0, 1
    return dist.get_rank(), dist.get_world_size()


def local_device():
    """GPU of this process: LOCAL_RANK under torchrun, else 0."""
    return int(os.environ.get('LOCAL_RANK', '0')) if _dist() is not None else 0


def init(backend=None):
    """Join the process group the launcher described in the environment (RANK, WORLD_SIZE,
    MASTER_ADDR, MASTER_PORT).  No-op for a single process."""
    import torch
    import torch.distributed as dist
    if dist.is_initialized() or int(os.environ.get('WORLD_SIZE', '1')) <= 1:
        return rank_world()
    if backend is None:
        backend = 'nccl' if torch.cuda.is_available() else 'gloo'
    if backend == 'nccl':
        local = int(os.environ.get('LOCAL_RANK', '0'))
        torch.cuda.set_device(local)
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    else:
        dist.init_process_group(backend)
    return rank_world()


def shard_range(n_total, rank, world):
    """[first_id, first_id + n) of `rank`: sizes differ by at most one."""
    base, rem = divmod(int(n_total), int(world))
    first = rank * base + min(rank, rem)
    return first, base + (1 if rank < rem else 0)


def broadcast_object(obj, src=0):
    """The same Python object on every rank (seeds, catalogue bookkeeping)."""
    dist = _dist()
    if dist is None or dist.get_world_size() == 1:
        return obj
    box = [obj]
    dist.broadcast_object_list(box, src=src)
    return box[0]


def _nccl_comm():
    """The C-ABI communicator of this process group (created on first use)."""
    dist = _dist()
    rank, world = dist.get_rank(), dist.get_world_size()
    if _comm['handle'] is not None and _comm['world'] == world:
        return _comm['lib'], _comm['handle']
    from . import _lib
    lib = _lib.load()
    uid = C.create_string_buffer(128)
    if rank == 0 and lib.nx_comm_unique_id(uid) != 0:
        raise RuntimeError('nx_comm_unique_id: ' + lib.nx_comm_last_error().decode())
    raw = broadcast_object(bytes(uid.raw), src=0)
    handle = C.c_void_p()
    rc = lib.nx_comm_create(local_device(), raw, rank, world, C.byref(handle))
    if rc != 0:
        raise RuntimeError(f'nx_comm_create failed ({rc}): ' + lib.nx_comm_last_error().decode())
    _comm.update(handle=handle, lib=lib, world=world)
    return lib, handle


def allreduce_sum(*arrays):
    """In-place SUM over the ranks of float64 / int64 host arrays -- call it ONCE per product.
    NCCL through the C ABI when the process group runs on GPUs, ``torch.distributed`` (gloo)
    otherwise.  Returns the arrays."""
    dist = _dist()
    if dist is None or dist.get_world_size() == 1:
        return arrays
    use_nccl = dist.get_backend() == 'nccl'
    for a in arrays:
        if not (isinstance(a, np.ndarray) and a.flags.c_contiguous and
                a.dtype in (np.float64, np.int64)):
            raise TypeError('allreduce_sum needs C-contiguous float64 / int64 ndarrays')
        if use_nccl:
            lib, comm = _nccl_comm()
            rc = lib.nx_allreduce_host(comm, a.ctypes.data_as(C.c_void_p), a.size,
                                       0 if a.dtype == np.float64 else 1)
            if rc != 0:
                raise RuntimeError(f'nx_allreduce_host failed ({rc}): ' +
                                   lib.nx_comm_last_error().decode())
        else:
            import torch
            t = torch.from_numpy(a)
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return arrays


def combine_ranks(arrays, *scalars):
    """Sum a product's host ``arrays`` over the ranks in place, with ``scalars`` (totalsource,
    ...) riding along in one float64 array: ONE all-reduce, a no-op for a single process.
    Returns the summed scalars as a tuple of floats."""
    tot = np.array(scalars, dtype=np.float64)
    allreduce_sum(*arrays, tot)
    return tuple(float(v) for v in tot)


def nccl_comm():
    """``(lib, nx_comm handle)`` when this process group runs over NCCL, else ``None`` (single
    process, or the gloo backend of the CPU tests)."""
    dist = _dist()
    if dist is None or dist.get_world_size() == 1 or dist.get_backend() != 'nccl':
        return None
    return _nccl_comm()


def allreduce_products(*tensors):
    """In-place SUM all-reduce of torch tensors (device tensors under NCCL); kept for callers
    that hold their products as tensors (bench.py)."""
    dist = _dist()
    if dist is not None and dist.get_world_size() > 1:
        for t in tensors:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return tensors
