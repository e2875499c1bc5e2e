"""
Multi-GPU plumbing: one process per GPU (torchrun), photons of every (run, g) job sharded by
`photon_index % world == rank` (disjoint Philox counters), and ONE NCCL all-reduce (sum, fp64) of the tallies over
NVLink at the end -- the only exchange step this path has (SURVEY.md 8e).  The reference's counterpart is the
process pool of er3t/rtm/mca/mca_run.py:144-159 (no collective at all).
"""

import os

import numpy as np

__all__ = ['init_from_env', 'allreduce_results', 'shard_from_env', 'tally_views']


def shard_from_env():
    return int(os.environ.get('RANK', '0')), int(os.environ.get('WORLD_SIZE', '1'))


def init_from_env(backend=None):
    """Initialise torch.distributed from the torchrun environment (no-op for world size 1).  Returns (rank, world, local_rank)."""
    rank, world = shard_from_env()
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if world > 1:
        import torch
        import torch.distributed as dist
        if not dist.is_initialized():
            if backend is None:
                backend = 'nccl' if torch.cuda.is_available() else 'gloo'
            if backend == 'nccl':
                torch.cuda.set_device(local)
            dist.init_process_group(backend=backend, rank=rank, world_size=world)
    return rank, world, local


class _DeviceDoubles:
    """Zero-copy view of `n` doubles at a device address for torch (`torch.as_tensor` honours __cuda_array_interface__)."""

    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {'shape': (int(n),), 'typestr': '<f8', 'data': (int(ptr), False), 'version': 2}


def tally_views(solver):
    """torch tensors that ALIAS the library-owned tally buffers (b200rt_tally_ptrs): {'flux' | 'rad' | 'heat': tensor or None}."""
    import torch
    out = {}
    for key, (ptr, n) in solver.tally_ptrs().items():
        out[key] = torch.as_tensor(_DeviceDoubles(ptr, n), device='cuda:%d' % solver.device) if (ptr and n) else None
    return out


def allreduce_results(solver, to_host=True):
    """
    Sum the tallies of all ranks.  With NCCL the all-reduce runs IN PLACE on the library's own device buffers (no staging
    tensor, no device-to-device copy): afterwards every rank's handle holds the global tallies and `solver.results()` /
    `b200rt_read_*` return them.  After a Jacobian run (`Solver.run_jac`), a path-length run (`Solver.run_plen`) or an
    actinic run (`Solver.run_act`) its tally is reduced too (`res['jac']` / `res['plen']` / `res['act']`).  With gloo (CPU tests) the host arrays are reduced.  The run is waited for first
    (`solver.sync()`: NaN guard + fresh event counters), and the event counters are reduced with the same collective.
    """
    import torch
    import torch.distributed as dist
    res = {'flux': None, 'rad': None, 'heat': None}
    world = dist.get_world_size() if dist.is_initialized() else 1
    use_cuda = world > 1 and dist.get_backend() == 'nccl'
    if hasattr(solver, 'sync'):
        solver.sync()
    st = solver.stats()
    xt = getattr(solver, '_xt_key', None)       # 'jac' / 'plen' / 'act': the extra tally of a Jacobian / path-length / actinic run
    keys = ('flux', 'rad', 'heat') + ((xt,) if xt else ())
    if use_cuda:
        views = tally_views(solver)
        if xt:
            ptr, n = getattr(solver, xt + '_ptr')()
            views[xt] = torch.as_tensor(_DeviceDoubles(ptr, n), device='cuda:%d' % solver.device)
        for key in keys:
            t = views[key]
            if t is None:
                continue
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            res[key] = t
        if to_host:
            torch.cuda.synchronize()
            host = solver.results()
            for key in keys:
                res[key] = host[key]
    else:
        host = solver.results()
        for key in keys:
            a = host[key]
            if a is None:
                continue
            if world > 1:
                t = torch.from_numpy(np.ascontiguousarray(a))
                dist.all_reduce(t, op=dist.ReduceOp.SUM)
                a = t.numpy()
            res[key] = a
    if world > 1:
        keys = [k for k in st.keys() if k not in ('elapsed_ms', 'launches')]
        v = torch.tensor([float(st[k]) for k in keys], dtype=torch.float64, device='cuda' if use_cuda else 'cpu')
        dist.all_reduce(v, op=dist.ReduceOp.SUM)
        for k, x in zip(keys, v.cpu().tolist()):
            st[k] = type(st[k])(x)
    if res['flux'] is not None and hasattr(solver, 'scene') and not hasattr(res['flux'], 'is_cuda'):
        res['flux'] = res['flux'].reshape(solver.scene.flux_shape(solver.options.nslab))
    res['stats'] = st
    return res
