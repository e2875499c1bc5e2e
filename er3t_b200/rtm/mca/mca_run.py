"""
Job execution with the role of er3t/rtm/mca/mca_run.py.

The reference builds one shell command per (run, g) job -- `mcarats <photons> <solver> <inp> <out>` (mca_run.py:110-113)
-- orders them with `rearrange_jobs` and feeds them to a process pool (mca_run.py:144-159).  Here a job is a
`b200rt_job` record and all jobs of a scene run in ONE persistent-kernel launch per GPU, so no ordering heuristic is
needed on one GPU; `rearrange_jobs` is kept (restated) because callers and tests use it, and because it is the
whole-job load balancer across GPUs when photon-sharding is switched off.
"""

import numpy as np

from er3t_b200 import abi
from er3t_b200.solver import Solver

__all__ = ['mca_run', 'rearrange_jobs']


class mca_run:

    """
    scene   : abi.HostScene
    options : abi.Options
    photons : photons per job (array, job order = run-major like the reference's flattened fnames lists)
    seeds   : Philox key per job
    slabs   : output slab per job
    abs1d, flx_scale, rad_scale : per-job arrays / factors (see include/b200rt.h)
    kd      : keywords of abi.make_kd (spectral run, b200rt_run_kd: every job serves all these terms) or None
    jac_edges : layer-group edges of a Jacobian run (b200rt_run_jac) or None
    plen    : (tpmin, tpmax, ntp), metres, of a path-length run (b200rt_run_plen) or None

    Ncpu, mp_mode are accepted for signature compatibility and ignored.
    """

    def __init__(self, scene, options, photons, seeds, slabs, abs1d=None, flx_scale=None, rad_scale=None,
                 device=0, solver_obj=None, Ncpu=None, mp_mode='py', verbose=False, quiet=False, run=True, kd=None,
                 jac_edges=None, plen=None):
        self.scene = scene
        self.options = options
        self.quiet = quiet
        self.verbose = verbose
        self.jobs, self._keep = abi.make_jobs(photons, seeds, slabs, abs1d=abs1d, flx_scale=flx_scale, rad_scale=rad_scale)
        self.jac_edges = jac_edges
        self.plen = plen
        self.kd = None
        if kd is not None:
            self.kd, keep = abi.make_kd(njob=len(self.jobs), **kd)
            self._keep += keep
        self.solver = solver_obj if solver_obj is not None else Solver(device=device)
        self._own = solver_obj is None
        self.results = None
        if run:
            self.run()

    def launch(self):
        """upload the scene and trace all jobs (synchronous); the tallies stay on the device"""
        self.solver.upload_scene(self.scene, self.options)
        if self.kd is not None:
            self.solver.run_kd(self.jobs, self.kd)
        elif self.jac_edges is not None:
            self.solver.run_jac(self.jobs, self.jac_edges)
        elif self.plen is not None:
            self.solver.run_plen(self.jobs, *self.plen)
        else:
            self.solver.run(self.jobs)

    def run(self):
        self.launch()
        self.results = self.solver.results()
        return self.results

    def close(self):
        if self._own and self.solver is not None:
            self.solver.close()
            self.solver = None


def rearrange_jobs(Ncpu, weights_in):
    """
    Order jobs so that `Ncpu` workers finish at about the same time (restatement of er3t/rtm/mca/mca_run.py:185-315):
    greedy longest-processing-time assignment, then round-by-round emission in which the worker that has received the
    least work so far is served first.  Returns the job indices in execution order.
    """
    w = np.array(np.asarray(weights_in).ravel(), dtype=np.float64)
    w = w + w.min()
    order = np.argsort(w)[::-1]
    loads = np.zeros(Ncpu, dtype=np.float32)
    workers = [[] for _ in range(Ncpu)]
    for j in order:
        k = int(np.argmin(((loads + w[j]) - loads.min()) ** 2))
        loads[k] += w[j]
        workers[k].append((int(j), w[j]))
    # workers with more jobs first (stable on ties like np.argsort(...)[::-1])
    nj = np.array([len(x) for x in workers])
    workers = [workers[i] for i in np.argsort(nj)[::-1]]
    out = []
    nxt = np.arange(Ncpu)
    base = None
    while max(len(x) for x in workers) > 0:
        wr, ir = [], []
        for i in nxt:
            if workers[i]:
                j, wj = workers[i].pop(0)
                out.append(j)
                wr.append(wj)
                ir.append(i)
        wr = np.array(wr, dtype=np.float64)
        ir = np.array(ir, dtype=np.int32)
        base = wr.copy() if base is None else base[:wr.size] + wr
        nxt = ir[np.argsort(base)]
    return np.array(out)
