"""
Config 5 (flux with gas absorption under broken 3-D clouds, workloads.c5) and config 1 (plane-parallel flux, workloads.c1)
at their named shapes, each traced two ways with the same seeds: a plain run and one that also tallies the actinic flux
(mcarats_ng(actinic=True)).  The two modes alternate within every repetition, so that drifts of the shared machine hit
both.  Per config and mode: kernel time (CUDA events, stats()['elapsed_ms']) per repetition and its median, and tally
updates that reach global memory.  Also checked: the actinic runs reproduce the plain fluxes.  The GPU's name, power
limit and maximum SM clock are read in the same process.

    python tools/bench_actinic.py --out actinic.json [--scale 1.0] [--reps 3]
"""

import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import workloads  # noqa: E402
from er3t_b200.rtm import mca as bmca  # noqa: E402
from er3t_b200.solver import Solver  # noqa: E402


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else 'unknown'


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True)
    ap.add_argument('--scale', type=float, default=1.0)
    ap.add_argument('--reps', type=int, default=3, help='repetitions of the alternating plain / actinic pair')
    a = ap.parse_args()
    solver = Solver(device=0)
    res = {'gpu': gpu_info(), 'scale': a.scale, 'reps': a.reps}
    for cfg, builder in (('C5', workloads.c5), ('C1', workloads.c1)):
        kw, _ = builder(scale=a.scale)
        kw = dict(kw, solver_obj=solver)
        for act in (False, True):       # warm-up: module load, shared-memory attributes
            bmca.mcarats_ng(**dict(kw, actinic=act, photons=1e5))
        out = {'plain': dict(kernel_ms_reps=[]), 'actinic': dict(kernel_ms_reps=[])}
        f0 = None
        for rep in range(a.reps):
            for name, act in (('plain', False), ('actinic', True)):
                m = bmca.mcarats_ng(**dict(kw, actinic=act))
                st = m.stats
                d = out[name]
                d['kernel_ms_reps'].append(st['elapsed_ms'])
                d['histories'], d['n_tally'] = int(st['photons']), int(st['n_tally'])
                f = [np.asarray(x) for x in m.fused['flux']]
                if not act:
                    f0 = f
                else:
                    diff = max(float(np.max(np.abs(x - y)) / np.max(np.abs(y))) for x, y in zip(f, f0))
                    d['max_rel_flux_diff_vs_plain'] = max(diff, d.get('max_rel_flux_diff_vs_plain', 0.0))
                    act_t = np.asarray(m.fused['actinic'][0])[:, :, :, 1]
                    d['domain_mean_actinic_total_per_layer_run0'] = act_t[..., 0].mean(axis=(0, 1)).tolist()
        for name in out:
            d = out[name]
            d['kernel_ms'] = float(np.median(d['kernel_ms_reps']))
            d['kernel_ratio_vs_plain'] = d['kernel_ms'] / out['plain']['kernel_ms']
            d['kernel_ratio_vs_plain_reps'] = [x / y for x, y in zip(d['kernel_ms_reps'], out['plain']['kernel_ms_reps'])]
        out['shape'] = dict(nx=int(m.Nx), ny=int(m.Ny), nz=int(m.scene.struct.nz), Nrun=int(m.Nrun), Ng=int(m.Ng))
        res[cfg] = out
    solver.close()
    with open(a.out, 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: (v if not isinstance(v, dict) else {q: ({x: y for x, y in w.items() if not x.startswith('domain')}
                                                                 if isinstance(w, dict) else w) for q, w in v.items()})
                      for k, v in res.items()}))


if __name__ == '__main__':
    main()
