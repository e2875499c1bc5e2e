"""
Config 4 (OCO-2 O2 A-band sweep, workloads.c4: 8 wavelengths, per-g jobs) traced three ways with the same seeds: a plain
radiance run, a run that also tallies the gas-absorption Jacobian of 4 layer groups (mcarats_ng(gas_jacobian=levels)),
and one with one group per layer (gas_jacobian=True: 40 groups).  Per mode: kernel time (CUDA events,
stats()['elapsed_ms'], summed over the 8 calls) and tally updates.  The finite-difference alternative costs ngrp + 1 plain
runs (one per group plus the unperturbed one), so its kernel time is reported as (ngrp + 1) x the plain time, with the
ratio to the Jacobian run.  Also checked: the Jacobian runs reproduce the plain radiance.  The GPU's name and power limit
are read in the same process.

    python tools/bench_jacobian.py --out jacobian.json [--scale 1.0] [--reps 1]
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


def run_mode(cases, gas_jacobian, solver, reps):
    ms, tallies, hist = 0.0, 0, 0
    per_wvl, rads = [], []
    for rep in range(reps):
        for iw, (kw, abs0) in enumerate(cases):
            m = bmca.mcarats_ng(**dict(kw, solver_obj=solver, gas_jacobian=gas_jacobian, seed=kw['seed'] + 7919 * rep))
            st = m.stats
            ms += st['elapsed_ms']
            tallies += int(st['n_tally'])
            hist += int(st['photons'])
            if rep == 0:
                rads.append(np.asarray(m.fused['radiance'][0]))
                row = dict(wvl=iw, Ng=m.Ng, kernel_ms=st['elapsed_ms'], n_tally=int(st['n_tally']))
                if gas_jacobian is not None:
                    jac = np.asarray(m.fused['jacobian'][0])                  # (nx, ny, ngrp, 1, Nrun)
                    row['ngrp'] = int(jac.shape[2])
                    row['mean_rad'] = float(rads[-1].mean())
                    row['mean_jac_per_group'] = [float(v) for v in jac.mean(axis=(0, 1, 3, 4))]
                per_wvl.append(row)
    return dict(kernel_ms=ms / reps, histories=hist // reps, n_tally=tallies // reps, per_wavelength=per_wvl), rads


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True)
    ap.add_argument('--scale', type=float, default=1.0)
    ap.add_argument('--reps', type=int, default=1, help='repetitions with other seeds (times are averaged)')
    a = ap.parse_args()
    cases = workloads.c4(scale=a.scale)
    lev = cases[0][0]['atm_1ds'][0].atm.lev['altitude']['data']
    four = [float(lev[0]), 2.0, 5.0, 10.0, float(lev[-1])]                   # km: 4 layer groups
    solver = Solver(device=0)
    # warm-up of the three kernels on the first wavelength (module load, smem attributes)
    for gj in (None, four, True):
        kw, _ = cases[0]
        bmca.mcarats_ng(**dict(kw, solver_obj=solver, gas_jacobian=gj, photons=1e5))
    res = {'gpu': gpu_info(), 'config': 'C4', 'scale': a.scale, 'reps': a.reps, 'levels_4_km': four}
    res['plain'], r0 = run_mode(cases, None, solver, a.reps)
    for name, gj in (('jac_4', four), ('jac_layers', True)):
        res[name], r = run_mode(cases, gj, solver, a.reps)
        ngrp = res[name]['per_wavelength'][0]['ngrp']
        res[name]['ngrp'] = ngrp
        res[name]['max_rel_rad_diff_vs_plain'] = max(float(np.max(np.abs(x - y)) / np.max(np.abs(y))) for x, y in zip(r, r0))
        res[name]['kernel_ratio_vs_plain'] = res[name]['kernel_ms'] / res['plain']['kernel_ms']
        res[name]['fd_kernel_ms'] = (ngrp + 1) * res['plain']['kernel_ms']
        res[name]['fd_over_jac'] = res[name]['fd_kernel_ms'] / res[name]['kernel_ms']
    solver.close()
    with open(a.out, 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: (v if not isinstance(v, dict) else {q: w for q, w in v.items() if q != 'per_wavelength'}) for k, v in res.items()}))


if __name__ == '__main__':
    main()
