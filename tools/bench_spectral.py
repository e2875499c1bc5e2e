"""
Config 4 (OCO-2 O2 A-band sweep, workloads.c4) traced per g (one job per (run, g): 279 jobs over the 8 wavelengths) and
in spectral mode (mcarats_ng(spectral=True): one job per run, every history serves all g of its wavelength: 24 jobs).
Both modes trace the same number of histories.  Per mode: kernel time (CUDA events, stats()['elapsed_ms'], summed over
the 8 calls), histories/s, the per-pixel standard deviation over the 3 runs of the fused radiance, and the figure of merit
1 / (mean sigma^2 * t_kernel); then the ratio of the two figures of merit.  The GPU's name and power limit are read in the
same process.

    python tools/bench_spectral.py --out spectral.json [--scale 1.0] [--reps 1]
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


def run_mode(cases, spectral, solver, reps):
    ms, hist, var, npx = 0.0, 0, 0.0, 0
    per_wvl = []
    for rep in range(reps):
        for iw, (kw, abs0) in enumerate(cases):
            m = bmca.mcarats_ng(**dict(kw, solver_obj=solver, spectral=spectral, seed=kw['seed'] + 7919 * rep))
            st = m.stats
            rad = np.asarray(m.fused['radiance'][0])[:, :, 0, 0, :]          # (nx, ny, Nrun)
            sd = rad.std(axis=-1, ddof=1)
            ms += st['elapsed_ms']
            hist += int(st['photons'])
            var += float((sd ** 2).sum())
            npx += sd.size
            if rep == 0:
                per_wvl.append(dict(wvl=iw, Ng=m.Ng, jobs=m.Nrun if spectral else m.Nrun * m.Ng, kernel_ms=st['elapsed_ms'],
                                    mean_rad=float(rad.mean()), mean_sigma=float(sd.mean())))
    mean_var = var / npx
    t = ms / 1e3
    return dict(kernel_ms=ms / reps, histories=hist // reps, histories_per_s=hist / t, mean_sigma2=mean_var,
                fom=1.0 / (mean_var * (t / reps)), per_wavelength=per_wvl)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True)
    ap.add_argument('--scale', type=float, default=1.0)
    ap.add_argument('--reps', type=int, default=1, help='repetitions with other seeds (sigma^2 and time are averaged)')
    a = ap.parse_args()
    cases = workloads.c4(scale=a.scale)
    solver = Solver(device=0)
    # warm-up of both kernels on the first wavelength (module load, smem attributes)
    for sp in (False, True):
        kw, _ = cases[0]
        bmca.mcarats_ng(**dict(kw, solver_obj=solver, spectral=sp, photons=1e5))
    res = {'gpu': gpu_info(), 'config': 'C4', 'scale': a.scale, 'reps': a.reps}
    res['per_g'] = run_mode(cases, False, solver, a.reps)
    res['spectral'] = run_mode(cases, True, solver, a.reps)
    res['fom_ratio'] = res['spectral']['fom'] / res['per_g']['fom']
    solver.close()
    with open(a.out, 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: (v if not isinstance(v, dict) else {q: w for q, w in v.items() if q != 'per_wavelength'}) for k, v in res.items()}))


if __name__ == '__main__':
    main()
