"""
Config 4 (OCO-2 O2 A-band sweep, workloads.c4: 8 wavelengths, per-g jobs) traced three ways with the same seeds: a plain
radiance run and runs that also tally the path-length distribution behind every pixel (mcarats_ng(path_length=...)) with
16 and 64 bins.  The three modes alternate within every repetition, so that drifts of the shared machine hit all of them.
Per mode: kernel time (CUDA events, stats()['elapsed_ms'], summed over the 8 calls) per repetition and its median, and
tally updates.  Also checked: the path-length runs reproduce the plain radiance, and the bins + underflow + overflow of
the tally sum to it.  The GPU's name and power limit are read in the same process.

    python tools/bench_plen.py --out plen.json [--scale 1.0] [--reps 3]
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

TPMAX_KM = 200.0


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else 'unknown'


def run_mode(cases, path_length, solver):
    """one sweep over the wavelengths: (kernel ms, histories, tally updates, radiance per wavelength, per-wavelength rows)"""
    ms, tallies, hist = 0.0, 0, 0
    rads, rows = [], []
    for iw, (kw, abs0) in enumerate(cases):
        m = bmca.mcarats_ng(**dict(kw, solver_obj=solver, path_length=path_length))
        st = m.stats
        ms += st['elapsed_ms']
        tallies += int(st['n_tally'])
        hist += int(st['photons'])
        rad = np.asarray(m.fused['radiance'][0])
        rads.append(rad)
        row = dict(wvl=iw, kernel_ms=st['elapsed_ms'], n_tally=int(st['n_tally']))
        if path_length is not None:
            pl = np.asarray(m.fused['path_length'][0])                     # (nx, ny, ntp+3, 1, Nrun)
            ntp = pl.shape[2] - 3
            row['max_rel_sum_identity'] = float(np.max(np.abs(pl[:, :, :ntp + 2].sum(axis=2) - rad[:, :, 0])) / np.max(np.abs(rad)))
            row['mean_path_km'] = float(pl[:, :, ntp + 2].sum() / rad.sum() / 1000.0)
            row['overflow_share'] = float(pl[:, :, ntp + 1].sum() / rad.sum())
        rows.append(row)
    return ms, hist, tallies, rads, rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True)
    ap.add_argument('--scale', type=float, default=1.0)
    ap.add_argument('--reps', type=int, default=3, help='repetitions of the alternating plain / 16-bin / 64-bin sweep')
    a = ap.parse_args()
    cases = workloads.c4(scale=a.scale)
    modes = (('plain', None), ('plen_16', (0.0, TPMAX_KM, 16)), ('plen_64', (0.0, TPMAX_KM, 64)))
    solver = Solver(device=0)
    # warm-up of the kernels on the first wavelength (module load, smem attributes)
    for _, pl in modes:
        kw, _ = cases[0]
        bmca.mcarats_ng(**dict(kw, solver_obj=solver, path_length=pl, photons=1e5))
    res = {'gpu': gpu_info(), 'config': 'C4', 'scale': a.scale, 'reps': a.reps, 'tpmax_km': TPMAX_KM}
    for name, _ in modes:
        res[name] = dict(kernel_ms_reps=[])
    r0 = None
    for rep in range(a.reps):
        for name, pl in modes:
            ms, hist, tallies, rads, rows = run_mode(cases, pl, solver)
            d = res[name]
            d['kernel_ms_reps'].append(ms)
            d['histories'], d['n_tally'] = hist, tallies
            if rep == 0:
                d['per_wavelength'] = rows
            if pl is None:
                r0 = rads
            else:
                diff = max(float(np.max(np.abs(x - y)) / np.max(np.abs(y))) for x, y in zip(rads, r0))
                d['max_rel_rad_diff_vs_plain'] = max(diff, d.get('max_rel_rad_diff_vs_plain', 0.0))
    for name, _ in modes:
        d = res[name]
        d['kernel_ms'] = float(np.median(d['kernel_ms_reps']))
        d['kernel_ratio_vs_plain'] = d['kernel_ms'] / res['plain']['kernel_ms']
        d['kernel_ratio_vs_plain_reps'] = [x / y for x, y in zip(d['kernel_ms_reps'], res['plain']['kernel_ms_reps'])]
    solver.close()
    with open(a.out, 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: (v if not isinstance(v, dict) else {q: w for q, w in v.items() if q != 'per_wavelength'}) for k, v in res.items()}))


if __name__ == '__main__':
    main()
