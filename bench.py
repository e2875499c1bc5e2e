#!/usr/bin/env python
"""
bench.py -- headline benchmark of the photon-transport path: photons/s on the 3-D LES cloud radiance config
(BASELINE.json configs[1]: 480 x 480 x 100 voxels at 100 m, nadir radiance at 650 nm, 1e8 photons per set, 3 runs,
16 g weighted -- projects/05_cnn-les_rad-sim shape, examples/00_er3t_mca.py::example_05).

    python bench.py --gpus N --steps K --warmup W            # this repo (CUDA, sm_100a)
    python bench.py --impl reference --gpus N ...            # CPU arm: the oracle port on the host cores
    python bench.py ... --dump-outputs DIR                   # also write the tallies of the last timed step to DIR

One "step" = one complete `mcarats_ng` job set (Nrun x Ng jobs = 3 x 1e8 photons) over the synthetic scene.
`--dump-outputs DIR`: after the timed steps, every tally the timed step returns (`Solver.results()`: radiance, and flux /
heating when the target has them) is written as DIR/<name>.npy in float64.  The inputs and photon seeds are fixed, so two
builds run with the same arguments can be compared array for array; above 64 MB in all, a fixed seeded sample is written.
`value`  : photons/s with the scene already resident in HBM (b200rt_run only; CUDA events on the launching stream).
`e2e`    : photons/s through the public API, starting from the RAW cloud fields (extinction, effective radius) as host
           numpy arrays: mca_atm_3d(device_props=True) + mcarats_ng + mca_out_ng -- the input builder, scene packing
           (omega / apf derived on the GPU), H2D, transport, D2H and the run statistics are all inside the timed region.
`strong` : the FIXED 3e8-photon job set sharded over the N ranks (N > 1 only; `value` stays weak-scaled).
`c4_sweep`: (N > 1) the config-4 wavelength x g sweep sharded over the ranks, photon sharding vs whole wavelengths per rank.
`accuracy`: error of the GPU path against the deterministic adding-doubling fixture (plane-parallel Mie cloud) and
           against the CPU oracle on a scaled copy of this workload.
Inputs are larger than L2 (3-D fields 370 MB in HBM vs 126 MB L2), so no explicit L2 flush between iterations.
Rank 0 prints ONE JSON line.
"""

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED = 20260101


def build_workload(nx=480, ny=480, nz3=100, photons=1e8, nrun=3, parts=False):
    """BASELINE.json configs[1] as synthetic input (SURVEY.md 8d 'C2', workloads.c2): kwargs for mcarats_ng + abs object
    (+ the raw cloud / atmosphere / phase objects the e2e leg rebuilds mca_atm_3d from, with parts=True)."""
    import workloads
    out = workloads.c2(scale=1.0, photons=photons, nx=nx, ny=ny, nz3=nz3, nrun=nrun, parts=parts)
    out[0]['fdir'] = 'tmp-data/bench'
    return out


class ClockSampler:
    """nvidia-smi sampler running DURING the timed region (B200_PROFILING.md recipe)."""

    Q = 'index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,' \
        'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, gpu_index=0):
        self.f = tempfile.NamedTemporaryFile('w+', suffix='.csv', delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(['nvidia-smi', '-i', str(gpu_index), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits', '-lms', '200'],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        out = {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, smmax, reasons, power = [], [], set(), []
        for line in self.f.read().splitlines():
            w = [x.strip() for x in line.split(',')]
            if len(w) < 9:
                continue
            try:
                sm.append(float(w[1])); smmax.append(float(w[2])); power.append(float(w[3]))
            except ValueError:
                continue
            for name, val in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), w[5:9]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        self.f.close()
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        if sm:
            # median over samples taken under load (power above the idle floor)
            load = [s for s, p in zip(sm, power) if p > 0.5 * max(power)] or sm
            out.update(sm_mhz=float(np.median(load)), sm_max_mhz=float(max(smmax)), reasons=sorted(reasons), samples=len(sm),
                       power_w_max=float(max(power)))
        return out


def measured_peak():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.isfile(p):
        try:
            return float(json.load(open(p))['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
        except Exception:
            pass
    return 6650.0, 'fallback (B200_PROFILING.md)'


def ncu_traffic(key='transport_kernel_dram_bytes_per_launch'):
    """per-launch DRAM bytes of the transport kernel (or the headline counters) from the committed ncu captures, or None."""
    p = os.path.join(ROOT, 'profiles', 'traffic.json')
    if os.path.isfile(p):
        try:
            return json.load(open(p)).get(key)
        except Exception:
            return None
    return None


def host_cores():
    """Host threads this process may use.  Passed to the oracle explicitly: torchrun exports OMP_NUM_THREADS=1."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return os.cpu_count() or 1


def cpu_oracle_rate(kw, abs0, seconds=15.0, nthreads=0):
    """Bounded sample of the same workload on the host cores with the oracle port; returns (photons/s, photons, cores)."""
    import oracle
    from er3t_b200.rtm.mca import mcarats_ng
    cores = nthreads = nthreads if nthreads > 0 else host_cores()
    rate = None
    nphot = 40000
    total_t = 0.0
    while True:
        k = dict(kw)
        k.update(photons=nphot, Nrun=1, dry_run=True)
        m = mcarats_ng(**k)
        from er3t_b200 import abi
        jobs, keep = abi.make_jobs(**m.jobs_args)
        t0 = time.time()
        oracle.run(m.scene, m.options, jobs, nthreads=nthreads)
        dt = time.time() - t0
        total_t += dt
        rate = nphot / dt
        if total_t >= 0.6 * seconds or nphot >= 5e7:
            return rate, nphot, cores
        nphot = int(max(nphot * 2, min(5e7, rate * (seconds - total_t) * 0.8)))


# the only throughput the reference publishes (docs/source/other/contest.rst:15-24; BASELINE.md): 3e8 photons in <= 45 s on
# 24 CPUs for a 480 x 480 x 4 scene -- a derived lower bound on another scene, quoted for context only
PUBLISHED = {'value': 6.7e6, 'unit': 'photons/s', 'cores': 24, 'what': 'MCARaTS, derived lower bound, 480x480x4 scene (contest.rst:15-24)'}


def accuracy_summary(sol):
    """Error of the CUDA path (a) against the converged deterministic solution of the plane-parallel Mie-cloud case
    (tests/golden/ad_fixtures.npz, oracle/adding_doubling.py) at 4e8 photons, (b) against the CPU oracle on a scaled
    copy of the bench workload (per-pixel z-scores, domain-mean radiance)."""
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    import scenes
    import oracle
    import workloads
    from er3t_b200 import abi
    from er3t_b200.rtm.mca import mcarats_ng
    out = {}
    # (a) deterministic
    fx = scenes.ad_fixture('mie')
    nslab = 8
    sc = scenes.ad_scene(fx)
    opt = abi.make_options(target=abi.TARGET_FLUX | abi.TARGET_RADIANCE, nslab=nslab, wmin=0.2)
    jobs, keep = scenes.multi_seed_jobs(50000000, nslab, abs1d=fx['absg'])
    sol.upload_scene(sc, opt)
    sol.run(jobs)
    r = sol.results()
    nlev = fx['z'].size
    flux = r['flux'].reshape(nslab, 3, nlev)
    rad = r['rad'].reshape(nslab, -1)
    mu0 = float(fx['mu0'])
    fm = flux.mean(axis=0)
    rm, rs = rad.mean(axis=0), rad.std(axis=0, ddof=1) / np.sqrt(nslab)
    out['vs_adding_doubling'] = {
        'case': 'config-1 atmosphere, tau = 10 cloud with the 498-angle Mie table, SZA 30, 4e8 photons',
        'flux_up_max_rel_err': float(np.max(np.abs(fm[2] - fx['f_up']) / np.maximum(fx['f_up'], 0.05 * mu0))),
        'flux_down_max_rel_err': float(np.max(np.abs(fm[1] - fx['f_down']) / np.maximum(fx['f_down'], 0.05 * mu0))),
        'radiance_rel_err': [float(v) for v in (rm / fx['rad_views'] - 1.0)],
        'radiance_rel_sem': [float(v) for v in (rs / fx['rad_views'])],
        'views_vza_dphi': fx['views'].tolist()}
    # (b) oracle on a scaled copy of the workload (north_star: domain mean within 0.5 %, pixels within 3 combined sigma)
    kws, _ = workloads.c2(scale=0.004, photons=1e8)
    nrep = 6
    m = mcarats_ng(**dict(kws, Nrun=nrep, dry_run=True))
    ja = dict(m.jobs_args)
    jobs, keep = abi.make_jobs(**ja)
    sol.upload_scene(m.scene, m.options)
    sol.run(jobs)
    g = sol.results()['rad'].reshape(nrep, -1)
    c = oracle.run(m.scene, m.options, jobs, nthreads=host_cores())['rad'].reshape(nrep, -1)
    gm, cm = g.mean(axis=0), c.mean(axis=0)
    se = np.sqrt(g.var(axis=0, ddof=1) / nrep + c.var(axis=0, ddof=1) / nrep)
    ok = se > 0
    z = (gm[ok] - cm[ok]) / se[ok]
    out['vs_oracle_c2_scaled'] = {
        'case': '%d x %d x %d voxels, %d photons x %d runs (workloads.c2 scale 0.004)' % (m.scene.struct.nx, m.scene.struct.ny, m.scene.struct.nz3,
                                                                                            int(np.sum(ja['nphot']) / nrep), nrep),
        'domain_mean_rel_err': float(gm.mean() / cm.mean() - 1.0), 'pixel_z_rms': float(np.sqrt(np.mean(z ** 2))),
        'pixel_z_max_abs': float(np.max(np.abs(z))), 'pixels_beyond_3_sigma_frac': float(np.mean(np.abs(z) > 3.0))}
    return out


DUMP_LIMIT = 64 << 20


def dump_outputs(outdir, results):
    """Write the non-empty tally arrays of `results` as outdir/<name>.npy (float64).  When they exceed DUMP_LIMIT bytes in
    all, each array is flattened and cut to the same fraction by a sorted sample of positions drawn with a fixed seed."""
    arrays = {k: np.ascontiguousarray(v, dtype=np.float64) for k, v in results.items() if k != 'stats' and v is not None}
    total = sum(a.nbytes for a in arrays.values())
    os.makedirs(outdir, exist_ok=True)
    for name, a in sorted(arrays.items()):
        if total > DUMP_LIMIT:
            keep = a.size * DUMP_LIMIT // total
            a = a.ravel()[np.sort(np.random.default_rng(SEED).choice(a.size, size=keep, replace=False, shuffle=False))]
        np.save(os.path.join(outdir, name + '.npy'), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--photons', type=float, default=1e8, help='photons per set (BASELINE: 1e8)')
    ap.add_argument('--nx', type=int, default=480)
    ap.add_argument('--nz3', type=int, default=100)
    ap.add_argument('--e2e-steps', type=int, default=2)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-accuracy', action='store_true')
    ap.add_argument('--c4-photons', type=float, default=1e9, help='N > 1: photons of the config-4 sweep leg (0 = skip)')
    ap.add_argument('--sv', type=str, default='0,0,0')
    ap.add_argument('--empty-runs', type=int, default=0, help='A/B switch of the resident leg: -1 = no vertical merging of empty coarse cells')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the tallies of the last timed step as DIR/<name>.npy (float64, at most 64 MB in all)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs needs the CUDA arm: the reference arm sizes its photon sample from a timing probe')

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    workload = 'C2 3D LES-like cloud %dx%dx%d voxels @100 m (3-D block 0.5-4.5 km), nadir radiance 650 nm, %g photons/set x 3 runs x 16 g' % (
        args.nx, args.nx, args.nz3, args.photons)
    config = {'workload': workload, 'nx': args.nx, 'ny': args.nx, 'nz3': args.nz3, 'photons_per_set': args.photons, 'Nrun': 3, 'Ng': 16,
              'l2': 'inputs larger than L2 (no flush)', 'parallelism': 'photons sharded over %d GPU(s), one NCCL all-reduce of tallies' % world}

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == 'reference':
        if rank != 0:
            return
        kw, abs0 = build_workload(args.nx, args.nx, args.nz3, args.photons)
        import oracle
        from er3t_b200 import abi
        from er3t_b200.rtm.mca import mcarats_ng
        cores = host_cores()
        # size the per-step sample from a probe so that the whole run ends within a few minutes
        probe, _, _ = cpu_oracle_rate(kw, abs0, seconds=6.0, nthreads=cores)
        nstep = max(1, args.steps + args.warmup)
        sample = int(max(2e4, min(args.photons, probe * 100.0 / nstep)))
        k = dict(kw); k.update(photons=sample, Nrun=1, dry_run=True)
        m = mcarats_ng(**k)
        jobs, keep = abi.make_jobs(**m.jobs_args)
        for _ in range(args.warmup):
            oracle.run(m.scene, m.options, jobs, nthreads=cores)
        t0 = time.time()
        for _ in range(args.steps):
            oracle.run(m.scene, m.options, jobs, nthreads=cores)
        dt = time.time() - t0
        val = sample * args.steps / dt
        line = {'impl': 'reference', 'metric': 'photons/s', 'value': val, 'unit': 'photons/s', 'n_gpus': args.gpus, 'steps': args.steps,
                'warmup': args.warmup, 'ms_per_step': 1e3 * dt / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
                'dtype': 'f64', 'data': 'synthetic', 'config': config,
                'cpu_baseline': {'value': val, 'unit': 'photons/s', 'cores': cores, 'kind': 'port', 'published_reference': PUBLISHED,
                                 'sample': '%d photons per step of the same scene (1 run x 16 g), oracle/oracle_mc.cpp with OpenMP; MCARaTS itself cannot be built offline' % sample},
                'e2e': {'value': val, 'unit': 'photons/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
        print(json.dumps(line))
        return

    # ------------------------------------------------------------------ this repo (CUDA)
    import torch
    from er3t_b200 import abi, dist as edist
    from er3t_b200.solver import Solver
    from er3t_b200.rtm.mca import mcarats_ng, mca_out_ng

    if not torch.cuda.is_available():
        raise OSError('Error [bench]: no CUDA device; the product path has no CPU fallback (use --impl reference for the CPU arm).')
    rank, world, local = edist.init_from_env()
    torch.cuda.set_device(local)
    # weak scaling: every GPU traces the full BASELINE photon count, the job set grows with the number of GPUs
    kw, abs0, parts = build_workload(args.nx, args.nx, args.nz3, args.photons * world, parts=True)
    # the e2e leg's inputs -- the raw cloud fields -- live in page-locked host memory (the contract's "pinned host
    # inputs"); mca_atm_3d(device_props=True) hands them to the library without a host copy
    from er3t_b200.util import pin_array
    for key in ('extinction', 'cer'):
        parts['cld'].lay[key]['data'] = pin_array(np.asarray(parts['cld'].lay[key]['data'], dtype=np.float32))
    kw['device'] = local
    kw['supervoxel'] = tuple(int(v) for v in args.sv.split(','))
    kw['shard'] = (rank, world)

    sol = Solver(device=local)
    prep = mcarats_ng(**dict(kw, dry_run=True))
    jobs, keep = abi.make_jobs(**prep.jobs_args)
    prep.options.empty_runs = args.empty_runs
    sol.upload_scene(prep.scene, prep.options)
    photons_step = int(np.sum(prep.jobs_args['nphot']))          # whole job set, all ranks

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def step_resident():
        sol.run(jobs, sync=False)
        if world > 1:
            return edist.allreduce_results(sol, to_host=False)
        sol.sync()
        return None

    for _ in range(args.warmup):
        step_resident()
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kern_ms, bytes_alg, launches = [], [], 0
    ev0.record()
    for _ in range(args.steps):
        step_resident()
        st = sol.stats() if world == 1 else None
        if st is not None:
            kern_ms.append(st['elapsed_ms']); bytes_alg.append(st['bytes_alg']); launches += int(st['launches'])
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    if world > 1:
        sol.sync()
        st = sol.stats()
        kern_ms.append(st['elapsed_ms']); bytes_alg.append(st['bytes_alg']); launches = int(st['launches']) * args.steps
        t = torch.tensor([ms], dtype=torch.float64, device='cuda')
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        ms = float(t.item())
    clocks = sampler.stop() if sampler is not None else None
    value = photons_step * args.steps / (ms * 1e-3)
    if args.dump_outputs and rank == 0:
        # before the legs below upload other scenes into the same handle
        dump_outputs(args.dump_outputs, sol.results())

    # ---- strong scaling (N > 1): the FIXED BASELINE job set (3 x 1e8 photons) sharded over the ranks, same timing rules
    strong = None
    if world > 1:
        kws = dict(kw, photons=args.photons)
        preps = mcarats_ng(**dict(kws, dry_run=True))
        jobs_s, keep_s = abi.make_jobs(**preps.jobs_args)
        sol.upload_scene(preps.scene, preps.options)

        def step_strong():
            sol.run(jobs_s, sync=False)
            return edist.allreduce_results(sol, to_host=False)
        for _ in range(args.warmup):
            step_strong()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            step_strong()
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device='cuda')
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        ms_s = float(t.item())
        sol.sync()
        nphot_s = int(np.sum(preps.jobs_args['nphot']))
        strong = {'value': nphot_s * args.steps / (ms_s * 1e-3), 'unit': 'photons/s', 'photons_per_step': nphot_s, 'ms_per_step': ms_s / args.steps,
                  'kernel_ms_per_launch_rank0': float(sol.stats()['elapsed_ms']),
                  'efficiency_vs_weak': (nphot_s * args.steps / (ms_s * 1e-3)) / value,
                  'note': 'same job set as N = 1 (3 x 1e8 photons), photons of every job split over the ranks, one in-place NCCL all-reduce of the tallies per step'}

    # ---- end to end through the public API (host inputs, H2D and D2H inside the timed region).  The step starts from the
    #      raw cloud fields: mca_atm_3d(device_props=True) hands extinction + effective radius to the library, whose
    #      packing kernel derives (omega, apf) on the GPU (er3t/rtm/mca/mca_atm.py:231-337 is the host loop it replaces)
    e2e = None
    esteps = max(1, args.e2e_steps)
    h2d = d2h = 0
    from er3t_b200.rtm.mca import mca_atm_3d

    def step_e2e():
        a3 = mca_atm_3d(cld_obj=parts['cld'], atm_obj=parts['atm'], pha_obj=parts['pha'], quiet=True, device_props=True)
        m = mcarats_ng(**dict(kw, atm_3ds=[a3], solver_obj=sol, reduce=(lambda s: edist.allreduce_results(s)) if world > 1 else None))
        out = mca_out_ng(mca_obj=m, abs_obj=abs0, mode='mean', squeeze=True)
        return m, out
    step_e2e()
    barrier()
    t0 = time.time()
    for _ in range(esteps):
        m, out = step_e2e()
    barrier()
    dt = time.time() - t0
    if world > 1:
        t = torch.tensor([dt], dtype=torch.float64, device='cuda')
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        dt = float(t.item())
    h2d = int(m.h2d_bytes)
    d2h = int(8 * prep.scene.rad_size(prep.nslab))
    e2e = {'value': photons_step * esteps / dt, 'unit': 'photons/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
           'steps': esteps, 'ms_per_step': 1e3 * dt / esteps,
           'api': 'er3t_b200.rtm.mca: mca_atm_3d(cld, atm, pha, device_props=True) + mcarats_ng(...) + mca_out_ng(...) from host numpy '
                  'extinction / effective-radius fields: the input builder is INSIDE the timed region'}

    # ---- accuracy (rank 0, N = 1): the number the metric is quoted with ("photons/s ...; flux/radiance err")
    accuracy = None
    if world == 1 and not args.no_accuracy:
        accuracy = accuracy_summary(sol)

    # ---- config-4 sweep sharded over the ranks (N > 1): photon sharding vs whole wavelengths per rank (tools/c4_sweep.py)
    c4 = None
    if world > 1 and args.c4_photons > 0:
        try:
            sys.path.insert(0, os.path.join(ROOT, 'tools'))
            from c4_sweep import sweep_both
            c4 = sweep_both(sol, rank, world, scale=1.0, reps=1, photons=args.c4_photons)
        except Exception as e:                                 # never lose the headline line to the extra leg
            c4 = {'error': repr(e)[:300]}

    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()
    if rank != 0:
        return
    peak, peak_src = measured_peak()
    t_kernel = float(np.mean(kern_ms)) * 1e-3
    achieved = float(np.mean(bytes_alg)) / t_kernel / 1e9
    cap = ncu_traffic('ncu_capture') or {}
    wipp = cap.get('warp_instructions_per_photon')
    sm_hz = 1e6 * float((clocks or {}).get('sm_mhz') or 1965.0)
    issue = None
    if wipp:
        # issue-slot roofline: warp instructions per photon (ncu) x photons/s of the kernel / (148 SMs x 4 schedulers x SM clock)
        ach = wipp * (photons_step / world) / t_kernel
        issue = {'achieved': ach, 'peak': 148 * 4 * sm_hz, 'unit': 'warp instructions/s', 'frac': ach / (148 * 4 * sm_hz),
                 'warp_instructions_per_photon': wipp, 'source': cap.get('file')}
    roofline = {'bound': 'hbm', 'limiter': 'instruction issue / dependent-gather latency (the HBM fraction only says that bytes are not the limit)',
                'issue': issue,
                'kernel': 'transport_kernel', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak,
                'traffic': ncu_traffic(), 'peak_source': peak_src, 'bytes_alg_per_launch': float(np.mean(bytes_alg)),
                'kernel_ms_per_launch': float(np.mean(kern_ms)),
                'bytes_alg_per_photon': float(np.mean(bytes_alg)) / (photons_step / world),
                'ncu': cap}
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        r, n, cores = cpu_oracle_rate(kw, abs0, seconds=15.0)
        cpu = {'value': r, 'unit': 'photons/s', 'cores': cores, 'kind': 'port', 'published_reference': PUBLISHED,
               'sample': '%d photons of the same scene (1 run x 16 g) on the host cores, oracle/oracle_mc.cpp (fp64, exact traversal, OpenMP)' % n}
    line = {'metric': 'photons/s', 'value': value, 'unit': 'photons/s', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32 (fp64 tallies)', 'data': 'synthetic', 'config': config,
            'e2e': e2e, 'gpu_launches': launches, 'clocks': clocks, 'roofline': roofline, 'cpu_baseline': cpu,
            'photons_per_step': photons_step, 'accuracy': accuracy, 'strong': strong, 'c4_sweep': c4}
    print(json.dumps(line))


if __name__ == '__main__':
    # stdout carries exactly ONE line (the JSON of rank 0): whatever libraries print while the benchmark runs (NCCL's
    # version banner goes to stdout) is sent to stderr instead
    sys.stdout.flush()
    _saved_stdout = os.dup(1)
    os.dup2(2, 1)
    _real_print = print

    def print(*a, **k):                                    # noqa: A001  (only the JSON line is printed in this file)
        sys.stdout.flush()
        os.dup2(_saved_stdout, 1)
        _real_print(*a, **k)
        sys.stdout.flush()
        os.dup2(2, 1)
    main()
