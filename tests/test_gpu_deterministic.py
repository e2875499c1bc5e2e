"""
The CUDA path against a DETERMINISTIC solver, an order of magnitude tighter than the GPU-vs-oracle parity tests.

tests/golden/ad_fixtures.npz holds converged adding-doubling results (oracle/adding_doubling.py::solve_beam, 320 streams,
96 azimuthal Fourier modes; made by tests/golden/make_ad_fixtures.py) for the config-1 atmosphere of BASELINE.json --
Rayleigh + gas absorption + a tau = 10 cloud in 1-2 km over a Lambertian surface, SZA 30 deg -- with (a) the 498-angle
Mie table of r_eff = 10 um at 650 nm and (b) Henyey-Greenstein g = 0.85: flux at all 21 levels and TOA radiance at nadir
and four oblique views.  The GPU traces >= 1e9 photons per case (seconds), which resolves ~1e-4 -- enough to expose any
bias of the fp32 flight, the fast-math intrinsics, the 24-bit uniforms or the fp32 cumulative profiles that the
0.5 % / 3 sigma tests cannot see.  The reference's counterpart: examples/00_er3t_bmk.py:470-579 (MCARaTS vs libRadtran).

Tolerance, written where it is used: |GPU - deterministic| <= 2e-4 relative (3e-4 for the nadir radiance of the Mie
case, the least converged entry of the fixture) + 4 standard errors of the GPU run itself (from 8 independent slabs).
"""

import numpy as np
import pytest

import scenes
from er3t_b200 import abi

pytestmark = pytest.mark.gpu

NSLAB = 8
RTOL = 2.0e-4


def run_case(solver, fx, nphot_total, hom3d=False):
    sc = scenes.ad_scene(fx, hom3d=hom3d)
    opt = abi.make_options(target=abi.TARGET_FLUX | abi.TARGET_RADIANCE, nslab=NSLAB, wmin=0.2)
    jobs, keep = scenes.multi_seed_jobs(int(nphot_total // NSLAB), NSLAB, abs1d=fx['absg'])
    solver.upload_scene(sc, opt)
    solver.run(jobs)
    r = solver.results()
    st = r['stats']
    bal = (st['w_toa_up'] + st['w_sfc_abs'] + st['w_atm_abs'] - st['w_roulette']) / st['photons'] - 1.0
    assert abs(bal) < 1e-9, bal
    nlev = fx['z'].size
    flux = r['flux'].reshape(NSLAB, 3, nlev, -1).mean(axis=-1)        # domain mean (1 or 2 x 2 columns)
    nview = fx['views'].shape[0]
    rad = r['rad'].reshape(NSLAB, nview, -1).mean(axis=-1)
    return flux, rad, st


def check(fx, flux, rad, rtol_rad0):
    mu0 = float(fx['mu0'])
    worst = {}
    for var, key in ((2, 'f_up'), (1, 'f_down'), (0, 'f_down_direct')):
        m, s = scenes.mean_sem(flux[:, var])
        ref = fx[key]
        tol = RTOL * np.maximum(ref, 0.05 * mu0) + 4.0 * s
        worst[key] = float(np.max(np.abs(m - ref) / np.maximum(ref, 0.05 * mu0)))
        assert np.all(np.abs(m - ref) <= tol), (key, worst[key], np.max(np.abs(m - ref) / tol))
    m, s = scenes.mean_sem(rad)
    ref = fx['rad_views']
    rt = np.full(ref.size, RTOL)
    rt[0] = rtol_rad0
    tol = rt * ref + 4.0 * s
    worst['rad'] = (m / ref - 1.0).tolist()
    assert np.all(np.abs(m - ref) <= tol), (worst['rad'], (s / ref).tolist())
    return worst


@pytest.mark.parametrize('name,rtol_nadir', [('mie', 3.0e-4), ('hg', 2.0e-4)])
def test_plane_parallel_1e9_photons_against_adding_doubling(solver, name, rtol_nadir):
    fx = scenes.ad_fixture(name)
    flux, rad, st = run_case(solver, fx, 1.2e9)
    w = check(fx, flux, rad, rtol_nadir)
    print('\n%s 1-D: %.0f M photons/s; worst relative deviations %s' % (name, st['photons'] / st['elapsed_ms'] / 1e3, w))


@pytest.mark.parametrize('name,rtol_nadir', [('mie', 3.0e-4), ('hg', 2.0e-4)])
def test_homogeneous_3d_block_1e9_photons_against_adding_doubling(solver, name, rtol_nadir):
    """The same atmosphere with the cloud as a 2 x 2-column 3-D block (the cld_gen_hom variant of config 1): exercises
    the voxel flight, the null-collision tracking and the local-estimate ray through the 3-D block at the same tolerance."""
    fx = scenes.ad_fixture(name)
    flux, rad, st = run_case(solver, fx, 1.0e9, hom3d=True)
    w = check(fx, flux, rad, rtol_nadir)
    print('\n%s hom-3D: %.0f M photons/s; worst relative deviations %s' % (name, st['photons'] / st['elapsed_ms'] / 1e3, w))


def test_reflectance_vs_cot_benchmark_against_adding_doubling(solver):
    """The reference's own benchmark (examples/00_er3t_bmk.py:24-46,470-579: func_ref_vs_cot over 35 COT values 0 ... 400 at
    650 nm, SZA 28.2797 deg, nadir, albedo 0.03, r_eff 10 um cloud in 1-2 km; there MCARaTS against libRadtran) through this
    repo's func_ref_vs_cot -- all 35 columns in ONE IPA launch with the tabulated Mie function -- against the deterministic
    adding-doubling curve of tests/golden/ad_cot_sweep.npz (made by tests/golden/make_cot_sweep.py from the same 1-D
    inputs) and, as the reference's class does, beside the two-stream estimate cal_r_twostream (er3t/util/util.py:1135).

    The local estimate of a nadir radiance under a Mie phase function has heavy-tailed noise (rare near-forward
    contributions; profiles/diag_cot_r02_k.txt: 0.1-0.35 % per point at 8e7 photons per COT, no systematic sign), so the
    test has two parts: every point within 1.5e-3 relative + 3 x the fixture's convergence estimate + 6 standard errors
    (8 runs), and the MEAN relative deviation over the cloudy points -- where the noise averages down -- within 2.5e-3."""
    import os
    import sys
    gdir = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
    sys.path.insert(0, gdir)
    import make_cot_sweep as mk
    import er3t_b200.rtm.mca as bmca
    fx = np.load(os.path.join(gdir, 'ad_cot_sweep.npz'))
    atm0, abs0, pha0 = mk.inputs()
    nrun = 8
    f = bmca.func_ref_vs_cot(fx['cot'], cer0=float(fx['cer']), fdir=None, date=mk.DATE, wavelength=650.0, surface_albedo=float(fx['albedo']),
                             solar_zenith_angle=float(fx['sza']), solar_azimuth_angle=238.9053, sensor_zenith_angle=0.0,
                             sensor_azimuth_angle=261.9049, cloud_top_height=2.0, cloud_geometrical_thickness=1.0, Nphoton=2e6,
                             seed=7, solver_obj=solver, atm0=atm0, pha0=pha0, abs0=abs0, Nrun=nrun)
    ref, sem = f.ref, f.ref_std / np.sqrt(nrun)
    tol = 1.5e-3 * fx['ref'] + 3.0 * fx['ref_conv'] + 6.0 * sem
    dev = np.abs(ref - fx['ref'])
    cloudy = fx['cot'] >= 2.0
    mean_rel = float(np.mean(ref[cloudy] / fx['ref'][cloudy] - 1.0))
    print('ref vs COT: max |dev| / ref %.2e, max dev / tol %.2f, mean relative deviation (COT >= 2) %+.2e' % (
        float(np.max(dev / fx['ref'])), float(np.max(dev / tol)), mean_rel))
    assert np.all(dev <= tol), (ref.tolist(), fx['ref'].tolist(), (dev / tol).tolist())
    assert abs(mean_rel) < 2.5e-3, mean_rel
    assert np.all(np.diff(ref) > -6.0 * np.hypot(sem[1:], sem[:-1])) and ref[-1] < 1.0        # monotone within the noise
    # two-stream estimate of the reference's class: same limits, same order of magnitude in between
    assert np.all(np.diff(f.ref_2s) > 0) and np.max(np.abs(f.ref_2s - ref)) < 0.12
    st = f.mca.stats
    assert abs((st['w_toa_up'] + st['w_sfc_abs'] + st['w_atm_abs'] - st['w_roulette']) / st['photons'] - 1.0) < 1e-9
