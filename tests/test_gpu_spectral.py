"""
Spectral runs (b200rt_run_kd, mcarats_ng(spectral=True)): one photon history serves every k-distribution term of a
wavelength.  On the GPU: exact reduction to b200rt_run (one term, or terms that sum to one, without gas absorption),
a closed form for a non-scattering atmosphere, statistical parity with the per-g jobs on a C4-like scene, and sharding.
Without a GPU: the documented errors of mcarats_ng and the ctypes layout of b200rt_kd.
"""

import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import workloads
from er3t_b200 import abi
from er3t_b200.rtm import mca as bmca

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), '..'))


def _balance(st):
    return (st['w_toa_up'] + st['w_sfc_abs'] + st['w_atm_abs'] - st['w_roulette']) / st['photons'] - 1.0


def _c2_small():
    """C2-like scene at small scale with an oblique extra view: (scene, options, nz)"""
    kw, _ = workloads.c2(scale=0.01, nrun=1)
    kw = dict(kw, extra_sensors=[dict(sensor_zenith_angle=35.0, sensor_azimuth_angle=60.0)], dry_run=True)
    m = bmca.mcarats_ng(**kw)
    return m.scene, m.options, m.scene.struct.nz


def _run(solver, scene, opt, nphot, seed, kd=None):
    jobs, keep = abi.make_jobs([nphot], [seed], [0])
    solver.upload_scene(scene, opt)
    if kd is None:
        solver.run(jobs)
    else:
        k, keep2 = abi.make_kd(njob=1, **kd)
        solver.run_kd(jobs, k)
    return solver.read_rad().copy(), solver.stats()


COUNTERS = ('photons', 'n_cell', 'n_tent', 'n_coll', 'n_sfc', 'n_le', 'n_le_visit', 'n_tally', 'n_roulette_kill')


@pytest.mark.gpu
def test_one_term_without_absorption_equals_run(solver):
    scene, opt, nz = _c2_small()
    r0, s0 = _run(solver, scene, opt, 200000, 11)
    r1, s1 = _run(solver, scene, opt, 200000, 11, kd=dict(abs1d=np.zeros((1, nz)), wkd=[1.0], rad_scale=[1.0]))
    assert r0.max() > 0
    np.testing.assert_allclose(r1, r0, rtol=1e-12, atol=0)
    for k in COUNTERS:
        assert s0[k] == s1[k], k
    assert abs(_balance(s1)) < 1e-9


@pytest.mark.gpu
def test_terms_that_sum_to_one_split_the_same_histories(solver):
    scene, opt, nz = _c2_small()
    r0, s0 = _run(solver, scene, opt, 200000, 11)
    w = [0.125, 0.125, 0.25, 0.5]
    r4, s4 = _run(solver, scene, opt, 200000, 11, kd=dict(abs1d=np.zeros((4, nz)), wkd=w, rad_scale=w))
    np.testing.assert_allclose(r4, r0, rtol=1e-12, atol=0)
    for k in COUNTERS:
        assert s0[k] == s4[k], k


@pytest.mark.gpu
@pytest.mark.parametrize('block3d', [False, True])
def test_non_scattering_atmosphere_closed_form(solver, block3d):
    """Every history goes straight to the Lambertian surface: its only contribution is
    sum_g rad_scale_g (alpha / pi) mu0 exp(-tau_g / mu0) exp(-tau_g / mu_v) per unit domain-mean radiance."""
    nx = ny = 16
    zgrd = np.linspace(0.0, 10000.0, 11)
    nz = zgrd.size - 1
    kw = {}
    if block3d:
        # a transparent 3-D block: oblique local estimates walk it voxel by voxel (le_tau_generic)
        kw = dict(iz3l=2, ext3d=np.zeros((nx, ny, 3), np.float32), omg3d=np.ones((nx, ny, 3), np.float32),
                  apf3d=np.zeros((nx, ny, 3), np.float32))
    alpha, sza = 0.3, 40.0
    views = (0.0, 30.0)
    sensors = [dict(kind=2, the=180.0 - v, phi=270.0 - 45.0, zloc=705000.0, nxr=nx, nyr=ny) for v in views]
    scene = abi.HostScene(zgrd, np.zeros((1, nz)), np.ones((1, nz)), np.zeros((1, nz)), nx=nx, ny=ny, dx=1000.0, dy=1000.0,
                          sfc_type=abi.SFC_LAMBERT, sfc_param=(alpha, 0, 0, 0, 0), src_the=180.0 - sza, src_phi=200.0, src_qmax=0.0,
                          sensors=sensors, **kw)
    opt = abi.make_options(target=abi.TARGET_RADIANCE, wmin=0.0, smem_tally=-1)
    tau = np.geomspace(1e-3, 10.0, 6)
    prof = np.linspace(2.0, 0.5, nz)                     # absorption decreasing with height
    abs1d = tau[:, None] * (prof / (prof * np.diff(zgrd)).sum())[None, :]
    rs = np.array([0.3, 0.1, 0.2, 0.15, 0.05, 0.2])
    r, st = _run(solver, scene, opt, 100000, 5, kd=dict(abs1d=abs1d, wkd=np.full(tau.size, 1.0 / tau.size), rad_scale=rs))
    mu0 = np.cos(np.radians(sza))
    n = nx * ny
    for k, v in enumerate(views):
        muv = np.cos(np.radians(v))
        exp = np.sum(rs * alpha / np.pi * mu0 * np.exp(-tau / mu0) * np.exp(-tau / muv))
        got = r[k * n:(k + 1) * n].mean()
        assert abs(got / exp - 1.0) < 1e-5, (v, got, exp)
    assert abs(_balance(st)) < 1e-9


@pytest.mark.gpu
def test_statistical_parity_with_per_g_jobs(solver, tmp_path):
    """C4-like scene (line centre: column gas optical depths 1e-3 ... 10): spectral and per-g runs estimate the same fused
    radiance."""
    kw, abs0 = workloads.c4(scale=0.014, nwvl=2)[1]
    nrun = 24
    kw = dict(kw, Nrun=nrun, photons=1e6, fdir=str(tmp_path), solver_obj=solver)
    ms = bmca.mcarats_ng(**dict(kw, seed=101, spectral=True))
    rs = np.array(ms.fused['radiance'][0])[:, :, 0, 0, :]
    bs = _balance(ms.stats)
    mg = bmca.mcarats_ng(**dict(kw, seed=9001))
    rg = np.array(mg.fused['radiance'][0])[:, :, 0, 0, :]
    assert ms.stats['photons'] == nrun * int(1e6)
    assert abs(bs) < 1e-9 and abs(_balance(mg.stats)) < 1e-9
    a, b = rs.mean(axis=(0, 1)), rg.mean(axis=(0, 1))    # domain mean per run
    assert abs(a.mean() / b.mean() - 1.0) < 0.003, (a.mean(), b.mean())
    sm, ss = rs.mean(axis=-1), rs.std(axis=-1, ddof=1) / np.sqrt(nrun)
    gm, gs = rg.mean(axis=-1), rg.std(axis=-1, ddof=1) / np.sqrt(nrun)
    den = np.hypot(ss, gs)
    z = (sm - gm)[den > 0] / den[den > 0]
    assert z.size > 0.9 * sm.size
    assert np.mean(np.abs(z) > 4.0) < 1e-3, np.sort(np.abs(z))[-10:]


@pytest.mark.gpu
def test_shards_add_up(solver):
    scene, opt, nz = _c2_small()
    rng = np.random.default_rng(3)
    kd = dict(abs1d=rng.uniform(0, 2e-5, (5, nz)), wkd=rng.uniform(0.1, 1, 5), rad_scale=rng.uniform(0.5, 1.5, 5))
    full, _ = _run(solver, scene, opt, 150000, 21, kd=kd)
    parts = []
    for rank in (0, 1):
        o = abi.make_options(target=opt.target, nslab=opt.nslab, wmin=opt.wmin, wfac=opt.wfac, iso_ss=opt.iso_ss, iso_max=opt.iso_max,
                             shard_rank=rank, shard_world=2)
        parts.append(_run(solver, scene, o, 150000, 21, kd=kd)[0])
    assert full.max() > 0
    np.testing.assert_allclose(parts[0] + parts[1], full, rtol=1e-12, atol=1e-300)
    # accumulate: the second shard adds onto the tallies of the first
    jobs, keep = abi.make_jobs([150000], [21], [0])
    k, keep2 = abi.make_kd(njob=1, **kd)
    o = abi.make_options(target=opt.target, nslab=opt.nslab, wmin=opt.wmin, wfac=opt.wfac, iso_ss=opt.iso_ss, iso_max=opt.iso_max,
                         shard_rank=0, shard_world=1)
    solver.upload_scene(scene, o)
    solver.run_kd(jobs, k)
    solver.run_kd(jobs, k, accumulate=True)
    np.testing.assert_allclose(solver.read_rad(), 2.0 * full, rtol=1e-12)


@pytest.mark.gpu
def test_unsupported_targets_are_rejected_by_the_library(solver):
    scene, opt, nz = _c2_small()
    jobs, keep = abi.make_jobs([1000], [1], [0])
    k, keep2 = abi.make_kd(np.zeros((2, nz)), [0.5, 0.5])
    o = abi.make_options(target=abi.TARGET_RADIANCE | abi.TARGET_FLUX)
    solver.upload_scene(scene, o)
    with pytest.raises(OSError, match='radiance targets only'):
        solver.run_kd(jobs, k)
    solver.upload_scene(scene, opt)
    k33, keep3 = abi.make_kd(np.zeros((33, nz)), np.ones(33))
    with pytest.raises(OSError, match='nkd must be 1 ... 32'):
        solver.run_kd(jobs, k33)
    jobs_abs, keep4 = abi.make_jobs([1000], [1], [0], abs1d=[np.zeros(nz)])
    with pytest.raises(OSError, match='must be NULL'):
        solver.run_kd(jobs_abs, k)


# ---------------------------------------------------------------------------------------------------- host only
@pytest.fixture(scope='module')
def c4_kw():
    kw, abs0 = workloads.c4(scale=0.0005, nwvl=1)[0]
    return dict(kw, Nrun=1, photons=1e4, spectral=True)


@pytest.mark.parametrize('change, msg', [
    (dict(raw=True), 'raw'),
    (dict(target='flux'), 'radiance'),
    (dict(target='heating rate'), 'radiance'),
    (dict(sensor_type='all-sky camera'), 'satellite'),
])
def test_spectral_errors(c4_kw, tmp_path, change, msg):
    with pytest.raises(OSError, match=r'Error \[mcarats_ng\]: .*' + msg):
        bmca.mcarats_ng(**dict(c4_kw, fdir=str(tmp_path), **change))


def test_spectral_rejects_write_files(c4_kw, tmp_path):
    with pytest.raises(OSError, match=r'Error \[mcarats_ng\]: .*write_files'):
        bmca.mcarats_ng(**dict(c4_kw, fdir=str(tmp_path / 'out'), write_files=True))


def test_spectral_needs_an_absorption_object(c4_kw, tmp_path):
    atm = c4_kw['atm_1ds'][0]
    saved = atm.abs
    try:
        atm.abs = None
        with pytest.raises(OSError, match=r'Error \[mcarats_ng\]: .*absorption'):
            bmca.mcarats_ng(**dict(c4_kw, fdir=str(tmp_path)))
    finally:
        atm.abs = saved


def test_spectral_dry_run_builds_one_job_per_run(c4_kw, tmp_path):
    m = bmca.mcarats_ng(**dict(c4_kw, Nrun=3, fdir=str(tmp_path), dry_run=True))
    ja = m.jobs_args
    assert ja['slabs'] == [0, 1, 2] and ja['nphot'] == [int(1e4)] * 3
    assert ja['seeds'] == [int(m.seeds[ir, 0]) for ir in range(3)]
    assert all(a is None for a in ja['abs1d']) and all(f is None for f in ja['flx_scale'])
    kd = m.kd_args
    assert kd['abs1d'].shape == (m.Ng, m.scene.struct.nz)
    np.testing.assert_allclose(kd['wkd'], m.weights)
    k, keep = abi.make_kd(njob=3, **kd)
    assert len(k) == 3 and k[2].nkd == m.Ng


def test_kd_struct_layout_matches_header(tmp_path):
    probe = tmp_path / 'probe.c'
    probe.write_text('''
#include <stdio.h>
#include <stddef.h>
#include "b200rt.h"
int main(void) {
  printf("%zu %zu %zu %zu %zu\\n", sizeof(b200rt_kd), offsetof(b200rt_kd, nkd), offsetof(b200rt_kd, wkd),
         offsetof(b200rt_kd, abs1d), offsetof(b200rt_kd, rad_scale));
  return 0;
}''')
    exe = tmp_path / 'probe'
    subprocess.check_call(['gcc', '-I', os.path.join(ROOT, 'include'), str(probe), '-o', str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).decode().split()]
    K = abi.Kd
    assert got == [C.sizeof(K), K.nkd.offset, K.wkd.offset, K.abs1d.offset, K.rad_scale.offset]
