"""
Radiance Jacobians with respect to the gas absorption of layer groups (b200rt_run_jac, Solver.run_jac,
mcarats_ng(gas_jacobian=...)), tallied inside the histories of the radiance run.  On the GPU: the same histories as
b200rt_run, a closed form for a non-scattering atmosphere, common-random-number finite differences (no roulette: the
trajectories do not depend on the absorption), additivity over groups, roulette, shards / accumulate, the end-to-end path
through mcarats_ng and mca_out_ng, library-side rejections and a two-rank NCCL reduction.
"""

import copy
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

import workloads
from er3t_b200 import abi
from er3t_b200.rtm import mca as bmca

pytestmark = pytest.mark.gpu
ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), '..'))
COUNTERS = ('photons', 'n_cell', 'n_tent', 'n_coll', 'n_sfc', 'n_le', 'n_le_visit', 'n_roulette_kill')


def _c2_small(photons=2e5, wmin=None):
    """C2-like scene at small scale, an oblique extra view, 16 per-g jobs with gas absorption: (scene, options, jobs_args)"""
    kw, _ = workloads.c2(scale=0.01, nrun=1)
    kw = dict(kw, extra_sensors=[dict(sensor_zenith_angle=35.0, sensor_azimuth_angle=60.0)], dry_run=True, photons=photons, wmin=wmin)
    m = bmca.mcarats_ng(**kw)
    return m.scene, m.options, m.jobs_args


def _scaled(jobs_args, fac):
    """jobs_args with abs1d multiplied by fac (a (nz,) array or a scalar)"""
    return dict(jobs_args, abs1d=[None if a is None else a * fac for a in jobs_args['abs1d']])


def _run(solver, scene, opt, jobs_args, edges=None, accumulate=False, upload=True):
    jobs, keep = abi.make_jobs(**jobs_args)
    if upload:
        solver.upload_scene(scene, opt)
    if edges is None:
        solver.run(jobs, accumulate=accumulate)
        return solver.read_rad().copy(), None, solver.stats()
    solver.run_jac(jobs, edges, accumulate=accumulate)
    return solver.read_rad().copy(), solver.read_jac().copy(), solver.stats()


def test_same_histories_as_run(solver):
    scene, opt, ja = _c2_small()
    nz = scene.struct.nz
    assert any(a is not None and a.max() > 0 for a in ja['abs1d'])
    r0, _, s0 = _run(solver, scene, opt, ja)
    r1, j1, s1 = _run(solver, scene, opt, ja, edges=np.arange(nz + 1))
    assert r0.max() > 0
    np.testing.assert_allclose(r1, r0, rtol=1e-12, atol=0)
    for k in COUNTERS:
        assert s0[k] == s1[k], k
    assert s1['n_tally'] > s0['n_tally']
    assert j1.shape == (opt.nslab, scene.rad_size(1), nz)
    assert np.all(j1.sum(axis=-1) <= 0) and j1.min() < 0            # more absorption never brightens a pixel


@pytest.mark.parametrize('block3d', [False, True])
def test_non_scattering_atmosphere_closed_form(solver, block3d):
    """Every history goes straight to the Lambertian surface and its local estimate straight to the sensor:
    I = (alpha / pi) mu0 exp(-tau / mu0) exp(-tau / mu_v) and dI / dln(a_j) = -I tau_j (1 / mu0 + 1 / mu_v)."""
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
    tau = np.geomspace(1e-3, 10.0, 6)
    prof = np.linspace(2.0, 0.5, nz)                     # absorption decreasing with height
    abs1d = tau[:, None] * (prof / (prof * np.diff(zgrd)).sum())[None, :]
    opt = abi.make_options(target=abi.TARGET_RADIANCE, nslab=tau.size, wmin=0.0, smem_tally=-1)
    ja = dict(nphot=[50000] * tau.size, seeds=list(range(5, 5 + tau.size)), slabs=list(range(tau.size)), abs1d=list(abs1d))
    r, jac, st = _run(solver, scene, opt, ja, edges=np.arange(nz + 1))
    mu0 = np.cos(np.radians(sza))
    n = nx * ny
    r = r.reshape(tau.size, -1)
    for s in range(tau.size):
        tau_j = abs1d[s] * np.diff(zgrd)
        for k, v in enumerate(views):
            muv = np.cos(np.radians(v))
            rad = alpha / np.pi * mu0 * np.exp(-tau[s] / mu0) * np.exp(-tau[s] / muv)
            got = r[s, k * n:(k + 1) * n].mean()
            assert abs(got / rad - 1.0) < 1e-5, (s, v, got, rad)
            exp = -rad * tau_j * (1.0 / mu0 + 1.0 / muv)
            gj = jac[s, k * n:(k + 1) * n].mean(axis=0)
            np.testing.assert_allclose(gj, exp, rtol=1e-5, err_msg='slab %d view %g' % (s, v))


def _group_edges(nz, ngrp):
    return np.unique(np.round(np.linspace(0, nz, ngrp + 1)).astype(int))


def test_common_random_number_finite_difference(solver):
    """wmin = 0: the trajectories do not depend on the absorption, so a central difference with the absorption of group j
    scaled by 1 +- eps and the same seeds follows the same histories as the Jacobian run."""
    scene, opt, ja = _c2_small(photons=3e5, wmin=0.0)
    nz = scene.struct.nz
    edges = _group_edges(nz, 4)
    _, jac, _ = _run(solver, scene, opt, ja, edges=edges)
    eps = 1e-2
    for j in range(edges.size - 1):
        fac = np.ones(nz)
        fac[edges[j]:edges[j + 1]] = 1.0 + eps
        rp, _, _ = _run(solver, scene, opt, _scaled(ja, fac))
        fac[edges[j]:edges[j + 1]] = 1.0 - eps
        rm, _, _ = _run(solver, scene, opt, _scaled(ja, fac))
        fd = ((rp - rm) / (2.0 * eps)).reshape(jac.shape[:-1])
        jj = jac[..., j]
        assert jj.min() < 0
        assert abs(jj.mean() / fd.mean() - 1.0) < 2e-3, (j, jj.mean(), fd.mean())
        big = np.abs(fd) > 1e-3 * np.abs(fd).max()
        rel = np.abs(jj[big] - fd[big]) / np.abs(fd[big])
        assert np.mean(rel < 2e-2) > 0.99, (j, np.sort(rel)[-10:])


def test_groups_add_up_and_no_absorption_gives_zero(solver):
    scene, opt, ja = _c2_small()
    nz = scene.struct.nz
    _, j_all, _ = _run(solver, scene, opt, ja, edges=np.arange(nz + 1))
    _, j_one, _ = _run(solver, scene, opt, ja, edges=[0, nz])
    _, j_four, _ = _run(solver, scene, opt, ja, edges=_group_edges(nz, 4))
    tot = j_all.sum(axis=-1)
    scale = np.abs(tot).max()
    np.testing.assert_allclose(j_one[..., 0], tot, rtol=1e-5, atol=1e-6 * scale)
    np.testing.assert_allclose(j_four.sum(axis=-1), tot, rtol=1e-5, atol=1e-6 * scale)
    # jobs without gas absorption: no Jacobian update at all, the same tally traffic as b200rt_run
    clear = _scaled(ja, 1.0)
    clear['abs1d'] = [None] * len(clear['abs1d'])
    r0, _, s0 = _run(solver, scene, opt, clear)
    r1, j1, s1 = _run(solver, scene, opt, clear, edges=_group_edges(nz, 4))
    np.testing.assert_allclose(r1, r0, rtol=1e-12, atol=0)
    assert not np.any(j1) and s1['n_tally'] == s0['n_tally']


def test_roulette_leaves_the_jacobian_unbiased(solver):
    """Domain-mean Jacobian per group with the default Pho_wmin against wmin = 0, over independent slabs"""
    nslab = 12
    means = {}
    for wmin in (None, 0.0):
        scene, opt, ja = _c2_small(photons=1e5, wmin=wmin)
        nz = scene.struct.nz
        edges = _group_edges(nz, 4)
        o = abi.make_options(target=opt.target, nslab=nslab, wmin=opt.wmin, wfac=opt.wfac, iso_ss=opt.iso_ss, iso_max=opt.iso_max)
        nj = len(ja['nphot'])
        rep = dict(nphot=list(ja['nphot']) * nslab, seeds=[int(s) + 7919 * k + (0 if wmin is None else 104729) for k in range(nslab) for s in ja['seeds']],
                   slabs=[k for k in range(nslab) for _ in range(nj)], abs1d=list(ja['abs1d']) * nslab, rad_scale=list(ja['rad_scale']) * nslab)
        _, jac, _ = _run(solver, scene, o, rep, edges=edges)
        means[wmin] = jac.mean(axis=1)                                    # (nslab, ngrp)
    a, b = means[None], means[0.0]
    assert np.all(a.mean(axis=0) < 0)
    sig = np.hypot(a.std(axis=0, ddof=1), b.std(axis=0, ddof=1)) / np.sqrt(nslab)
    z = (a.mean(axis=0) - b.mean(axis=0)) / sig
    assert np.all(np.abs(z) < 4.0), z


def test_shards_add_up_and_accumulate(solver):
    scene, opt, ja = _c2_small(photons=1.5e5)
    nz = scene.struct.nz
    edges = _group_edges(nz, 5)
    full_r, full_j, _ = _run(solver, scene, opt, ja, edges=edges)
    parts = []
    for rank in (0, 1):
        o = abi.make_options(target=opt.target, nslab=opt.nslab, wmin=opt.wmin, wfac=opt.wfac, iso_ss=opt.iso_ss, iso_max=opt.iso_max,
                             shard_rank=rank, shard_world=2)
        parts.append(_run(solver, scene, o, ja, edges=edges))
    assert full_j.min() < 0
    np.testing.assert_allclose(parts[0][0] + parts[1][0], full_r, rtol=1e-12, atol=1e-300)
    np.testing.assert_allclose(parts[0][1] + parts[1][1], full_j, rtol=1e-12, atol=1e-300)
    # accumulate: the second run adds onto the tallies of the first
    _run(solver, scene, opt, ja, edges=edges)
    r2, j2, _ = _run(solver, scene, opt, ja, edges=edges, accumulate=True, upload=False)
    np.testing.assert_allclose(r2, 2.0 * full_r, rtol=1e-12)
    np.testing.assert_allclose(j2, 2.0 * full_j, rtol=1e-12)
    assert 'jac' in solver.results()
    # a plain run afterwards: no Jacobian any more
    _run(solver, scene, opt, ja, upload=False)
    assert 'jac' not in solver.results()
    with pytest.raises(OSError, match='not a Jacobian run'):
        solver.read_jac()


def test_mcarats_ng_end_to_end_matches_crn_finite_difference(solver, tmp_path):
    """Small C4 case (per-g jobs, wmin = 0): the sum over the groups of the fused Jacobian is d I / dln(a) for the whole
    absorption object, which a central difference with the absorption object scaled by 1 +- eps gives for the same
    histories."""
    kw, abs0 = workloads.c4(scale=0.002, nwvl=2)[1]
    kw = dict(kw, Nrun=2, photons=4e5, fdir=str(tmp_path), solver_obj=solver, wmin=0.0, seed=77,
              extra_sensors=[dict(sensor_zenith_angle=30.0, sensor_azimuth_angle=45.0)])
    atm0 = kw['atm_1ds'][0].atm
    lev = atm0.lev['altitude']['data']
    m = bmca.mcarats_ng(**dict(kw, gas_jacobian=[lev[0], 2.0, 5.0, lev[-1]]))
    jac = np.asarray(m.fused['jacobian'][0])
    nx, ny = m.Nx, m.Ny
    assert jac.shape == (nx, ny, 3, 1, 2)
    np.testing.assert_allclose(m.jac_levels, [lev[0], 2.0, 5.0, lev[-1]])
    assert len(m.jac_extra) == 1 and m.jac_extra[0].shape == (nx, ny, 3, 2)
    rad = np.asarray(m.fused['radiance'][0])
    eps = 1e-3
    out = []
    for f in (1.0 + eps, 1.0 - eps):
        a = copy.deepcopy(abs0)
        a.coef['abso_coef']['data'] = a.coef['abso_coef']['data'] * f
        mf = bmca.mcarats_ng(**dict(kw, atm_1ds=[bmca.mca_atm_1d(atm_obj=atm0, abs_obj=a)]))
        out.append((np.asarray(mf.fused['radiance'][0]), mf.rad_extra[0]))
    m0 = bmca.mcarats_ng(**kw)
    np.testing.assert_allclose(rad, np.asarray(m0.fused['radiance'][0]), rtol=1e-12)      # gas_jacobian changes no radiance
    for got, fd in ((jac.sum(axis=2)[:, :, 0, :], (out[0][0] - out[1][0])[:, :, 0, 0, :] / (2 * eps)),
                    (m.jac_extra[0].sum(axis=2), (out[0][1] - out[1][1]) / (2 * eps))):
        assert fd.mean() < 0
        assert abs(got.mean() / fd.mean() - 1.0) < 2e-3, (got.mean(), fd.mean())
    o = bmca.mca_out_ng(mca_obj=m, abs_obj=abs0, mode='mean')
    assert o.data['rad_jac']['data'].shape == (nx, ny, 3)
    assert o.data['rad_jac_std']['data'].shape == (nx, ny, 3)
    np.testing.assert_allclose(o.data['jac_levels']['data'], m.jac_levels)
    o0 = bmca.mca_out_ng(mca_obj=m0, abs_obj=abs0, mode='mean')
    assert not any(k.startswith('rad_jac') or k == 'jac_levels' for k in o0.data)


def test_unsupported_runs_are_rejected_by_the_library(solver):
    scene, opt, ja = _c2_small(photons=1e4)
    nz = scene.struct.nz
    jobs, keep = abi.make_jobs(**ja)
    solver.upload_scene(scene, abi.make_options(target=abi.TARGET_RADIANCE | abi.TARGET_FLUX))
    with pytest.raises(OSError, match='radiance targets only'):
        solver.run_jac(jobs, [0, nz])
    solver.upload_scene(scene, opt)
    for edges, msg in (([1, nz], 'start at layer 0'), ([0, nz - 1], 'end at nz'), ([0, 3, 3, nz], 'strictly increasing'),
                       (np.r_[np.arange(65), nz], 'ngrp must be 1 ... 64')):
        with pytest.raises(OSError, match=msg):
            solver.run_jac(jobs, edges)
    solver.run(jobs)
    with pytest.raises(OSError, match='not a Jacobian run'):
        solver.read_jac()
    with pytest.raises(OSError, match='accumulate needs the previous run to be a Jacobian run'):
        solver.run_jac(jobs, [0, nz], accumulate=True)
    solver.run_jac(jobs, [0, nz])
    with pytest.raises(OSError, match='same edges'):
        solver.run_jac(jobs, [0, 1, nz], accumulate=True)
    # the all-sky camera
    kw, _ = workloads.c2(scale=0.01, nrun=1)
    mc = bmca.mcarats_ng(**dict(kw, sensor_type='all-sky camera', camera_pixels=(8, 8), dry_run=True, photons=1e4))
    o = abi.make_options(target=mc.options.target, smem_tally=-1)
    solver.upload_scene(mc.scene, o)
    jc, keep2 = abi.make_jobs(**mc.jobs_args)
    with pytest.raises(OSError, match='all-sky camera'):
        solver.run_jac(jc, [0, mc.scene.struct.nz])


# ---------------------------------------------------------------------------------------------------- two ranks
def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _worker(rank, world, port, out):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    import torch.distributed as dist
    from er3t_b200 import abi, dist as edist
    from er3t_b200.solver import Solver
    edist.init_from_env(backend='nccl')
    scene, opt, ja = _c2_small(photons=1e5)
    o = abi.make_options(target=opt.target, nslab=opt.nslab, wmin=opt.wmin, wfac=opt.wfac, iso_ss=opt.iso_ss, iso_max=opt.iso_max,
                         shard_rank=rank, shard_world=world)
    jobs, keep = abi.make_jobs(**ja)
    s = Solver(device=rank)
    s.upload_scene(scene, o)
    s.run_jac(jobs, _group_edges(scene.struct.nz, 4), sync=False)
    res = edist.allreduce_results(s)
    assert np.array_equal(s.read_jac(), res['jac'])
    if rank == 0:
        np.savez(out, rad=res['rad'], jac=res['jac'], photons=res['stats']['photons'])
    dist.barrier()
    dist.destroy_process_group()
    s.close()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs two GPUs')
def test_two_nccl_ranks_reduce_the_jacobian(solver, tmp_path):
    out = str(tmp_path / 'j.npz')
    mp.spawn(_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    got = np.load(out)
    scene, opt, ja = _c2_small(photons=1e5)
    r, j, st = _run(solver, scene, opt, ja, edges=_group_edges(scene.struct.nz, 4))
    assert int(got['photons']) == st['photons']
    assert np.allclose(got['rad'], r, rtol=1e-9, atol=1e-15)
    assert np.allclose(got['jac'], j, rtol=1e-9, atol=1e-15)
