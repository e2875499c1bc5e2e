"""
Radiance path-length distributions (b200rt_run_plen, Solver.run_plen, mcarats_ng(path_length=...)), tallied inside the
histories of the radiance run.  On the GPU: the same histories as b200rt_run, a closed form for a non-scattering
atmosphere, the first moment against the gas-absorption Jacobian of the same histories and against common-random-number
finite differences, roulette, shards / accumulate, the end-to-end path through mcarats_ng and mca_out_ng, library-side
rejections and a two-rank NCCL reduction.
"""

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
BINS = (0.0, 200000.0, 64)           # tpmin, tpmax (m), ntp


def _c2_small(photons=2e5, wmin=None):
    """C2-like scene at small scale, an oblique extra view, 16 per-g jobs with gas absorption: (scene, options, jobs_args)"""
    kw, _ = workloads.c2(scale=0.01, nrun=1)
    kw = dict(kw, extra_sensors=[dict(sensor_zenith_angle=35.0, sensor_azimuth_angle=60.0)], dry_run=True, photons=photons, wmin=wmin)
    m = bmca.mcarats_ng(**kw)
    return m.scene, m.options, m.jobs_args


def _uniform(jobs_args, nz, k):
    """jobs_args with the gas absorption coefficient k (1/m) in every layer of every job"""
    return dict(jobs_args, abs1d=[np.full(nz, k) for _ in jobs_args['abs1d']])


def _run(solver, scene, opt, jobs_args, bins=None, accumulate=False, upload=True):
    jobs, keep = abi.make_jobs(**jobs_args)
    if upload:
        solver.upload_scene(scene, opt)
    if bins is None:
        solver.run(jobs, accumulate=accumulate)
        return solver.read_rad().copy(), None, solver.stats()
    solver.run_plen(jobs, *bins, accumulate=accumulate)
    return solver.read_rad().copy(), solver.read_plen().copy(), solver.stats()


def _views(scene):
    """slices of the radiance pixels of every sensor"""
    out, off = [], 0
    for se in scene.sensors:
        n = se.nxr * se.nyr
        out.append(slice(off, off + n))
        off += n
    return out


def test_same_histories_as_run(solver):
    scene, opt, ja = _c2_small()
    ntp = BINS[2]
    r0, _, s0 = _run(solver, scene, opt, ja)
    r1, p1, s1 = _run(solver, scene, opt, ja, bins=BINS)
    assert r0.max() > 0
    np.testing.assert_allclose(r1, r0, rtol=1e-12, atol=0)
    for k in COUNTERS:
        assert s0[k] == s1[k], k
    assert s1['n_tally'] == s0['n_tally'] + 2 * s1['n_le']
    assert p1.shape == (opt.nslab, scene.rad_size(1), ntp + 3)
    # bins + underflow + overflow sum to the radiance, pixel by pixel
    np.testing.assert_allclose(p1[..., :ntp + 2].sum(axis=-1), r1.reshape(p1.shape[:2]), rtol=1e-12, atol=0)
    assert np.all(p1 >= 0) and p1[..., :ntp].sum() > 0.5 * p1[..., :ntp + 2].sum()


@pytest.mark.parametrize('block3d', [False, True])
def test_non_scattering_atmosphere_closed_form(solver, block3d):
    """Every history goes straight to the Lambertian surface and its local estimate straight to the sensor, so every
    contribution has the path L = H / mu0 + H / mu_v, with or without gas absorption."""
    nx = ny = 16
    H = 10000.0
    zgrd = np.linspace(0.0, H, 11)
    nz = zgrd.size - 1
    kw = {}
    if block3d:
        # a transparent 3-D block: flights cross it cell by cell, oblique local estimates walk it voxel by voxel
        kw = dict(iz3l=2, ext3d=np.zeros((nx, ny, 3), np.float32), omg3d=np.ones((nx, ny, 3), np.float32),
                  apf3d=np.zeros((nx, ny, 3), np.float32))
    alpha, sza = 0.3, 40.0
    views = (0.0, 30.0)
    sensors = [dict(kind=2, the=180.0 - v, phi=270.0 - 45.0, zloc=705000.0, nxr=nx, nyr=ny) for v in views]
    scene = abi.HostScene(zgrd, np.zeros((1, nz)), np.ones((1, nz)), np.zeros((1, nz)), nx=nx, ny=ny, dx=1000.0, dy=1000.0,
                          sfc_type=abi.SFC_LAMBERT, sfc_param=(alpha, 0, 0, 0, 0), src_the=180.0 - sza, src_phi=200.0, src_qmax=0.0,
                          sensors=sensors, **kw)
    # slab 0 without gas absorption, slab 1 with it
    prof = np.linspace(2.0, 0.5, nz)
    abs1d = [None, 0.5 * prof / (prof * np.diff(zgrd)).sum()]
    opt = abi.make_options(target=abi.TARGET_RADIANCE, nslab=2, wmin=0.0, smem_tally=-1)
    ja = dict(nphot=[50000] * 2, seeds=[5, 6], slabs=[0, 1], abs1d=abs1d)
    bins = (0.0, 40000.0, 40)                              # 1 km bins
    r, pl, st = _run(solver, scene, opt, ja, bins=bins)
    ntp = bins[2]
    mu0 = np.cos(np.radians(sza))
    r = r.reshape(2, -1)
    for s in range(2):
        for k, (v, sl) in enumerate(zip(views, _views(scene))):
            L = H / mu0 + H / np.cos(np.radians(v))
            b = int(L // 1000.0)
            assert min(L - 1000.0 * b, 1000.0 * (b + 1) - L) >= 10.0
            rad = r[s, sl].sum()
            assert rad > 0
            t = pl[s, sl]
            np.testing.assert_allclose(t[:, b], r[s, sl], rtol=1e-12, err_msg='slab %d view %g' % (s, v))
            others = np.delete(t[:, :ntp + 2], b, axis=1)
            assert not np.any(others), (s, v)
            assert abs(t[:, ntp + 2].sum() / rad / L - 1.0) < 1e-5, (s, v, t[:, ntp + 2].sum() / rad, L)


def test_first_moment_matches_the_jacobian_of_a_uniform_absorber(solver):
    """With an absorber uniform in height and one layer group, every history has T + tau_LE = k L, so the Jacobian run
    gives jac = -k moment per pixel from the same histories (to fp32 path arithmetic)."""
    scene, opt, ja = _c2_small()
    nz = scene.struct.nz
    k = 2e-5
    ju = _uniform(ja, nz, k)
    ntp = BINS[2]
    r0, pl, _ = _run(solver, scene, opt, ju, bins=BINS)
    jobs, keep = abi.make_jobs(**ju)
    solver.upload_scene(scene, opt)
    solver.run_jac(jobs, [0, nz])
    jac = solver.read_jac()[..., 0]
    np.testing.assert_allclose(solver.read_rad(), r0, rtol=1e-12, atol=0)
    exp = -k * pl[..., ntp + 2]
    big = np.abs(exp) > 0
    rel = np.abs(jac[big] / exp[big] - 1.0)
    print('worst relative difference jac / (-k moment) - 1 over %d pixels: %.3g' % (big.sum(), rel.max()))
    assert big.sum() > 0
    assert rel.max() < 1e-4, np.sort(rel)[-5:]


def test_first_moment_matches_crn_finite_difference(solver):
    """wmin = 0: the trajectories do not depend on the absorption, so plain runs with a uniform absorber k (1 +- eps) and
    the same seeds follow the same histories; dI / dk = -E[c L] = -moment."""
    scene, opt, ja = _c2_small(photons=3e5, wmin=0.0)
    nz = scene.struct.nz
    k, eps = 2e-5, 1e-2
    ntp = BINS[2]
    _, pl, _ = _run(solver, scene, opt, _uniform(ja, nz, k), bins=BINS)
    rp, _, _ = _run(solver, scene, opt, _uniform(ja, nz, k * (1.0 + eps)))
    rm, _, _ = _run(solver, scene, opt, _uniform(ja, nz, k * (1.0 - eps)))
    fd = (-(rp - rm) / (2.0 * eps * k)).reshape(pl.shape[:2])
    mom = pl[..., ntp + 2]
    assert fd.mean() > 0
    assert abs(mom.mean() / fd.mean() - 1.0) < 2e-3, (mom.mean(), fd.mean())
    big = np.abs(fd) > 1e-3 * np.abs(fd).max()
    rel = np.abs(mom[big] - fd[big]) / np.abs(fd[big])
    assert np.mean(rel < 2e-2) > 0.99, np.sort(rel)[-10:]


def test_roulette_leaves_the_mean_path_unbiased(solver):
    """Domain-mean <L> per view with Pho_wmin = 0.2 against wmin = 0, over independent slabs"""
    nslab = 12
    ntp = BINS[2]
    means = {}
    for wmin in (0.2, 0.0):
        scene, opt, ja = _c2_small(photons=1e5, wmin=wmin)
        o = abi.make_options(target=opt.target, nslab=nslab, wmin=wmin, wfac=opt.wfac, iso_ss=opt.iso_ss, iso_max=opt.iso_max)
        nj = len(ja['nphot'])
        rep = dict(nphot=list(ja['nphot']) * nslab, seeds=[int(s) + 7919 * k + (0 if wmin else 104729) for k in range(nslab) for s in ja['seeds']],
                   slabs=[k for k in range(nslab) for _ in range(nj)], abs1d=list(ja['abs1d']) * nslab, rad_scale=list(ja['rad_scale']) * nslab)
        _, pl, st = _run(solver, scene, o, rep, bins=BINS)
        if wmin:
            assert st['n_roulette_kill'] > 0
        means[wmin] = np.stack([pl[:, sl, ntp + 2].sum(axis=1) / pl[:, sl, :ntp + 2].sum(axis=(1, 2)) for sl in _views(scene)], axis=1)
    a, b = means[0.2], means[0.0]                                            # (nslab, nview)
    sig = np.hypot(a.std(axis=0, ddof=1), b.std(axis=0, ddof=1)) / np.sqrt(nslab)
    z = (a.mean(axis=0) - b.mean(axis=0)) / sig
    assert np.all(np.abs(z) < 4.0), z


def test_shards_add_up_and_accumulate(solver):
    scene, opt, ja = _c2_small(photons=1.5e5)
    full_r, full_p, _ = _run(solver, scene, opt, ja, bins=BINS)
    parts = []
    for rank in (0, 1):
        o = abi.make_options(target=opt.target, nslab=opt.nslab, wmin=opt.wmin, wfac=opt.wfac, iso_ss=opt.iso_ss, iso_max=opt.iso_max,
                             shard_rank=rank, shard_world=2, smem_tally=opt.smem_tally)
        parts.append(_run(solver, scene, o, ja, bins=BINS))
    assert full_p.max() > 0
    np.testing.assert_allclose(parts[0][0] + parts[1][0], full_r, rtol=1e-12, atol=1e-300)
    np.testing.assert_allclose(parts[0][1] + parts[1][1], full_p, rtol=1e-12, atol=1e-300)
    # accumulate: the second run adds onto the tallies of the first
    _run(solver, scene, opt, ja, bins=BINS)
    r2, p2, _ = _run(solver, scene, opt, ja, bins=BINS, accumulate=True, upload=False)
    np.testing.assert_allclose(r2, 2.0 * full_r, rtol=1e-12)
    np.testing.assert_allclose(p2, 2.0 * full_p, rtol=1e-12)
    assert 'plen' in solver.results() and 'jac' not in solver.results()
    # a plain run afterwards: no path-length tally any more
    _run(solver, scene, opt, ja, upload=False)
    assert 'plen' not in solver.results()
    with pytest.raises(OSError, match='not a path-length run'):
        solver.read_plen()


def test_mcarats_ng_end_to_end(solver, tmp_path):
    kw, abs0 = workloads.c4(scale=0.002, nwvl=2)[1]
    kw = dict(kw, Nrun=2, photons=2e5, fdir=str(tmp_path), solver_obj=solver, seed=77,
              extra_sensors=[dict(sensor_zenith_angle=30.0, sensor_azimuth_angle=45.0)])
    ntp = 32
    m = bmca.mcarats_ng(**dict(kw, path_length=(0.0, 160.0, ntp)))
    pl = np.asarray(m.fused['path_length'][0])
    nx, ny = m.Nx, m.Ny
    assert pl.shape == (nx, ny, ntp + 3, 1, 2)
    assert len(m.plen_extra) == 1 and m.plen_extra[0].shape == (nx, ny, ntp + 3, 2)
    np.testing.assert_allclose(m.plen_edges, np.linspace(0.0, 160.0, ntp + 1))
    assert all(n['Rad_mplen'] == 1 and n['Rad_ntp'] == ntp and n['Rad_tpmin'] == 0.0 and n['Rad_tpmax'] == 160000.0 for n in m.nml)
    rad = np.asarray(m.fused['radiance'][0])
    np.testing.assert_allclose(pl[:, :, :ntp + 2].sum(axis=2), rad[:, :, 0], rtol=1e-12, atol=0)
    np.testing.assert_allclose(m.plen_extra[0][:, :, :ntp + 2].sum(axis=2), m.rad_extra[0], rtol=1e-12, atol=0)
    m0 = bmca.mcarats_ng(**kw)
    np.testing.assert_allclose(rad, np.asarray(m0.fused['radiance'][0]), rtol=1e-12)      # path_length changes no radiance
    o = bmca.mca_out_ng(mca_obj=m, abs_obj=abs0, mode='mean')
    for key, shape in (('rad_plen', (nx, ny, ntp)), ('rad_plen_std', (nx, ny, ntp)), ('rad_plen_out', (nx, ny, 2)),
                       ('rad_mean_plen', (nx, ny))):
        assert o.data[key]['data'].shape == shape, key
    np.testing.assert_allclose(o.data['plen_edges']['data'], m.plen_edges)
    exp = pl[:, :, ntp + 2, 0].sum(axis=-1) / rad[:, :, 0, 0].sum(axis=-1) / 1000.0
    np.testing.assert_allclose(o.data['rad_mean_plen']['data'], exp, rtol=1e-12)
    assert np.all(np.isnan(exp) == (rad[:, :, 0, 0].sum(axis=-1) == 0))
    assert np.nanmin(exp) > 0.0 and np.isfinite(exp).any()
    o0 = bmca.mca_out_ng(mca_obj=m0, abs_obj=abs0, mode='mean')
    assert not any('plen' in k for k in o0.data)


def test_unsupported_runs_are_rejected_by_the_library(solver):
    scene, opt, ja = _c2_small(photons=1e4)
    nz = scene.struct.nz
    jobs, keep = abi.make_jobs(**ja)
    solver.upload_scene(scene, abi.make_options(target=abi.TARGET_RADIANCE | abi.TARGET_FLUX))
    with pytest.raises(OSError, match='run_plen: radiance targets only'):
        solver.run_plen(jobs, *BINS)
    with pytest.raises(OSError, match=r'options.kernel must be 0 \(auto\) or 8'):
        solver.upload_scene(scene, abi.make_options(target=opt.target, smem_tally=-1, kernel=9))
    solver.upload_scene(scene, opt)
    for bins, msg in (((0.0, 1e5, 0), 'ntp must be 1 ... 1024'), ((0.0, 1e5, 1025), 'ntp must be 1 ... 1024'),
                      ((-1.0, 1e5, 8), '0 <= tpmin < tpmax'), ((1e5, 1e5, 8), '0 <= tpmin < tpmax'),
                      ((2e5, 1e5, 8), '0 <= tpmin < tpmax'), ((0.0, np.inf, 8), 'finite'), ((np.nan, 1e5, 8), 'finite'),
                      ((0.0, 1e39, 8), 'finite')):
        with pytest.raises(OSError, match=msg):
            solver.run_plen(jobs, *bins)
    solver.run(jobs)
    with pytest.raises(OSError, match='not a path-length run'):
        solver.read_plen()
    assert solver.plen_ptr() == (None, 0)
    with pytest.raises(OSError, match='accumulate needs the previous run to be a path-length run'):
        solver.run_plen(jobs, *BINS, accumulate=True)
    solver.run_jac(jobs, [0, nz])
    with pytest.raises(OSError, match='accumulate needs the previous run to be a path-length run'):
        solver.run_plen(jobs, *BINS, accumulate=True)
    solver.run_plen(jobs, *BINS)
    with pytest.raises(OSError, match='not a Jacobian run'):
        solver.read_jac()
    with pytest.raises(OSError, match='accumulate needs the previous run to be a Jacobian run'):
        solver.run_jac(jobs, [0, nz], accumulate=True)
    for bins in ((0.0, 1e5, BINS[2]), (0.0, BINS[1], 32)):
        with pytest.raises(OSError, match='same binning'):
            solver.run_plen(jobs, *bins, accumulate=True)
    solver.run_plen(jobs, *BINS, accumulate=True)
    # the all-sky camera
    kw, _ = workloads.c2(scale=0.01, nrun=1)
    mc = bmca.mcarats_ng(**dict(kw, sensor_type='all-sky camera', camera_pixels=(8, 8), dry_run=True, photons=1e4))
    solver.upload_scene(mc.scene, abi.make_options(target=mc.options.target, smem_tally=-1))
    jc, keep2 = abi.make_jobs(**mc.jobs_args)
    with pytest.raises(OSError, match='run_plen: the all-sky camera'):
        solver.run_plen(jc, *BINS)


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
                         shard_rank=rank, shard_world=world, smem_tally=opt.smem_tally)
    jobs, keep = abi.make_jobs(**ja)
    s = Solver(device=rank)
    s.upload_scene(scene, o)
    s.run_plen(jobs, *BINS, sync=False)
    res = edist.allreduce_results(s)
    assert np.array_equal(s.read_plen(), res['plen'])
    if rank == 0:
        np.savez(out, rad=res['rad'], plen=res['plen'], photons=res['stats']['photons'])
    dist.barrier()
    dist.destroy_process_group()
    s.close()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs two GPUs')
def test_two_nccl_ranks_reduce_the_path_length_tally(solver, tmp_path):
    out = str(tmp_path / 'p.npz')
    mp.spawn(_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    got = np.load(out)
    scene, opt, ja = _c2_small(photons=1e5)
    r, p, st = _run(solver, scene, opt, ja, bins=BINS)
    assert int(got['photons']) == st['photons']
    assert np.allclose(got['rad'], r, rtol=1e-9, atol=1e-15)
    assert np.allclose(got['plen'], p, rtol=1e-9, atol=1e-15)
