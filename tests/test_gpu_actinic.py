"""
Actinic flux (b200rt_run_act, Solver.run_act, mcarats_ng(actinic=True)), tallied by track length inside the histories of
the flux / heating run.  On the GPU: the same histories as b200rt_run, closed forms for the direct beam and for the
light a Lambertian surface sends up through a non-scattering absorbing atmosphere, Gershun's law against the flux
divergence, the heating identity, roulette, shards / accumulate / tally paths, library-side rejections, the end-to-end
path through mcarats_ng and mca_out_ng, and a two-rank NCCL reduction.
"""

import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp
from scipy.special import expn

import scenes
import workloads
from er3t_b200 import abi
from er3t_b200.rtm import mca as bmca

pytestmark = pytest.mark.gpu
ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), '..'))
COUNTERS = ('photons', 'n_cell', 'n_tent', 'n_coll', 'n_sfc', 'n_le', 'n_le_visit', 'n_roulette_kill')
FH = abi.TARGET_FLUX | abi.TARGET_HEATING


def _run(solver, scene, opt, ja, act=True, accumulate=False, upload=True):
    jobs, keep = abi.make_jobs(**ja)
    if upload:
        solver.upload_scene(scene, opt)
    if act:
        solver.run_act(jobs, accumulate=accumulate)
    else:
        solver.run(jobs, accumulate=accumulate)
    res = solver.results()
    return {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in res.items()}


def _c5_small(photons=2e5):
    kw, _ = workloads.c5(scale=0.02, photons=photons)
    m = bmca.mcarats_ng(**dict(kw, Nrun=1, dry_run=True, target='heating rate'))
    return m.scene, m.options, m.jobs_args


def _pp(omega=1.0, nslab=8, nphot=100000, wmin=None, smem_tally=0, cot=10.0):
    """plane-parallel cloud over gas absorption in the lowest layers; flux + heating, one job per slab"""
    sc, absg = scenes.plane_parallel(omega=omega, absorb=True, with_sensor=False, cot=cot)
    absg = absg * 30.0                        # strong enough that every step loses a visible share of its weight
    kw = dict(target=FH, nslab=nslab, smem_tally=smem_tally)
    if wmin is not None:
        kw['wmin'] = wmin
    opt = abi.make_options(**kw)
    ja = dict(nphot=[nphot] * nslab, seeds=list(range(11, 11 + nslab)), slabs=list(range(nslab)), abs1d=[absg] * nslab)
    return sc, opt, ja, absg


@pytest.mark.parametrize('which', ['3d', 'plane'])
def test_same_histories_as_run(solver, which):
    if which == '3d':
        scene, opt, ja = _c5_small()
    else:
        scene, opt, ja, _ = _pp(omega=0.95, nslab=2, nphot=50000)
    r0 = _run(solver, scene, opt, ja, act=False)
    r1 = _run(solver, scene, opt, ja)
    assert 'act' not in r0 and r1['act'].shape == (opt.nslab, 2, scene.struct.nz, scene.struct.ny, scene.struct.nx)
    for k in ('flux', 'heat'):
        assert r0[k].max() > 0
        np.testing.assert_allclose(r1[k], r0[k], rtol=1e-12, atol=1e-300 if k == 'flux' else 1e-18)
    for k in COUNTERS:
        assert r0['stats'][k] == r1['stats'][k], k
    assert r1['stats']['n_tally'] >= r0['stats']['n_tally']
    a = r1['act']
    assert np.all(a >= 0) and a[:, 1].sum() > 0
    assert np.all(a[:, 0] <= a[:, 1] * (1 + 1e-12) + 1e-300)


def _clear_scene(kind, albedo=0.0, nslab=4, nphot=100000, sza=40.0):
    """non-scattering 10 km atmosphere with gas absorption, collimated beam; kind: 'pp', 'block3d' (transparent 3-D block of
    12 x 12 columns: the generic step and column splitting) or 'ipa'"""
    zgrd = np.linspace(0.0, 10000.0, 11)
    nz = zgrd.size - 1
    n = 12 if kind != 'pp' else 4
    kw = {}
    if kind != 'pp':
        kw = dict(iz3l=2, ext3d=np.zeros((n, n, 3), np.float32), omg3d=np.ones((n, n, 3), np.float32),
                  apf3d=np.zeros((n, n, 3), np.float32))
    scene = abi.HostScene(zgrd, np.zeros((1, nz)), np.ones((1, nz)), np.zeros((1, nz)), nx=n, ny=n, dx=1000.0, dy=1000.0,
                          sfc_type=abi.SFC_LAMBERT, sfc_param=(albedo, 0, 0, 0, 0), src_the=180.0 - sza, src_phi=200.0,
                          src_qmax=0.0, sensors=[], **kw)
    prof = np.linspace(2.0, 0.5, nz)
    k = 0.6 * prof / (prof * np.diff(zgrd)).sum()          # total gas optical depth 0.6
    opt = abi.make_options(target=abi.TARGET_FLUX, nslab=nslab, wmin=0.0,
                           solver=abi.SOLVER_IPA if kind == 'ipa' else abi.SOLVER_3D)
    ja = dict(nphot=[nphot] * nslab, seeds=list(range(3, 3 + nslab)), slabs=list(range(nslab)), abs1d=[k] * nslab)
    return scene, opt, ja, zgrd, k


@pytest.mark.parametrize('kind', ['pp', 'block3d', 'ipa'])
def test_direct_beam_closed_form(solver, kind):
    sza = 40.0
    scene, opt, ja, zgrd, k = _clear_scene(kind, sza=sza)
    a = _run(solver, scene, opt, ja)['act']                  # (nslab, 2, nz, ny, nx)
    mu0 = np.cos(np.radians(sza))
    tl = k * np.diff(zgrd)
    ttop = np.concatenate([np.cumsum(tl[::-1])[::-1][1:], [0.0]])
    exp = np.exp(-ttop / mu0) * mu0 / tl * (1.0 - np.exp(-tl / mu0))
    np.testing.assert_allclose(a[:, 0], a[:, 1], rtol=1e-12)  # nothing scatters, the surface is black: all direct
    dom = a[:, 1].mean(axis=(0, 2, 3))
    np.testing.assert_allclose(dom, exp, rtol=1e-5)
    ncol = a.shape[-1] * a.shape[-2]
    col = a[:, 1].mean(axis=0)                                # (nz, ny, nx)
    sig = exp[:, None, None] * np.sqrt(ncol / (opt.nslab * ja['nphot'][0]))
    assert np.all(np.abs(col - exp[:, None, None]) < 4.0 * sig), np.abs(col - exp[:, None, None]).max() / sig.min()


def test_lambertian_surface_closed_form(solver):
    sza, alpha = 40.0, 0.5
    scene, opt, ja, zgrd, k = _clear_scene('pp', albedo=alpha, nslab=8, nphot=200000, sza=sza)
    a = _run(solver, scene, opt, ja)['act']
    mu0 = np.cos(np.radians(sza))
    tl = k * np.diff(zgrd)
    tstar = tl.sum()
    tb = np.concatenate([[0.0], np.cumsum(tl)])              # optical depth above the surface at every level
    I0 = alpha * mu0 * np.exp(-tstar / mu0) / np.pi
    exp = 2.0 * np.pi * I0 * (expn(3, tb[:-1]) - expn(3, tb[1:])) / tl
    diff = (a[:, 1] - a[:, 0]).mean(axis=(2, 3))              # (nslab, nz)
    m, sem = diff.mean(axis=0), diff.std(axis=0, ddof=1) / np.sqrt(diff.shape[0])
    assert np.all(np.abs(m - exp) < 4.0 * sem + 1e-12 * exp), (m / exp - 1, sem / exp)
    assert np.all(np.abs(m / exp - 1.0) < 0.01)


def test_gershun_law(solver):
    """absorbed power of a layer (net-flux divergence, flux tally) = (k_gas + sigma_a) dz x actinic flux (actinic tally)"""
    sc, opt, ja, absg = _pp(omega=0.9, nslab=32, nphot=200000)
    r = _run(solver, sc, opt, ja)
    z = np.asarray(sc.zgrd, dtype=np.float64) if hasattr(sc, 'zgrd') else scenes.std_z()
    dz = np.diff(z)
    nz = dz.size
    f = r['flux'][:, :, :, 0, 0]                             # (nslab, 3, nz+1)
    net = f[:, 1] - f[:, 2]
    absorbed = net[:, 1:] - net[:, :-1]                       # (nslab, nz)
    ext = np.zeros((2, nz))
    ext[0] = scenes.rayleigh_ext(z)
    ext[1, 1] = 10.0 / 1000.0
    sig_a = ext[1] * (1.0 - 0.9)
    est = ((absg + sig_a) * dz)[None, :] * r['act'][:, 1, :, 0, 0]
    d = absorbed - est
    m, sem = d.mean(axis=0), d.std(axis=0, ddof=1) / np.sqrt(d.shape[0])
    assert np.all(np.abs(m) <= 4.0 * sem + 1e-9), (m, sem)
    assert absorbed.mean(axis=0)[1] > 0.01


def test_heating_identity(solver):
    """omega = 1 everywhere: heating is gas absorption only, heat = k dz x actinic flux, layer by layer (one column)"""
    sc, opt, ja, absg = _pp(omega=1.0, nslab=2, nphot=200000)
    r = _run(solver, sc, opt, ja)
    dz = np.diff(scenes.std_z())
    heat = r['heat'][:, :, 0, 0]
    est = (absg * dz)[None, :] * r['act'][:, 1, :, 0, 0]
    on = absg > 0
    assert heat[:, on].min() > 0
    np.testing.assert_allclose(est[:, on], heat[:, on], rtol=1e-5)
    np.testing.assert_allclose(est[:, on].sum(axis=1), heat[:, on].sum(axis=1), rtol=1e-5)
    assert np.all(heat[:, ~on] == 0)


def test_roulette_leaves_it_unbiased(solver):
    sc, opt, ja, _ = _pp(omega=0.95, nslab=8, nphot=100000)
    a = _run(solver, sc, opt, ja)['act'][:, 1, :, 0, 0]
    sc, opt0, ja, _ = _pp(omega=0.95, nslab=8, nphot=100000, wmin=0.0)
    b = _run(solver, sc, opt0, ja)['act'][:, 1, :, 0, 0]
    d = a.mean(axis=0) - b.mean(axis=0)
    s = np.sqrt(a.var(axis=0, ddof=1) / a.shape[0] + b.var(axis=0, ddof=1) / b.shape[0])
    assert np.all(np.abs(d) <= 4.0 * s + 1e-12), d / s


@pytest.mark.parametrize('which', ['plane', '3d'])
def test_shards_accumulate_and_tally_paths(solver, which):
    if which == '3d':
        scene, opt, ja = _c5_small(photons=1e5)
    else:
        scene, opt, ja, _ = _pp(omega=0.95, nslab=2, nphot=50000)
    full = _run(solver, scene, opt, ja)
    parts = []
    for rank in (0, 1):
        o = abi.make_options(target=opt.target, nslab=opt.nslab, wmin=opt.wmin, wfac=opt.wfac, iso_ss=opt.iso_ss, iso_max=opt.iso_max,
                             solver=opt.solver, shard_rank=rank, shard_world=2, smem_tally=opt.smem_tally)
        parts.append(_run(solver, scene, o, ja)['act'])
    np.testing.assert_allclose(parts[0] + parts[1], full['act'], rtol=1e-12, atol=1e-300)
    _run(solver, scene, opt, ja)
    acc = _run(solver, scene, opt, ja, accumulate=True, upload=False)
    np.testing.assert_allclose(acc['act'], 2.0 * full['act'], rtol=1e-12, atol=1e-300)
    np.testing.assert_allclose(acc['flux'], 2.0 * full['flux'], rtol=1e-12, atol=1e-300)
    # global atomics instead of the block-private shared tally
    o = abi.make_options(target=opt.target, nslab=opt.nslab, wmin=opt.wmin, wfac=opt.wfac, iso_ss=opt.iso_ss, iso_max=opt.iso_max,
                         solver=opt.solver, smem_tally=-1)
    g = _run(solver, scene, o, ja)
    np.testing.assert_allclose(g['act'], full['act'], rtol=1e-12, atol=1e-300)
    _run(solver, scene, opt, ja, act=False, upload=False)
    assert 'act' not in solver.results()
    with pytest.raises(OSError, match='not an actinic run'):
        solver.read_act()
    assert solver.act_ptr() == (None, 0)


def test_unsupported_runs_are_rejected_by_the_library(solver):
    scene, opt, ja, _ = _pp(nslab=1, nphot=1000)
    jobs, keep = abi.make_jobs(**ja)
    sc_rad, _ = scenes.plane_parallel(with_sensor=True)
    solver.upload_scene(sc_rad, abi.make_options(target=abi.TARGET_RADIANCE, smem_tally=-1))
    with pytest.raises(OSError, match='run_act: needs the flux or heating target'):
        solver.run_act(jobs)
    solver.upload_scene(sc_rad, abi.make_options(target=abi.TARGET_RADIANCE | abi.TARGET_FLUX))
    with pytest.raises(OSError, match='run_act: no radiance sensors'):
        solver.run_act(jobs)
    with pytest.raises(OSError, match=r'options.kernel must be 0 \(auto\) or 8'):
        solver.upload_scene(scene, abi.make_options(target=FH, kernel=9))
    solver.upload_scene(scene, opt)
    solver.run(jobs)
    with pytest.raises(OSError, match='accumulate needs the previous run to be an actinic run'):
        solver.run_act(jobs, accumulate=True)
    solver.run_act(jobs)
    solver.run_act(jobs, accumulate=True)
    kw, _ = workloads.c2(scale=0.01, nrun=1)
    mc = bmca.mcarats_ng(**dict(kw, sensor_type='all-sky camera', camera_pixels=(8, 8), dry_run=True, photons=1e4))
    solver.upload_scene(mc.scene, abi.make_options(target=mc.options.target | abi.TARGET_FLUX, smem_tally=-1))
    jc, keep2 = abi.make_jobs(**mc.jobs_args)
    with pytest.raises(OSError, match='run_act: the all-sky camera'):
        solver.run_act(jc)


@pytest.mark.parametrize('target', ['flux', 'heating rate'])
def test_mcarats_ng_end_to_end(solver, tmp_path, target):
    kw, abs0 = workloads.c5(scale=0.02, photons=2e5)
    kw = dict(kw, Nrun=2, fdir=str(tmp_path), solver_obj=solver, target=target)
    m = bmca.mcarats_ng(**dict(kw, actinic=True))
    a = np.asarray(m.fused['actinic'][0])
    nx, ny, nz = m.Nx, m.Ny, m.scene.struct.nz
    assert a.shape == (nx, ny, nz, 2, 2)
    m0 = bmca.mcarats_ng(**kw)
    assert 'actinic' not in m0.fused
    for i in range(3):
        np.testing.assert_allclose(m.fused['flux'][i], m0.fused['flux'][i], rtol=1e-12, atol=1e-300)
    o = bmca.mca_out_ng(mca_obj=m, abs_obj=abs0, mode='mean')
    o0 = bmca.mca_out_ng(mca_obj=m0, abs_obj=abs0, mode='mean')
    for key in ('f_act', 'f_act_direct', 'f_act_diffuse', 'f_act_std', 'f_act_direct_std', 'f_act_diffuse_std'):
        assert o.data[key]['data'].shape == (nx, ny, nz), key
        assert key not in o0.data
    np.testing.assert_allclose(o.data['f_act_direct']['data'] + o.data['f_act_diffuse']['data'], o.data['f_act']['data'],
                               rtol=1e-5, atol=1e-6 * o.data['f_act']['data'].max())
    assert o.data['f_act']['data'].max() > 0
    assert set(o.data) - set(o0.data) == {'f_act', 'f_act_direct', 'f_act_diffuse', 'f_act_std', 'f_act_direct_std',
                                          'f_act_diffuse_std'}
    for key in o0.data:
        np.testing.assert_allclose(np.asarray(o.data[key]['data']), np.asarray(o0.data[key]['data']), rtol=1e-6, err_msg=key)


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
    scene, opt, ja = _c5_small(photons=1e5)
    o = abi.make_options(target=opt.target, nslab=opt.nslab, wmin=opt.wmin, wfac=opt.wfac, iso_ss=opt.iso_ss, iso_max=opt.iso_max,
                         solver=opt.solver, shard_rank=rank, shard_world=world, smem_tally=opt.smem_tally)
    jobs, keep = abi.make_jobs(**ja)
    s = Solver(device=rank)
    s.upload_scene(scene, o)
    s.run_act(jobs, sync=False)
    res = edist.allreduce_results(s)
    assert np.array_equal(s.read_act(), res['act'])
    if rank == 0:
        np.savez(out, act=res['act'], photons=res['stats']['photons'])
    dist.barrier()
    dist.destroy_process_group()
    s.close()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs two GPUs')
def test_two_nccl_ranks_reduce_the_actinic_tally(solver, tmp_path):
    out = str(tmp_path / 'a.npz')
    mp.spawn(_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    got = np.load(out)
    scene, opt, ja = _c5_small(photons=1e5)
    r = _run(solver, scene, opt, ja)
    assert int(got['photons']) == r['stats']['photons']
    assert np.allclose(got['act'], r['act'], rtol=1e-9, atol=1e-15)
