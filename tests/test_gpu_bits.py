"""Bit-exact and deterministic parts of the CUDA path, through the C-ABI: Philox streams, photon -> job mapping and
sharding, the phase-function / BRDF device functions against the oracle's fp64 versions, error reporting."""

import ctypes as C

import numpy as np
import pytest

import oracle
import scenes
from oracle import philox_np
from er3t_b200 import abi

pytestmark = pytest.mark.gpu


def test_philox_device_bit_exact(solver):
    for seed, first, c2, c3 in [(0, 0, 0, 0), (20260101, 5, 3, 0xB200), (0xDEADBEEFCAFEF00D, (1 << 32) - 7, 17, 0xB200)]:
        got = solver.philox(seed, first, 4096, c2=c2, c3=c3)
        assert np.array_equal(got, philox_np.photon_block(seed, first, 4096, c2=c2, c3=c3))
        assert np.array_equal(got[:64], oracle.philox(seed, first, 64, c2=c2, c3=c3))


def test_phase_functions_match_oracle(solver):
    ang, pha = scenes.synthetic_mie_table()
    sc = abi.HostScene(np.array([0.0, 1000.0]), [[1e-6]], [[1.0]], [[0.0]], ang=ang, pha=pha)
    solver.upload_scene(sc, abi.make_options(target=abi.TARGET_FLUX, nslab=1))
    lib = oracle.load()
    mu = np.linspace(-1.0, 1.0, 2001)
    xi = (np.arange(5000) + 0.5) / 5000
    for apf in (-1.0, 0.0, 0.6, 0.86, 1.0, 2.0, 2.4, 3.0):
        ref = np.zeros_like(mu)
        lib.oracle_phase_eval(C.addressof(sc.struct), apf, mu.ctypes.data, ref.ctypes.data, mu.size)
        got = solver.phase_eval(apf, mu)
        assert np.allclose(got, ref, rtol=3e-4, atol=1e-5), apf            # fp32 vs fp64, forward peak up to ~1e3
        if apf == int(apf):                                                  # (fractional indices pick a table at random)
            refs = np.zeros_like(xi)
            lib.oracle_phase_sample(C.addressof(sc.struct), apf, xi.ctypes.data, refs.ctypes.data, xi.size)
            gots = solver.phase_sample(apf, xi)
            if apf >= 1.0:
                # the device integrates the tabulated CDF from the forward direction (fp32 resolution sits in the
                # forward peak), the oracle from the backward one: sample_gpu(xi) == sample_oracle(1 - xi)
                refs = refs[::-1]
            assert np.max(np.abs(gots - refs)) < 2e-4, apf


def test_phase_tables_on_the_498_angle_mie_grid(solver):
    """The O(1) guide tables must find the SAME interval a full search finds, also on the reference's forward-dense
    default grid (er3t/pre/pha/pha_mie.py:106-113: 0.01 deg steps below 2 deg, where float32 cosines coincide)."""
    from er3t_b200.pre.pha import mie_angles_default
    ang = mie_angles_default()
    mu_t = np.cos(np.deg2rad(ang))
    tabs = []
    for g in (0.86, 0.8):
        # forward peak (diffraction-like) + broad HG + a rainbow bump + backscatter rise
        hg = lambda gg: (1 - gg * gg) / (1 + gg * gg - 2 * gg * mu_t) ** 1.5
        tabs.append(0.45 * hg(0.995) + 0.5 * hg(g) + 0.04 * np.exp(-0.5 * ((ang - 140.0) / 3.0) ** 2) + 0.01 * hg(-0.6))
    sc = abi.HostScene(np.array([0.0, 1000.0]), [[1e-6]], [[1.0]], [[0.0]], ang=ang, pha=np.stack(tabs, axis=1))
    solver.upload_scene(sc, abi.make_options(target=abi.TARGET_FLUX, nslab=1))
    lib = oracle.load()
    rng = np.random.default_rng(11)
    # evaluation: uniform in mu, dense in the forward peak, and exactly ON the grid points
    mu = np.concatenate([np.linspace(-1.0, 1.0, 4001), np.cos(np.deg2rad(rng.uniform(0.0, 3.0, 3000))), mu_t, 0.5 * (mu_t[1:] + mu_t[:-1])])
    xi = np.concatenate([(np.arange(20000) + 0.5) / 20000, rng.uniform(0.0, 1e-3, 2000), 1.0 - rng.uniform(0.0, 1e-3, 2000)])
    xi = np.sort(xi)
    for apf in (1.0, 2.0):
        ref = np.zeros_like(mu)
        lib.oracle_phase_eval(C.addressof(sc.struct), apf, mu.ctypes.data, ref.ctypes.data, mu.size)
        got = solver.phase_eval(apf, mu)
        # float32 cosines resolve the forward peak only to ~0.02 deg: compare where the table is smooth at that scale,
        # and bound the peak region by the table's own range
        smooth = mu < np.cos(np.deg2rad(1.0))
        assert np.allclose(got[smooth], ref[smooth], rtol=2e-3, atol=1e-5), apf
        assert np.all(got[~smooth] <= 1.0001 * ref.max()) and np.all(got[~smooth] >= 0.999 * ref[~smooth].min()), apf
        gots = solver.phase_sample(apf, xi)
        # device CDF runs from the forward direction, the oracle's from the backward one (see above)
        refs1 = np.zeros_like(xi)
        x1 = np.ascontiguousarray(1.0 - xi)
        lib.oracle_phase_sample(C.addressof(sc.struct), apf, x1.ctypes.data, refs1.ctypes.data, xi.size)
        assert np.max(np.abs(np.arccos(np.clip(gots, -1, 1)) - np.arccos(np.clip(refs1, -1, 1)))) < np.deg2rad(0.05), apf
        # sampling is monotone in xi (a wrong interval from the guide table would break this)
        assert np.all(np.diff(gots) <= 1e-6), apf


def test_brdf_matches_oracle(solver):
    lib = oracle.load()
    rng = np.random.default_rng(3)
    n = 4000
    def hemi(sign):
        mu = 0.05 + 0.95 * rng.random(n)
        ph = 2 * np.pi * rng.random(n)
        st = np.sqrt(1 - mu * mu)
        return np.stack([st * np.cos(ph), st * np.sin(ph), sign * mu], axis=1)
    din, dout = hemi(-1.0), hemi(+1.0)
    for t, prm in ((abi.SFC_LAMBERT, [0.3, 0, 0, 0, 0]), (abi.SFC_LSRT, [0.2, 0.03, 0.1, 0, 0]), (abi.SFC_DSM, [0.22, 0.05, 1.34, 1e-7, 0.04])):
        prm = np.array(prm, dtype=np.float32)
        ref = np.zeros(n)
        lib.oracle_brdf_eval(t, prm.ctypes.data, np.ascontiguousarray(din).ctypes.data, np.ascontiguousarray(dout).ctypes.data, ref.ctypes.data, n)
        got = solver.brdf_eval(t, prm, din, dout)
        assert np.allclose(got, ref, rtol=2e-3, atol=1e-6), t


def test_every_photon_is_traced_once_and_shards_add_up(solver):
    sc = scenes.scene_3d(nx=8, ny=6)
    nphot = [30011, 7, 0, 12345]
    jobs, keep = abi.make_jobs(nphot, [11, 12, 13, 14], [0, 1, 0, 1])
    opt = abi.make_options(target=abi.TARGET_RADIANCE | abi.TARGET_FLUX, nslab=2, wmin=0.2)
    solver.upload_scene(sc, opt); solver.run(jobs)
    full = solver.results()
    assert full['stats']['photons'] == sum(nphot)
    parts = []
    for r in range(3):
        o = abi.make_options(target=abi.TARGET_RADIANCE | abi.TARGET_FLUX, nslab=2, wmin=0.2, shard_rank=r, shard_world=3)
        solver.upload_scene(sc, o); solver.run(jobs)
        parts.append(solver.results())
    assert sum(p['stats']['photons'] for p in parts) == sum(nphot)
    rad = sum(p['rad'] for p in parts)
    flux = sum(p['flux'] for p in parts)
    # identical photon set (counter-based streams keyed by the global photon index): only the summation order differs
    assert np.allclose(rad, full['rad'], rtol=1e-9, atol=1e-15)
    assert np.allclose(flux, full['flux'], rtol=1e-9, atol=1e-15)
    # and a rerun reproduces the run
    solver.upload_scene(sc, opt); solver.run(jobs)
    again = solver.results()
    assert np.allclose(again['rad'], full['rad'], rtol=1e-9, atol=1e-15)
    for k in ('n_coll', 'n_sfc', 'n_tent', 'n_roulette_kill'):
        assert again['stats'][k] == full['stats'][k]


def test_block_private_tallies_equal_global_atomics(solver):
    """Small flux / heating tallies are accumulated per block in shared memory and flushed once; the photon set is the
    same (counter-based streams), so the result must equal the global-atomics path up to the summation order."""
    sc, absg = scenes.plane_parallel(absorb=True, with_sensor=False)
    jobs, keep = abi.make_jobs([150000, 50000, 30000], [5, 6, 7], [0, 1, 1], abs1d=[absg] * 3)
    res = []
    for st in (0, -1):
        opt = abi.make_options(target=abi.TARGET_FLUX | abi.TARGET_HEATING, nslab=2, wmin=0.2, smem_tally=st)
        solver.upload_scene(sc, opt); solver.run(jobs)
        res.append(solver.results())
    a, b = res
    assert a['stats']['n_tally'] < b['stats']['n_tally'] / 100        # flushed entries vs one global atomic per crossing
    assert np.allclose(a['flux'], b['flux'], rtol=1e-10, atol=1e-15)
    assert np.allclose(a['heat'], b['heat'], rtol=1e-10, atol=1e-15)
    for k in ('n_coll', 'n_sfc', 'n_roulette_kill', 'photons'):
        assert a['stats'][k] == b['stats'][k]


def test_accumulate_flag(solver):
    sc = scenes.scene_3d(nx=8, ny=6)
    opt = abi.make_options(target=abi.TARGET_RADIANCE, nslab=1, wmin=0.2)
    j1, k1 = abi.make_jobs([20000], [1], [0])
    j2, k2 = abi.make_jobs([20000], [2], [0])
    solver.upload_scene(sc, opt)
    solver.run(j1); a = solver.read_rad().copy()
    solver.run(j2); b = solver.read_rad().copy()
    solver.run(j1); solver.run(j2, accumulate=True); c = solver.read_rad().copy()
    assert np.allclose(c, a + b, rtol=1e-9)


def test_errors_are_reported_not_swallowed(solver):
    z = np.array([0.0, 1000.0, 500.0])
    with pytest.raises(OSError, match='strictly increasing'):
        solver.upload_scene(abi.HostScene(z, [[1e-5, 1e-5]], [[1, 1]], [[0, 0]]), abi.make_options())
    with pytest.raises(OSError, match='out of range'):
        solver.upload_scene(abi.HostScene(np.array([0.0, 1000.0]), [[-1.0]], [[1.0]], [[0.0]]), abi.make_options())
    with pytest.raises(OSError, match='3-D field out of range'):
        e3 = np.full((2, 2, 1), -0.1, dtype=np.float32)
        solver.upload_scene(abi.HostScene(np.array([0.0, 1000.0]), [[1e-5]], [[1.0]], [[0.0]], nx=2, ny=2, dx=10., dy=10., iz3l=1,
                                          ext3d=e3, omg3d=np.ones_like(e3), apf3d=np.zeros_like(e3)), abi.make_options())
    with pytest.raises(OSError, match='exceeds the atmosphere'):
        e3 = np.full((2, 2, 2), 0.1, dtype=np.float32)
        solver.upload_scene(abi.HostScene(np.array([0.0, 1000.0]), [[1e-5]], [[1.0]], [[0.0]], nx=2, ny=2, dx=10., dy=10., iz3l=1,
                                          ext3d=e3, omg3d=np.ones_like(e3), apf3d=np.zeros_like(e3)), abi.make_options())
    with pytest.raises(OSError, match='travel downward'):
        solver.upload_scene(abi.HostScene(np.array([0.0, 1000.0]), [[1e-5]], [[1.0]], [[0.0]], src_the=60.0), abi.make_options())
    sc, _ = scenes.plane_parallel()
    with pytest.raises(OSError, match=r'options.kernel must be 0 \(auto\) or 8'):
        solver.upload_scene(sc, abi.make_options(target=abi.TARGET_FLUX, nslab=1, kernel=9))
    with pytest.raises(OSError, match=r'pool_slots must be 0 \(auto\), 64, 96 or 128'):
        solver.upload_scene(sc, abi.make_options(target=abi.TARGET_FLUX, nslab=1, pool_slots=1024))
    solver.upload_scene(sc, abi.make_options(target=abi.TARGET_FLUX, nslab=1))
    with pytest.raises(OSError, match='slab out of range'):
        jobs, keep = abi.make_jobs([10], [1], [5])
        solver.run(jobs)
    with pytest.raises(OSError, match='not part of the target'):
        jobs, keep = abi.make_jobs([10], [1], [0])
        solver.run(jobs)
        solver.read_rad()


def test_public_api_on_gpu_matches_oracle_backed_run(solver, tmp_path):
    """mcarats_ng + mca_out_ng on the GPU against the same call driven through the oracle test double."""
    import datetime
    import er3t_b200.pre as bpre
    from er3t_b200.rtm import mca as bmca
    from oracle_solver import OracleSolver
    atm0 = bpre.atm_atmmod(levels=np.linspace(0, 20, 21))
    abs0 = bpre.abs_16g(wavelength=650.0, atm_obj=atm0)
    cld0 = bpre.cld_gen_hem(Nx=10, Ny=8, dx=0.1, dy=0.1, altitude=np.arange(1.25, 2.8, 0.5), radii=[0.3], cloud_frac_tgt=0.3, seed=3)
    pha0 = bpre.pha_mie_wc(wavelength=650.0, reff=[8.0, 12.0, 16.0], nr=48)
    kw = dict(date=datetime.datetime(2017, 8, 13), atm_1ds=[bmca.mca_atm_1d(atm_obj=atm0, abs_obj=abs0)],
              atm_3ds=[bmca.mca_atm_3d(cld_obj=cld0, atm_obj=atm0, pha_obj=pha0, quiet=True)], Ng=16, target='radiance', surface_albedo=0.05,
              sca=bmca.mca_sca(pha_obj=pha0), solar_zenith_angle=30.0, solar_azimuth_angle=45.0, fdir=str(tmp_path), Nrun=6, weights=abs0.coef['weight']['data'],
              solver='3D', quiet=True)
    g = bmca.mca_out_ng(mca_obj=bmca.mcarats_ng(photons=2e6, seed=3, solver_obj=solver, **kw), abs_obj=abs0, mode='all').data['rad']['data']
    c = bmca.mca_out_ng(mca_obj=bmca.mcarats_ng(photons=2e5, seed=9, solver_obj=OracleSolver(), **kw), abs_obj=abs0, mode='all').data['rad']['data']
    gm, gs = g.mean(axis=-1), g.std(axis=-1, ddof=1) / np.sqrt(6)
    cm, cs = c.mean(axis=-1), c.std(axis=-1, ddof=1) / np.sqrt(6)
    z = (gm - cm) / np.sqrt(gs ** 2 + cs ** 2)
    assert np.mean(np.abs(z) > 3.0) <= 0.05 and np.max(np.abs(z)) < 7.0
    assert abs(gm.mean() / cm.mean() - 1.0) < 0.01


def test_device_derived_omega_apf_equal_host_interpolation(solver):
    """mca_atm_3d(device_props=True): (omega, apf) of the cloudy voxels are derived from the effective radius by the
    scene-packing kernel (scene.cer3d) instead of the host loop of er3t/rtm/mca/mca_atm.py:291-303.  Same float32 values
    => the same photon histories => identical tallies and event counts, bit for bit up to the fp64 summation order."""
    import datetime
    import er3t_b200.pre as bpre
    from er3t_b200.rtm import mca as bmca
    atm0 = bpre.atm_atmmod(levels=np.linspace(0, 20, 21))
    abs0 = bpre.abs_16g(wavelength=650.0, atm_obj=atm0)
    cld0 = bpre.cld_gen_les(Nx=40, Ny=36, dx=0.1, dy=0.1, altitude=np.arange(1.25, 3.8, 0.5), seed=5, atm_obj=atm0)
    # float32-representable radii: the GPU receives the field as float32 (include/b200rt.h)
    cld0.lay['cer']['data'] = np.asarray(cld0.lay['cer']['data'], dtype=np.float32).astype(np.float64)
    pha0 = bpre.pha_mie_wc(wavelength=650.0, reff=[4.0, 8.0, 12.0, 16.0, 20.0], nr=32)
    out = []
    for dev in (False, True):
        a3 = bmca.mca_atm_3d(cld_obj=cld0, atm_obj=atm0, pha_obj=pha0, quiet=True, device_props=dev)
        m = bmca.mcarats_ng(date=datetime.datetime(2017, 8, 13), atm_1ds=[bmca.mca_atm_1d(atm_obj=atm0, abs_obj=abs0)], atm_3ds=[a3], Ng=16,
                            target='radiance', surface_albedo=0.05, sca=bmca.mca_sca(pha_obj=pha0), solar_zenith_angle=30.0,
                            solar_azimuth_angle=45.0, Nrun=2, weights=abs0.coef['weight']['data'], solver='3D', quiet=True, photons=4e5, seed=11,
                            solver_obj=solver, iz3l_fix=True)
        out.append((m, a3))
    (m0, a0), (m1, a1) = out
    assert m1.scene.cer3d is not None and m1.scene.omg3d is None            # the device path really was taken
    for k in ('n_coll', 'n_tent', 'n_sfc', 'n_roulette_kill', 'photons', 'n_cell'):
        assert m0.stats[k] == m1.stats[k], k
    assert np.allclose(m0.fused['radiance'][0], m1.fused['radiance'][0], rtol=1e-10, atol=1e-16)
    # and the lazily evaluated namelist payload of the device variant equals the host arrays
    assert np.array_equal(np.asarray(a1.nml['Atm_omgp3d']['data']), a0.nml['Atm_omgp3d']['data'])
    assert np.array_equal(np.asarray(a1.nml['Atm_apfp3d']['data']), a0.nml['Atm_apfp3d']['data'])
    assert np.array_equal(np.asarray(a1.nml['Atm_tmpa3d']['data']), a0.nml['Atm_tmpa3d']['data'])
