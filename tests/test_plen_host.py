"""
Host side of the path-length tally (mcarats_ng(path_length=...)): the documented errors, the Rad_mplen / Rad_ntp /
Rad_tpmin / Rad_tpmax namelist entries, and the mca_out_ng keys that exist only when a path length was asked for.  No GPU
needed.
"""

import numpy as np
import pytest

import workloads
from er3t_b200 import abi
from er3t_b200.rtm import mca as bmca

PLEN = (0.0, 120.0, 24)


@pytest.fixture(scope='module')
def c4_kw():
    kw, abs0 = workloads.c4(scale=0.0005, nwvl=1)[0]
    return dict(kw, Nrun=2, photons=1e4, path_length=PLEN)


@pytest.mark.parametrize('change, msg', [
    (dict(spectral=True), 'spectral'),
    (dict(gas_jacobian=True), 'gas_jacobian'),
    (dict(raw=True), 'raw'),
    (dict(target='flux'), 'radiance'),
    (dict(target='heating rate'), 'radiance'),
    (dict(sensor_type='all-sky camera'), 'satellite'),
    (dict(path_length=(0.0, 120.0)), r'\(tpmin_km, tpmax_km, ntp\)'),
    (dict(path_length='all'), r'\(tpmin_km, tpmax_km, ntp\)'),
    (dict(path_length=(0.0, 120.0, 0)), 'ntp, 1 ... 1024'),
    (dict(path_length=(0.0, 120.0, 1025)), 'ntp, 1 ... 1024'),
    (dict(path_length=(0.0, 120.0, 2.5)), 'integer number of bins'),
    (dict(path_length=(-1.0, 120.0, 8)), '0 <= tpmin_km < tpmax_km'),
    (dict(path_length=(50.0, 50.0, 8)), '0 <= tpmin_km < tpmax_km'),
    (dict(path_length=(0.0, np.inf, 8)), 'finite'),
])
def test_path_length_errors(c4_kw, tmp_path, change, msg):
    with pytest.raises(OSError, match=r'Error \[mcarats_ng\]: .*' + msg):
        bmca.mcarats_ng(**dict(c4_kw, fdir=str(tmp_path), **change))


def test_path_length_rejects_write_files(c4_kw, tmp_path):
    with pytest.raises(OSError, match=r'Error \[mcarats_ng\]: .*write_files'):
        bmca.mcarats_ng(**dict(c4_kw, fdir=str(tmp_path / 'out'), write_files=True))


def test_path_length_needs_an_absorption_object(c4_kw, tmp_path):
    atm = c4_kw['atm_1ds'][0]
    saved = atm.abs
    try:
        atm.abs = None
        with pytest.raises(OSError, match=r'Error \[mcarats_ng\]: .*absorption'):
            bmca.mcarats_ng(**dict(c4_kw, fdir=str(tmp_path)))
    finally:
        atm.abs = saved


def test_namelist_records_the_request(c4_kw, tmp_path):
    m = bmca.mcarats_ng(**dict(c4_kw, fdir=str(tmp_path), dry_run=True))
    assert len(m.nml) == m.Ng
    for n in m.nml:
        assert n['Rad_mplen'] == 1 and n['Rad_ntp'] == 24
        assert n['Rad_tpmin'] == 0.0 and n['Rad_tpmax'] == 120000.0          # metres, as MCARaTS takes them
    np.testing.assert_allclose(m.plen_edges, np.linspace(0.0, 120.0, 25))
    assert m.plen == (0.0, 120000.0, 24)
    assert m.options.smem_tally == -1
    # without path_length nothing changes
    m0 = bmca.mcarats_ng(**dict(c4_kw, fdir=str(tmp_path), dry_run=True, path_length=None))
    assert all(n['Rad_mplen'] == 0 and 'Rad_ntp' not in n and 'Rad_tpmin' not in n and 'Rad_tpmax' not in n for n in m0.nml)
    assert m0.plen is None and m0.plen_edges is None and m0.options.smem_tally == 0


def _fake_fused(m, ntp, plen):
    """radiance and, when asked, a path-length tally consistent with it (bins + underflow + overflow = radiance)"""
    rng = np.random.default_rng(0)
    nx, ny, nrun = m.Nx, m.Ny, m.Nrun
    parts = rng.uniform(0, 1, (nx, ny, ntp + 2, 1, nrun))
    parts[0, 0] = 0.0                                                      # one pixel without radiance
    rad = parts.sum(axis=2, keepdims=True)
    m.fused = {'flux': None, 'radiance': [rad], 'heating': None}
    if plen:
        moment = rad * rng.uniform(20e3, 80e3, rad.shape)
        m.fused['path_length'] = [np.concatenate([parts, moment], axis=2)]
    return m


@pytest.mark.parametrize('mode', ['mean', 'all'])
def test_mca_out_keys_only_with_a_path_length(c4_kw, tmp_path, mode):
    ntp = PLEN[2]
    m = bmca.mcarats_ng(**dict(c4_kw, fdir=str(tmp_path), dry_run=True))
    _fake_fused(m, ntp, True)
    o = bmca.mca_out_ng(mca_obj=m, abs_obj=m.abs, mode=mode)
    nx, ny, nrun = m.Nx, m.Ny, m.Nrun
    pl = m.fused['path_length'][0][:, :, :, 0, :]
    bins = pl[:, :, :ntp].astype(np.float32)
    out = pl[:, :, ntp:ntp + 2].astype(np.float32)
    np.testing.assert_allclose(o.data['plen_edges']['data'], np.linspace(0.0, 120.0, ntp + 1))
    if mode == 'mean':
        np.testing.assert_allclose(o.data['rad_plen']['data'], bins.mean(axis=-1), rtol=1e-6)
        np.testing.assert_allclose(o.data['rad_plen_std']['data'], bins.std(axis=-1), rtol=1e-5, atol=1e-7)
        np.testing.assert_allclose(o.data['rad_plen_out']['data'], out.mean(axis=-1), rtol=1e-6)
        assert o.data['rad_plen']['dims_info'] == ['Nx', 'Ny', 'Nbin']
        assert o.data['rad_plen_out']['dims_info'] == ['Nx', 'Ny', 'Nout']
    else:
        assert o.data['rad_plen']['data'].shape == (nx, ny, ntp, nrun)
        assert o.data['rad_plen_out']['data'].shape == (nx, ny, 2, nrun)
        assert 'rad_plen_std' not in o.data
    # the mean path is the ratio of the sums over runs (km), NaN where there is no radiance
    rad = m.fused['radiance'][0][:, :, 0, 0, :]
    with np.errstate(invalid='ignore'):
        exp = pl[:, :, ntp + 2].sum(axis=-1) / rad.sum(axis=-1) / 1000.0
    got = o.data['rad_mean_plen']['data']
    assert got.shape == (nx, ny) and o.data['rad_mean_plen']['units'] == 'km'
    assert np.isnan(got[0, 0]) and np.isnan(exp[0, 0])
    np.testing.assert_allclose(got, exp, rtol=1e-12)
    assert np.nanmin(got) >= 20.0 and np.nanmax(got) <= 80.0
    # the same simulation without a path length: the keys are absent
    m0 = bmca.mcarats_ng(**dict(c4_kw, fdir=str(tmp_path), dry_run=True, path_length=None))
    _fake_fused(m0, ntp, False)
    o0 = bmca.mca_out_ng(mca_obj=m0, abs_obj=m0.abs, mode=mode)
    new = {'rad_plen', 'rad_plen_out', 'rad_mean_plen', 'plen_edges'} | ({'rad_plen_std'} if mode == 'mean' else set())
    assert set(o.data) - set(o0.data) == new
    for k in o0.data:
        a, b = o.data[k]['data'], o0.data[k]['data']
        np.testing.assert_array_equal(a, b, err_msg=k)


def test_run_plen_prototype():
    lib = abi.load_library()
    assert len(lib.b200rt_run_plen.argtypes) == 8
    assert {'b200rt_run_plen', 'b200rt_read_plen', 'b200rt_plen_ptr'} <= set(abi.EXPORTS)


@pytest.mark.parametrize('mode', ['mean', 'all'])
def test_a_single_bin_keeps_its_axis(c4_kw, tmp_path, mode):
    m = bmca.mcarats_ng(**dict(c4_kw, fdir=str(tmp_path), dry_run=True, path_length=(0.0, 120.0, 1)))
    _fake_fused(m, 1, True)
    o = bmca.mca_out_ng(mca_obj=m, abs_obj=m.abs, mode=mode)
    nx, ny, nrun = m.Nx, m.Ny, m.Nrun
    assert o.data['rad_plen']['data'].shape == ((nx, ny, 1) if mode == 'mean' else (nx, ny, 1, nrun))
    assert o.data['rad_plen']['dims_info'][:3] == ['Nx', 'Ny', 'Nbin']
    np.testing.assert_allclose(o.data['plen_edges']['data'], [0.0, 120.0])
