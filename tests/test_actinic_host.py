"""
Host side of the actinic flux (mcarats_ng(actinic=True)): the documented errors and the mca_out_ng keys that exist only
when the actinic flux was asked for.  No GPU needed.
"""

import numpy as np
import pytest

import workloads
from er3t_b200 import abi
from er3t_b200.rtm import mca as bmca


@pytest.fixture(scope='module')
def c5_kw():
    kw, abs0 = workloads.c5(scale=0.01, photons=1e4)
    return dict(kw, Nrun=2, actinic=True)


@pytest.mark.parametrize('change, msg', [
    (dict(target='radiance'), 'not radiance'),
    (dict(spectral=True), 'spectral'),
    (dict(raw=True), 'raw'),
])
def test_actinic_errors(c5_kw, tmp_path, change, msg):
    with pytest.raises(OSError, match=r'Error \[mcarats_ng\]: <actinic=True>.*' + msg):
        bmca.mcarats_ng(**dict(c5_kw, fdir=str(tmp_path), **change))


def test_actinic_rejects_write_files(c5_kw, tmp_path):
    with pytest.raises(OSError, match=r'Error \[mcarats_ng\]: <actinic=True>.*write_files'):
        bmca.mcarats_ng(**dict(c5_kw, fdir=str(tmp_path / 'out'), write_files=True))


def test_actinic_needs_an_absorption_object(c5_kw, tmp_path):
    atm = c5_kw['atm_1ds'][0]
    saved = atm.abs
    try:
        atm.abs = None
        with pytest.raises(OSError, match=r'Error \[mcarats_ng\]: <actinic=True>.*absorption'):
            bmca.mcarats_ng(**dict(c5_kw, fdir=str(tmp_path)))
    finally:
        atm.abs = saved


@pytest.mark.parametrize('target', ['flux', 'flux0', 'heating rate'])
def test_targets_with_fluxes_are_accepted(c5_kw, tmp_path, target):
    m = bmca.mcarats_ng(**dict(c5_kw, fdir=str(tmp_path), dry_run=True, target=target))
    assert m.actinic and m.options.target & (abi.TARGET_FLUX | abi.TARGET_HEATING)


def _fake_fused(m, act):
    rng = np.random.default_rng(0)
    nx, ny, nz, nrun = m.Nx, m.Ny, m.scene.struct.nz, m.Nrun
    flux = [rng.uniform(0, 1, (nx, ny, nz + 1, 1, nrun)) for _ in range(3)]
    m.fused = {'flux': flux, 'radiance': None, 'heating': [rng.uniform(0, 1, (nx, ny, nz, 1, nrun))]}
    if act:
        direct = rng.uniform(0, 1, (nx, ny, nz, 1, nrun))
        m.fused['actinic'] = [np.concatenate([direct, direct + rng.uniform(0, 1, direct.shape)], axis=3)]
    return m


@pytest.mark.parametrize('mode', ['mean', 'all'])
def test_mca_out_keys_only_with_the_actinic_flux(c5_kw, tmp_path, mode):
    m = _fake_fused(bmca.mcarats_ng(**dict(c5_kw, fdir=str(tmp_path), dry_run=True, target='heating rate')), True)
    o = bmca.mca_out_ng(mca_obj=m, abs_obj=m.abs, mode=mode)
    nx, ny, nz, nrun = m.Nx, m.Ny, m.scene.struct.nz, m.Nrun
    a = m.fused['actinic'][0].astype(np.float32)
    direct, total = a[:, :, :, 0, :], a[:, :, :, 1, :]
    if mode == 'mean':
        np.testing.assert_allclose(o.data['f_act']['data'], total.mean(axis=-1), rtol=1e-6)
        np.testing.assert_allclose(o.data['f_act_direct']['data'], direct.mean(axis=-1), rtol=1e-6)
        np.testing.assert_allclose(o.data['f_act_diffuse']['data'], (total - direct).mean(axis=-1), rtol=1e-5, atol=1e-7)
        np.testing.assert_allclose(o.data['f_act_std']['data'], total.std(axis=-1), rtol=1e-5, atol=1e-7)
        for k in ('f_act', 'f_act_direct', 'f_act_diffuse'):
            assert o.data[k]['data'].shape == (nx, ny, nz) and o.data[k]['dims_info'] == ['Nx', 'Ny', 'Nz']
            assert o.data[k]['units'] == 'W/m^2/nm'
    else:
        assert o.data['f_act']['data'].shape == (nx, ny, nz, nrun)
        assert 'f_act_std' not in o.data
    m0 = _fake_fused(bmca.mcarats_ng(**dict(c5_kw, fdir=str(tmp_path), dry_run=True, target='heating rate', actinic=False)), False)
    o0 = bmca.mca_out_ng(mca_obj=m0, abs_obj=m0.abs, mode=mode)
    new = {'f_act', 'f_act_direct', 'f_act_diffuse'}
    if mode == 'mean':
        new |= {k + '_std' for k in new}
    assert set(o.data) - set(o0.data) == new
    for k in o0.data:
        np.testing.assert_array_equal(np.asarray(o.data[k]['data']), np.asarray(o0.data[k]['data']), err_msg=k)


def test_run_act_prototype():
    lib = abi.load_library()
    assert len(lib.b200rt_run_act.argtypes) == 5
    assert {'b200rt_run_act', 'b200rt_read_act', 'b200rt_act_ptr'} <= set(abi.EXPORTS)
