"""
Host side of the gas-absorption Jacobian (mcarats_ng(gas_jacobian=...)): the documented errors, the layer-group edges
built from `gas_jacobian`, and the mca_out_ng keys that exist only when a Jacobian was asked for.  No GPU needed.
"""

import numpy as np
import pytest

import workloads
from er3t_b200 import abi
from er3t_b200.rtm import mca as bmca
from er3t_b200.rtm.mca.mcarats import jacobian_edges


@pytest.fixture(scope='module')
def c4_kw():
    kw, abs0 = workloads.c4(scale=0.0005, nwvl=1)[0]
    return dict(kw, Nrun=2, photons=1e4, gas_jacobian=True)


@pytest.mark.parametrize('change, msg', [
    (dict(spectral=True), 'spectral'),
    (dict(raw=True), 'raw'),
    (dict(target='flux'), 'radiance'),
    (dict(target='heating rate'), 'radiance'),
    (dict(sensor_type='all-sky camera'), 'satellite'),
    (dict(gas_jacobian=[0.0, 1.25, 20.0]), 'levels of the atmosphere'),
    (dict(gas_jacobian=[0.5, 20.0]), 'bottom and the top'),
    (dict(gas_jacobian=[0.0, 5.0, 2.0, 20.0]), 'strictly increasing'),
    (dict(gas_jacobian='all'), 'level heights'),
])
def test_jacobian_errors(c4_kw, tmp_path, change, msg):
    with pytest.raises(OSError, match=r'Error \[mcarats_ng\]: .*' + msg):
        bmca.mcarats_ng(**dict(c4_kw, fdir=str(tmp_path), **change))


def test_jacobian_rejects_write_files(c4_kw, tmp_path):
    with pytest.raises(OSError, match=r'Error \[mcarats_ng\]: .*write_files'):
        bmca.mcarats_ng(**dict(c4_kw, fdir=str(tmp_path / 'out'), write_files=True))


def test_jacobian_needs_an_absorption_object(c4_kw, tmp_path):
    atm = c4_kw['atm_1ds'][0]
    saved = atm.abs
    try:
        atm.abs = None
        with pytest.raises(OSError, match=r'Error \[mcarats_ng\]: .*absorption'):
            bmca.mcarats_ng(**dict(c4_kw, fdir=str(tmp_path)))
    finally:
        atm.abs = saved


def test_edges_from_gas_jacobian(c4_kw, tmp_path):
    m = bmca.mcarats_ng(**dict(c4_kw, fdir=str(tmp_path), dry_run=True))
    nz = m.scene.struct.nz
    np.testing.assert_array_equal(m.jac_edges, np.arange(nz + 1))
    np.testing.assert_allclose(m.jac_levels, m.scene.zgrd / 1000.0)
    assert m.options.smem_tally == -1
    lev = m.scene.zgrd / 1000.0
    m2 = bmca.mcarats_ng(**dict(c4_kw, fdir=str(tmp_path), dry_run=True, gas_jacobian=[lev[0], 2.0, 5.0, lev[-1]]))
    e = m2.jac_edges
    assert e[0] == 0 and e[-1] == nz and e.size == 4
    np.testing.assert_allclose(lev[e], [lev[0], 2.0, 5.0, lev[-1]])
    np.testing.assert_allclose(m2.jac_levels, [lev[0], 2.0, 5.0, lev[-1]])
    # without gas_jacobian nothing changes
    m3 = bmca.mcarats_ng(**dict(c4_kw, fdir=str(tmp_path), dry_run=True, gas_jacobian=None))
    assert m3.jac_edges is None and m3.options.smem_tally == 0


def test_jacobian_edges_function():
    z = np.arange(0.0, 100001.0, 1000.0)                 # 100 layers
    with pytest.raises(OSError, match='at most 64'):
        jacobian_edges(True, z)
    np.testing.assert_array_equal(jacobian_edges([0.0, 50.0, 100.0], z), [0, 50, 100])
    np.testing.assert_array_equal(jacobian_edges(True, z[:11]), np.arange(11))
    assert jacobian_edges(np.array([0.0, 100.0]), z).dtype == np.int32


def _fake_fused(m, ngrp, jac):
    rng = np.random.default_rng(0)
    nx, ny, nrun = m.Nx, m.Ny, m.Nrun
    m.fused = {'flux': None, 'radiance': [rng.uniform(0, 1, (nx, ny, 1, 1, nrun))], 'heating': None}
    if jac:
        m.fused['jacobian'] = [rng.uniform(-1, 0, (nx, ny, ngrp, 1, nrun))]
    return m


@pytest.mark.parametrize('mode', ['mean', 'all'])
def test_mca_out_keys_only_with_a_jacobian(c4_kw, tmp_path, mode):
    m = bmca.mcarats_ng(**dict(c4_kw, fdir=str(tmp_path), dry_run=True, gas_jacobian=[0.0, 2.0, 5.0, 20.0]))
    _fake_fused(m, 3, True)
    o = bmca.mca_out_ng(mca_obj=m, abs_obj=m.abs, mode=mode)
    nx, ny = m.Nx, m.Ny
    jac = np.asarray(m.fused['jacobian'][0], dtype=np.float32)[:, :, :, 0, :]
    np.testing.assert_allclose(o.data['jac_levels']['data'], [0.0, 2.0, 5.0, 20.0])
    if mode == 'mean':
        np.testing.assert_allclose(o.data['rad_jac']['data'], jac.mean(axis=-1), rtol=1e-6)
        np.testing.assert_allclose(o.data['rad_jac_std']['data'], jac.std(axis=-1), rtol=1e-5)
        assert o.data['rad_jac']['dims_info'] == ['Nx', 'Ny', 'Ngroup']
    else:
        assert o.data['rad_jac']['data'].shape == (nx, ny, 3, m.Nrun)
        assert 'rad_jac_std' not in o.data
    # the same simulation without a Jacobian: the keys are absent
    m0 = bmca.mcarats_ng(**dict(c4_kw, fdir=str(tmp_path), dry_run=True, gas_jacobian=None))
    _fake_fused(m0, 3, False)
    o0 = bmca.mca_out_ng(mca_obj=m0, abs_obj=m0.abs, mode=mode)
    assert not any(k.startswith('rad_jac') or k == 'jac_levels' for k in o0.data)
    assert set(o.data) - set(o0.data) == ({'rad_jac', 'rad_jac_std', 'jac_levels'} if mode == 'mean' else {'rad_jac', 'jac_levels'})


def test_run_jac_prototype():
    lib = abi.load_library()
    assert len(lib.b200rt_run_jac.argtypes) == 7
    assert 'b200rt_read_jac' in abi.EXPORTS and 'b200rt_jac_ptr' in abi.EXPORTS
