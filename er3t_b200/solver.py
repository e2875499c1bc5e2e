"""
Thin object wrapper over the C-ABI (include/b200rt.h): one Solver == one handle == one GPU.

This is what `mcarats_ng` drives instead of `mca_run` (er3t/rtm/mca/mca_run.py:41-181).  Errors from the
library surface as OSError carrying the library's message, in the reference's message style
(`'Error [mcarats_ng]: ...'`, er3t/rtm/mca/mcarats.py:144-145,481-483).
"""

import ctypes as C

import numpy as np

from . import abi

__all__ = ['Solver']


class Solver:

    def __init__(self, device=0, lib=None):
        self.lib = lib if lib is not None else abi.load_library()
        self.handle = C.c_void_p()
        rc = self.lib.b200rt_create(C.byref(self.handle), int(device))
        if rc != 0:
            self.handle = None
            raise OSError('Error [er3t_b200]: cannot create a solver on CUDA device %d (code %d). A B200 GPU is required; there is no CPU fallback.' % (device, rc))
        self.device = device
        self.scene = None
        self.options = None
        self._keep = None
        self._xt_key = None      # 'jac' / 'plen' / 'act' when the last run was a Jacobian / path-length / actinic run, else None
        self._xt_shape = None    # shape of that run's tally

    # ------------------------------------------------------------------ helpers
    def _check(self, rc, where):
        if rc != 0:
            msg = self.lib.b200rt_last_error(self.handle)
            msg = msg.decode() if msg else ''
            raise OSError('Error [er3t_b200]: %s failed (code %d): %s' % (where, rc, msg))

    def close(self):
        if getattr(self, 'handle', None):
            self.lib.b200rt_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ API
    def upload_scene(self, scene, options):
        """scene: abi.HostScene (or any object with `.struct`); options: abi.Options"""
        self._check(self.lib.b200rt_upload_scene(self.handle, C.byref(scene.struct), C.byref(options)), 'b200rt_upload_scene')
        self.scene = scene
        self.options = options

    def run(self, jobs, accumulate=False, stream=None, sync=True):
        """jobs: ctypes array of abi.Job (see abi.make_jobs)."""
        self._keep = jobs
        self._xt_key, self._xt_shape = None, None
        self._check(self.lib.b200rt_run(self.handle, jobs, len(jobs), 1 if accumulate else 0, stream), 'b200rt_run')
        if sync:
            self.sync()

    def run_kd(self, jobs, kd, accumulate=False, stream=None, sync=True):
        """Spectral run: jobs (abi.make_jobs, without abs1d / flx_scale) and kd (abi.make_kd, one record per job): every
        history serves all k-distribution terms of its job."""
        self._keep = (jobs, kd)
        self._xt_key, self._xt_shape = None, None
        self._check(self.lib.b200rt_run_kd(self.handle, jobs, kd, len(jobs), 1 if accumulate else 0, stream), 'b200rt_run_kd')
        if sync:
            self.sync()

    def run_jac(self, jobs, edges, accumulate=False, stream=None, sync=True):
        """b200rt_run that also tallies dI / dln(a_j) for the gas absorption of the layer groups [edges[j], edges[j+1]) (layer
        indices, 0 = edges[0] < ... < edges[-1] = nz, at most 64 groups): same histories, same radiance."""
        e = np.ascontiguousarray(edges, dtype=np.int32)
        if e.ndim != 1 or e.size < 2:
            raise ValueError('Error [er3t_b200]: <edges> must be a 1-D sequence of at least two layer indices.')
        self._keep = (jobs, e)
        self._check(self.lib.b200rt_run_jac(self.handle, jobs, len(jobs), e.ctypes.data, e.size - 1, 1 if accumulate else 0, stream),
                    'b200rt_run_jac')
        self._xt_key, self._xt_shape = 'jac', (self.options.nslab, self.scene.rad_size(1), e.size - 1)
        if sync:
            self.sync()

    def run_plen(self, jobs, tpmin, tpmax, ntp, accumulate=False, stream=None, sync=True):
        """b200rt_run that also tallies, per radiance pixel, the distribution of the geometric path lengths L (m) behind the
        radiance: ntp uniform bins on [tpmin, tpmax), underflow, overflow and the first moment sum(c L) (include/b200rt.h);
        same histories, same radiance."""
        self._keep = jobs
        self._check(self.lib.b200rt_run_plen(self.handle, jobs, len(jobs), float(tpmin), float(tpmax), int(ntp), 1 if accumulate else 0,
                                             stream), 'b200rt_run_plen')
        self._xt_key, self._xt_shape = 'plen', (self.options.nslab, self.scene.rad_size(1), int(ntp) + 3)
        if sync:
            self.sync()

    def run_act(self, jobs, accumulate=False, stream=None, sync=True):
        """b200rt_run that also tallies the actinic flux (spherical irradiance): the mean over every layer and column,
        direct and total, in the units of the flux (include/b200rt.h); same histories, same flux and heating."""
        self._keep = jobs
        self._check(self.lib.b200rt_run_act(self.handle, jobs, len(jobs), 1 if accumulate else 0, stream), 'b200rt_run_act')
        hs = self.scene.heat_shape(self.options.nslab)
        self._xt_key, self._xt_shape = 'act', (hs[0], 2) + tuple(hs[1:])
        if sync:
            self.sync()

    def sync(self):
        self._check(self.lib.b200rt_sync(self.handle), 'b200rt_sync')

    def stats(self):
        st = abi.Stats()
        self._check(self.lib.b200rt_stats_get(self.handle, C.byref(st)), 'b200rt_stats_get')
        return st.as_dict()

    def tally_ptrs(self):
        vp = C.c_void_p
        f, r, h = vp(), vp(), vp()
        nf, nr, nh = C.c_int64(), C.c_int64(), C.c_int64()
        self._check(self.lib.b200rt_tally_ptrs(self.handle, C.byref(f), C.byref(nf), C.byref(r), C.byref(nr), C.byref(h), C.byref(nh)),
                    'b200rt_tally_ptrs')
        return {'flux': (f.value, nf.value), 'rad': (r.value, nr.value), 'heat': (h.value, nh.value)}

    def read_flux(self, out=None):
        shape = self.scene.flux_shape(self.options.nslab)
        if out is None:
            out = np.empty(shape, dtype=np.float64)
        self._check(self.lib.b200rt_read_flux(self.handle, out.ctypes.data, out.size), 'b200rt_read_flux')
        return out

    def read_rad(self, out=None):
        n = self.scene.rad_size(self.options.nslab)
        if out is None:
            out = np.empty(n, dtype=np.float64)
        self._check(self.lib.b200rt_read_rad(self.handle, out.ctypes.data, out.size), 'b200rt_read_rad')
        return out

    _XT_RUN = {'jac': ('a Jacobian', 'run_jac'), 'plen': ('a path-length', 'run_plen'), 'act': ('an actinic', 'run_act')}

    def _read_xt(self, key, out):
        if self._xt_key != key:
            raise OSError('Error [er3t_b200]: read_%s: the last run was not %s run (%s).' % ((key,) + self._XT_RUN[key]))
        if out is None:
            out = np.empty(int(np.prod(self._xt_shape)), dtype=np.float64)
        self._check(getattr(self.lib, 'b200rt_read_' + key)(self.handle, out.ctypes.data, out.size), 'b200rt_read_' + key)
        return out.reshape(self._xt_shape)

    def _xt_ptr(self, key):
        if self._xt_key != key:
            return None, 0
        p, n = C.c_void_p(), C.c_int64()
        self._check(getattr(self.lib, 'b200rt_%s_ptr' % key)(self.handle, C.byref(p), C.byref(n)), 'b200rt_%s_ptr' % key)
        return p.value, n.value

    def read_jac(self, out=None):
        """Jacobian tally of the last run (run_jac): (nslab, sum_k nyr_k * nxr_k, ngrp), group fastest."""
        return self._read_xt('jac', out)

    def jac_ptr(self):
        """(device pointer, doubles) of the Jacobian tally of the last run (b200rt_jac_ptr), or (None, 0) when it was not a
        Jacobian run."""
        return self._xt_ptr('jac')

    def read_plen(self, out=None):
        """Path-length tally of the last run (run_plen): (nslab, sum_k nyr_k * nxr_k, ntp + 3), bins fastest: ntp bins,
        underflow, overflow, first moment."""
        return self._read_xt('plen', out)

    def plen_ptr(self):
        """(device pointer, doubles) of the path-length tally of the last run (b200rt_plen_ptr), or (None, 0) when it was not
        a path-length run."""
        return self._xt_ptr('plen')

    def read_act(self, out=None):
        """Actinic flux of the last run (run_act): (nslab, 2, nz, ny, nx), variable 0 direct, 1 total."""
        return self._read_xt('act', out)

    def act_ptr(self):
        """(device pointer, doubles) of the actinic tally of the last run (b200rt_act_ptr), or (None, 0) when it was not an
        actinic run."""
        return self._xt_ptr('act')

    def read_heat(self, out=None):
        shape = self.scene.heat_shape(self.options.nslab)
        if out is None:
            out = np.empty(shape, dtype=np.float64)
        self._check(self.lib.b200rt_read_heat(self.handle, out.ctypes.data, out.size), 'b200rt_read_heat')
        return out

    def results(self):
        """Everything the target asked for, as numpy arrays (same keys as oracle.run)."""
        res = {'flux': None, 'rad': None, 'heat': None}
        t = self.options.target
        if t & abi.TARGET_FLUX:
            res['flux'] = self.read_flux()
        if (t & abi.TARGET_RADIANCE) and self.scene.struct.nrad > 0:
            res['rad'] = self.read_rad()
        if t & abi.TARGET_HEATING:
            res['heat'] = self.read_heat()
        if self._xt_key:
            res[self._xt_key] = self._read_xt(self._xt_key, None)
        res['stats'] = self.stats()
        return res

    # diagnostics
    def philox(self, seed, first, n, c2=0, c3=0):
        out = np.zeros(4 * n, dtype=np.uint32)
        self._check(self.lib.b200rt_philox_fill(self.handle, int(seed), int(first), int(c2), int(c3), out.ctypes.data, int(n)), 'b200rt_philox_fill')
        return out.reshape(n, 4)

    def phase_eval(self, apf, mu):
        mu = np.ascontiguousarray(mu, dtype=np.float64)
        out = np.empty_like(mu)
        self._check(self.lib.b200rt_phase_eval(self.handle, float(apf), mu.ctypes.data, out.ctypes.data, mu.size), 'b200rt_phase_eval')
        return out

    def phase_sample(self, apf, xi):
        xi = np.ascontiguousarray(xi, dtype=np.float64)
        out = np.empty_like(xi)
        self._check(self.lib.b200rt_phase_sample(self.handle, float(apf), xi.ctypes.data, out.ctypes.data, xi.size), 'b200rt_phase_sample')
        return out

    def brdf_eval(self, sfc_type, param5, dir_in, dir_out):
        p = np.ascontiguousarray(param5, dtype=np.float32)
        di = np.ascontiguousarray(dir_in, dtype=np.float64).reshape(-1, 3)
        do = np.ascontiguousarray(dir_out, dtype=np.float64).reshape(-1, 3)
        out = np.empty(di.shape[0], dtype=np.float64)
        self._check(self.lib.b200rt_brdf_eval(self.handle, int(sfc_type), p.ctypes.data, di.ctypes.data, do.ctypes.data, out.ctypes.data, out.size),
                    'b200rt_brdf_eval')
        return out
