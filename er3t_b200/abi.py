"""
ctypes mirror of include/b200rt.h (the drop-in C-ABI) and the loader of libb200rt.so.

The product path has NO CPU fallback: if the CUDA library is missing or cannot be loaded,
`load_library()` raises OSError -- callers never silently route anywhere else.

Reference interface this replaces: the `mcarats` command line built at
er3t/rtm/mca/mca_run.py:110-113 and executed at :179-181 (env var MCARATS_V010_EXE, er3t/common.py:10).
"""

import os
import ctypes as C

import numpy as np

__all__ = ['Sensor', 'SceneStruct', 'Job', 'Kd', 'Options', 'Stats', 'load_library', 'library_path',
           'SFC_LAMBERT', 'SFC_DSM', 'SFC_RPV', 'SFC_LSRT',
           'SOLVER_3D', 'SOLVER_PARTIAL_3D', 'SOLVER_IPA',
           'TARGET_FLUX', 'TARGET_RADIANCE', 'TARGET_HEATING', 'HostScene', 'make_jobs', 'make_kd', 'make_options']

SFC_LAMBERT, SFC_DSM, SFC_RPV, SFC_LSRT = 1, 2, 3, 4
SOLVER_3D, SOLVER_PARTIAL_3D, SOLVER_IPA = 0, 1, 2
TARGET_FLUX, TARGET_RADIANCE, TARGET_HEATING = 1, 2, 4

_dp = C.POINTER(C.c_double)
_fp = C.POINTER(C.c_float)
_ip = C.POINTER(C.c_int32)


class Sensor(C.Structure):
    _fields_ = [('kind', C.c_int32), ('nxr', C.c_int32), ('nyr', C.c_int32), ('_pad', C.c_int32),
                ('the', C.c_double), ('phi', C.c_double), ('zloc', C.c_double), ('zref', C.c_double),
                ('psi', C.c_double), ('xpos', C.c_double), ('ypos', C.c_double), ('qmax', C.c_double),
                ('umax', C.c_double), ('vmax', C.c_double), ('apsize', C.c_double)]


class SceneStruct(C.Structure):
    _fields_ = [('nx', C.c_int32), ('ny', C.c_int32), ('nz', C.c_int32),
                ('iz3l', C.c_int32), ('nz3', C.c_int32),
                ('np1d', C.c_int32), ('np3d', C.c_int32), ('layout3d', C.c_int32),
                ('dx', C.c_double), ('dy', C.c_double),
                ('zgrd', C.c_void_p),
                ('ext1d', C.c_void_p), ('omg1d', C.c_void_p), ('apf1d', C.c_void_p),
                ('ext3d', C.c_void_p), ('omg3d', C.c_void_p), ('apf3d', C.c_void_p), ('abs3d', C.c_void_p),
                ('npf', C.c_int32), ('nang', C.c_int32),
                ('ang', C.c_void_p), ('pha', C.c_void_p),
                ('sfc_nx', C.c_int32), ('sfc_ny', C.c_int32),
                ('sfc_type', C.c_void_p), ('sfc_param', C.c_void_p),
                ('src_the', C.c_double), ('src_phi', C.c_double), ('src_qmax', C.c_double), ('src_flx', C.c_double),
                ('nrad', C.c_int32), ('_pad1', C.c_int32),
                ('sensors', C.POINTER(Sensor)),
                ('cer3d', C.c_void_p), ('nref', C.c_int32), ('_pad2', C.c_int32),
                ('ref_tab', C.c_void_p), ('ssa_tab', C.c_void_p), ('asy_tab', C.c_void_p)]


class Job(C.Structure):
    _fields_ = [('nphot', C.c_int64), ('seed', C.c_uint64), ('slab', C.c_int32), ('_pad', C.c_int32),
                ('abs1d', C.c_void_p), ('flx_scale', C.c_void_p), ('rad_scale', C.c_double)]


class Kd(C.Structure):
    _fields_ = [('nkd', C.c_int32), ('_pad', C.c_int32), ('wkd', C.c_void_p), ('abs1d', C.c_void_p), ('rad_scale', C.c_void_p)]


class Options(C.Structure):
    _fields_ = [('solver', C.c_int32), ('target', C.c_int32), ('nslab', C.c_int32),
                ('shard_rank', C.c_int32), ('shard_world', C.c_int32),
                ('svx', C.c_int32), ('svy', C.c_int32), ('svz', C.c_int32),
                ('cmx', C.c_int32), ('cmy', C.c_int32), ('cmz', C.c_int32), ('flight_steps', C.c_int32),
                ('event_min', C.c_int32), ('empty_runs', C.c_int32), ('pool_slots', C.c_int32),
                ('iso_ss', C.c_int32), ('iso_max', C.c_int32),
                ('threads_per_block', C.c_int32), ('blocks_per_sm', C.c_int32), ('smem_tally', C.c_int32),
                ('kernel', C.c_int32), ('_reserved', C.c_int32),
                ('wmin', C.c_double), ('wfac', C.c_double)]


class Stats(C.Structure):
    _fields_ = [('photons', C.c_uint64), ('n_cell', C.c_uint64), ('n_tent', C.c_uint64), ('n_coll', C.c_uint64),
                ('n_sfc', C.c_uint64), ('n_le', C.c_uint64), ('n_le_visit', C.c_uint64), ('n_tally', C.c_uint64),
                ('n_roulette_kill', C.c_uint64),
                ('w_toa_up', C.c_double), ('w_sfc_abs', C.c_double), ('w_atm_abs', C.c_double),
                ('w_roulette', C.c_double), ('elapsed_ms', C.c_double), ('bytes_alg', C.c_double),
                ('launches', C.c_uint64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


# every symbol include/b200rt.h declares (tests check the library exports all of them)
EXPORTS = ['b200rt_version', 'b200rt_create', 'b200rt_destroy', 'b200rt_last_error', 'b200rt_upload_scene',
           'b200rt_run', 'b200rt_run_kd', 'b200rt_run_jac', 'b200rt_run_plen', 'b200rt_sync', 'b200rt_read_flux', 'b200rt_read_rad',
           'b200rt_read_heat', 'b200rt_read_jac', 'b200rt_jac_ptr', 'b200rt_read_plen', 'b200rt_plen_ptr', 'b200rt_tally_ptrs',
           'b200rt_stats_get', 'b200rt_philox_fill', 'b200rt_phase_eval', 'b200rt_phase_sample', 'b200rt_brdf_eval']


def library_path():
    """Path of the CUDA library: $ER3T_B200_LIB (the analogue of $MCARATS_V010_EXE, er3t/common.py:10)
    or the in-tree build er3t_b200/csrc/libb200rt.so."""
    p = os.environ.get('ER3T_B200_LIB')
    if p:
        return p
    return os.path.join(os.path.dirname(os.path.abspath(__file__)), 'csrc', 'libb200rt.so')


_LIB = None


def load_library(path=None):
    """Load libb200rt.so and declare prototypes.  Raises OSError when the library is missing --
    there is deliberately no CPU fallback."""
    global _LIB
    if _LIB is not None and path is None:
        return _LIB
    p = path or library_path()
    if not os.path.isfile(p):
        msg = 'Error [er3t_b200]: CUDA library <%s> not found. Build it with `python -c "import __graft_entry__ as g; g.build()"` ' \
              'or point $ER3T_B200_LIB at libb200rt.so. There is no CPU fallback.' % p
        raise OSError(msg)
    lib = C.CDLL(p)
    vp = C.c_void_p
    lib.b200rt_version.restype = C.c_int
    lib.b200rt_create.argtypes = [C.POINTER(vp), C.c_int]
    lib.b200rt_destroy.argtypes = [vp]
    lib.b200rt_last_error.argtypes = [vp]
    lib.b200rt_last_error.restype = C.c_char_p
    lib.b200rt_upload_scene.argtypes = [vp, C.POINTER(SceneStruct), C.POINTER(Options)]
    lib.b200rt_run.argtypes = [vp, C.POINTER(Job), C.c_int, C.c_int, vp]
    lib.b200rt_run_kd.argtypes = [vp, C.POINTER(Job), C.POINTER(Kd), C.c_int, C.c_int, vp]
    lib.b200rt_run_jac.argtypes = [vp, C.POINTER(Job), C.c_int, vp, C.c_int, C.c_int, vp]
    lib.b200rt_run_plen.argtypes = [vp, C.POINTER(Job), C.c_int, C.c_double, C.c_double, C.c_int, C.c_int, vp]
    lib.b200rt_sync.argtypes = [vp]
    for name in ('b200rt_read_flux', 'b200rt_read_rad', 'b200rt_read_heat', 'b200rt_read_jac', 'b200rt_read_plen'):
        getattr(lib, name).argtypes = [vp, vp, C.c_int64]
    lib.b200rt_tally_ptrs.argtypes = [vp, C.POINTER(vp), C.POINTER(C.c_int64), C.POINTER(vp), C.POINTER(C.c_int64),
                                      C.POINTER(vp), C.POINTER(C.c_int64)]
    lib.b200rt_jac_ptr.argtypes = [vp, C.POINTER(vp), C.POINTER(C.c_int64)]
    lib.b200rt_plen_ptr.argtypes = [vp, C.POINTER(vp), C.POINTER(C.c_int64)]
    lib.b200rt_stats_get.argtypes = [vp, C.POINTER(Stats)]
    lib.b200rt_philox_fill.argtypes = [vp, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32, vp, C.c_int64]
    lib.b200rt_phase_eval.argtypes = [vp, C.c_double, vp, vp, C.c_int64]
    lib.b200rt_phase_sample.argtypes = [vp, C.c_double, vp, vp, C.c_int64]
    lib.b200rt_brdf_eval.argtypes = [vp, C.c_int32, vp, vp, vp, vp, C.c_int64]
    for name in EXPORTS:
        f = getattr(lib, name)
        if name not in ('b200rt_last_error',):
            f.restype = C.c_int
    if path is None:
        _LIB = lib
    return lib


def _arr(a, dtype):
    return np.ascontiguousarray(a, dtype=dtype)


def _ptr(a):
    return None if a is None else a.ctypes.data


class HostScene:
    """
    Owns contiguous host (numpy) copies of every scene array and the ctypes struct that points at them.

    Array conventions (same as the reference's files): 3-D fields are given as numpy arrays of shape
    (nx, ny, nz3, np3d) exactly like `Atm_extp3d` (er3t/rtm/mca/mca_atm.py:248-252) and are transposed here
    into the ABI layout [np3d][nz3][ny][nx] (x fastest == Fortran order of the reference's binary,
    mca_atm.py:383-388).
    """

    def __init__(self, zgrd, ext1d, omg1d, apf1d, nx=1, ny=1, dx=1.0e4, dy=1.0e4,
                 iz3l=1, ext3d=None, omg3d=None, apf3d=None, abs3d=None,
                 cer3d=None, cer_tables=None,
                 ang=None, pha=None,
                 sfc_type=1, sfc_param=(0.0, 0.0, 0.0, 0.0, 0.0),
                 src_the=150.0, src_phi=270.0, src_qmax=0.533133, src_flx=1.0,
                 sensors=()):
        self.zgrd = _arr(zgrd, np.float64)
        nz = self.zgrd.size - 1
        self.ext1d = np.atleast_2d(_arr(ext1d, np.float64))
        self.omg1d = np.atleast_2d(_arr(omg1d, np.float64))
        self.apf1d = np.atleast_2d(_arr(apf1d, np.float64))
        np1d = self.ext1d.shape[0]
        if self.ext1d.shape != (np1d, nz) or self.omg1d.shape != (np1d, nz) or self.apf1d.shape != (np1d, nz):
            raise ValueError('Error [HostScene]: 1-D profiles must have shape (np1d, nz).')

        s = SceneStruct()
        s.nx, s.ny, s.nz = int(nx), int(ny), int(nz)
        s.np1d = np1d
        s.dx, s.dy = float(dx), float(dy)
        s.zgrd = _ptr(self.zgrd)
        s.ext1d, s.omg1d, s.apf1d = _ptr(self.ext1d), _ptr(self.omg1d), _ptr(self.apf1d)

        self.cer3d = self.ref_tab = self.ssa_tab = self.asy_tab = None
        if ext3d is not None:
            e3 = np.asarray(ext3d)
            if e3.ndim == 3:
                e3 = e3[..., np.newaxis]
            if cer3d is not None:
                # (omega, apf) are derived on the GPU from the effective radius (scene.cer3d, include/b200rt.h)
                c3 = np.asarray(cer3d)
                if c3.ndim == 3:
                    c3 = c3[..., np.newaxis]
                if c3.shape != e3.shape or e3.shape[3] != 1 or cer_tables is None:
                    raise ValueError('Error [HostScene]: <cer3d> needs one 3-D component of the shape of <ext3d> and <cer_tables>.')
                self.cer3d = _arr(c3, np.float32)
                self.ref_tab, self.ssa_tab, self.asy_tab = [_arr(t, np.float64) for t in cer_tables]
                o3 = a3 = None
            else:
                o3 = np.asarray(omg3d)
                a3 = np.asarray(apf3d)
                if o3.ndim == 3:
                    o3 = o3[..., np.newaxis]
                if a3.ndim == 3:
                    a3 = a3[..., np.newaxis]
            if e3.shape[0] != nx or e3.shape[1] != ny or (o3 is not None and (o3.shape != e3.shape or a3.shape != e3.shape)):
                raise ValueError('Error [HostScene]: 3-D fields must have shape (nx, ny, nz3[, np3d]).')
            # zero-copy when the arrays are already float32 and C-contiguous (what mca_atm_3d produces): the library
            # transposes (nx, ny, nz3, np3d) -> [np3d][nz3][ny][nx] on the GPU (layout3d = 1)
            self.ext3d = _arr(e3, np.float32)
            self.omg3d = None if o3 is None else _arr(o3, np.float32)
            self.apf3d = None if a3 is None else _arr(a3, np.float32)
            s.layout3d = 1
            s.np3d, s.nz3 = self.ext3d.shape[3], self.ext3d.shape[2]
            s.iz3l = int(iz3l)
            s.ext3d, s.omg3d, s.apf3d = _ptr(self.ext3d), _ptr(self.omg3d), _ptr(self.apf3d)
            if self.cer3d is not None:
                s.cer3d, s.nref = _ptr(self.cer3d), int(self.ref_tab.size)
                s.ref_tab, s.ssa_tab, s.asy_tab = _ptr(self.ref_tab), _ptr(self.ssa_tab), _ptr(self.asy_tab)
            if abs3d is not None and np.asarray(abs3d).any():
                b3 = np.asarray(abs3d)
                if b3.ndim == 4:
                    b3 = b3[..., 0]
                self.abs3d = _arr(np.transpose(b3, (2, 1, 0)), np.float32)
                s.abs3d = _ptr(self.abs3d)
            else:
                self.abs3d = None
                s.abs3d = None
        else:
            self.ext3d = self.omg3d = self.apf3d = self.abs3d = None
            s.np3d, s.nz3, s.iz3l = 0, 0, 1

        if pha is not None:
            self.ang = _arr(ang, np.float64)
            p = np.asarray(pha, dtype=np.float64)
            if p.ndim == 1:
                p = p[:, np.newaxis]
            # (nang, npf) as in pha_obj.data['pha'] (er3t/rtm/mca/mca_sca.py:92-93) -> [npf][nang]
            self.pha = _arr(p.T, np.float64)
            s.npf, s.nang = self.pha.shape
            if self.ang.size != s.nang:
                raise ValueError('Error [HostScene]: <ang> and <pha> disagree in size.')
            s.ang, s.pha = _ptr(self.ang), _ptr(self.pha)
        else:
            self.ang = self.pha = None
            s.npf, s.nang = 0, 0

        st = np.asarray(sfc_type)
        if st.ndim == 0:
            self.sfc_type = np.full((1, 1), int(st), dtype=np.int32)
            self.sfc_param = _arr(np.asarray(sfc_param, dtype=np.float32).reshape(5, 1, 1), np.float32)
        else:
            # (nxb, nyb) and (nxb, nyb, 5) as in Sfc_jsfc2d / Sfc_psfc2d (er3t/rtm/mca/mca_sfc.py:94-101)
            self.sfc_type = _arr(st.T, np.int32)
            self.sfc_param = _arr(np.transpose(np.asarray(sfc_param), (2, 1, 0)), np.float32)
        s.sfc_ny, s.sfc_nx = self.sfc_type.shape
        s.sfc_type, s.sfc_param = _ptr(self.sfc_type), _ptr(self.sfc_param)

        s.src_the, s.src_phi, s.src_qmax, s.src_flx = float(src_the), float(src_phi), float(src_qmax), float(src_flx)

        self.sensors = (Sensor * max(1, len(sensors)))()
        for i, q in enumerate(sensors):
            se = self.sensors[i]
            se.kind = int(q.get('kind', 2))
            se.nxr, se.nyr = int(q.get('nxr', nx)), int(q.get('nyr', ny))
            se.the, se.phi = float(q.get('the', 180.0)), float(q.get('phi', 270.0))
            se.zloc, se.zref = float(q.get('zloc', 705000.0)), float(q.get('zref', 0.0))
            se.psi, se.xpos, se.ypos = float(q.get('psi', 0.0)), float(q.get('xpos', 0.5)), float(q.get('ypos', 0.5))
            se.qmax, se.umax, se.vmax = float(q.get('qmax', 180.0)), float(q.get('umax', 180.0)), float(q.get('vmax', 180.0))
            se.apsize = float(q.get('apsize', 0.0))
        s.nrad = len(sensors)
        s.sensors = C.cast(self.sensors, C.POINTER(Sensor))
        self.struct = s

    # dims of the output tallies
    @property
    def nxy(self):
        return self.struct.nx * self.struct.ny

    def nbytes(self):
        """bytes of scene arrays that cross the host -> device boundary in b200rt_upload_scene"""
        n = 0
        for name in ('zgrd', 'ext1d', 'omg1d', 'apf1d', 'ext3d', 'omg3d', 'apf3d', 'abs3d', 'cer3d', 'ang', 'pha', 'sfc_type', 'sfc_param'):
            arr = getattr(self, name, None)
            if arr is not None:
                n += arr.nbytes
        return n

    def flux_shape(self, nslab):
        return (nslab, 3, self.struct.nz + 1, self.struct.ny, self.struct.nx)

    def heat_shape(self, nslab):
        return (nslab, self.struct.nz, self.struct.ny, self.struct.nx)

    def rad_size(self, nslab):
        return nslab * sum(self.sensors[i].nxr * self.sensors[i].nyr for i in range(self.struct.nrad))


def make_jobs(nphot, seeds, slabs, abs1d=None, flx_scale=None, rad_scale=None):
    """Build a ctypes array of Job plus the list of numpy arrays that must stay alive."""
    n = len(nphot)
    jobs = (Job * n)()
    keep = []
    for i in range(n):
        jobs[i].nphot = int(nphot[i])
        jobs[i].seed = int(seeds[i]) & 0xFFFFFFFFFFFFFFFF
        jobs[i].slab = int(slabs[i])
        if abs1d is not None and abs1d[i] is not None:
            a = _arr(abs1d[i], np.float64)
            keep.append(a)
            jobs[i].abs1d = _ptr(a)
        if flx_scale is not None and flx_scale[i] is not None:
            f = _arr(flx_scale[i], np.float64)
            keep.append(f)
            jobs[i].flx_scale = _ptr(f)
        jobs[i].rad_scale = 1.0 if rad_scale is None else float(rad_scale[i])
    return jobs, keep


def make_kd(abs1d, wkd, rad_scale=None, njob=1):
    """The k-distribution terms of a spectral run (b200rt_run_kd): `abs1d` (nkd, nz) gas absorption per term (1/m), `wkd`
    (nkd,) term weights (Atm_wkd0), `rad_scale` (nkd,) per-term radiance factors (default 1).  Returns a ctypes array of
    `njob` identical Kd records (one per job) plus the list of numpy arrays that must stay alive."""
    a = _arr(np.atleast_2d(abs1d), np.float64)
    nkd = a.shape[0]
    w = _arr(np.ravel(wkd), np.float64)
    r = _arr(np.ones(nkd) if rad_scale is None else np.ravel(rad_scale), np.float64)
    if w.size != nkd or r.size != nkd:
        raise ValueError('Error [make_kd]: <abs1d>, <wkd> and <rad_scale> disagree in the number of terms.')
    kd = (Kd * int(njob))()
    for j in range(int(njob)):
        kd[j].nkd = nkd
        kd[j].wkd, kd[j].abs1d, kd[j].rad_scale = _ptr(w), _ptr(a), _ptr(r)
    return kd, [a, w, r]


def make_options(solver=SOLVER_3D, target=TARGET_FLUX, nslab=1, shard_rank=0, shard_world=1,
                 sv=(0, 0, 0), iso_ss=1, iso_max=0, wmin=0.2, wfac=1.0, threads_per_block=0, blocks_per_sm=0,
                 cm=(0, 0, 0), flight_steps=0, event_min=0, empty_runs=0, pool_slots=0, smem_tally=0, kernel=0):
    o = Options()
    o.solver, o.target, o.nslab = int(solver), int(target), int(nslab)
    o.shard_rank, o.shard_world = int(shard_rank), int(shard_world)
    o.svx, o.svy, o.svz = [int(v) for v in sv]
    o.cmx, o.cmy, o.cmz = [int(v) for v in cm]
    o.flight_steps = int(flight_steps)
    o.event_min, o.empty_runs = int(event_min), int(empty_runs)
    o.pool_slots = int(pool_slots)
    o.kernel = int(kernel)
    o.smem_tally = int(smem_tally)
    o.iso_ss, o.iso_max = int(iso_ss), int(iso_max)
    o.threads_per_block, o.blocks_per_sm = int(threads_per_block), int(blocks_per_sm)
    o.wmin, o.wfac = float(wmin), float(wfac)
    return o
