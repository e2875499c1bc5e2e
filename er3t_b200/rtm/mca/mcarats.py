"""
`mcarats_ng` with the constructor of er3t/rtm/mca/mcarats.py:62-99 -- construct == run, like the reference --
but the (run, g) jobs are traced in-process by the sm_100a solver (include/b200rt.h) instead of being written as
namelists and handed to the MCARaTS executable (mcarats.py:417-468, mca_run.py:110-181).

What is kept: every keyword of the reference, the per-g namelist dictionaries `self.nml[ig]` built by the same
`init_*` steps (they remain the parameter contract and can be dumped with `mca_inp_file`), the photon distribution
over g (`distribute_photon`), the attributes downstream code reads (`Ng Nrun date target fnames_inp fnames_out photons
photons_per_set Nx Ny dx dy wvl_info sfc_2d solver`), the error strings.

What is new (keyword-only, all optional): `seed` (reproducible Philox streams; default = wall clock like
mcarats.py:432), `device`, `raw` (keep per-job fields instead of g-weighted per-run sums), `write_files` (emit the
namelist text and MCARaTS-style .bin/.ctl outputs), `iz3l_fix`, `supervoxel`, `shard` / `reduce` (multi-GPU),
`extra_sensors`, `solver_obj` (reuse a handle), `camera_pixels` (all-sky camera grid instead of the reference's fixed
500 x 500), `spectral` (MCARaTS's multi-term mode, Atm_nkd = Ng: one history serves every g of the wavelength),
`gas_jacobian` (the radiance's derivatives with respect to the gas absorption of layer groups, from the same histories),
`path_length` (per-pixel histograms and mean of the photon path lengths behind the radiance, from the same histories).
"""

import datetime
import multiprocessing as mp
import numbers
import os
import time

import numpy as np

from er3t_b200 import abi
from er3t_b200.solver import Solver   # noqa: F401  (re-exported for callers that build their own handle)
from .mca_run import mca_run
from er3t_b200.util import add_reference
from .mca_inp import mca_inp_file, DEFAULTS
from .mca_out import cal_factors, write_mca_out_raw

__all__ = ['mcarats_ng', 'cal_mca_azimuth', 'distribute_photon']


class mcarats_ng:

    reference = '\nMCARaTS (Iwabuchi, 2006; Iwabuchi and Okamura, 2017):\n- Iwabuchi, H.: Efficient Monte Carlo methods for radiative transfer modeling, J. Atmos. Sci., 63, 2324-2339, https://doi.org/10.1175/JAS3755.1, 2006.\n- Iwabuchi, H., and Okamura, R.: Multispectral Monte Carlo radiative transfer simulation by using the maximum cross-section method, Journal of Quantitative Spectroscopy and Radiative Transfer, 193, 40-46, https://doi.org/10.1016/j.jqsrt.2017.01.025, 2017.'

    def __init__(self,
                 atm_1ds=[],
                 atm_3ds=[],
                 sca=None,
                 Ng=16,
                 weights=None,
                 fdir='tmp-data/sim',
                 Nrun=3,
                 Ncpu='auto',
                 mp_mode='py',
                 overwrite=True,
                 date=datetime.datetime.now(),
                 comment=False,
                 tune=False,
                 target='flux',
                 surface_albedo=0.03,
                 solar_zenith_angle=30.0,
                 solar_azimuth_angle=0.0,
                 sensor_zenith_angle=0.0,
                 sensor_azimuth_angle=0.0,
                 sensor_altitude=705000.0,
                 sensor_type='satellite',
                 sensor_xpos=0.5,
                 sensor_ypos=0.5,
                 solver='3d',
                 photons=1e7,
                 base_ratio=0.05,
                 verbose=False,
                 quiet=False,
                 *,
                 seed=None,
                 device=0,
                 raw=False,
                 write_files=False,
                 iz3l_fix=False,
                 supervoxel=(0, 0, 0),
                 shard=None,
                 reduce=None,
                 extra_sensors=None,
                 solver_obj=None,
                 wmin=None,
                 camera_pixels=None,
                 dry_run=False,
                 spectral=False,
                 gas_jacobian=None,
                 path_length=None,
                 actinic=False):
        """spectral=True: one job per run traces `photons` histories (not photons per g), each of which carries all Ng
        terms of the correlated-k set (Atm_nkd = Ng, Atm_wkd0 = weights; Iwabuchi and Okamura 2017).  `self.fused` has the
        same layout and meaning as without it.  Needs target='radiance' with the satellite sensor and an `abs` object;
        `raw`, `write_files`, flux / heating targets and the all-sky camera raise OSError.

        gas_jacobian: also estimate dI / dln(a_j) in the same histories, where a_j multiplies the gas absorption (Atm_abs1d)
        of every layer of group j, for every g.  True: one group per layer; a sequence of level heights (km), which must be
        levels of the atmosphere including its bottom and top: contiguous groups between them.  Results:
        `self.fused['jacobian']` (nx, ny, ngrp, 1, Nrun), `self.jac_extra` for the extra sensors (like `rad_extra`),
        `self.jac_levels` (km) and `self.jac_edges` (layer indices).  Atm_abst3d and particle absorption are not
        differentiated.  Needs target='radiance' with the satellite sensor and an `abs` object; `spectral`, `raw`,
        `write_files`, flux / heating targets and the all-sky camera raise OSError.

        path_length=(tpmin_km, tpmax_km, ntp): also tally, in the same histories, how long the photon paths behind each
        pixel's radiance were (MCARaTS's Rad_mplen / Rad_ntp / Rad_tpmin / Rad_tpmax, which this sets in `self.nml`).  The
        path of one local-estimate contribution runs from TOA along the whole history to the event and on to the sensor
        level.  Results: `self.fused['path_length']` (nx, ny, ntp+3, 1, Nrun): ntp uniform bins on [tpmin, tpmax), underflow,
        overflow and the first moment sum(c L) in metres (include/b200rt.h); `self.plen_extra` for the extra sensors and
        `self.plen_edges` (km).  Same rules as `gas_jacobian`, with which it cannot be combined.

        actinic=True: also tally, in the same histories, the actinic flux (spherical irradiance, the radiance integrated over
        all directions) as the mean over every layer and column, direct and total, in the units of the flux and with its
        g-weighting.  Result: `self.fused['actinic']` (nx, ny, nz, 2, Nrun), variable 0 direct, 1 total.  Needs
        target='flux', 'flux0' or 'heating rate' and an `abs` object; the radiance target, `spectral`, `raw` and
        `write_files` raise OSError."""

        add_reference(self.reference)

        fdir = os.path.abspath(fdir)
        self.write_files = write_files
        if write_files and not os.path.exists(fdir):
            os.makedirs(fdir)
            if not quiet:
                print('Message [mcarats_ng]: Directory <%s> is created.' % fdir)

        self.Ng = Ng
        self.date = date
        self.fdir = fdir
        self.verbose = verbose
        self.quiet = quiet
        self.overwrite = overwrite
        self.mp_mode = mp_mode.lower()
        self.sca = sca
        self.surface_albedo = surface_albedo
        self.solar_zenith_angle = solar_zenith_angle
        self.solar_azimuth_angle = solar_azimuth_angle
        self.sensor_zenith_angle = sensor_zenith_angle
        self.sensor_azimuth_angle = sensor_azimuth_angle
        self.sensor_altitude = sensor_altitude
        self.sensor_type = sensor_type
        self.sensor_xpos = sensor_xpos
        self.sensor_ypos = sensor_ypos
        self.Nrun = Nrun
        self.seed = seed
        self.device = device
        # write_files asks for MCARaTS-style per-job .bin/.ctl outputs: they only exist for un-fused (raw) slabs
        self.keep_raw = raw or write_files
        self.iz3l_fix = iz3l_fix
        self.supervoxel = supervoxel
        self.shard = shard if shard is not None else (0, 1)
        self.reduce = reduce
        self.extra_sensors = list(extra_sensors) if extra_sensors else []
        self._solver_obj = solver_obj
        self._wmin = wmin
        self.camera_pixels = camera_pixels
        self.dry_run = dry_run
        self.spectral = spectral
        self.gas_jacobian = gas_jacobian
        self.jac_edges = None
        self.jac_levels = None
        self.jac_extra = None
        self.path_length = path_length
        self.plen = None if path_length is None else path_length_bins(path_length)     # (tpmin, tpmax, ntp), metres
        self.plen_edges = None if self.plen is None else np.linspace(self.plen[0], self.plen[1], self.plen[2] + 1) / 1000.0
        self.plen_extra = None
        self.actinic = bool(actinic)
        self.atm_1ds = atm_1ds
        self.atm_3ds = atm_3ds

        s = solver.lower()
        if s in ['3d', '3 d', 'three d']:
            self.solver = '3D'
        elif s in ['p3d', 'p-3d', 'partial 3d', 'partial-3d']:
            self.solver = 'Partial 3D'
        elif s in ['ipa', 'independent pixel approximation']:
            self.solver = 'IPA'
        else:
            # (the reference formats self.solver here before assigning it, mcarats.py:144 -- SURVEY.md Appendix C)
            raise OSError('Error [mcarats_ng]: Cannot understand <solver=%s>.' % solver)

        self.target = target

        if len(atm_3ds) > 0:
            self.Nx = atm_3ds[0].nml['Atm_nx']['data']
            self.Ny = atm_3ds[0].nml['Atm_ny']['data']
        else:
            self.Nx = 1
            self.Ny = 1

        # photon distribution over the g of the correlated-k (mcarats.py:159-171)
        if weights is None:
            self.np_mode = 'evenly'
            weights = np.repeat(1.0 / self.Ng, Ng)
        else:
            self.np_mode = 'weighted'
        self.weights = np.asarray(weights, dtype=np.float64)
        photons_dist = distribute_photon(photons, weights, base_ratio=base_ratio)
        self.photons = np.tile(photons_dist, Nrun)
        self.photons_per_set = photons_dist.sum()

        # the reference refuses Ncpu == 1 (mcarats.py:177-186); any value is accepted here and ignored
        self.Ncpu_total = mp.cpu_count()
        self.Ncpu = self.Ncpu_total - 1 if Ncpu == 'auto' else Ncpu

        self.fnames_inp = [['%s/r%2.2d.g%3.3d.inp.txt' % (self.fdir, ir, ig) for ig in range(self.Ng)] for ir in range(self.Nrun)]
        self.fnames_out = [['%s/r%2.2d.g%3.3d.out.bin' % (self.fdir, ir, ig) for ig in range(self.Ng)] for ir in range(self.Nrun)]

        self.fused = None
        self.raw = None
        self.stats = None

        if not self.quiet and not self.overwrite:
            print('Message [mcarats_ng]: Reading mode ...')

        if overwrite:
            self.nml = [{} for ig in range(self.Ng)]
            self.init_wld(verbose=verbose, tune=tune, sensor_zenith_angle=sensor_zenith_angle, sensor_azimuth_angle=sensor_azimuth_angle,
                          sensor_type=sensor_type, sensor_altitude=sensor_altitude, sensor_xpos=sensor_xpos, sensor_ypos=sensor_ypos)
            self.init_sca(sca=sca)
            self.init_atm(atm_1ds=atm_1ds, atm_3ds=atm_3ds)
            self.init_sfc(surface_albedo=surface_albedo)
            self.init_src(solar_zenith_angle=solar_zenith_angle, solar_azimuth_angle=solar_azimuth_angle)
            self.gen_mca_inp(comment=comment)
            self.gen_mca_out()

        if self.mp_mode not in ['batch', 'shell', 'bash', 'hpc', 'sh']:
            self.run_check()

    # ------------------------------------------------------------------ namelist construction (mcarats.py:234-414)
    def init_wld(self, tune=False, verbose=False, sensor_zenith_angle=0.0, sensor_azimuth_angle=0.0,
                 sensor_type='satellite', sensor_altitude=705000.0, sensor_xpos=0.5, sensor_ypos=0.5):
        t = self.target.lower()
        if t in ['f', 'flux', 'irradiance']:
            self.target = 'flux'
        elif t in ['f0', 'flux0', 'irradiance0']:
            self.target = 'flux0'
        elif t in ['heating rate', 'hr']:
            self.target = 'heating rate'
        elif t in ['radiance', 'rad']:
            self.target = 'radiance'
        else:
            raise OSError('Error [mcarats_ng]: Cannot understand <target=%s>.' % self.target)

        for ig in range(self.Ng):
            n = self.nml[ig]
            n['Wld_mverb'] = 3 if verbose else 0
            n['Wld_moptim'] = 2 if tune else 0
            n['Wld_mbswap'] = 0
            n['Wld_njob'] = 1
            if self.target == 'flux':
                n['Wld_mtarget'], n['Flx_mflx'], n['Flx_mhrt'] = 1, 3, 0
            elif self.target == 'flux0':
                n['Wld_mtarget'], n['Flx_mflx'], n['Flx_mhrt'] = 1, 1, 0
            elif self.target == 'heating rate':
                n['Wld_mtarget'], n['Flx_mflx'], n['Flx_mhrt'] = 1, 3, 1
            else:
                n['Wld_mtarget'] = 2
                if 'satellite' in sensor_type.lower():
                    n['Rad_mrkind'] = 2
                elif 'all-sky' in sensor_type.lower():
                    n['Rad_mrkind'] = 1
                    n['Rad_qmax'] = 178.0
                    n['Rad_apsize'] = 0.05
                    n['Rad_xpos'] = sensor_xpos
                    n['Rad_ypos'] = sensor_ypos
                n['Rad_mplen'] = 0
                if self.plen is not None:
                    n['Rad_mplen'] = 1
                    n['Rad_tpmin'], n['Rad_tpmax'], n['Rad_ntp'] = self.plen
                n['Rad_mpmap'] = 1
                n['Rad_nrad'] = 1
                n['Rad_difr0'] = 7.5
                n['Rad_difr1'] = 0.0025
                n['Rad_the'] = 180.0 - sensor_zenith_angle
                n['Rad_phi'] = cal_mca_azimuth(sensor_azimuth_angle)
                n['Rad_zloc'] = sensor_altitude

    def init_sca(self, sca=None):
        for ig in range(self.Ng):
            if sca is None:
                self.nml[ig]['Sca_npf'] = 0
            else:
                for key in sca.nml.keys():
                    self.nml[ig][key] = sca.nml[key]['data']

    def init_atm(self, atm_1ds=[], atm_3ds=[]):
        if len(atm_1ds) == 0:
            raise OSError('Error [mcarats_ng]: need <atm_1ds> to proceed.')
        big = ['Atm_tmpa3d', 'Atm_abst3d', 'Atm_extp3d', 'Atm_omgp3d', 'Atm_apfp3d']
        for ig in range(self.Ng):
            for atm_1d in atm_1ds:
                for key in atm_1d.nml[ig].keys():
                    self.nml[ig][key] = atm_1d.nml[ig][key]['data']
            self.wvl_info = atm_1ds[-1].wvl_info
            for atm_3d in atm_3ds:
                for key in atm_3d.nml.keys():
                    if key not in big:
                        self.nml[ig][key] = atm_3d.nml[key]['data']
                self.Nx = atm_3d.nml['Atm_nx']['data']
                self.Ny = atm_3d.nml['Atm_ny']['data']
                self.dx = atm_3d.nml['Atm_dx']['data']
                self.dy = atm_3d.nml['Atm_dy']['data']
                if self.target == 'radiance':
                    if 'satellite' in self.sensor_type.lower():
                        self.nml[ig]['Rad_nxr'] = atm_3d.nml['Atm_nx']['data']
                        self.nml[ig]['Rad_nyr'] = atm_3d.nml['Atm_ny']['data']
                    elif 'all-sky' in self.sensor_type.lower():
                        self.nml[ig]['Rad_nxr'] = 500
                        self.nml[ig]['Rad_nyr'] = 500
        self.abs = getattr(atm_1ds[-1], 'abs', None)

    def init_src(self, solar_zenith_angle=0.0, solar_azimuth_angle=0.0):
        for ig in range(self.Ng):
            n = self.nml[ig]
            n['Src_flx'] = 1.0
            n['Src_qmax'] = 0.533133
            n['Src_dwlen'] = 0.0
            n['Src_mtype'] = 1
            n['Src_mphi'] = 0
            n['Src_the'] = 180.0 - solar_zenith_angle
            n['Src_phi'] = cal_mca_azimuth(solar_azimuth_angle)

    def init_sfc(self, surface_albedo=0.03):
        for ig in range(self.Ng):
            if self.verbose:
                print('Message [mcarats_ng]: Assume Lambertian surface ...')
            # (the reference accepts only float / np.float32 / np.float64 and raises ValueError for an int,
            #  mcarats.py:393,411-414; any real number is accepted here -- SURVEY.md Appendix C)
            if isinstance(surface_albedo, numbers.Real) or isinstance(surface_albedo, (np.floating, np.integer)):
                self.nml[ig]['Sfc_mbrdf'] = np.array([1, 0, 0, 0])
                self.nml[ig]['Sfc_mtype'] = 1
                self.nml[ig]['Sfc_param(1)'] = float(surface_albedo)
                self.sfc_2d = False
            elif hasattr(surface_albedo, 'nml') and 'Sfc_jsfc2d' in surface_albedo.nml:
                for key in surface_albedo.nml.keys():
                    if '2d' not in key:
                        self.nml[ig][key] = surface_albedo.nml[key]['data']
                self.sfc_2d = True
            else:
                raise ValueError('\nError [mcarats_ng]: Cannot ingest <surface_albedo>.')

    # ------------------------------------------------------------------ inputs: seeds (+ optional namelist dump)
    def gen_mca_inp(self, comment=False):
        if self.seed is None:
            # wall-clock seeds exactly like mcarats.py:432-437 (np.random.shuffle permutes the rows of the 2-D array)
            base = int(time.time())
            rands = np.arange(self.Nrun * self.Ng).reshape((self.Nrun, self.Ng))
            np.random.shuffle(rands)
        else:
            base = int(self.seed)
            rands = np.arange(self.Nrun * self.Ng).reshape((self.Nrun, self.Ng))
        self.seeds = base + rands
        if self.write_files:
            for ir in range(self.Nrun):
                for ig in range(self.Ng):
                    self.nml[ig]['Wld_jseed'] = int(self.seeds[ir, ig])
                    mca_inp_file(self.fnames_inp[ir][ig], self.nml[ig], comment=comment)
            if not self.quiet:
                print('Message [mcarats_ng]: Created MCARaTS input files under <%s>.' % self.fdir)

    # ------------------------------------------------------------------ scene hand-off
    def build_scene(self):
        """Translate namelist + input objects into the C-ABI scene (host arrays; the library copies them to HBM)."""
        n0 = self.nml[0]
        zgrd = np.asarray(n0['Atm_zgrd0'], dtype=np.float64)
        nz = zgrd.size - 1
        np1d = int(n0.get('Atm_np1d', 1))
        ext1d = np.stack([np.asarray(n0['Atm_ext1d(1:, %d)' % (k + 1)], dtype=np.float64) for k in range(np1d)])
        if 'Atm_fext1d' in n0:
            # Atm_fext1d(KNP1D): scaling factor for Atm_ext1d (mca_inp.py:232); er3t never sets it (default 1)
            ext1d = ext1d * np.broadcast_to(np.asarray(n0['Atm_fext1d'], dtype=np.float64), (np1d,))[:, None]
        omg1d = np.stack([np.asarray(n0['Atm_omg1d(1:, %d)' % (k + 1)], dtype=np.float64) for k in range(np1d)])
        apf1d = np.stack([np.asarray(n0['Atm_apf1d(1:, %d)' % (k + 1)], dtype=np.float64) for k in range(np1d)])
        if ext1d.shape[1] != nz:
            raise OSError('Error [mcarats_ng]: <Atm_zgrd0> and the 1D profiles disagree in size.')
        kw = {}
        if len(self.atm_3ds) > 0:
            a3 = self.atm_3ds[-1].nml
            iz3l = int(n0.get('Atm_iz3l', DEFAULTS['Atm_iz3l']))
            if self.iz3l_fix:
                iz3l -= 1
            kw.update(nx=int(a3['Atm_nx']['data']), ny=int(a3['Atm_ny']['data']), dx=float(a3['Atm_dx']['data']), dy=float(a3['Atm_dy']['data']),
                      iz3l=iz3l, ext3d=a3['Atm_extp3d']['data'])
            a3obj = self.atm_3ds[-1]
            if getattr(a3obj, 'cer3d', None) is not None and int(a3['Atm_np3d']['data']) == 1:
                # mca_atm_3d(device_props=True): the GPU derives (omega, apf) from the effective radius while packing the scene
                kw.update(cer3d=a3obj.cer3d, cer_tables=a3obj.cer_tables)
            else:
                kw.update(omg3d=a3['Atm_omgp3d']['data'], apf3d=a3['Atm_apfp3d']['data'])
            # Atm_abst3d: always looked at (a caller may have filled the array in place); only lazily created zeros
            # that nobody has touched are skipped
            b3d = a3['Atm_abst3d']['data']
            if hasattr(b3d, '_fn') and b3d._val is None:
                b3d = None                                    # lazy zeros nobody has touched
            elif b3d is not None and not np.any(np.asarray(b3d)):
                b3d = None
            kw.update(abs3d=b3d)
            fe3, fa3 = self.nml[0].get('Atm_fext3d', 1.0), self.nml[0].get('Atm_fabs3d', 1.0)
            if np.any(np.asarray(fe3) != 1.0):
                # Atm_fext3d(KNP3D): scaling factor for the 3-D extinction (mca_inp.py:233)
                e3s = np.asarray(kw['ext3d'], dtype=np.float32)
                e3s = e3s[..., np.newaxis] if e3s.ndim == 3 else e3s
                kw['ext3d'] = e3s * np.broadcast_to(np.asarray(fe3, dtype=np.float32), (e3s.shape[3],))
            if kw['abs3d'] is not None and float(fa3) != 1.0:
                kw['abs3d'] = np.asarray(kw['abs3d'], dtype=np.float32) * np.float32(fa3)
        if self.sca is not None and int(n0.get('Sca_npf', 0)) > 0:
            kw.update(ang=self.sca.pha.data['ang']['data'], pha=self.sca.pha.data['pha']['data'])
        if self.sfc_2d:
            s2 = self.surface_albedo.nml
            kw.update(sfc_type=np.asarray(s2['Sfc_jsfc2d']['data'], dtype=np.int32), sfc_param=s2['Sfc_psfc2d']['data'])
        else:
            kw.update(sfc_type=int(n0['Sfc_mtype']), sfc_param=(float(n0['Sfc_param(1)']), 0.0, 0.0, 0.0, 0.0))
        sensors = []
        if self.target == 'radiance':
            nxr = int(n0.get('Rad_nxr', kw.get('nx', 1)))
            nyr = int(n0.get('Rad_nyr', kw.get('ny', 1)))
            if int(n0.get('Rad_mrkind', 2)) == 1:
                # all-sky camera (mcarats.py:291-296,369-371): local radiance per solid angle at (xpos, ypos, zloc)
                if self.camera_pixels is not None:
                    nxr, nyr = int(self.camera_pixels[0]), int(self.camera_pixels[1])
                    for ig in range(self.Ng):
                        self.nml[ig]['Rad_nxr'], self.nml[ig]['Rad_nyr'] = nxr, nyr
                sensors.append(dict(kind=1, the=n0['Rad_the'], phi=n0['Rad_phi'], psi=n0.get('Rad_psi', DEFAULTS.get('Rad_psi', 0.0)),
                                    zloc=n0['Rad_zloc'], nxr=nxr, nyr=nyr, xpos=n0.get('Rad_xpos', 0.5), ypos=n0.get('Rad_ypos', 0.5),
                                    qmax=n0.get('Rad_qmax', 180.0), umax=n0.get('Rad_umax', DEFAULTS.get('Rad_umax', 180.0)),
                                    vmax=n0.get('Rad_vmax', DEFAULTS.get('Rad_vmax', 180.0)), apsize=n0.get('Rad_apsize', 0.0)))
            else:
                sensors.append(dict(kind=2, the=n0['Rad_the'], phi=n0['Rad_phi'], zloc=n0['Rad_zloc'], zref=n0.get('Rad_zref', DEFAULTS['Rad_zref']), nxr=nxr, nyr=nyr))
            for e in self.extra_sensors:
                sensors.append(dict(kind=2, the=180.0 - e['sensor_zenith_angle'], phi=cal_mca_azimuth(e['sensor_azimuth_angle']),
                                    zloc=e.get('sensor_altitude', n0['Rad_zloc']), zref=e.get('zref', 0.0), nxr=nxr, nyr=nyr))
        return abi.HostScene(zgrd, ext1d, omg1d, apf1d, src_the=n0['Src_the'], src_phi=n0['Src_phi'], src_qmax=n0['Src_qmax'],
                             src_flx=n0['Src_flx'], sensors=sensors, **kw)

    # ------------------------------------------------------------------ run (replaces mca_run + the MCARaTS process)
    def gen_mca_out(self):
        solvers = {'3D': abi.SOLVER_3D, 'Partial 3D': abi.SOLVER_PARTIAL_3D, 'IPA': abi.SOLVER_IPA}
        if not self.quiet:
            print('Message [mcarats_ng]: Running the in-process B200 solver ...')
            self.print_info()

        scene = self.build_scene()
        self.scene = scene
        nz = scene.struct.nz
        Ng, Nrun = self.Ng, self.Nrun
        if self.target in ('flux', 'flux0'):
            tflag = abi.TARGET_FLUX
        elif self.target == 'heating rate':
            tflag = abi.TARGET_FLUX | abi.TARGET_HEATING
        else:
            tflag = abi.TARGET_RADIANCE

        if self.actinic:
            if self.target == 'radiance':
                raise OSError('Error [mcarats_ng]: <actinic=True> supports target=\'flux\', \'flux0\' and \'heating rate\' only (not radiance).')
            if self.spectral:
                raise OSError('Error [mcarats_ng]: <actinic=True> is not available with <spectral=True>.')
            if self.keep_raw:
                raise OSError('Error [mcarats_ng]: <actinic=True> is tallied per run: <raw> and <write_files> are not available.')
            if self.abs is None:
                raise OSError('Error [mcarats_ng]: <actinic=True> needs the gas absorption object of <atm_1ds>.')
        if self.spectral:
            if self.keep_raw:
                raise OSError('Error [mcarats_ng]: <spectral=True> sums the g terms in every history: <raw> and <write_files> are not available.')
            if self.target != 'radiance':
                raise OSError('Error [mcarats_ng]: <spectral=True> supports target=\'radiance\' only (flux and heating rates are not available yet).')
            if 'satellite' not in self.sensor_type.lower():
                raise OSError('Error [mcarats_ng]: <spectral=True> supports the satellite sensor only (not the all-sky camera).')
            if self.abs is None:
                raise OSError('Error [mcarats_ng]: <spectral=True> needs the gas absorption object of <atm_1ds> (its g weights and solar factors).')
        jac = self.gas_jacobian is not None and self.gas_jacobian is not False
        if jac:
            if self.spectral:
                raise OSError('Error [mcarats_ng]: <gas_jacobian> is not available with <spectral=True>.')
            if self.keep_raw:
                raise OSError('Error [mcarats_ng]: <gas_jacobian> is tallied per run: <raw> and <write_files> are not available.')
            if self.target != 'radiance':
                raise OSError('Error [mcarats_ng]: <gas_jacobian> supports target=\'radiance\' only (flux and heating rates are not available).')
            if 'satellite' not in self.sensor_type.lower():
                raise OSError('Error [mcarats_ng]: <gas_jacobian> supports the satellite sensor only (not the all-sky camera).')
            if self.abs is None:
                raise OSError('Error [mcarats_ng]: <gas_jacobian> needs the gas absorption object of <atm_1ds>.')
            self.jac_edges = jacobian_edges(self.gas_jacobian, scene.zgrd)
            self.jac_levels = scene.zgrd[self.jac_edges] / 1000.0
        if self.plen is not None:
            if jac:
                raise OSError('Error [mcarats_ng]: <path_length> cannot be combined with <gas_jacobian> (one extra tally per run).')
            if self.spectral:
                raise OSError('Error [mcarats_ng]: <path_length> is not available with <spectral=True>.')
            if self.keep_raw:
                raise OSError('Error [mcarats_ng]: <path_length> is tallied per run: <raw> and <write_files> are not available.')
            if self.target != 'radiance':
                raise OSError('Error [mcarats_ng]: <path_length> supports target=\'radiance\' only (flux and heating rates are not available).')
            if 'satellite' not in self.sensor_type.lower():
                raise OSError('Error [mcarats_ng]: <path_length> supports the satellite sensor only (not the all-sky camera).')
            if self.abs is None:
                raise OSError('Error [mcarats_ng]: <path_length> needs the gas absorption object of <atm_1ds>.')
        fuse = (not self.keep_raw) and (self.abs is not None)
        self.fuse = fuse
        if fuse:
            f_lev, _ = cal_factors(self.date, self.abs, nz + 1, Ng)       # flux levels
            f_rad, _ = cal_factors(self.date, self.abs, 1, Ng)
            nslab = Nrun
        else:
            nslab = Nrun * Ng

        nphot, seeds, slabs, abs1d, fsc, rsc = [], [], [], [], [], []
        for ir in range(Nrun):
            for ig in range(Ng if not self.spectral else 0):
                nphot.append(int(self.photons[ir * Ng + ig]))
                seeds.append(int(self.seeds[ir, ig]))
                slabs.append(ir if fuse else ir * Ng + ig)
                key = 'Atm_abs1d(1:, 1)'
                a1 = np.asarray(self.nml[ig][key], dtype=np.float64) if key in self.nml[ig] else None
                if a1 is not None and 'Atm_fabs1d' in self.nml[ig]:
                    a1 = a1 * float(self.nml[ig]['Atm_fabs1d'])          # scaling factor for Atm_abs1d (mca_inp.py:234)
                abs1d.append(a1)
                fsc.append(f_lev[:, ig].astype(np.float64) if fuse else None)
                rsc.append(float(f_rad[0, ig]) if fuse else 1.0)
        kd = None
        if self.spectral:
            # one job per run; term g: Atm_abs1d(1:, 1) x Atm_fabs1d of self.nml[ig] as above, radiance factor f_rad[0, ig]
            key = 'Atm_abs1d(1:, 1)'
            terms = []
            for ig in range(Ng):
                a1 = np.asarray(self.nml[ig][key], dtype=np.float64) if key in self.nml[ig] else np.zeros(nz)
                if 'Atm_fabs1d' in self.nml[ig]:
                    a1 = a1 * float(self.nml[ig]['Atm_fabs1d'])
                terms.append(a1)
            kd = dict(abs1d=np.stack(terms), wkd=self.weights, rad_scale=f_rad[0, :].astype(np.float64))
            for ir in range(Nrun):
                nphot.append(int(self.photons_per_set))
                seeds.append(int(self.seeds[ir, 0]))
                slabs.append(ir)
                abs1d.append(None)
                fsc.append(None)
                rsc.append(1.0)
        wmin = DEFAULTS['Pho_wmin'] if self._wmin is None else self._wmin
        # (spectral: tiny radiance tallies go through global atomics; the kernels that keep them in shared memory are the
        # per-level ones, which have no spectral variant)
        opt = abi.make_options(solver=solvers[self.solver], target=tflag, nslab=nslab, shard_rank=self.shard[0], shard_world=self.shard[1],
                               sv=self.supervoxel, iso_ss=DEFAULTS['Pho_iso_SS'], iso_max=DEFAULTS['Pho_iso_max'], wmin=wmin, wfac=DEFAULTS['Pho_wfac'],
                               smem_tally=-1 if (self.spectral or jac or self.plen is not None) else 0)
        jobs_args = dict(nphot=nphot, seeds=seeds, slabs=slabs, abs1d=abs1d, flx_scale=fsc, rad_scale=rsc)
        self.kd_args = kd
        self.options, self.jobs_args, self.nslab = opt, jobs_args, nslab
        if self.dry_run:
            # everything is prepared (scene, options, jobs) but nothing is traced; used by bench.py to time the
            # device-resident path separately from the host-side packing
            self.fused = {}
            return
        # the reference hands the job list to `mca_run` (mcarats.py:468); so does this class -- one launch instead of a pool
        runner = mca_run(scene, opt, nphot, seeds, slabs, abs1d=abs1d, flx_scale=fsc, rad_scale=rsc, device=self.device,
                         solver_obj=self._solver_obj, Ncpu=self.Ncpu, mp_mode=self.mp_mode, quiet=True, run=False, kd=kd,
                         jac_edges=self.jac_edges, plen=self.plen, act=self.actinic)
        try:
            self.h2d_bytes = scene.nbytes() + sum(a.nbytes for a in runner._keep)
            runner.launch()
            if self.reduce is not None:
                res = self.reduce(runner.solver)     # multi-GPU: all-reduce of the tallies (er3t_b200.dist.allreduce_results)
            else:
                res = runner.solver.results()
        finally:
            runner.close()
        self.stats = res['stats']
        self._store(res, scene, nslab, fuse)

    def _store(self, res, scene, nslab, fuse):
        nx, ny, nz = scene.struct.nx, scene.struct.ny, scene.struct.nz
        Ng, Nrun = self.Ng, self.Nrun
        flux = rad = heat = None
        if res.get('flux') is not None:
            # [nslab][3][nz+1][ny][nx] -> (3, nx, ny, nz+1, 1, nslab)
            flux = np.transpose(res['flux'].reshape(nslab, 3, nz + 1, ny, nx), (1, 4, 3, 2, 0))[:, :, :, :, np.newaxis, :]
        if res.get('rad') is not None:
            se = scene.sensors[0]
            per = scene.rad_size(1)
            r = res['rad'].reshape(nslab, per)
            n0 = se.nxr * se.nyr
            rad = np.transpose(r[:, :n0].reshape(nslab, se.nyr, se.nxr), (2, 1, 0))[:, :, np.newaxis, np.newaxis, :]
            self.rad_extra = []
            off = n0
            for k in range(1, scene.struct.nrad):
                sk = scene.sensors[k]
                nk = sk.nxr * sk.nyr
                self.rad_extra.append(np.transpose(r[:, off:off + nk].reshape(nslab, sk.nyr, sk.nxr), (2, 1, 0)))
                off += nk
        if res.get('heat') is not None:
            heat = np.transpose(res['heat'].reshape(nslab, nz, ny, nx), (3, 2, 1, 0))[:, :, :, np.newaxis, :]
        if fuse:
            self.fused = {'flux': None if flux is None else [flux[0], flux[1], flux[2]],
                          'radiance': None if rad is None else [rad],
                          'heating': None if heat is None else [heat]}
            for key, name, extra in (('jac', 'jacobian', 'jac_extra'), ('plen', 'path_length', 'plen_extra')):
                if res.get(key) is None:
                    continue
                # [nslab][sum_k nyr_k * nxr_k][ngrp or ntp+3] -> (nxr, nyr, ngrp or ntp+3, 1, nslab) per sensor
                jr = np.asarray(res[key]).reshape(nslab, scene.rad_size(1), -1)
                ng = jr.shape[-1]
                off, views = 0, []
                for k in range(scene.struct.nrad):
                    sk = scene.sensors[k]
                    nk = sk.nxr * sk.nyr
                    views.append(np.transpose(jr[:, off:off + nk].reshape(nslab, sk.nyr, sk.nxr, ng), (2, 1, 3, 0)))
                    off += nk
                self.fused[name] = [views[0][:, :, :, np.newaxis, :]]
                setattr(self, extra, views[1:])
            if res.get('act') is not None:
                # [nslab][2][nz][ny][nx] -> (nx, ny, nz, 2, nslab)
                self.fused['actinic'] = [np.transpose(np.asarray(res['act']).reshape(nslab, 2, nz, ny, nx), (4, 3, 2, 1, 0))]
        else:
            self.raw = []
            for ir in range(Nrun):
                row = []
                for ig in range(Ng):
                    j = ir * Ng + ig
                    fields = []
                    if flux is not None:
                        fields += [flux[0][..., j].astype(np.float32), flux[1][..., j].astype(np.float32), flux[2][..., j].astype(np.float32)]
                    if rad is not None:
                        fields += [rad[..., j].astype(np.float32)]
                    if heat is not None:
                        fields += [heat[..., j].astype(np.float32)]
                    row.append(fields)
                    if self.write_files:
                        names = []
                        if flux is not None:
                            names += [('a1', 'Fdn0 downward direct flux density'), ('a2', 'Fdn downward total flux density'), ('a3', 'Fup upward flux density')]
                        if rad is not None:
                            names += [('b1', 'Radiance')]
                        if heat is not None:
                            names += [('c1', 'Absorbed flux per layer')]
                        write_mca_out_raw(self.fnames_out[ir][ig], [(nm, ds, f[..., 0]) for (nm, ds), f in zip(names, fields)])
                self.raw.append(row)

    def run_check(self):
        if self.fused is None and self.raw is None:
            missing = [f for row in self.fnames_out for f in row if not os.path.exists(f)]
            if missing:
                raise OSError('Error [mcarats_ng]: Missing some output files.')

    def print_info(self):
        """One-paragraph summary of the run (the reference prints a boxed banner here, mcarats.py:486-523)."""
        rows = [('simulation', '%s %s' % (self.solver, self.target)),
                ('wavelength', str(self.wvl_info)),
                ('date', '%s (day of year %d)' % (self.date.strftime('%Y-%m-%d'), self.date.timetuple().tm_yday)),
                ('sun', 'zenith %.4f deg, azimuth %.4f deg (from north, clockwise)' % (self.solar_zenith_angle, self.solar_azimuth_angle))]
        if self.target == 'radiance':
            rows.append(('sensor', 'zenith %.4f deg (%s), azimuth %.4f deg, altitude %.1f km' % (
                self.sensor_zenith_angle, 'looking down' if self.sensor_zenith_angle < 90.0 else 'looking up',
                self.sensor_azimuth_angle, self.sensor_altitude / 1000.0)))
        rows.append(('surface', '2-D map' if self.sfc_2d else 'Lambertian, albedo %.2f' % self.surface_albedo))
        rows.append(('phase function', 'Henyey-Greenstein' if self.sca is None else self.sca.pha.ID))
        if (self.Nx > 1) or (self.Ny > 1):
            rows.append(('domain', '%d x %d columns of %.2f km x %.2f km' % (self.Nx, self.Ny, self.dx / 1000.0, self.dy / 1000.0)))
        rows.append(('photons', '%.1e per set (%s over %d g) x %d sets' % (self.photons_per_set, self.np_mode, self.Ng, self.Nrun)))
        rows.append(('solver', 'in-process CUDA (sm_100a), device %d' % self.device))
        width = max(len(k) for k, _ in rows)
        print('Message [mcarats_ng]: run summary')
        for k, v in rows:
            print('    %s : %s' % (k.rjust(width), v))


def jacobian_edges(gas_jacobian, zgrd_m):
    """Layer-group edges (layer indices, 0 ... nz) of `mcarats_ng(gas_jacobian=...)`: True gives one group per layer; a
    sequence of level heights in km, which must be levels of the atmosphere (`zgrd_m`, metres) and include its bottom and
    top, gives the contiguous groups between them."""
    zgrd_m = np.asarray(zgrd_m, dtype=np.float64)
    nz = zgrd_m.size - 1
    if gas_jacobian is True:
        edges = np.arange(nz + 1)
    else:
        try:
            lev = np.asarray(gas_jacobian, dtype=np.float64).ravel() * 1000.0
        except (TypeError, ValueError):
            raise OSError('Error [mcarats_ng]: <gas_jacobian> must be True or a sequence of level heights in km.')
        if lev.size < 2 or np.any(np.diff(lev) <= 0.0):
            raise OSError('Error [mcarats_ng]: <gas_jacobian> levels must be at least two strictly increasing heights in km.')
        idx = np.abs(lev[:, None] - zgrd_m[None, :]).argmin(axis=1)
        if np.any(np.abs(zgrd_m[idx] - lev) > 1e-6 * np.maximum(1.0, np.abs(lev))):
            raise OSError('Error [mcarats_ng]: <gas_jacobian> levels must be levels of the atmosphere (Atm_zgrd0).')
        if idx[0] != 0 or idx[-1] != nz:
            raise OSError('Error [mcarats_ng]: <gas_jacobian> levels must include the bottom and the top of the atmosphere.')
        edges = idx
    if edges.size - 1 > 64:
        raise OSError('Error [mcarats_ng]: <gas_jacobian> supports at most 64 layer groups (%d asked for).' % (edges.size - 1))
    return edges.astype(np.int32)


def path_length_bins(path_length):
    """(tpmin, tpmax, ntp), tpmin and tpmax in metres, of `mcarats_ng(path_length=(tpmin_km, tpmax_km, ntp))`:
    1 <= ntp <= 1024, 0 <= tpmin < tpmax, finite."""
    try:
        lo, hi, n = path_length
        lo, hi = float(lo) * 1000.0, float(hi) * 1000.0
        ntp = int(n)
    except (TypeError, ValueError):
        raise OSError('Error [mcarats_ng]: <path_length> must be (tpmin_km, tpmax_km, ntp).')
    if ntp != n or not 1 <= ntp <= 1024:
        raise OSError('Error [mcarats_ng]: <path_length> needs an integer number of bins ntp, 1 ... 1024.')
    if not (np.isfinite(lo) and np.isfinite(hi) and 0.0 <= lo < hi):
        raise OSError('Error [mcarats_ng]: <path_length> needs finite 0 <= tpmin_km < tpmax_km.')
    return lo, hi, ntp


def cal_mca_azimuth(normal_azimuth_angle):
    """Compass azimuth (0 = north, clockwise) -> MCARaTS azimuth 270 - az in [0, 360): the direction of travel counted
    counter-clockwise from +x = east (er3t/rtm/mca/mcarats.py:527-549)."""
    while normal_azimuth_angle < 0.0:
        normal_azimuth_angle += 360.0
    while normal_azimuth_angle > 360.0:
        normal_azimuth_angle -= 360.0
    mca_azimuth = 270.0 - normal_azimuth_angle
    if mca_azimuth < 0.0:
        mca_azimuth += 360.0
    return mca_azimuth


def distribute_photon(Nphoton, weights, base_ratio=0.05):
    """Photons per g: int(N (1 - b) w_g) + int(N b / Ng); the remainder goes to the g with the smallest weight (or is
    taken from the largest when negative) (er3t/rtm/mca/mcarats.py:553-565)."""
    weights = np.asarray(weights)
    Ndist = weights.size
    photons_dist = np.int_(Nphoton * (1.0 - base_ratio) * weights) + np.int_(Nphoton * base_ratio / Ndist)
    Ndiff = Nphoton - photons_dist.sum()
    if Ndiff >= 0:
        photons_dist[np.argmin(weights)] += Ndiff
    else:
        photons_dist[np.argmax(weights)] += Ndiff
    return photons_dist
