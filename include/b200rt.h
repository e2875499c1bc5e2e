/*
 * b200rt.h -- C-ABI of the in-process photon-transport solver that replaces the
 * `mcarats <nphotons> <solver> <input.txt> <output.bin>` subprocess of er3t.rtm.mca.
 *
 * What each entry point replaces in the reference (paths relative to the er3t repo):
 *   b200rt_create / b200rt_destroy   <- process spawn per job, er3t/rtm/mca/mca_run.py:110-113,179-181
 *   b200rt_upload_scene              <- namelist text + 3 binaries written per job
 *                                       (er3t/rtm/mca/mca_inp.py:636-697, mca_atm.py:373-392,
 *                                        mca_sca.py:82-95, mca_sfc.py:136-146)
 *   b200rt_run                       <- mp.Pool.imap(execute_command) over Nrun*Ng jobs,
 *                                       er3t/rtm/mca/mca_run.py:144-159 (photon counts, solver mode,
 *                                       per-job seed of mcarats.py:432-437)
 *   b200rt_run_kd                    <- MCARaTS's multi-term mode (Atm_nkd > 1, Atm_wkd0; Iwabuchi and Okamura 2017):
 *                                       one job per run serves all Ng terms of a wavelength
 *   b200rt_run_jac                   <- finite differences of whole runs with the gas absorption of a layer group
 *                                       scaled (no counterpart in MCARaTS: Rad_mplen stays 0, as er3t sets it)
 *   b200rt_run_plen                  <- MCARaTS's path-length statistics (Rad_mplen, Rad_ntp, Rad_tpmin, Rad_tpmax),
 *                                       which er3t switches off (Rad_mplen = 0); own layout, not MCARaTS's record
 *   b200rt_run_act                   <- nothing: MCARaTS reports no actinic flux (mean radiance); own definition and layout
 *   b200rt_read_flux / _rad / _heat  <- `.bin` + `.ctl` parsing, er3t/rtm/mca/mca_out.py:48-103
 *                                       (and, through job.flx_scale / job.rad_scale, the g-weighting of
 *                                        mca_out.py:319-327,354-366,444-452,475-481)
 *   b200rt_stats                     <- nothing (the reference discards the exit status, mca_run.py:181)
 *   b200rt_last_error                <- OSError('Missing some output files'), mcarats.py:471-483
 *
 * Conventions (SURVEY.md Appendix B): metres; x east, y north, z up; 3-D arrays are laid out
 * [component][iz3][iy][ix] with ix fastest (the reference's Fortran order, mca_atm.py:383-388);
 * angles in degrees; `the`/`phi` are polar/azimuth of the PROPAGATION (source) or VIEWING (sensor)
 * vector (mcarats.py:305-306,382-383).
 *
 * Every input pointer may be a host pointer or a CUDA device pointer (the library copies with
 * cudaMemcpyDefault into its own packed layout and keeps no caller pointer after the call returns).
 * Outputs are copied into caller-owned buffers (host or device) by the b200rt_read_* calls.
 * No torch / C++ types cross this boundary.
 */
#ifndef B200RT_H
#define B200RT_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200RT_VERSION 103 /* 0.1.3: scene.cer3d + (ref, ssa, asy) tables: (omega, apf) of the 3-D field derived on the GPU; Atm_abst3d
                              supported; options.kernel; b200rt_run stream-asynchronous (one run in flight per handle) */

/* error codes (0 = ok, negative = failure; message via b200rt_last_error) */
enum {
    B200RT_OK            = 0,
    B200RT_ERR_ARG       = -1, /* invalid argument / inconsistent scene            */
    B200RT_ERR_CUDA      = -2, /* CUDA runtime error (never swallowed)             */
    B200RT_ERR_STATE     = -3, /* call order (e.g. run before upload_scene)        */
    B200RT_ERR_NUMERIC   = -4, /* NaN/Inf found in tallies                         */
    B200RT_ERR_NOMEM     = -5
};

/* surface types: Sfc_mtype / Sfc_jsfc2d of er3t/rtm/mca/mca_sfc.py:94,112,126 */
enum { B200RT_SFC_LAMBERT = 1, B200RT_SFC_DSM = 2, B200RT_SFC_RPV = 3, B200RT_SFC_LSRT = 4 };

/* solver modes: er3t/rtm/mca/mcarats.py:450-454 */
enum { B200RT_SOLVER_3D = 0, B200RT_SOLVER_PARTIAL_3D = 1, B200RT_SOLVER_IPA = 2 };

/* target bit flags: Wld_mtarget / Flx_mflx / Flx_mhrt of mcarats.py:267-287 */
enum { B200RT_TARGET_FLUX = 1, B200RT_TARGET_RADIANCE = 2, B200RT_TARGET_HEATING = 4 };

/* One radiance sensor (Rad_* of mcarats.py:285-307; docs er3t/rtm/mca/mca_inp.py:141-171,305-364).
 * kind 2 = "2nd kind": radiance averaged over the horizontal cross-section of a column,
 * parallel projection along the viewing vector; pixel = where the line of sight meets z = zref.
 * kind 1 = "1st kind" (all-sky camera, mcarats.py:291-296,369-371): local radiance at the point
 * (xpos * Lx, ypos * Ly, zloc) averaged over the solid angle of each pixel; camera frame = Z-Y-Z rotation by
 * (phi, the, psi), the camera looks along its +z axis (the, phi as for kind 2); field of view = cone of FULL
 * angle qmax; polar pixel mapping (Rad_mpmap = 1): U = theta cos(az), V = theta sin(az) with U in
 * [-umax/2, umax/2], V in [-vmax/2, vmax/2] (degrees) spread over nxr x nyr pixels. */
typedef struct b200rt_sensor {
    int32_t kind;       /* Rad_mrkind: 2 (satellite) or 1 (all-sky camera)                      */
    int32_t nxr, nyr;   /* Rad_nxr, Rad_nyr                                                     */
    int32_t _pad;
    double  the, phi;   /* Rad_the (=180-vza), Rad_phi (=270-vaa): viewing vector               */
    double  zloc;       /* Rad_zloc: sensor altitude (m); >= TOA means "above the atmosphere"   */
    double  zref;       /* Rad_zref: reference level for pixel registration (m), default 0      */
    /* kind 1 only */
    double  psi;        /* Rad_psi: rotation about the camera axis (deg)                        */
    double  xpos, ypos; /* Rad_xpos, Rad_ypos: relative position in the domain, 0 ... 1         */
    double  qmax;       /* Rad_qmax: full angle of the field-of-view cone (deg)                 */
    double  umax, vmax; /* Rad_umax, Rad_vmax: full angular width of the pixel grid (deg)       */
    double  apsize;     /* Rad_apsize: aperture size (m): lower bound of the distance in 1/R^2  */
} b200rt_sensor;

/* The scene = everything that is identical for all (run, g) jobs (SURVEY.md Appendix B,
 * "Per-g differences": only Atm_abs1d and the seed differ between jobs). */
typedef struct b200rt_scene {
    /* grid: Atm_nx, Atm_ny, Atm_nz, Atm_dx, Atm_dy, Atm_zgrd0, Atm_iz3l (1-based), Atm_nz3 */
    int32_t nx, ny, nz;
    int32_t iz3l, nz3;            /* nz3 == 0: no 3-D block                                    */
    int32_t np1d, np3d;           /* Atm_np1d, Atm_np3d                                        */
    int32_t layout3d;             /* memory order of ext3d/omg3d/apf3d: 0 = [np3d][nz3][ny][nx] (the reference's file
                                     order, x fastest); 1 = C order of the reference's in-memory arrays
                                     (nx, ny, nz3, np3d) (mca_atm.py:248-252), transposed on the GPU */
    double  dx, dy;               /* m                                                         */
    const double* zgrd;           /* [nz+1] level heights, m, strictly increasing              */
    /* 1-D components, mca_atm.py:85-139 */
    const double* ext1d;          /* [np1d][nz] 1/m                                            */
    const double* omg1d;          /* [np1d][nz]                                                */
    const double* apf1d;          /* [np1d][nz]  -1 Rayleigh | (-1,1) HG g | >=1 table index   */
    /* 3-D components, mca_atm.py:248-337 (float32 exactly as the reference stores them) */
    const float*  ext3d;          /* 1/m, see layout3d                                         */
    const float*  omg3d;
    const float*  apf3d;
    const float*  abs3d;          /* [nz3][ny][nx] Atm_abst3d: absorption coefficient added inside the 3-D block, 1/m,
                                     >= 0 (treated as one more component with omega = 0); may be NULL            */
    /* tabulated phase functions, mca_sca.py:82-95 */
    int32_t npf, nang;            /* Sca_npf, Sca_nangi (npf == 0: none)                       */
    const double* ang;            /* [nang] scattering angle, degrees, increasing from 0 to 180 */
    const double* pha;            /* [npf][nang] phase function (any normalisation)            */
    /* surface, mcarats.py:386-414 and mca_sfc.py:81-146 */
    int32_t sfc_nx, sfc_ny;       /* Sfc_nxb, Sfc_nyb; 1 x 1 = uniform                         */
    const int32_t* sfc_type;      /* [sfc_ny][sfc_nx]                                          */
    const float*   sfc_param;     /* [5][sfc_ny][sfc_nx]  (Sfc_psfc2d, parameter index slowest) */
    /* source, mcarats.py:374-383 */
    double src_the, src_phi;      /* Src_the (=180-sza), Src_phi (=270-saa)                    */
    double src_qmax;              /* full cone angle, degrees                                  */
    double src_flx;               /* flux density normal to the beam                           */
    /* sensors */
    int32_t nrad;                 /* Rad_nrad                                                  */
    int32_t _pad1;
    const b200rt_sensor* sensors; /* [nrad] host pointer                                       */
    /* Optional: let the library derive (omega, apf) of the (single) 3-D component from the droplet effective radius,
     * exactly as mca_atm_3d does on the host (er3t/rtm/mca/mca_atm.py:291-303): voxels with ext > 0 get
     * omega = interp(ssa_tab)(cer), apf = interp(asy_tab)(cer) (linear, linearly extrapolated: Henyey-Greenstein with
     * the Mie asymmetry parameter); clear voxels get omega = 1, apf = -1.  omg3d / apf3d are ignored (may be NULL). */
    const float*  cer3d;          /* same layout as ext3d (np3d must be 1), um; NULL = use omg3d / apf3d */
    int32_t nref;                 /* entries of the three tables (>= 2)                          */
    int32_t _pad2;
    const double* ref_tab;        /* [nref] effective radius, strictly increasing; host pointer  */
    const double* ssa_tab;        /* [nref] single-scattering albedo                             */
    const double* asy_tab;        /* [nref] asymmetry parameter                                  */
} b200rt_scene;

/* One (run, g) job = one MCARaTS invocation of the reference (mca_run.py:110-113). */
typedef struct b200rt_job {
    int64_t  nphot;               /* photons of this job (whole job, before sharding)          */
    uint64_t seed;                /* Philox key; Wld_jseed of mcarats.py:437                   */
    int32_t  slab;                /* output slab the job accumulates into (run index, or job index for raw output) */
    int32_t  _pad;
    const double* abs1d;          /* [nz] gas absorption coefficient 1/m (Atm_abs1d(1:,1)), NULL = 0; host pointer */
    const double* flx_scale;      /* [nz+1] per-level factor (mca_out.py:324-327), NULL = 1; host pointer;
                                     entry iz also scales the heating tally of layer iz                             */
    double   rad_scale;           /* factor for radiance (mca_out.py:449-452, iz = 0)          */
} b200rt_job;

/* Atm_nkd k-distribution terms of one job (b200rt_run_kd): gas absorption never changes a trajectory, so one history
 * serves every term.  Run r estimates sum_g rad_scale[g] * E[radiance of term g]; Russian roulette and the energy sums of
 * b200rt_stats act on the term-weighted weight W = w * sum_g q_g exp(-T_g), q_g = wkd[g] / sum(wkd), T_g = the history's
 * gas-absorption optical path in term g. */
typedef struct b200rt_kd {
    int32_t nkd, _pad;              /* 1 ... 32                                                                        */
    const double* wkd;              /* [nkd] Atm_wkd0: weights of roulette and energy sums (normalised by the library) */
    const double* abs1d;            /* [nkd][nz] gas absorption per term, 1/m, host pointer                            */
    const double* rad_scale;        /* [nkd] per-term radiance factor                                                  */
} b200rt_kd;

typedef struct b200rt_options {
    int32_t solver;               /* B200RT_SOLVER_*                                           */
    int32_t target;               /* OR of B200RT_TARGET_*                                     */
    int32_t nslab;                /* number of output slabs                                    */
    int32_t shard_rank;           /* this process handles photon indices i with               */
    int32_t shard_world;          /*   i % shard_world == shard_rank  (1 GPU: 0 / 1)           */
    int32_t svx, svy, svz;        /* fine majorant cell in voxels / layers; 0 = auto           */
    int32_t cmx, cmy, cmz;        /* coarse (empty-space) cell in fine cells (x, y: power of two); 0 = auto */
    int32_t flight_steps;         /* max cell crossings per lane in one flight phase; 0 = auto      */
    int32_t event_min;            /* lanes parked at an event that end a flight phase early; 0 = auto */
    int32_t empty_runs;           /* vertical merging of empty coarse cells into one box: 0 = auto (on when the 3-D
                                     layers are equally thick and no per-level tally is asked for), -1 = off        */
    int32_t pool_slots;           /* photon slots in shared memory per warp: 64, 96 or 128; 0 = auto (96)             */
    int32_t iso_ss;               /* Pho_iso_SS: partial-3D switches to 1-D after this order   */
    int32_t iso_max;              /* Pho_iso_max: max scattering order sampled (0 = 1e6)       */
    int32_t threads_per_block;    /* 0 = auto                                                  */
    int32_t blocks_per_sm;        /* 0 = auto                                                  */
    int32_t smem_tally;           /* block-private tallies in shared memory for plane-parallel and few-column (<= 64 columns)
                                     scenes whose whole flux + heating tally is <= 2048 doubles (radiance: <= 512): lanes of a
                                     warp that hit the same address are summed first, one flush per block.  0 = auto (on),
                                     -1 = off (global atomics only), 2 = additionally one private copy per warp           */
    int32_t kernel;               /* transport kernel: 0 = auto (8), 8 = every warp runs every phase on its own photon pool;
                                     other values are rejected at upload                                               */
    int32_t _reserved;
    double  wmin;                 /* Pho_wmin: Russian roulette threshold (0 = no roulette)    */
    double  wfac;                 /* Pho_wfac: weight given to roulette survivors              */
} b200rt_options;

/* Event counters: the inputs of the algorithmic-bytes formula of SURVEY.md 8(d). */
typedef struct b200rt_stats {
    uint64_t photons;             /* histories started on this GPU                             */
    uint64_t n_cell;              /* majorant-cell visits (4 B each)                           */
    uint64_t n_tent;              /* tentative collisions = voxel extinction look-ups (4 B)    */
    uint64_t n_coll;              /* real collisions (8 B: omega + apf)                        */
    uint64_t n_sfc;               /* surface hits                                              */
    uint64_t n_le;                /* local-estimate rays                                       */
    uint64_t n_le_visit;          /* voxels crossed (or table look-ups) by local-estimate rays */
    uint64_t n_tally;             /* tally updates that reached global memory (8 B)            */
    uint64_t n_roulette_kill;
    double   w_toa_up;            /* sum of weights leaving through TOA   (R * photons)        */
    double   w_sfc_abs;           /* sum of weights absorbed by surface   (T_net * photons)    */
    double   w_atm_abs;           /* sum of weights absorbed in atmosphere (A * photons)       */
    double   w_roulette;          /* net weight created(+)/destroyed(-) by roulette + cut-offs */
    double   elapsed_ms;          /* device time of the last b200rt_run (CUDA events)          */
    double   bytes_alg;           /* algorithmic bytes of the last run (SURVEY.md 8d formula)  */
    uint64_t launches;            /* kernels launched by the last b200rt_run                   */
} b200rt_stats;

int          b200rt_version(void);
int          b200rt_create(void** handle, int device);
int          b200rt_destroy(void* handle);
const char*  b200rt_last_error(void* handle);

/* Copy + repack the scene into HBM; builds majorant grid, phase-function CDFs, tau-to-sensor
 * tables. May be called again to replace the scene. */
int          b200rt_upload_scene(void* handle, const b200rt_scene* scene, const b200rt_options* opt);

/* Trace all jobs asynchronously on `cuda_stream` (a cudaStream_t or NULL for the default stream): the per-job tables are
 * staged in page-locked memory and uploaded with cudaMemcpyAsync on that stream, nothing in the call waits for the GPU.
 * Tallies are zeroed first unless `accumulate` != 0.  ONE run may be in flight per handle: a second b200rt_run,
 * b200rt_upload_scene or b200rt_read_* first waits for the stream of the run in flight. */
int          b200rt_run(void* handle, const b200rt_job* jobs, int njob, int accumulate, void* cuda_stream);

/* b200rt_run with kd[j] the k-distribution terms of jobs[j] (radiance target with satellite sensors only: flux / heating
 * targets and the all-sky camera are rejected).  jobs[j].abs1d and .flx_scale must be NULL; jobs[j].rad_scale is a factor
 * common to all terms.  Same asynchronous contract as b200rt_run. */
int          b200rt_run_kd(void* handle, const b200rt_job* jobs, const b200rt_kd* kd, int njob, int accumulate, void* cuda_stream);

/* b200rt_run that also tallies the radiance's derivatives with respect to the gas absorption of ngrp layer groups:
 * jac = dI / dln(a_j), where a_j multiplies jobs[].abs1d of layers edges[j] ... edges[j+1]-1 (host array of ngrp+1 layer
 * indices, 0 = edges[0] < ... < edges[ngrp] = nz, 1 <= ngrp <= 64).  Estimated inside the same histories, without bias:
 * every local estimate with contribution c (as tallied into the radiance) adds -c (T_j + tau_j) to pixel and group j, where
 * T_j is the gas optical path the history has collected in group j and tau_j that of the segment toward the sensor.  The
 * radiance, draws and event counters are those of b200rt_run (stats.n_tally also counts the Jacobian updates).  Atm_abst3d
 * and particle absorption are not differentiated.  Radiance target with satellite sensors only (flux / heating targets,
 * options.smem_tally >= 0 on scenes whose radiance tally fits shared memory and the all-sky camera are rejected).  With
 * accumulate != 0 the previous run since the last upload, if any, must be a Jacobian run with the same edges.  Same
 * asynchronous contract as b200rt_run. */
int          b200rt_run_jac(void* handle, const b200rt_job* jobs, int njob, const int32_t* edges, int ngrp, int accumulate,
                            void* cuda_stream);

/* b200rt_run that also tallies the distribution of the photon path lengths behind every radiance pixel.  L (metres) is
 * the geometric path of one local-estimate contribution c (as tallied into the radiance, job.rad_scale and the pixel
 * factor included): from the photon's entry at TOA along every leg of its history to the event, then along the
 * event -> sensor segment to the sensor's target level min(Rad_zloc, TOA).  Per pixel the tally holds ntp + 3 doubles:
 *   0 ... ntp-1  c summed into uniform bins of width (tpmax - tpmin) / ntp on [tpmin, tpmax)
 *   ntp          underflow, L < tpmin
 *   ntp + 1      overflow, L >= tpmax
 *   ntp + 2      the first moment, sum of c L
 * so that entries 0 ... ntp+1 sum to the radiance and <L> = moment / radiance.  The bin index is computed in fp32 from
 * the fp32 path.  1 <= ntp <= 1024, 0 <= tpmin < tpmax, all finite.  The radiance, draws and event counters are those of
 * b200rt_run (stats.n_tally also counts the two updates per local estimate).  Radiance target with satellite sensors only,
 * every solver mode (flux / heating targets, options.smem_tally >= 0 on scenes whose radiance tally fits shared memory,
 * and the all-sky camera are rejected).  With accumulate != 0 the previous run since the last upload, if any, must be a
 * path-length run with the same tpmin, tpmax and ntp.  Same asynchronous contract as b200rt_run. */
int          b200rt_run_plen(void* handle, const b200rt_job* jobs, int njob, double tpmin, double tpmax, int ntp, int accumulate,
                             void* cuda_stream);

/* b200rt_run that also tallies the actinic flux (spherical irradiance, F_act = integral of the radiance over 4 pi sr) as
 * the volume mean over every layer iz and atmosphere column, from the track length of every flight move in the voxel:
 * sum of the integral of the weight along the track / dz, the weight falling with the layer's gas absorption along it.
 * Same units and per-job factors as the flux (job.flx_scale of layer iz included): per unit Src_flx normal to the beam,
 * so that a direct beam in vacuum gives Src_flx.  Two variables: 0 direct (photons that have not scattered), 1 total.
 * Trajectories never change, so flux, heating, draws and event counters are those of b200rt_run (stats.n_tally also
 * counts the actinic updates that go to global memory).  Flux and / or heating target only: radiance sensors in the same
 * run and the all-sky camera are rejected.  With accumulate != 0 the previous run since the last upload, if any, must be
 * an actinic run.  Same asynchronous contract as b200rt_run. */
int          b200rt_run_act(void* handle, const b200rt_job* jobs, int njob, int accumulate, void* cuda_stream);

/* Wait for the stream of the last run; checks tallies for NaN/Inf. */
int          b200rt_sync(void* handle);

/* Output dims: flux [nslab][3][nz+1][ny][nx] (0 direct-down, 1 total-down, 2 up; mca_out.py:350-352),
 * radiance [nslab][nrad][nyr][nxr], heating [nslab][nz][ny][nx] (absorbed power per unit area per layer).
 * `dst` is a host or device pointer to doubles; `count` = number of doubles the caller provides. */
int          b200rt_read_flux(void* handle, double* dst, int64_t count);
int          b200rt_read_rad (void* handle, double* dst, int64_t count);
int          b200rt_read_heat(void* handle, double* dst, int64_t count);
/* Jacobian tally of the last run, which must have been a b200rt_run_jac: [nslab][nrad][nyr][nxr][ngrp] (group fastest),
 * count = doubles the caller provides.  b200rt_jac_ptr: its device pointer and size (in-place NCCL all-reduce). */
int          b200rt_read_jac(void* handle, double* dst, int64_t count);
int          b200rt_jac_ptr(void* handle, double** p, int64_t* n);
/* Path-length tally of the last run, which must have been a b200rt_run_plen: [nslab][nrad][nyr][nxr][ntp+3] (bin
 * fastest).  b200rt_plen_ptr: its device pointer and size. */
int          b200rt_read_plen(void* handle, double* dst, int64_t count);
int          b200rt_plen_ptr(void* handle, double** p, int64_t* n);
/* Actinic flux of the last run, which must have been a b200rt_run_act: [nslab][2][nz][ny][nx] (variable 0 direct, 1 total;
 * laid out like the heating tally with the variable axis added).  b200rt_act_ptr: its device pointer and size. */
int          b200rt_read_act(void* handle, double* dst, int64_t count);
int          b200rt_act_ptr(void* handle, double** p, int64_t* n);
/* Device pointers to the library-owned tallies (for in-place NCCL all-reduce by the caller). */
int          b200rt_tally_ptrs(void* handle, double** flux, int64_t* nflux, double** rad, int64_t* nrad,
                               double** heat, int64_t* nheat);

int          b200rt_stats_get(void* handle, b200rt_stats* out);

/* Diagnostics / test hooks (bit-exact against oracle/): */
/* Philox4x32-10: out[4*i..4*i+3] = philox(key=(seed_lo,seed_hi), ctr=(i_lo,i_hi,c2,c3)). */
int          b200rt_philox_fill(void* handle, uint64_t seed, uint64_t first, uint32_t c2, uint32_t c3,
                                uint32_t* out_host, int64_t n);
/* Evaluate the normalised phase function / sample cos(theta) exactly as the kernel does. */
int          b200rt_phase_eval(void* handle, double apf, const double* mu, double* p_out, int64_t n);
int          b200rt_phase_sample(void* handle, double apf, const double* xi, double* mu_out, int64_t n);
/* Surface BRDF value f_r(in -> out) [1/sr] as the kernel evaluates it for local estimates. */
int          b200rt_brdf_eval(void* handle, int32_t type, const float* param5,
                              const double* dir_in3, const double* dir_out3, double* f_out, int64_t n);

#ifdef __cplusplus
}
#endif
#endif /* B200RT_H */
