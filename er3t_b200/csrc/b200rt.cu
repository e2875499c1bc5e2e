// b200rt.cu -- sm_100a photon-transport solver behind the C-ABI of include/b200rt.h.
//
// Replaces the external MCARaTS process that er3t launches at er3t/rtm/mca/mca_run.py:110-113,179-181.
// Kernels (DESIGN.md has the roofline of each):
//   pack_scene_tiled_kernel per-voxel total extinction + (omega, apf) records, tiled (ix, k) transpose of the caller's
//                          C-order fields, (omega, apf) optionally derived from the effective radius  (HBM streaming)
//   pack_scene_kernel      the same for any other layout / several components / Atm_abst3d           (HBM streaming)
//   majorant_kernel, empty_kernel, run_kernel, mark_empty_kernel
//                          fine majorant grid, coarse emptiness, vertical runs of empty cells        (HBM streaming)
//   tau_up_kernel          optical depth from each voxel to the top of the 3-D block (vertical local estimates)
//   transport_kernel       persistent-thread photon transport with in-place regeneration, Philox streams,
//                          two-level majorant grid + null-collision tracking, local-estimate radiance, fp64 tallies
//                          (and, on request, track-length actinic flux, radiance Jacobians, path-length distributions)
//   check_finite_kernel    NaN/Inf guard over the tallies
// No CPU fallback exists: every entry point fails with an error code if CUDA fails.

#include "../../include/b200rt.h"
#include "rt_device.cuh"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#define MAX_SENS 16
// Launch shape of the transport kernel.  Warps are independent (per-warp photon pools, no block-level synchronisation
// after the table staging), so the block size only sets the granularity.  A B200 SM sub-partition holds 16 K registers:
// 5 warps per scheduler need <= 96 registers per thread (tools/sweep_pool.py: 20 warps/SM at 96 registers beat 16 warps
// at 123 registers by 4.5 % although ptxas then spills a few words per thread; 22 or 24 warps at 80 registers lose 30 %,
// profiles/README.md).  Shared memory per block: 82.6 KB of pools + tables + accumulators = 92.8 KB on config 2, so two
// blocks stay under the 200 KB carve-out and ~56 KB of L1 remain for the voxel / majorant gathers.
#ifndef RT_TPB
#define RT_TPB 320
#endif
#ifndef RT_MINB
#define RT_MINB 2
#endif

// ============================================================================ device structs
struct DevSensor {
    float3 s;            // direction of photon travel toward the sensor (= -viewing vector)
    float inv_sz;        // 1 / |s.z|
    float inv_szs;       // 1 / s.z (signed)
    float zt;            // target level of the transmittance integral: clamp(zloc, z0, ztoa)
    float zref;
    int lt;              // layer that contains zt (nz-1 when zt == ztoa)
    int nxr, nyr;
    int vertical_up;     // s == (0,0,1): precomputed tau-to-top table applies in 3-D mode
    int fast_ok;         // zt is at/above the top of the 3-D block
    long long off;       // offset of this sensor inside a radiance slab
    double npix;         // kind 2: nxr * nyr ; kind 1: domain area Lx * Ly (m^2)
    // all-sky camera (kind 1): `s` is the viewing axis, (ex, ey) complete the camera frame
    int kind;
    float3 cpos, ex, ey;
    float cos_half_fov;  // cos(qmax / 2)
    float u_half, v_half;        // umax / 2, vmax / 2 (rad)
    float pix_per_u, pix_per_v;  // nxr / umax, nyr / vmax (pixels per rad)
    float ap2;           // apsize^2
};

struct DevJob {
    unsigned long long first;   // prefix sum of local photon counts
    unsigned long long count;   // photons of this job handled by this GPU
    unsigned long long seed;
    double norm;                // mu0 * src_flx / nphot(job, all GPUs)
    double rad_fac;             // norm * rad_scale
    int slab;
    int has_abs;
    int has_fscale;
    int _pad;
    unsigned long long flux_off;   // slab * 3 * (nz + 1) * nx * ny: start of the job's slab in the flux tally
    unsigned long long heat_off;   // slab * nz * nx * ny
};

struct DevStats {
    unsigned long long photons, n_cell, n_tent, n_coll, n_sfc, n_le, n_le_visit, n_tally, n_kill;
    double w_toa, w_sfc, w_atm, w_rr;
};

struct DevScene {
    int nx, ny, nz, iz0, nz3, np1d, np3d;
    float dx, dy, Lx, Ly, inv_dx, inv_dy, inv_Lx, inv_Ly;
    int svx, svy, svz, ncx, ncy, ncz;
    unsigned svx_mul, svy_mul;   // fine column -> fine cell without a divide: fx / svx == div_exact(fx, svx_mul, svx_sh)
    int svx_sh, svy_sh;
    float Sx, Sy, inv_Sx, inv_Sy;
    float Lux, Luy;           // domain size in units of fine cells (nx / svx, ny / svy; the last cell may be partial)
    int nslab_z;
    int ngroup;               // coarse z groups of fine slabs
    int nCx, nCy, shx, shy;   // coarse (emptiness) grid: 2^shx x 2^shy fine cells per coarse cell
    int flight_steps;         // max cell crossings per lane between two event phases
    int event_min;            // parked lanes that end the flight loop early
    // vertical runs of empty coarse cells (only when the 3-D layers are equally thick): a photon's fine z slab follows
    // from its height by one multiply, so a box may span several coarse z groups
    int uz_ok;                // 1: runs enabled, slab = uz_s0 + clamp(int((z - uz_z0) * uz_inv), 0, ncz - 1)
    int uz_s0;                // index of the first fine slab of the 3-D block
    float uz_z0, uz_inv;
    float maj1d_blk;          // 1-D majorant of the whole 3-D block (used by boxes that span several groups)
    // small flux / heating tallies (plane-parallel and few-column scenes) are kept per block in shared memory and flushed
    // once: all photons would otherwise hammer the same few L2 addresses
    int ntal_flux_smem, ntal_heat_smem;   // doubles of the whole flux / heating tally held in shared memory (0: global atomics)
    int ntal_rad_smem;        // doubles of the whole radiance tally held in shared memory (tiny sensors: 1 x 1-pixel views)
    int tal_per_warp;         // 1: every warp of a block keeps its own copy (very small tallies), 0: one copy per block
    // small 1-D tables (global copies; staged into shared memory by the transport kernel)
    const float* zgrd;        // [nz+1]
    const float* e1tot;       // [nz]
    const float* e1cum;       // [nz+1]
    const float* e1;          // [np1d][nz]
    const float* o1;          // [np1d][nz]
    const float* a1;          // [np1d][nz]
    const int* slab_lay0;     // [nslab_z+1]
    const int* slab_cz;       // [nslab_z]
    const float* slab_maj1d;  // [nslab_z]
    const int* slab_cg;       // [nslab_z]
    const float* group_maj1d; // [ngroup]
    const int* group_lo;      // [ngroup+1]
    const int* group_cz;      // [ngroup]
    const unsigned char* empty3; // [nCz][nCy][nCx] 1 = coarse cell holds no 3-D extinction
    // 3-D block in HBM
    const float* ext3tot;     // [nz3][ny][nx]
    const float2* prop3;      // [np3d][nz3][ny][nx]  (omega, apf)
    const float* ext3;        // [np3d][nz3][ny][nx]  (only read when np3d > 1)
    const float* maj;         // [ncz][ncy][ncx]
    const float* tu3;         // [nz3+1][ny][nx]
    PhaseTab pt;
    int sfc_nx, sfc_ny;
    const int* sfc_type;
    const float* sfc_param;   // [5][sfc_ny][sfc_nx]
    float3 src;
    float src_cos_half, mu0;
    int nrad;
    DevSensor sens[MAX_SENS];
    long long rad_slab;       // doubles per radiance slab
    int solver, target;
    float wmin, wfac;
    int iso_ss, iso_max;
    int shard_rank, shard_world;
    // jobs
    int njob;
    const DevJob* jobs;
    const float* job_abs;     // [njob][nz]
    const float* job_cabs;    // [njob][nz+1]
    const double* job_fscale; // [njob][nz+1]  norm * (columns in the domain) * per-level factor: the complete tally scale
    unsigned long long nphot_local;
    // outputs
    double* flux;
    double* rad;
    double* heat;
    unsigned long long* counter;
    DevStats* stats;
    // spectral runs (b200rt_run_kd, read by the KD kernels only): kd_n gas-absorption terms per job, zero-padded
    int kd_n;
    const float2* kd_tab;     // [njob][nz+2][kd_n] row 0: (normalised Atm_wkd0, 0); row 1 + iz: (cumulative gas optical depth at
                              // level iz, absorption coefficient of layer iz)
    const double* kd_rf;      // [njob][kd_n] norm x job.rad_scale x kd.rad_scale[g]
    float* kd_r;              // [block][warp][pool slot][kd_n] per-term state of the photon in each slot (see kd_leg)
    // radiance Jacobians (b200rt_run_jac, read by the JAC kernels only): jac_n groups of contiguous layers
    int jac_n;
    const int* jac_lev;       // [jac_n+1] group edges as layer indices, 0 = jac_lev[0] < ... < jac_lev[jac_n] = nz
    const unsigned char* jac_grp;   // [nz] group of every layer
    // per-slot state and per-pixel tally of the JAC and PLEN kernels
    float* xs;                // JAC: [block][warp][pool slot][jac_n] gas optical path of the slot's history per group (see jac_leg)
                              // PLEN: [block][warp][pool slot] geometric path of the slot's history so far (m)
    double* xt;               // JAC: [nslab][rad_slab][jac_n] tally of dI / dln(a_j); PLEN: [nslab][rad_slab][pl_ntp+3] (plen_deposit);
                              // ACT: [nslab][2][nz][ny][nx] actinic flux (act_move)
    // path-length distributions (b200rt_run_plen, read by the PLEN kernels only): pl_ntp bins on [pl_lo, pl_hi) metres
    int pl_ntp;
    float pl_lo, pl_hi, pl_inv_w;   // pl_inv_w = pl_ntp / (pl_hi - pl_lo)
    // actinic flux (b200rt_run_act, read by the ACT kernels only): the tally is xt, [nslab][2][nz][ny][nx]; doubles of it held
    // in the block-private shared tally next to flux and heating (0: global atomics)
    int ntal_act_smem;
};

// ============================================================================ setup kernels
// (omega, apf) of a voxel from its droplet effective radius, as mca_atm_3d derives them on the host
// (er3t/rtm/mca/mca_atm.py:291-303: scipy interp1d(..., fill_value='extrapolate') of ssa and asy against the table radii;
// HG with the Mie asymmetry parameter).  fp64 without fused multiply-adds so that the float32 results equal numpy's.
#define CER_MAX 64
struct CerTab {
    int n;
    double ref[CER_MAX], ssa[CER_MAX], asy[CER_MAX];
};
__device__ __forceinline__ float2 cer_props(const CerTab& T, float ext, float cer) {
    if (!(ext > 0.0f)) return make_float2(1.0f, -1.0f);              // clear voxel: conservative Rayleigh placeholder
    const double x = double(cer);
    int lo = 0, hi = T.n;                                            // first index with ref > x  (searchsorted side='right')
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (T.ref[mid] <= x) lo = mid + 1; else hi = mid;
    }
    const int i = min(T.n - 2, max(0, lo - 1));
    const double t = __ddiv_rn(__dsub_rn(x, T.ref[i]), __dsub_rn(T.ref[i + 1], T.ref[i]));
    const double o = __dadd_rn(T.ssa[i], __dmul_rn(t, __dsub_rn(T.ssa[i + 1], T.ssa[i])));
    const double a = __dadd_rn(T.asy[i], __dmul_rn(t, __dsub_rn(T.asy[i + 1], T.asy[i])));
    return make_float2(float(o), float(a));
}

// layout 0: [np3d][nz3][ny][nx] (x fastest, the byte order of the reference's binary file, mca_atm.py:383-388)
// layout 1: numpy C order of the reference's in-memory arrays (nx, ny, nz3, np3d) (mca_atm.py:248-252): no host transpose
// abs3 (optional, [nz3][ny][nx]): Atm_abst3d >= 0 becomes one more component with omega = 0 -- absorption as a collision
// process (implicit capture) instead of the path integral used for the 1-D gas profile; same expectation
// cer (optional, layout of ext, np3d == 1): (omega, apf) from the effective radius instead of omg / apf
__global__ void pack_scene_kernel(const float* __restrict__ ext, const float* __restrict__ omg,
                                  const float* __restrict__ apf, const float* __restrict__ abs3, const float* __restrict__ cer,
                                  const __grid_constant__ CerTab T, int np3d, int nx, int ny, int nz3, int layout,
                                  float* __restrict__ ext3tot, float2* __restrict__ prop3, float* __restrict__ ext3,
                                  int* __restrict__ bad) {
    const size_t nvox = size_t(nz3) * ny * nx;
    const size_t stride = size_t(gridDim.x) * blockDim.x;
    for (size_t v = size_t(blockIdx.x) * blockDim.x + threadIdx.x; v < nvox; v += stride) {
        const int ix = int(v % nx), iy = int((v / nx) % ny), k = int(v / (size_t(nx) * ny));
        float tot = 0.0f;
        for (int c = 0; c < np3d; ++c) {
            const size_t src = layout == 0 ? size_t(c) * nvox + v : ((size_t(ix) * ny + iy) * nz3 + k) * np3d + c;
            const float e = ext[src];
            float2 pr;
            if (cer) {
                const float r = cer[src];
                if (e > 0.0f && !isfinite(r)) atomicOr(bad, 1);
                pr = cer_props(T, e, r);
            } else pr = make_float2(omg[src], apf[src]);
            if (!(e >= 0.0f) || !(pr.x >= 0.0f && pr.x <= 1.0f) || !isfinite(pr.y)) atomicOr(bad, 1);
            tot += e;
            prop3[size_t(c) * nvox + v] = pr;
            if (ext3) ext3[size_t(c) * nvox + v] = e;
        }
        if (abs3) {
            const float e = abs3[v];
            if (!(e >= 0.0f) || !isfinite(e)) atomicOr(bad, 2);
            tot += e;
            prop3[size_t(np3d) * nvox + v] = make_float2(0.0f, 0.0f);
            ext3[size_t(np3d) * nvox + v] = e;
        }
        ext3tot[v] = tot;
    }
}

// The common case -- ONE 3-D component handed over in the reference's in-memory order (nx, ny, nz3) -- as a tiled
// transpose: a 32 x 32 tile of the (ix, k) plane of one iy is read with k fastest (the input's contiguous axis) and
// written with ix fastest (the packed layout's), both as full 128-byte rows.  HBM streaming: 12 B read (or 8 B with
// cer) + 12 B written per voxel.
__global__ void __launch_bounds__(256) pack_scene_tiled_kernel(const float* __restrict__ ext, const float* __restrict__ omg,
                                                               const float* __restrict__ apf, const float* __restrict__ cer,
                                                               const __grid_constant__ CerTab T, int nx, int ny, int nz3,
                                                               float* __restrict__ ext3tot, float2* __restrict__ prop3,
                                                               int* __restrict__ bad) {
    __shared__ float te[32][33];
    __shared__ float2 tp[32][33];
    const int k0 = blockIdx.x * 32, ix0 = blockIdx.y * 32, iy = blockIdx.z;
    const int tx = threadIdx.x, ty = threadIdx.y;           // (32, 8)
    int isbad = 0;
#pragma unroll
    for (int r = 0; r < 32; r += 8) {
        const int ix = ix0 + ty + r, k = k0 + tx;
        if (ix < nx && k < nz3) {
            const size_t src = (size_t(ix) * ny + iy) * nz3 + k;
            const float e = ext[src];
            float2 pr;
            if (cer) {
                const float rr = cer[src];
                if (e > 0.0f && !isfinite(rr)) isbad = 1;
                pr = cer_props(T, e, rr);
            } else pr = make_float2(omg[src], apf[src]);
            if (!(e >= 0.0f) || !(pr.x >= 0.0f && pr.x <= 1.0f) || !isfinite(pr.y)) isbad = 1;
            te[ty + r][tx] = e;
            tp[ty + r][tx] = pr;
        }
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < 32; r += 8) {
        const int k = k0 + ty + r, ix = ix0 + tx;
        if (ix < nx && k < nz3) {
            const size_t v = (size_t(k) * ny + iy) * nx + ix;
            ext3tot[v] = te[tx][ty + r];
            prop3[v] = tp[tx][ty + r];
        }
    }
    if (isbad) atomicOr(bad, 1);
}

__global__ void majorant_kernel(const float* __restrict__ ext3tot, int nx, int ny, int nz3, int svx, int svy, int svz,
                                int ncx, int ncy, int ncz, float* __restrict__ maj) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= ncx * ncy * ncz) return;
    const int cix = c % ncx, ciy = (c / ncx) % ncy, ciz = c / (ncx * ncy);
    float m = 0.0f;
    for (int kz = ciz * svz; kz < min(nz3, (ciz + 1) * svz); ++kz)
        for (int ky = ciy * svy; ky < min(ny, (ciy + 1) * svy); ++ky)
            for (int kx = cix * svx; kx < min(nx, (cix + 1) * svx); ++kx)
                m = fmaxf(m, ext3tot[(size_t(kz) * ny + ky) * nx + kx]);
    maj[c] = m;
}

__global__ void empty_kernel(const float* __restrict__ maj, int ncx, int ncy, int shx, int shy, int nCx, int nCy, int nCz,
                             const int* __restrict__ gz_lo, unsigned char* __restrict__ empty3) {
    // gz_lo[K] .. gz_lo[K+1]: fine z indices (in the majorant grid) covered by coarse z cell K
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= nCx * nCy * nCz) return;
    const int Cx = c % nCx, Cy = (c / nCx) % nCy, Cz = c / (nCx * nCy);
    float m = 0.0f;
    for (int kz = gz_lo[Cz]; kz < gz_lo[Cz + 1]; ++kz)
        for (int ky = Cy << shy; ky < min(ncy, (Cy + 1) << shy); ++ky)
            for (int kx = Cx << shx; kx < min(ncx, (Cx + 1) << shx); ++kx)
                m = fmaxf(m, maj[(size_t(kz) * ncy + ky) * ncx + kx]);
    empty3[c] = m > 0.0f ? 0 : 1;
}

// vertical runs of empty coarse cells, one thread per coarse column: runcode = first | last << 12 (z group numbers) of
// the maximal run of empty coarse cells that contains the cell (a run of one when `merge` is off)
__global__ void run_kernel(const unsigned char* __restrict__ empty3, int nCx, int nCy, int nCz, int gid0, int merge,
                           int* __restrict__ runcode) {
    const int col = blockIdx.x * blockDim.x + threadIdx.x;
    const int ncol = nCx * nCy;
    if (col >= ncol) return;
    for (int K = 0; K < nCz;) {
        if (!empty3[size_t(K) * ncol + col]) { runcode[size_t(K) * ncol + col] = -1; ++K; continue; }
        int E = K + 1;
        if (merge) while (E < nCz && empty3[size_t(E) * ncol + col]) ++E;
        for (int q = K; q < E; ++q) runcode[size_t(q) * ncol + col] = (gid0 + K) | ((gid0 + E - 1) << 12);
        K = E;
    }
}

// fold the emptiness flag into the fine majorant grid: cells inside an empty coarse cell get the negative value
// -(1 + runcode), exactly representable (24 bits), so that ONE look-up gives either the majorant or the empty box
__global__ void mark_empty_kernel(float* __restrict__ maj, int ncx, int ncy, int ncz, int shx, int shy, int nCx, int nCy,
                                  const int* __restrict__ fine2coarse_z, const int* __restrict__ runcode) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= ncx * ncy * ncz) return;
    const int cix = c % ncx, ciy = (c / ncx) % ncy, ciz = c / (ncx * ncy);
    const int code = runcode[(size_t(fine2coarse_z[ciz]) * nCy + (ciy >> shy)) * nCx + (cix >> shx)];
    if (code >= 0) maj[c] = -float(1 + code);
}

__global__ void tau_up_kernel(const float* __restrict__ ext3tot, const float* __restrict__ zgrd, int iz0, int nx, int ny,
                              int nz3, float* __restrict__ tu3) {
    const int col = blockIdx.x * blockDim.x + threadIdx.x;
    const size_t nxy = size_t(nx) * ny;
    if (col >= nxy) return;
    float acc = 0.0f;
    tu3[size_t(nz3) * nxy + col] = 0.0f;
    for (int k = nz3 - 1; k >= 0; --k) {
        acc += ext3tot[size_t(k) * nxy + col] * (zgrd[iz0 + k + 1] - zgrd[iz0 + k]);
        tu3[size_t(k) * nxy + col] = acc;
    }
}

__global__ void check_finite_kernel(const double* __restrict__ a, size_t n, int* __restrict__ bad) {
    const size_t stride = size_t(gridDim.x) * blockDim.x;
    int b = 0;
    for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride)
        if (!isfinite(a[i])) b = 1;
    if (b) atomicOr(bad, 1);
}

// ============================================================================ transport kernel
// Shared-memory view of one thread block: 1-D tables, per-thread accumulators and the per-warp photon pools.
struct Smem {
    const float* z;       // [nz+1]
    const float* e1tot;   // [nz]
    const float* e1cum;   // [nz+1]
    const float* e1;      // [np1d][nz]
    const float* o1;
    const float* a1;
    // packed per-cell records: one 16-byte shared-memory load each instead of a chain of dependent look-ups
    const float4* slabA;  // [nslab_z]   (zlo, zhi, 1-D majorant, bits: fine z index in the majorant grid | group << 16; sign bit: 1-D slab)
    const int4* slabB;    // [nslab_z]   (first layer, one-past-last layer, coarse group, -)
    const float4* grpA;   // [ngroup]    (zlo, zhi, 1-D majorant, bits: first fine slab | one-past-last fine slab << 16)
    const int4* grpB;     // [ngroup]    (first fine slab, one-past-last fine slab, first layer, one-past-last layer)
    double* acc;          // energy sums [4][32]: toa, sfc, (unused), roulette; one slot per lane and block
    double* acc_atm;      // atmospheric absorption: one slot per thread
    double* ftal;         // block- or warp-private flux tally (same layout as the global one) or nullptr
    double* htal;         // block- or warp-private heating tally or nullptr
    double* rtal;         // block- or warp-private radiance tally or nullptr
    double* atal;         // block- or warp-private actinic tally or nullptr (ACT kernels only)
    int tal_mode;         // 1: one copy per block (shared atomics); 2: one copy per warp (plain read-modify-write)
    unsigned* cnt;        // event counters [8][32]: one slot per lane and block (flushed to 64-bit totals per block)
};
enum { ACC_TOA = 0, ACC_SFC = 1, ACC_ATM = 2, ACC_RR = 3 };
enum { CNT_PHOT = 0, CNT_TENT = 1, CNT_COLL = 2, CNT_SFC = 3, CNT_LE = 4, CNT_VISIT = 5, CNT_TALLY = 6, CNT_KILL = 7 };
// Energy sums and event counters: one slot per LANE and block (not per thread), updated with shared-memory atomics -- the
// lanes of a warp hit 32 different addresses, warps of a block rarely collide.  2 KB per block instead of 20 KB: with
// the photon pools this brings two blocks under the 196 KB shared-memory carve-out and leaves 60 KB of L1 to the voxel
// and majorant gathers instead of 22 KB.
// The atmospheric-absorption sum is touched at every collision and keeps a plain per-THREAD slot (load, add, store).
#define ACC_ADD(k, v)                                                                        \
    {                                                                                        \
        if ((k) == ACC_ATM) sm.acc_atm[threadIdx.x] += (v);                                  \
        else tally_add_shared(&sm.acc[(k) * 32 + (threadIdx.x & 31)], (v));                  \
    }
#define CNT_ADD(k, v) cnt_add_shared(&sm.cnt[(k) * 32 + (threadIdx.x & 31)], (v))

// One copy of the Philox rounds for the whole transport kernel: the six draw sites would otherwise inline ~70 instructions
// each.  The hot loop (~38 KB of SASS) is larger than the instruction cache, and throughput reacts to its layout: measured
// on config 2 with prebuilt variants (tools/gpu_variants.sh, profiles/README.md r01_m), this Philox + an out-of-line
// abs_tau_at give 1478 M photons/s against 1430 M with both inlined; moving further cold code out of line lost again.
__device__ __noinline__ float4 philox_u01x4(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t k0, uint32_t k1) {
    const uint4 r = philox4x32_10(c0, c1, c2, 0xB200u, k0, k1);
    return make_float4(u01(r.x), u01(r.y), u01(r.z), u01(r.w));
}

// A photon in registers (while a lane works on it).  Between phases it lives in its warp's shared-memory pool.
struct Photon {
    float x, y, z;
    float3 d;
    float w;
    float tau;        // optical depth left until the next tentative collision
    int cix, ciy;     // fine majorant cell (3-D slabs) -- the column itself when frozen
    int is;           // fine z slab
    int iz;           // layer of the last event / crossing
    int order;
    int job;
    int flags;        // FL_*
    float za;         // start of the current straight leg (for path-integrated gas absorption)
    int iza;
    float leg;        // length of the current leg
    uint32_t rc0, rc1, rc2;   // Philox counter: global photon index (lo, hi), draw number
    float M;          // majorant of the cell in which the photon parked at a tentative collision
};
enum { FL_DIRECT = 1, FL_FROZEN = 2, FL_STALE = 4, FL_ABS = 8, FL_FSCALE = 16, FL_IN3 = 32, FL_EMPTY = 64 };

// pool record: NFIELD 32-bit words per slot, structure-of-arrays ([field][slot]) so that lanes touch distinct banks
enum { F_X = 0, F_Y, F_Z, F_DX, F_DY, F_DZ, F_W, F_TAU, F_CELL, F_LAY, F_ORD, F_JOB, F_ZA, F_LEG, F_RC0, F_RC1, F_RC2, F_M, F_AUX, NFIELD };
// 32-bit words of shared memory per warp: the pool + five queues (DEAD, FLY, TENTATIVE, COLLISION, SURFACE) of 16-bit
// slot numbers
#define POOL_WORDS(np) (NFIELD * (np) + 5 * (np) / 2)
enum { EV_NONE = 0, EV_COLL = 1, EV_SFC = 2, EV_ESC = 3, EV_TENT = 4 };

// The pool keeps the horizontal position in units of fine majorant cells (what the flight phase works in); the event
// and regeneration phases convert to metres on load and back on store.  Both happen at fixed points of a photon's
// history, so a trajectory does not depend on which other photons share its warp (reproducibility).
template <int NP>
__device__ __forceinline__ void pool_load(const float* __restrict__ f, int s, Photon& p, float Sx, float Sy) {
    p.x = f[F_X * NP + s] * Sx; p.y = f[F_Y * NP + s] * Sy; p.z = f[F_Z * NP + s];
    p.d.x = f[F_DX * NP + s]; p.d.y = f[F_DY * NP + s]; p.d.z = f[F_DZ * NP + s];
    p.w = f[F_W * NP + s]; p.tau = f[F_TAU * NP + s];
    const unsigned c = __float_as_uint(f[F_CELL * NP + s]);
    p.cix = int(c & 0xffffu); p.ciy = int(c >> 16);
    const unsigned l = __float_as_uint(f[F_LAY * NP + s]);
    p.is = int(l & 0xffffu); p.iz = int(l >> 16);
    const unsigned o = __float_as_uint(f[F_ORD * NP + s]);
    p.flags = int(o & 0xffu); p.order = int(o >> 8);
    const unsigned j = __float_as_uint(f[F_JOB * NP + s]);
    p.job = int(j & 0xffffu); p.iza = int(j >> 16);
    p.za = f[F_ZA * NP + s]; p.leg = f[F_LEG * NP + s];
    p.rc0 = __float_as_uint(f[F_RC0 * NP + s]); p.rc1 = __float_as_uint(f[F_RC1 * NP + s]); p.rc2 = __float_as_uint(f[F_RC2 * NP + s]);
    p.M = f[F_M * NP + s];
}
template <int NP>
__device__ __forceinline__ void pool_store(float* __restrict__ f, int s, const Photon& p, float inv_Sx, float inv_Sy) {
    f[F_X * NP + s] = p.x * inv_Sx; f[F_Y * NP + s] = p.y * inv_Sy; f[F_Z * NP + s] = p.z;
    f[F_DX * NP + s] = p.d.x; f[F_DY * NP + s] = p.d.y; f[F_DZ * NP + s] = p.d.z;
    f[F_W * NP + s] = p.w; f[F_TAU * NP + s] = p.tau;
    f[F_CELL * NP + s] = __uint_as_float(unsigned(p.cix) | (unsigned(p.ciy) << 16));
    f[F_LAY * NP + s] = __uint_as_float(unsigned(p.is) | (unsigned(p.iz) << 16));
    f[F_ORD * NP + s] = __uint_as_float(unsigned(p.flags) | (unsigned(p.order) << 8));
    f[F_JOB * NP + s] = __uint_as_float(unsigned(p.job) | (unsigned(p.iza) << 16));
    f[F_ZA * NP + s] = p.za; f[F_LEG * NP + s] = p.leg;
    f[F_RC0 * NP + s] = __uint_as_float(p.rc0); f[F_RC1 * NP + s] = __uint_as_float(p.rc1); f[F_RC2 * NP + s] = __uint_as_float(p.rc2);
    f[F_M * NP + s] = p.M;
}

// the flight phase reads and writes only the geometric part of the record
template <int NP, bool PL>
__device__ __forceinline__ void pool_load_flight(const float* __restrict__ f, int s, Photon& p) {
    p.x = f[F_X * NP + s]; p.y = f[F_Y * NP + s]; p.z = f[F_Z * NP + s];
    p.d.x = f[F_DX * NP + s]; p.d.y = f[F_DY * NP + s]; p.d.z = f[F_DZ * NP + s];
    p.tau = f[F_TAU * NP + s];
    const unsigned c = __float_as_uint(f[F_CELL * NP + s]);
    p.cix = int(c & 0xffffu); p.ciy = int(c >> 16);
    const unsigned l = __float_as_uint(f[F_LAY * NP + s]);
    p.is = int(l & 0xffffu); p.iz = int(l >> 16);
    const unsigned o = __float_as_uint(f[F_ORD * NP + s]);
    p.flags = int(o & 0xffu); p.order = int(o >> 8);
    p.leg = f[F_LEG * NP + s];
    p.M = 0.0f;
    if (PL) {
        p.w = f[F_W * NP + s];
        p.job = int(__float_as_uint(f[F_JOB * NP + s]) & 0xffffu);
    }
}
template <int NP, bool PL>
__device__ __forceinline__ void pool_store_flight(float* __restrict__ f, int s, const Photon& p) {
    f[F_X * NP + s] = p.x; f[F_Y * NP + s] = p.y; f[F_Z * NP + s] = p.z;
    f[F_TAU * NP + s] = p.tau;
    f[F_CELL * NP + s] = __uint_as_float(unsigned(p.cix) | (unsigned(p.ciy) << 16));
    f[F_LAY * NP + s] = __uint_as_float(unsigned(p.is) | (unsigned(p.iz) << 16));
    f[F_ORD * NP + s] = __uint_as_float(unsigned(p.flags) | (unsigned(p.order) << 8));
    f[F_LEG * NP + s] = p.leg;
    f[F_M * NP + s] = p.M;
    if (PL) f[F_W * NP + s] = p.w;
}
// a rejected (null) collision changes the optical-depth budget, the draw counter and the layer only
template <int NP>
__device__ __forceinline__ void pool_store_reject(float* __restrict__ f, int s, const Photon& p) {
    f[F_TAU * NP + s] = p.tau;
    f[F_RC2 * NP + s] = __uint_as_float(p.rc2);
    f[F_LAY * NP + s] = __uint_as_float(unsigned(p.is) | (unsigned(p.iz) << 16));
}

// an accepted collision hands over to the collision phase: new weight / order / cell / layer, the next optical-depth
// budget and draw counter, plus (in fields the finished leg no longer needs) the phase-function code, the two random
// numbers of the scattering direction and the 3-D extinction of the voxel
template <int NP>
__device__ __forceinline__ void pool_store_accept(float* __restrict__ f, int s, const Photon& p, float apf, float uz, float uw, float s3) {
    f[F_W * NP + s] = p.w; f[F_TAU * NP + s] = p.tau;
    f[F_RC2 * NP + s] = __uint_as_float(p.rc2);
    f[F_CELL * NP + s] = __uint_as_float(unsigned(p.cix) | (unsigned(p.ciy) << 16));
    f[F_LAY * NP + s] = __uint_as_float(unsigned(p.is) | (unsigned(p.iz) << 16));
    f[F_ORD * NP + s] = __uint_as_float(unsigned(p.flags) | (unsigned(p.order) << 8));
    f[F_LEG * NP + s] = apf; f[F_ZA * NP + s] = uz; f[F_AUX * NP + s] = uw; f[F_M * NP + s] = s3;
}

// x / d for 0 <= x < 2^31 and a divisor fixed per scene, in two instructions instead of the ~28 of a run-time integer
// divide: (mul, sh) from div_magic() on the host, which also checks the result over the range it is used on
__device__ __forceinline__ int div_exact(int x, unsigned mul, int sh) {
    return int((__umulhi(unsigned(x), mul) + unsigned(x)) >> sh);
}

__device__ __forceinline__ float wrapf(float x, float L, float invL) {
    x -= L * floorf(x * invL);
    if (x >= L) x = 0.0f;
    if (x < 0.0f) x = 0.0f;
    return x;
}

__device__ __forceinline__ void tally_add(double* p, double v) { atomicAdd(p, v); }
__device__ __forceinline__ void cnt_add_shared(unsigned* p, unsigned v) {
    const unsigned a = unsigned(__cvta_generic_to_shared(p));
    asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}
__device__ __forceinline__ void tally_add_shared(double* p, double v) {
    const unsigned a = unsigned(__cvta_generic_to_shared(p));
    asm volatile("red.shared.add.f64 [%0], %1;" ::"r"(a), "d"(v) : "memory");
}

// ---- tallies -------------------------------------------------------------------------------------------------------
// Warp-aggregated add: lanes of the (currently converged) warp that target the SAME address are summed first
// (__match_any_sync, then every group walks its own member list with shuffles) and ONE lane per address performs the
// update.  Plane-parallel and few-column scenes send most of a warp to the same few addresses (all lanes of a freshly
// regenerated batch cross the same level; every local estimate of a 1 x 1-pixel sensor hits one pixel): without this a
// shared-memory fp64 add (a CAS loop) or an L2 reduction serialises 32 ways.
//   mode 0: global atomic; mode 1: shared-memory atomic (block-private tally); mode 2: plain read-modify-write
//   (warp-private tally: no other warp touches it and, after aggregation, no two lanes of this warp do)
__device__ __forceinline__ void tally_agg(double* p, double v, int mode) {
    const unsigned am = __activemask();
    const unsigned grp = __match_any_sync(am, reinterpret_cast<unsigned long long>(p));
    const int lane = threadIdx.x & 31;
    const int leader = __ffs(grp) - 1;
    double s = v;
    if (grp & (grp - 1)) {                        // more than one lane on this address
        s = 0.0;
        for (unsigned r = grp; r; r &= r - 1) s += __shfl_sync(grp, v, __ffs(r) - 1);
    }
    if (lane == leader) {
        if (mode == 2) *p += s;
        else if (mode == 1) tally_add_shared(p, s);
        else tally_add(p, s);
    }
}

// Everything a flux / heating tally of one photon needs beyond (variable, level, column, weight); loaded once per phase
// visit instead of once per tally.
struct TallyCtx {
    const double* fs;             // complete per-level scale of the photon's job: norm x columns x caller's factor
    unsigned long long foff, hoff;   // start of the job's slab in the flux / heating tally
};
__device__ __forceinline__ TallyCtx tally_ctx(const DevScene& S, int job) {
    TallyCtx t;
    t.fs = S.job_fscale + size_t(job) * (S.nz + 1);
    t.foff = S.jobs[job].flux_off;
    t.hoff = S.jobs[job].heat_off;
    return t;
}
// column of the atmosphere grid from the horizontal position in units of fine cells (svx x svy columns each)
__device__ __forceinline__ int tally_col_u(const DevScene& S, float ux, float uy) {
    const int fx = min(S.nx - 1, max(0, __float2int_rd(ux * float(S.svx))));
    const int fy = min(S.ny - 1, max(0, __float2int_rd(uy * float(S.svy))));
    return fy * S.nx + fx;
}
__device__ __forceinline__ int tally_col_m(const DevScene& S, const Photon& p) {
    if (p.flags & FL_FROZEN) return p.ciy * S.nx + p.cix;
    return min(S.ny - 1, max(0, int(p.y * S.inv_dy))) * S.nx + min(S.nx - 1, max(0, int(p.x * S.inv_dx)));
}
// tal_mode: 0 global atomics, 1 block-private shared tally, 2 warp-private shared tally
// (updates that reach global memory are counted in the block's shared event counter; private ones at the flush)
// SMT: the kernel may hold block-private tallies (plane-parallel / few-column scenes only, see transport_kernel); the other
// kernels do not even contain the aggregation code -- the per-level kernel of config 5 is instruction-fetch bound and gained
// 27 % when that never-executed code left it (profiles/README.md r02_t)
template <bool SMT>
__device__ __forceinline__ void flux_add(const DevScene& S, const Smem& sm, const TallyCtx& t, int var, int lev, int col, float w) {
    const double v = double(w) * __ldg(t.fs + lev);
    const size_t idx = size_t(t.foff) + size_t(var * (S.nz + 1) + lev) * size_t(S.nx * S.ny) + size_t(col);
    if (SMT && sm.ftal) tally_agg(sm.ftal + idx, v, sm.tal_mode);
    else { tally_add(S.flux + idx, v); CNT_ADD(CNT_TALLY, 1u); }
}
template <bool SMT>
__device__ __forceinline__ void heat_add(const DevScene& S, const Smem& sm, const TallyCtx& t, int iz, int col, double dep) {
    const double v = dep * __ldg(t.fs + iz);
    const size_t idx = size_t(t.hoff) + size_t(iz) * size_t(S.nx * S.ny) + size_t(col);
    if (SMT && sm.htal) tally_agg(sm.htal + idx, v, sm.tal_mode);
    else { tally_add(S.heat + idx, v); CNT_ADD(CNT_TALLY, 1u); }
}

// one flux / heating tally of a photon whose position is in metres (p.x, p.y)
template <bool SMT>
__device__ __forceinline__ void flux_tally(const DevScene& S, const Smem& sm, const Photon& p, int var, int lev) {
    const TallyCtx t = tally_ctx(S, p.job);
    flux_add<SMT>(S, sm, t, var, lev, tally_col_m(S, p), p.w);
}
template <bool SMT>
__device__ __forceinline__ void heat_tally(const DevScene& S, const Smem& sm, const Photon& p, int iz, double dep) {
    const TallyCtx t = tally_ctx(S, p.job);
    heat_add<SMT>(S, sm, t, iz, tally_col_m(S, p), dep);
}
// radiance tally (idx: position inside the whole radiance tally).  The block-private copy exists in the per-level kernels
// of plane-parallel / few-column scenes only (SMT) -- tiny sensors belong to such scenes, which the host routes there -- so
// that the kernels of the large 3-D scenes carry neither the branch nor the aggregation code.
template <bool SMT>
__device__ __forceinline__ void rad_add(const DevScene& S, const Smem& sm, size_t idx, double v) {
    if (SMT && sm.rtal) tally_agg(sm.rtal + idx, v, sm.tal_mode);
    else { tally_add(S.rad + idx, v); CNT_ADD(CNT_TALLY, 1u); }
}

// layer that contains z among layers [l0, l1)
__device__ __forceinline__ int find_layer(const Smem& sm, int l0, int l1, float z) {
    int lo = l0, hi = l1 - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (z >= sm.z[mid]) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// gas-absorption optical depth of a straight leg from (za, layer iza) to (zb, layer izb) of length `dist`.
// Out of line and by value (three call sites; keeps the hot loop small).
__device__ __noinline__ float abs_tau_at(const float* __restrict__ ab, const float* __restrict__ cb, float za, float zla, int iza,
                                         float zb, float zlb, int izb, float dist, float inv_absdz) {
    if (iza == izb) return __ldg(ab + iza) * dist;
    const float ca = __ldg(cb + iza) + __ldg(ab + iza) * (za - zla);
    const float c2 = __ldg(cb + izb) + __ldg(ab + izb) * (zb - zlb);
    return fabsf(c2 - ca) * inv_absdz;
}
__device__ __forceinline__ float abs_tau(const DevScene& S, const Smem& sm, int job, float za, int iza, float zb, int izb,
                                         float dist, float inv_absdz) {
    return abs_tau_at(S.job_abs + size_t(job) * S.nz, S.job_cabs + size_t(job) * (S.nz + 1), za, sm.z[iza], iza, zb, sm.z[izb], izb,
                      dist, inv_absdz);
}

// ---- spectral runs: kd_n gas-absorption terms (Atm_nkd) share one history -------------------------------------------
// Gas absorption never changes a trajectory, so every term can ride on the same flights, collisions and draws.  Per term
// g the photon carries r_g = a_g / sum_h q_h a_h, where a_g = exp(-T_g) is its gas transmission so far in term g and q the
// normalised term weights, while p.w holds the term-weighted weight W = w sum_h q_h a_h (w: the gas-free weight).  Then
// w a_g = W r_g for every term, and everything that acts on p.w -- single-scattering albedo, surface reflection, Russian
// roulette, the energy sums -- acts on W unchanged: roulette on W keeps histories that are absorbed in every term from
// running forever, and the factor it applies (wfac / W) is common to all terms.  r_g <= 1 / q_g, so the state never
// overflows.  Regeneration sets r_g = 1.
// Where a leg ends (collision, surface, escape): e_g = exp(-tau_g(leg)), s = sum_g q_g r_g e_g, W <- W s,
// r_g <- r_g e_g / s.  Returns s; UPD = false (escape) leaves r alone.  Two passes over the slot's terms, out of line (the
// terms live in global scratch, DevScene::kd_r, not in registers).  tab: the job's rows of DevScene::kd_tab; dza, dzb:
// heights of the leg's ends above the bottom of their layers iza, izb; f: the leg's length when iza == izb, else 1 / |u_z|.
template <bool UPD>
__device__ __noinline__ float kd_leg(const float2* __restrict__ tab, float* __restrict__ r, int nkd, float dza, int iza, float dzb, int izb,
                                     float f) {
    const float2* ta = tab + size_t(1 + iza) * nkd;
    const float2* tb = tab + size_t(1 + izb) * nkd;
    float s = 0.0f;
    for (int g = 0; g < nkd; ++g) {
        const float2 A = __ldg(ta + g);
        float t;
        if (iza == izb) t = A.y * f;
        else {
            const float2 B = __ldg(tb + g);
            t = fabsf((B.x + B.y * dzb) - (A.x + A.y * dza)) * f;
        }
        const float re = r[g] * __expf(-t);
        s = fmaf(__ldg(tab + g).x, re, s);
        if (UPD) r[g] = re;
    }
    if (UPD) {
        const float inv = s > 0.0f ? 1.0f / s : 0.0f;
        for (int g = 0; g < nkd; ++g) r[g] *= inv;
    }
    return s;
}
// Radiance factor of one local estimate from the event (dz above the bottom of layer iz) to the sensor level (dzt above the
// bottom of layer lt), summed over the terms: sum_g rf_g r_g exp(-tau_abs_g), tau_abs_g = |C_g(zt) - C_g(z)| / |mu_v| from
// the cumulative gas profiles (O(1) per term).
__device__ __noinline__ double kd_le_sum(const float2* __restrict__ tab, const double* __restrict__ rf, const float* __restrict__ r,
                                         int nkd, float dz, int iz, float dzt, int lt, float inv_sz) {
    const float2* ta = tab + size_t(1 + iz) * nkd;
    const float2* tb = tab + size_t(1 + lt) * nkd;
    double sum = 0.0;
    for (int g = 0; g < nkd; ++g) {
        const float2 A = __ldg(ta + g), B = __ldg(tb + g);
        const float t = fabsf((B.x + B.y * dzt) - (A.x + A.y * dz)) * inv_sz;
        sum += __ldg(rf + g) * double(r[g] * __expf(-t));
    }
    return sum;
}
__device__ __noinline__ void kd_init(float* __restrict__ r, int nkd) {
    for (int g = 0; g < nkd; ++g) r[g] = 1.0f;
}
// the per-term state of pool slot `slot` of the calling warp (a slot belongs to one warp; __syncwarp after every queue pop
// orders these accesses as it orders the pool)
template <int NP>
__device__ __forceinline__ float* kd_state(const DevScene& S, int slot) {
    return S.kd_r + ((size_t(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5)) * NP + size_t(slot)) * S.kd_n;
}

// ---- radiance Jacobians: dI / dln(a_j), a_j a factor on the gas absorption (job.abs1d) of every layer of group j -------
// Gas absorption never changes a trajectory, so a local estimate's contribution c = w0 exp(-T_hist - tau_LE) ... depends
// on a_j only through the gas optical paths, and d c / d ln(a_j) = -c (T_j + tau_LE_j): T_j the gas optical path the
// history has collected inside group j since it started, tau_LE_j that of the event -> sensor segment.  The score is the
// photon weight times a function of the history, so Russian roulette (which keeps the expected weight given the past)
// leaves it unbiased.  The slot carries T_j in global scratch (DevScene::xs), updated where a leg ends at a collision
// or the surface; an escape leg needs nothing (no local estimate follows it).
// jac_leg splits the gas optical path of the leg from (dza above the bottom of layer iza) to (dzb above the bottom of izb)
// over the groups it crosses, exactly as abs_tau_at computes the leg's whole path: inside one layer abs * f (f = length),
// else clamped differences of the cumulative profile times f = 1 / |u_z|, so that sum_j of the increments is the leg's
// tau to rounding.  ab, cb: the job's rows of DevScene::job_abs / job_cabs.
__device__ __noinline__ void jac_leg(const float* __restrict__ ab, const float* __restrict__ cb, const int* __restrict__ lev,
                                     const unsigned char* __restrict__ grp, float* __restrict__ t, float dza, int iza, float dzb,
                                     int izb, float f) {
    if (iza == izb) {
        t[__ldg(grp + iza)] += __ldg(ab + iza) * f;
        return;
    }
    const float ca = __ldg(cb + iza) + __ldg(ab + iza) * dza;
    const float c2 = __ldg(cb + izb) + __ldg(ab + izb) * dzb;
    const float lo = fminf(ca, c2), hi = fmaxf(ca, c2);
    const int g1 = __ldg(grp + max(iza, izb));
    for (int j = __ldg(grp + min(iza, izb)); j <= g1; ++j) {
        const float a = fmaxf(lo, __ldg(cb + __ldg(lev + j))), b = fminf(hi, __ldg(cb + __ldg(lev + j + 1)));
        if (b > a) t[j] += (b - a) * f;
    }
}
// Deposit -c (T_j + tau_LE_j) for every group with a non-zero path into out[0 .. ngrp) (the groups of one radiance pixel,
// adjacent).  tau_LE_j: overlap of [event (dz above the bottom of layer iz), sensor level (dzt above the bottom of lt)]
// with group j from the cumulative profile, times inv_sz.  Returns the number of tally updates.
__device__ __noinline__ unsigned jac_deposit(double* __restrict__ out, const float* __restrict__ t, int ngrp, const float* __restrict__ ab,
                                             const float* __restrict__ cb, const int* __restrict__ lev,
                                             const unsigned char* __restrict__ grp, float dz, int iz, float dzt, int lt, float inv_sz,
                                             double c) {
    const float ca = __ldg(cb + iz) + __ldg(ab + iz) * dz;
    const float cs = __ldg(cb + lt) + __ldg(ab + lt) * dzt;
    const float lo = fminf(ca, cs), hi = fmaxf(ca, cs);
    const int g0 = __ldg(grp + min(iz, lt)), g1 = __ldg(grp + max(iz, lt));
    unsigned n = 0;
    for (int j = 0; j < ngrp; ++j) {
        float tau = t[j];
        if (j >= g0 && j <= g1) {
            const float a = fmaxf(lo, __ldg(cb + __ldg(lev + j))), b = fminf(hi, __ldg(cb + __ldg(lev + j + 1)));
            if (b > a) tau += (b - a) * inv_sz;
        }
        if (tau != 0.0f) {
            tally_add(out + j, -c * double(tau));
            ++n;
        }
    }
    return n;
}
__device__ __noinline__ void jac_init(float* __restrict__ t, int ngrp) {
    for (int j = 0; j < ngrp; ++j) t[j] = 0.0f;
}
// the per-group state of pool slot `slot` of the calling warp (ordered like kd_state)
template <int NP>
__device__ __forceinline__ float* jac_state(const DevScene& S, int slot) {
    return S.xs + ((size_t(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5)) * NP + size_t(slot)) * S.jac_n;
}

// ---- radiance path-length distributions: the geometric path L (m) behind every local-estimate contribution c -------------
// L runs from the photon's entry at TOA along every leg of its history to the event, then along the event -> sensor segment
// to the sensor's target level.  L is geometry only (it never changes a trajectory) and the score is the photon weight times
// a function of the history, so Russian roulette leaves it unbiased, as for the Jacobian.  The slot carries the path of its
// finished legs in global scratch (DevScene::xs), updated where a leg ends at a collision or the surface; an escape leg needs
// nothing.  plen_deposit adds c to the bin of L (index ntp: L < lo, ntp + 1: L >= hi) and c L to the first moment (ntp + 2)
// of one radiance pixel's row out[0 .. ntp+3); the bin index is computed in fp32 from the fp32 path.
__device__ __forceinline__ void plen_deposit(double* __restrict__ out, int ntp, float lo, float hi, float inv_w, float L, double c) {
    const int b = L < lo ? ntp : (L >= hi ? ntp + 1 : min(ntp - 1, int((L - lo) * inv_w)));
    tally_add(out + b, c);
    tally_add(out + ntp + 2, c * double(L));
}
// the path of pool slot `slot` of the calling warp (ordered like kd_state)
template <int NP>
__device__ __forceinline__ float* plen_state(const DevScene& S, int slot) {
    return S.xs + (size_t(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5)) * NP + size_t(slot);
}

// ---- actinic flux: track-length estimate of the layer-and-column mean of F_act = integral of I over 4 pi ----------------
// A flight move of length `len` inside layer iz adds the integral of the weight along the track, per column it crosses,
// divided by the layer's thickness dz and scaled like the heating (fs = the job's heating scale of the layer).  With gas absorption k
// the weight falls along the move: a segment of length l starting at weight w_a adds w_a (1 - exp(-k l)) / k, then
// w_a <- w_a exp(-k l) -- the heating deposit of the segment over k, so that sum over the layer of k dz act = heating.
// The kernel's own weight update stays the only one (this never touches the photon).  The move starts at (ux, uy) in fine
// cells (svx x svy columns each) and runs along (dux, duy) per metre; the walk crosses column faces, periodic wraps
// included.  col >= 0: the column of a frozen photon (no walk).  A move that crosses more than ACT_MAX_CROSS faces (a
// near-horizontal photon in a transparent 1-D layer wraps the domain many times) puts the rest of its track into the
// column where the walk stops: the domain mean stays exact.  out: the (slab, var 0, iz) plane of the tally, vstride the
// distance to the var-1 (total) plane; direct photons add to both.  mode as tally_agg (0: global atomics).  Returns the
// number of global updates.
#define ACT_MAX_CROSS 65536
__device__ __noinline__ unsigned act_move(double* __restrict__ out, size_t vstride, int mode, int direct, int nx, int ny, int svx,
                                          int svy, float ux, float uy, float dux, float duy, float len, float w, float k,
                                          double fs, float dz, int col) {
    const double sc = fs / double(dz);
    const float ik = k > 0.0f ? 1.0f / k : 0.0f;
    float px = ux * float(svx), py = uy * float(svy);
    const float vx = dux * float(svx), vy = duy * float(svy);
    int ix = col >= 0 ? col % nx : min(nx - 1, max(0, __float2int_rd(px)));
    int iy = col >= 0 ? col / nx : min(ny - 1, max(0, __float2int_rd(py)));
    const int stx = vx > 0.0f ? 1 : -1, sty = vy > 0.0f ? 1 : -1;
    const float ax = fabsf(1.0f / vx), ay = fabsf(1.0f / vy);      // metres per column crossed (|v| >= 1e-20 per fine cell)
    float tx = col >= 0 ? RT_INF : fmaxf(0.0f, (float(ix + (stx > 0 ? 1 : 0)) - px) / vx);
    float ty = col >= 0 ? RT_INF : fmaxf(0.0f, (float(iy + (sty > 0 ? 1 : 0)) - py) / vy);
    float rem = len, wa = w;
    unsigned n = 0;
    for (int c = 0;; ++c) {
        const float l = c < ACT_MAX_CROSS ? fmaxf(0.0f, fminf(rem, fminf(tx, ty))) : rem;
        if (l > 0.0f) {
            const float f = -expm1f(-k * l);                // fraction of w_a absorbed over the segment
            const double d = double(k > 0.0f ? wa * f * ik : wa * l) * sc;
            double* o = out + size_t(iy) * size_t(nx) + size_t(ix);
            if (mode == 0) {
                tally_add(o + vstride, d);
                n++;
                if (direct) { tally_add(o, d); n++; }
            } else {
                tally_agg(o + vstride, d, mode);
                if (direct) tally_agg(o, d, mode);
            }
            wa -= wa * f;
        }
        rem -= l;
        if (!(rem > 0.0f) || !(wa > 0.0f)) break;
        if (tx <= ty) {
            ix += stx; ix = ix >= nx ? 0 : (ix < 0 ? nx - 1 : ix);
            ty -= l; tx = ax;
        } else {
            iy += sty; iy = iy >= ny ? 0 : (iy < 0 ? ny - 1 : iy);
            tx -= l; ty = ay;
        }
    }
    return n;
}
// one flight move of photon p (still at its start, weight before the move) in its layer p.is; col as act_move
template <bool SMT>
__device__ __forceinline__ unsigned act_add(const DevScene& S, const Smem& sm, const TallyCtx& t, const Photon& p, float ux, float uy,
                                            float dux, float duy, float len, int col) {
    const size_t nxy = size_t(S.nx) * size_t(S.ny);
    const bool priv = SMT && sm.atal;
    double* out = (priv ? sm.atal : S.xt) + 2 * size_t(t.hoff) + size_t(p.is) * nxy;
    const float k = (p.flags & FL_ABS) ? __ldg(S.job_abs + size_t(p.job) * S.nz + p.is) : 0.0f;
    return act_move(out, size_t(S.nz) * nxy, priv ? sm.tal_mode : 0, p.flags & FL_DIRECT, S.nx, S.ny, S.svx, S.svy, ux, uy, dux, duy,
                    len, p.w, k, __ldg(t.fs + p.is), sm.z[p.is + 1] - sm.z[p.is], col);
}

// Exact optical depth toward a sensor for oblique views and sensors inside the atmosphere.
//   * 1-D extinction and gas absorption are horizontally uniform: their integral over the whole segment is a difference
//     of the cumulative profiles, O(1) whatever the number of layers;
//   * the 3-D extinction is integrated by an incremental voxel DDA (ray parameters of the next x / y / z face, one
//     add per crossing) over the part of the segment inside the 3-D block only; the load of the next voxel is issued
//     before the current one is consumed.
// Kept out of line: it is the cold path of le_tau and large.  Everything is passed by value so that the photon never
// has to live in local memory.
struct RayTarget { float3 s; float zt; int lt; };   // unit direction of travel; level at which the integral stops and its layer
__device__ __noinline__ float le_tau_generic(const DevScene& S, const float* __restrict__ smz, const float* __restrict__ sme1tot,
                                             const float* __restrict__ sme1cum, const RayTarget se, float x, float y, float z, int iz,
                                             int job, int has_abs, int frozen, int fx, int fy, bool in3, unsigned* n_visit_out) {
    const bool up = se.s.z > 0.0f;
    const float isz = 1.0f / se.s.z;
    // ---- 1-D part, closed form
    float c_a = sme1cum[iz] + sme1tot[iz] * (z - smz[iz]);
    float c_b = sme1cum[se.lt] + sme1tot[se.lt] * (se.zt - smz[se.lt]);
    if (has_abs) {
        const float* ab = S.job_abs + size_t(job) * S.nz;
        const float* cb = S.job_cabs + size_t(job) * (S.nz + 1);
        c_a += __ldg(cb + iz) + __ldg(ab + iz) * (z - smz[iz]);
        c_b += __ldg(cb + se.lt) + __ldg(ab + se.lt) * (se.zt - smz[se.lt]);
    }
    float tau = fabsf((c_b - c_a) * isz);
    *n_visit_out = 0;
    if (S.nz3 <= 0) return tau;
    // ---- 3-D part: the piece of [z, zt] inside the block
    const float zb0 = smz[S.iz0], zb1 = smz[S.iz0 + S.nz3];
    const float za = up ? fmaxf(z, zb0) : fminf(z, zb1);            // where the 3-D integral starts
    const float ze = up ? fminf(se.zt, zb1) : fmaxf(se.zt, zb0);    // ... and ends
    const float T = (ze - za) * isz;                                 // ray parameter (path length) of the 3-D piece
    if (!(T > 0.0f)) return tau;
    int l;                                                           // layer of the start point of the 3-D piece
    if (za == z) {
        l = min(S.iz0 + S.nz3 - 1, max(S.iz0, iz));
        if (up && z >= smz[l + 1] && l + 1 < S.iz0 + S.nz3) l++;
        if (!up && z <= smz[l] && l > S.iz0) l--;
    } else l = up ? S.iz0 : S.iz0 + S.nz3 - 1;
    const int nxy = S.nx * S.ny;
    unsigned n_visit = 0;
    if (frozen) {
        // column-frozen photon: the ray stays in its column
        const float* col = S.ext3tot + fy * S.nx + fx;
        float zc = za;
        for (;;) {
            const float zn = up ? fminf(smz[l + 1], ze) : fmaxf(smz[l], ze);
            tau += __ldg(col + (l - S.iz0) * nxy) * (zn - zc) * isz;
            ++n_visit;
            zc = zn;
            if (up) { if (zn >= ze || ++l >= S.iz0 + S.nz3) break; }
            else { if (zn <= ze || --l < S.iz0) break; }
        }
        *n_visit_out = n_visit;
        return tau;
    }
    if (za != z || !in3) {
        const float d0 = (za - z) * isz;
        x = wrapf(x + se.s.x * d0, S.Lx, S.inv_Lx); y = wrapf(y + se.s.y * d0, S.Ly, S.inv_Ly);
        fx = min(S.nx - 1, max(0, int(x * S.inv_dx)));
        fy = min(S.ny - 1, max(0, int(y * S.inv_dy)));
    }
    // ray parameters of the next faces, measured from the start of the 3-D piece
    const bool px = se.s.x > 0.0f, py = se.s.y > 0.0f;
    const float isx = se.s.x != 0.0f ? 1.0f / se.s.x : RT_INF, isy = se.s.y != 0.0f ? 1.0f / se.s.y : RT_INF;
    float tmx = se.s.x != 0.0f ? fmaxf(0.0f, (float(fx + (px ? 1 : 0)) * S.dx - x) * isx) : RT_INF;
    float tmy = se.s.y != 0.0f ? fmaxf(0.0f, (float(fy + (py ? 1 : 0)) * S.dy - y) * isy) : RT_INF;
    const float tdx = se.s.x != 0.0f ? fabsf(S.dx * isx) : 0.0f, tdy = se.s.y != 0.0f ? fabsf(S.dy * isy) : 0.0f;
    // one branch-free step per voxel (lanes of a warp cross different faces; selects keep them in one instruction stream)
    const int sx = px ? 1 : -1, sy = py ? 1 : -1, dl = up ? 1 : -1;
    const float* zl = smz + S.iz0 + (up ? 1 : 0);                    // zl[k]: the face of block layer k ahead of the ray
    int lz = l - S.iz0;
    const int lzend = up ? S.nz3 : -1;                               // first layer outside the block
    float tmz = fminf(T, (zl[lz] - za) * isz);
    const float* base = S.ext3tot;
    float t = 0.0f, tau3 = 0.0f;
// one voxel: SEG = path length inside the current voxel, IDX = index of the next one, DONE = the current one is the last
#define LE_STEP(SEG, IDX, DONE)                                               \
    {                                                                         \
        const float tn = fminf(fminf(tmx, tmy), tmz);                         \
        SEG = tn - t;                                                         \
        t = tn;                                                               \
        ++n_visit;                                                            \
        const bool cx = tmx <= tmy && tmx <= tmz;                             \
        const bool cy = !cx && tmy <= tmz;                                    \
        const bool cz = !(cx || cy);                                          \
        int nfx = fx + sx, nfy = fy + sy;                                     \
        nfx = nfx >= S.nx ? 0 : (nfx < 0 ? S.nx - 1 : nfx);                   \
        nfy = nfy >= S.ny ? 0 : (nfy < 0 ? S.ny - 1 : nfy);                   \
        fx = cx ? nfx : fx;                                                   \
        fy = cy ? nfy : fy;                                                   \
        lz = cz ? lz + dl : lz;                                               \
        tmx = cx ? tmx + tdx : tmx;                                           \
        tmy = cy ? tmy + tdy : tmy;                                           \
        DONE = tn >= T || lz == lzend;                                        \
        const int lzc = min(S.nz3 - 1, max(0, lz));                           \
        tmz = cz ? fminf(T, (zl[lzc] - za) * isz) : tmz;                      \
        IDX = (lzc * S.ny + fy) * S.nx + fx;                                  \
    }
    float e = __ldg(base + (lz * S.ny + fy) * S.nx + fx);
    for (;;) {
        float seg;
        int inext;
        bool done;
        LE_STEP(seg, inext, done);
        const float en = done ? 0.0f : __ldg(base + inext);   // next voxel: in flight while this one is consumed
        tau3 = fmaf(e, seg, tau3);
        if (done) break;
        e = en;
    }
#undef LE_STEP
    *n_visit_out = n_visit;
    return tau + tau3;
}

// Optical depth (extinction + gas absorption) from the photon position along the sensor direction to the sensor's
// target level.  fx, fy: fine column if the start point lies in a 3-D layer (else recomputed); s3: 3-D extinction of
// the start voxel.  KD: without the gas term (kd_le_sum adds it per term).
template <bool KD>
__device__ __forceinline__ float le_tau(const DevScene& S, const Smem& sm, const DevSensor& se, const Photon& p, int fx, int fy,
                                        float s3) {
    const int iz = p.iz;
    const bool frozen = (p.flags & FL_FROZEN) != 0;
    const bool in3 = (S.nz3 > 0) && iz >= S.iz0 && iz < S.iz0 + S.nz3;
    if (se.fast_ok && se.s.z > 0.0f && (frozen || se.vertical_up)) {
        // ---- vertical (or column-frozen) fast path: O(1) look-ups in the precomputed tables
        float t1 = (sm.e1cum[se.lt] + sm.e1tot[se.lt] * (se.zt - sm.z[se.lt])) - (sm.e1cum[iz] + sm.e1tot[iz] * (p.z - sm.z[iz]));
        if (!KD && (p.flags & FL_ABS)) {
            const float* ab = S.job_abs + size_t(p.job) * S.nz;
            const float* cb = S.job_cabs + size_t(p.job) * (S.nz + 1);
            t1 += (__ldg(cb + se.lt) + __ldg(ab + se.lt) * (se.zt - sm.z[se.lt])) - (__ldg(cb + iz) + __ldg(ab + iz) * (p.z - sm.z[iz]));
        }
        if (S.nz3 > 0 && iz < S.iz0 + S.nz3) {
            const int nxy = S.nx * S.ny;
            if (!in3) {
                fx = frozen ? p.cix : min(S.nx - 1, max(0, int(p.x * S.inv_dx)));
                fy = frozen ? p.ciy : min(S.ny - 1, max(0, int(p.y * S.inv_dy)));
                t1 += __ldg(S.tu3 + fy * S.nx + fx);
            } else {
                t1 += __ldg(S.tu3 + (iz - S.iz0 + 1) * nxy + fy * S.nx + fx) + s3 * (sm.z[iz + 1] - p.z);
            }
            CNT_ADD(CNT_VISIT, 1u);
        }
        return fmaxf(0.0f, t1) * se.inv_sz;
    }
    if (frozen) { fx = p.cix; fy = p.ciy; }
    unsigned nv = 0;
    const RayTarget rt = {se.s, se.zt, se.lt};
    const float t = le_tau_generic(S, sm.z, sm.e1tot, sm.e1cum, rt, p.x, p.y, p.z, iz, p.job, KD ? 0 : (p.flags & FL_ABS), frozen ? 1 : 0, fx,
                                   fy, in3, &nv);
    CNT_ADD(CNT_VISIT, nv);
    return t;
}

// deposit one local-estimate contribution (fw = weight x angular density toward the sensor, 1/sr)
// KD: kdr = the photon's per-term state; the radiance factor is the sum over the terms (kd_le_sum) instead of the job's
// JAC: kdr = the photon's per-group gas optical paths; the same contribution also goes to the Jacobian tally (jac_deposit)
// PLEN: kdr = the photon's path so far; the same contribution also goes to the path-length tally (plen_deposit)
template <bool SMT, bool KD = false, bool JAC = false, bool PLEN = false>
__device__ __forceinline__ void le_deposit(const DevScene& S, const Smem& sm, const DevSensor& se, const Photon& p, float fw,
                                           int fx, int fy, float s3, const float* kdr = nullptr) {
    const float tau = le_tau<KD>(S, sm, se, p, fx, fy, s3);
    const float contrib = fw * __expf(-tau) * se.inv_sz;
    int px, py;
    if (p.flags & FL_FROZEN) {
        px = min(se.nxr - 1, int((float(p.cix) + 0.5f) / float(S.nx) * float(se.nxr)));
        py = min(se.nyr - 1, int((float(p.ciy) + 0.5f) / float(S.ny) * float(se.nyr)));
    } else {
        const float t = (se.zref - p.z) * se.inv_szs;
        const float xr = wrapf(p.x + se.s.x * t, S.Lx, S.inv_Lx), yr = wrapf(p.y + se.s.y * t, S.Ly, S.inv_Ly);
        px = min(se.nxr - 1, max(0, int(xr * S.inv_Lx * float(se.nxr))));
        py = min(se.nyr - 1, max(0, int(yr * S.inv_Ly * float(se.nyr))));
    }
    const DevJob& J = S.jobs[p.job];
    const size_t idx = size_t(J.slab) * S.rad_slab + se.off + py * se.nxr + px;
    if (KD) {
        const double fac = kd_le_sum(S.kd_tab + size_t(p.job) * (S.nz + 2) * S.kd_n, S.kd_rf + size_t(p.job) * S.kd_n, kdr, S.kd_n,
                                     p.z - sm.z[p.iz], p.iz, se.zt - sm.z[se.lt], se.lt, se.inv_sz);
        rad_add<SMT>(S, sm, idx, double(contrib) * fac * se.npix);
    } else if (JAC) {
        const double c = double(contrib) * J.rad_fac * se.npix;
        rad_add<SMT>(S, sm, idx, c);
        if (p.flags & FL_ABS) {
            const unsigned n = jac_deposit(S.xt + idx * S.jac_n, kdr, S.jac_n, S.job_abs + size_t(p.job) * S.nz,
                                           S.job_cabs + size_t(p.job) * (S.nz + 1), S.jac_lev, S.jac_grp, p.z - sm.z[p.iz], p.iz,
                                           se.zt - sm.z[se.lt], se.lt, se.inv_sz, c);
            CNT_ADD(CNT_TALLY, n);
        }
    } else if (PLEN) {
        const double c = double(contrib) * J.rad_fac * se.npix;
        rad_add<SMT>(S, sm, idx, c);
        plen_deposit(S.xt + idx * (S.pl_ntp + 3), S.pl_ntp, S.pl_lo, S.pl_hi, S.pl_inv_w, *kdr + (se.zt - p.z) * se.inv_szs, c);
        CNT_ADD(CNT_TALLY, 2u);
    } else rad_add<SMT>(S, sm, idx, double(contrib) * J.rad_fac * se.npix);
    CNT_ADD(CNT_LE, 1u);
}

// All-sky camera (Rad_mrkind = 1): contribution of one event, per unit photon weight, to the radiance the camera at
// se.cpos records in the pixel that sees the event.  Returns 0 when the event lies outside the field of view.
//   I_pix += w * f(event -> camera) * exp(-tau) / (R^2 * dOmega_pix)          [times the power one photon carries]
// Periodic domain: the nearest image of the camera is used.  Polar pixel mapping: U = theta cos(az), V = theta sin(az);
// a pixel of size dU x dV subtends dOmega = (sin(theta) / theta) dU dV.
__device__ __noinline__ float camera_le(const DevScene& S, const float* __restrict__ smz, const float* __restrict__ sme1tot,
                                        const float* __restrict__ sme1cum,
                                        const DevSensor& se, float x, float y, float z, int iz, int job, int has_abs, int fx, int fy,
                                        bool in3, const float3 din, int evk, float apf, int sfc_type, float p0, float p1, float p2,
                                        float p3, float p4, int* pix_out, unsigned* n_visit_out) {
    *n_visit_out = 0;
    float dx = se.cpos.x - x, dy = se.cpos.y - y;
    dx -= S.Lx * rintf(dx * S.inv_Lx);
    dy -= S.Ly * rintf(dy * S.inv_Ly);
    const float dz = se.cpos.z - z;
    const float R2 = dx * dx + dy * dy + dz * dz;
    if (!(R2 > 1e-6f) || fabsf(dz) < 1e-3f) return 0.0f;
    const float invR = rsqrtf(R2);
    const float3 sdir = make_float3(dx * invR, dy * invR, dz * invR);          // event -> camera
    if (fabsf(sdir.z) < 1e-4f) return 0.0f;
    // direction in which the camera sees the event
    const float3 v = make_float3(-sdir.x, -sdir.y, -sdir.z);
    const float cq = v.x * se.s.x + v.y * se.s.y + v.z * se.s.z;
    if (cq < se.cos_half_fov) return 0.0f;
    const float theta = acosf(fminf(1.0f, cq));
    const float vx = v.x * se.ex.x + v.y * se.ex.y + v.z * se.ex.z, vy = v.x * se.ey.x + v.y * se.ey.y + v.z * se.ey.z;
    const float rho = sqrtf(vx * vx + vy * vy);
    const float U = rho > 0.0f ? theta * vx / rho : 0.0f, V = rho > 0.0f ? theta * vy / rho : 0.0f;
    if (fabsf(U) >= se.u_half || fabsf(V) >= se.v_half) return 0.0f;
    const int px = min(se.nxr - 1, max(0, int((U + se.u_half) * se.pix_per_u)));
    const int py = min(se.nyr - 1, max(0, int((V + se.v_half) * se.pix_per_v)));
    *pix_out = py * se.nxr + px;
    float f;
    if (evk == EV_COLL) f = phase_eval(S.pt, apf, din.x * sdir.x + din.y * sdir.y + din.z * sdir.z) * (0.25f / RT_PI);
    else f = sdir.z > 0.0f ? brdf_eval(sfc_type, p0, p1, p2, p3, p4, make_float3(-din.x, -din.y, -din.z), sdir) * sdir.z : 0.0f;
    if (!(f > 0.0f)) return 0.0f;
    const RayTarget rt = {sdir, se.cpos.z, se.lt};
    const float tau = le_tau_generic(S, smz, sme1tot, sme1cum, rt, x, y, z, iz, job, has_abs, 0, fx, fy, in3, n_visit_out);
    const float sinc = theta > 1e-4f ? __sinf(theta) / theta : 1.0f;
    const float domega = sinc / (se.pix_per_u * se.pix_per_v);
    return f * __expf(-tau) / (fmaxf(R2, se.ap2) * domega);
}

__device__ __forceinline__ float3 inv_dir(const float3 d) {
    return make_float3(d.x != 0.0f ? 1.0f / d.x : RT_INF, d.y != 0.0f ? 1.0f / d.y : RT_INF, d.z != 0.0f ? 1.0f / d.z : RT_INF);
}

// sample the reflected direction `wo` at a surface of the given type; returns the weight factor (BRDF cos / pdf)
__device__ __noinline__ float surface_sample(int sfc_type, float p0, float p1, float p2, float p3, float p4, const float3 wi,
                                             const float4 u, float3* wo_out) {
    const float prm[5] = {p0, p1, p2, p3, p4};
    float3 wo = make_float3(0.f, 0.f, 1.f);
    float fac = 0.0f;
    bool diffuse = true;
    if (sfc_type == B200RT_SFC_DSM && u.z >= prm[1]) diffuse = false;
    if (diffuse) {
        // cosine-weighted direction: Lambertian (type 1), whitecap part of DSM, LSRT with weight = pi * f_r
        const float ct = sqrtf(u.x), st = sqrtf(1.0f - u.x);
        float sp, cp;
        __sincosf(RT_2PI * u.y, &sp, &cp);
        wo = make_float3(st * cp, st * sp, fmaxf(ct, 1e-6f));
        fac = (sfc_type == B200RT_SFC_LSRT) ? lsrt_kernel_sum(prm, wi, wo) : prm[0];
    } else {
        // Cox-Munk facet: slope from the isotropic Gaussian, mirror reflection, weight F cos(gamma) / (mu_i mu_n) S
        const float sig2 = fmaxf(1e-6f, prm[4]);
        const float r = sqrtf(-sig2 * __logf(1.0f - u.x * 0.99999994f));
        float sp, cp;
        __sincosf(RT_2PI * u.y, &sp, &cp);
        const float zx = r * cp, zy = r * sp;
        const float nn = rsqrtf(1.0f + zx * zx + zy * zy);
        const float3 n = make_float3(-zx * nn, -zy * nn, nn);
        const float cosg = wi.x * n.x + wi.y * n.y + wi.z * n.z;
        if (cosg > 0.0f) {
            wo = make_float3(2.0f * cosg * n.x - wi.x, 2.0f * cosg * n.y - wi.y, 2.0f * cosg * n.z - wi.z);
            if (wo.z > 0.0f) fac = fresnel_unpol(cosg, prm[2], prm[3]) * cosg / (wi.z * n.z) * cm_shadow(wi.z, wo.z, sig2);
        }
    }
    *wo_out = wo;
    return fac;
}

// which of several 3-D components scatters (np3d > 1 only; cold for the single-component scenes er3t builds, so out of line)
__device__ __noinline__ float2 pick_component3(const float* __restrict__ ext3, const float2* __restrict__ prop3, int np3d, size_t n3,
                                               unsigned vox, float uc) {
    for (int k = 0; k < np3d; ++k) {
        const float e = __ldg(ext3 + size_t(k) * n3 + vox);
        if (uc < e || k == np3d - 1) return __ldg(prop3 + size_t(k) * n3 + vox);
        uc -= e;
    }
    return make_float2(1.0f, 0.0f);
}

// Persistent-thread photon transport with queue-based path regeneration.
//
// Every WARP owns a pool of NP photon slots in shared memory (NP = 3 x the warp width by default) and every slot is in
// one of five LIFO queues: DEAD (waiting for regeneration), FLY (waiting for the flight phase), TENTATIVE (parked at a
// tentative collision or at TOA), COLLISION (accepted, waiting for the scattering event) and SURFACE.  The warp
// repeatedly picks the FULLEST queue, loads up to 32 photons of it into registers -- one per lane --, runs that ONE
// phase convergently and writes the photons back with their new state:
//   regeneration   next global photon indices from one 64-bit atomic counter (one atomicAdd per batch of 32),
//                  Philox streams keyed by (job seed, global photon index): reproducible on any GPU count,
//   flight         pure geometry on the two-level majorant grid with vertical runs of empty cells (no RNG, no 3-D field
//                  look-ups); lanes that reach a tentative collision / the surface / TOA park; ends when `event_min`
//                  lanes are parked,
//   tentative      Philox draw + layer search + voxel extinction look-up + null-collision rejection; accepted
//                  collisions read (omega, apf), apply implicit capture and hand over through the pool,
//   collision /    local estimates toward every sensor, new direction (phase function / surface BRDF), roulette;
//   surface        the two kinds come from separate queues, so a warp works on one kind at a time.
// With NP >= 96 some queue always holds a full warp of work, so the phases run at (close to) 32 active lanes instead of
// the ~11 a one-photon-per-lane loop reaches (profiles/README.md).  Nothing in the pool is shared between warps: the
// only synchronisation is __syncwarp.
// RAD: radiance sensors present (false only in per-level kernels of pure flux / heating runs: no local-estimate code).
// NO3: no 3-D block at all (plane-parallel flux runs, config 1): neither the generic cell step nor the voxel look-ups exist.
// PL: flux / heating target (every level crossing is tallied, cells are single layers, absorption applied per step).
// FZ: column-frozen photons may occur (IPA and partial-3D solver modes).
// UZ (per-level kernels): the tight 1-D layer step is compiled in (plane-parallel and few-column scenes).
// UZ (other kernels): the 3-D layers are equally thick, vertical runs of empty cells are on (S.uz_ok) and every coarse z cell is one fine
//     slab: the fine slab of a photon that left a box sideways follows from its height, and the layer search for unequal
//     layers is not part of the flight loop at all (the other kernels keep both, decided at run time).  Measured on config 2: the ~35 never-executed instructions of that search cost 3.4 % (the loop is
//     instruction-fetch sensitive, profiles/README.md r02_f), hence a template parameter instead of a run-time test.
// XM: what the radiance kernels carry besides the radiance (XM_NONE for every other kernel).
//   XM_KD (b200rt_run_kd): every history serves S.kd_n gas-absorption terms (kd_leg, kd_le_sum).
//   XM_JAC (b200rt_run_jac): every history also tallies the radiance's derivatives with respect to the gas absorption of
//     S.jac_n layer groups (jac_leg, jac_deposit); radiance, draws and event counters are those of XM_NONE.
//   XM_PLEN (b200rt_run_plen): every history also tallies the distribution of the geometric path lengths behind each
//     pixel's radiance (plen_state, plen_deposit); radiance, draws and event counters are those of XM_NONE.
//   XM_ACT (b200rt_run_act, per-level kernels without radiance): every flight move also adds its track to the actinic flux
//     tally (act_add); flux, heating, draws and event counters are those of XM_NONE.
//   With XM_NONE none of that code exists, so the other kernels are unchanged.
enum { XM_NONE = 0, XM_KD = 1, XM_JAC = 2, XM_PLEN = 3, XM_ACT = 4 };
template <bool PL, bool FZ, int NP, bool CAM, bool UZ, bool RAD, bool NO3, int XM>
__global__ void __launch_bounds__(RT_TPB, RT_MINB) transport_kernel(const __grid_constant__ DevScene S) {
    extern __shared__ float4 smem_f4[];
    constexpr bool KD = XM == XM_KD, JAC = XM == XM_JAC, PLEN = XM == XM_PLEN, ACT = XM == XM_ACT;
    constexpr bool SMT = PL && UZ;      // block-private tallies exist only in the kernels of plane-parallel / few-column scenes
    Smem sm;
    float* pool;
    unsigned short *qD, *qF, *qE, *qC, *qS;
    {
        // 16-byte records first, then the double accumulators, then 4-byte tables, then the photon pools
        float4* q4 = smem_f4;
        float4* slabA = q4; q4 += S.nslab_z;
        int4* slabB = reinterpret_cast<int4*>(q4); q4 += S.nslab_z;
        float4* grpA = q4; q4 += S.ngroup;
        int4* grpB = reinterpret_cast<int4*>(q4); q4 += S.ngroup;
        double* acc = reinterpret_cast<double*>(q4);
        double* acc_atm = acc + 4 * 32;
        double* tal = acc_atm + blockDim.x;
        // private tallies: one copy per block (shared atomics) or one per warp (tal_per_warp)
        const int ntal1 = SMT ? S.ntal_flux_smem + S.ntal_heat_smem + S.ntal_rad_smem + (ACT ? S.ntal_act_smem : 0) : 0;
        const int ntal = ntal1 * (S.tal_per_warp ? int(blockDim.x >> 5) : 1);
        unsigned* cnt = reinterpret_cast<unsigned*>(tal + ntal);
        float* q = reinterpret_cast<float*>(cnt + 8 * 32);
        float* z = q; q += S.nz + 1;
        float* e1tot = q; q += S.nz;
        float* e1cum = q; q += S.nz + 1;
        float* e1 = q; q += S.np1d * S.nz;
        float* o1 = q; q += S.np1d * S.nz;
        float* a1 = q; q += S.np1d * S.nz;
        const int warp = threadIdx.x >> 5;
        pool = q + size_t(warp) * POOL_WORDS(NP);
        qD = reinterpret_cast<unsigned short*>(pool + NFIELD * NP);
        qF = qD + NP;
        qE = qF + NP;
        qC = qE + NP;
        qS = qC + NP;
        for (int i = threadIdx.x; i <= S.nz; i += blockDim.x) { z[i] = S.zgrd[i]; e1cum[i] = S.e1cum[i]; }
        for (int i = threadIdx.x; i < S.nz; i += blockDim.x) e1tot[i] = S.e1tot[i];
        for (int i = threadIdx.x; i < S.np1d * S.nz; i += blockDim.x) { e1[i] = S.e1[i]; o1[i] = S.o1[i]; a1[i] = S.a1[i]; }
        for (int i = threadIdx.x; i < S.nslab_z; i += blockDim.x) {
            const int l0 = S.slab_lay0[i], l1 = S.slab_lay0[i + 1];
            const int cz = S.slab_cz[i];
            const int w = cz >= 0 ? (cz | (S.slab_cg[i] << 16)) : int(0x80000000u | (unsigned(S.slab_cg[i]) << 16));
            slabA[i] = make_float4(S.zgrd[l0], S.zgrd[l1], S.slab_maj1d[i], __int_as_float(w));
            slabB[i] = make_int4(l0, l1, S.slab_cg[i], 0);
        }
        for (int i = threadIdx.x; i < S.ngroup; i += blockDim.x) {
            const int s0 = S.group_lo[i], s1 = S.group_lo[i + 1];
            const int l0 = S.slab_lay0[s0], l1 = S.slab_lay0[s1];
            grpA[i] = make_float4(S.zgrd[l0], S.zgrd[l1], S.group_maj1d[i], __int_as_float(int(unsigned(s0) | (unsigned(s1) << 16))));
            grpB[i] = make_int4(s0, s1, l0, l1);
        }
        if (threadIdx.x < 32) {
            for (int k = 0; k < 4; ++k) acc[k * 32 + threadIdx.x] = 0.0;
            for (int k = 0; k < 8; ++k) cnt[k * 32 + threadIdx.x] = 0u;
        }
        acc_atm[threadIdx.x] = 0.0;
        for (int i = threadIdx.x; i < ntal; i += blockDim.x) tal[i] = 0.0;
        {
            double* mine = tal + (S.tal_per_warp ? warp * ntal1 : 0);
            const int nf = SMT ? S.ntal_flux_smem : 0, nh = SMT ? S.ntal_heat_smem : 0;
            sm.ftal = nf > 0 ? mine : nullptr;
            sm.htal = nh > 0 ? mine + nf : nullptr;
            sm.rtal = (SMT && S.ntal_rad_smem > 0) ? mine + nf + nh : nullptr;
            sm.atal = (ACT && SMT && S.ntal_act_smem > 0) ? mine + nf + nh + S.ntal_rad_smem : nullptr;
            sm.tal_mode = S.tal_per_warp ? 2 : 1;
        }
        for (int i = (threadIdx.x & 31); i < NP; i += 32) qD[i] = (unsigned short)i;
        sm.z = z; sm.e1tot = e1tot; sm.e1cum = e1cum; sm.e1 = e1; sm.o1 = o1; sm.a1 = a1;
        sm.slabA = slabA; sm.slabB = slabB; sm.grpA = grpA; sm.grpB = grpB; sm.acc = acc; sm.acc_atm = acc_atm; sm.cnt = cnt;
    }
    __syncthreads();

    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const unsigned lt_mask = (1u << lane) - 1u;
    const bool want_flux = PL && (S.target & B200RT_TARGET_FLUX) != 0;
    const bool want_rad = RAD && (S.target & B200RT_TARGET_RADIANCE) != 0 && S.nrad > 0;
    const bool want_heat = PL && (S.target & B200RT_TARGET_HEATING) != 0;
    const int nxy = S.nx * S.ny;

    unsigned n_cell = 0;
    // queue lengths (warp-uniform): DEAD, FLY, TENTATIVE (+ escapes), COLLISION, SURFACE.  Queues are LIFO stacks of slot numbers.
    // Once the photon counter is exhausted nD becomes a large negative number: the dead queue never wins again and is no
    // longer written.
    int nD = NP, nF = 0, nE = 0, nC = 0, nS = 0;
    const int ND_DONE = -(1 << 29);

#define POP_SYNC() __syncwarp()
#define RNG4(out)                                                                                     \
    {                                                                                                 \
        const unsigned long long seed_ = S.jobs[p.job].seed;                                          \
        out = philox_u01x4(p.rc0, p.rc1, p.rc2, unsigned(seed_), unsigned(seed_ >> 32));              \
        p.rc2++;                                                                                      \
    }
// KD: factor of W for the gas absorption of the leg from (p.za, p.iza) to (zb, layer izb) of photon p in pool slot `slot`
#define KD_LEG(zb, izb, upd)                                                                                              \
    kd_leg<upd>(S.kd_tab + size_t(p.job) * (S.nz + 2) * S.kd_n, kd_state<NP>(S, slot), S.kd_n, p.za - sm.z[p.iza], p.iza,             \
                (zb) - sm.z[(izb)], (izb), p.iza == (izb) ? p.leg : inv_absdz)
// JAC: add the gas optical path of that leg, per layer group, to the state of pool slot `slot`
#define JAC_LEG(zb, izb)                                                                                                  \
    jac_leg(S.job_abs + size_t(p.job) * S.nz, S.job_cabs + size_t(p.job) * (S.nz + 1), S.jac_lev, S.jac_grp, jac_state<NP>(S, slot), \
            p.za - sm.z[p.iza], p.iza, (zb) - sm.z[(izb)], (izb), p.iza == (izb) ? p.leg : inv_absdz)
// push the slots of the lanes for which `cond` holds onto queue `q` (length `cnt`); `val` is the queue entry
#define QPUSH(q, cnt, cond, val)                                              \
    {                                                                         \
        const unsigned m_ = __ballot_sync(FULL, (cond));                      \
        if (cond) (q)[(cnt) + __popc(m_ & lt_mask)] = (unsigned short)(val);   \
        (cnt) += __popc(m_);                                                  \
    }
// the dead queue: not written once the photon source is exhausted (nD < 0)
#define QPUSH_DEAD(cond, val)                                                          \
    {                                                                                  \
        const unsigned m_ = __ballot_sync(FULL, (cond));                               \
        if ((cond) && nD >= 0) qD[nD + __popc(m_ & lt_mask)] = (unsigned short)(val);   \
        nD += __popc(m_);                                                              \
    }

    for (;;) {
        // =========================================================== pick the fullest queue
        __syncwarp();
        int phase = 0, nbest = nD;
        if (nF >= nbest) { phase = 1; nbest = nF; }
        if (nE >= nbest) { phase = 2; nbest = nE; }
        if (nC >= nbest) { phase = 3; nbest = nC; }
        if (nS > nbest) { phase = 4; nbest = nS; }
        if (nbest == 0) break;

        Photon p;
        if (phase == 0) {
            // ======================================================= regeneration
            const int n = min(nD, 32);
            const bool have = lane < n;
            const int slot = have ? int(qD[nD - 1 - lane]) : 0;
            nD -= n;
            POP_SYNC();                         // queue entries are read before any lane pushes (memory ordering, not just convergence)
            unsigned long long base = 0;
            if (lane == 0) base = atomicAdd(S.counter, (unsigned long long)n);
            base = __shfl_sync(FULL, base, 0);
            const bool exhausted = base + (unsigned long long)n >= S.nphot_local;
            const unsigned long long idx = base + (unsigned long long)lane;
            const bool born = have && idx < S.nphot_local;
            if (born) {
                int lo = 0, hi = S.njob - 1;
                while (lo < hi) {
                    const int mid = (lo + hi + 1) >> 1;
                    if (S.jobs[mid].first <= idx) lo = mid; else hi = mid - 1;
                }
                p.job = lo;
                const DevJob& J = S.jobs[lo];
                p.flags = FL_DIRECT | (J.has_abs ? FL_ABS : 0) | (J.has_fscale ? FL_FSCALE : 0);
                const unsigned long long gidx = (unsigned long long)S.shard_rank + (idx - J.first) * (unsigned long long)S.shard_world;
                p.rc0 = unsigned(gidx); p.rc1 = unsigned(gidx >> 32); p.rc2 = 0;
                float4 u, v;
                RNG4(u);
                RNG4(v);
                p.x = u.x * S.Lx; p.y = u.y * S.Ly; p.z = sm.z[S.nz];
                if (S.src_cos_half < 1.0f) p.d = rotate_dir(S.src, 1.0f - u.z * (1.0f - S.src_cos_half), RT_2PI * u.w);
                else p.d = S.src;
                p.w = 1.0f; p.order = 0;
                p.is = S.nslab_z - 1; p.iz = S.nz - 1;
                p.za = p.z; p.iza = p.iz; p.leg = 0.0f; p.M = 0.0f;
                p.cix = min(S.ncx - 1, int(p.x * S.inv_Sx));
                p.ciy = min(S.ncy - 1, int(p.y * S.inv_Sy));
                if (FZ && S.solver == B200RT_SOLVER_IPA) {
                    p.flags |= FL_FROZEN;
                    p.x = (float(p.cix) + 0.5f) * S.dx; p.y = (float(p.ciy) + 0.5f) * S.dy;
                }
                p.tau = -__logf(v.x);
                CNT_ADD(CNT_PHOT, 1u);
                if (want_flux) { flux_tally<SMT>(S, sm, p, 0, S.nz); flux_tally<SMT>(S, sm, p, 1, S.nz); }
                pool_store<NP>(pool, slot, p, S.inv_Sx, S.inv_Sy);
                if (KD) kd_init(kd_state<NP>(S, slot), S.kd_n);
                if (JAC && (p.flags & FL_ABS)) jac_init(jac_state<NP>(S, slot), S.jac_n);
                if (PLEN) *plen_state<NP>(S, slot) = 0.0f;
            }
            QPUSH(qF, nF, born, slot);
            if (exhausted) nD = ND_DONE;
            else QPUSH_DEAD(have && !born, slot);
            continue;
        }

        if (phase == 1) {
            // ======================================================= flight: geometry only
            // Horizontal position in units of fine majorant cells (ux, uy): faces are integers, so a face distance is one
            // int->float conversion, one subtraction and one multiplication.  1-D slabs behave like one empty coarse
            // cell that spans the whole domain: the periodic wrap is an ordinary face crossing.  One branch-free
            // instruction stream serves fine cells, empty coarse cells and 1-D slab groups.
            const int n = min(nF, 32);
            const bool have = lane < n;
            const int slot = have ? int(qF[nF - 1 - lane]) : 0;
            nF -= n;
            POP_SYNC();
            if (have) pool_load_flight<NP, PL>(pool, slot, p);
            const bool frozen = FZ && (p.flags & FL_FROZEN);
            // direction per fine cell; zero components are replaced by a tiny value (no special cases in the loop)
            float dux = frozen ? 0.0f : p.d.x * S.inv_Sx, duy = frozen ? 0.0f : p.d.y * S.inv_Sy, dzg = p.d.z;
            if (fabsf(dux) < 1e-20f) dux = 1e-20f;
            if (fabsf(duy) < 1e-20f) duy = 1e-20f;
            if (fabsf(dzg) < 1e-12f) dzg = 1e-12f;
            const float kx = 1.0f / dux, ky = 1.0f / duy, kz = 1.0f / dzg;
            const bool upz = dzg > 0.0f;
            const int ox = dux > 0.0f ? 1 : 0, oy = duy > 0.0f ? 1 : 0;
            const int upmx = -ox, upmy = -oy;
            float ux = p.x, uy = p.y;                                  // cell units in the pool
            const float Lux = S.Lux, Luy = S.Luy;
            const int ncx = S.ncx, ncy = S.ncy;
            const int cmx = (1 << S.shx) - 1, cmy = (1 << S.shy) - 1;
            const float inv_Lux = 1.0f / Lux, inv_Luy = 1.0f / Luy;
            const float* __restrict__ majp = S.maj;
            TallyCtx tcf;                                              // per-level kernels: the photon's tally context, once per visit
            if (PL && have) tcf = tally_ctx(S, p.job);
            int ev = EV_NONE;
#pragma unroll 1
            for (int kstep = 0; kstep < S.flight_steps; ++kstep) {
                bool plane = false;
                if (PL && UZ && have && ev == EV_NONE) {
                    // ---- per-level targets: a 1-D layer as its own tight step.  Every level must be tallied, so 1-D layers
                    //      cannot be merged into one box as in the radiance kernels; what can go is the generic cell step
                    //      per layer (a flux run spends most of its steps between TOA and the cloud layer): here a layer
                    //      costs its look-up, the absorption factor and the tallies.  Same physics as the generic step
                    //      below; the periodic wrap is a floor instead of a face crossing.  One layer per pass of the loop,
                    //      so that parked lanes still end the phase early (event_min) and lanes stay in lock-step.
                    const float4 A1 = sm.slabA[p.is];
                    plane = __float_as_int(A1.w) < 0;
                }
                // (The choice is per LANE: which step a photon takes must not depend on the other photons of its warp, or a
                // trajectory would no longer be reproducible to the bit -- a warp-uniform choice was measured and broke
                // tests/test_gpu_bits.py::test_every_photon_is_traced_once_and_shards_add_up.  A warp that mixes 1-D and 3-D
                // lanes therefore pays for both instruction streams, which is why this step is compiled in only for
                // plane-parallel and few-column scenes -- template flag UZ of the per-level kernels: on config 5, whose
                // warps mix most of the time, it cost 18-24 %.)
                if (PL && UZ && plane) {
                    const float4 A1 = sm.slabA[p.is];
                    {
                        const float zf = upz ? A1.y : A1.x;
                        const float seg = fmaxf(0.0f, (zf - p.z) * kz);
                        const float M = A1.z;
                        const bool hit = p.tau < M * seg;
                        const float dmove = hit ? __fdividef(p.tau, M) : seg;
                        if (ACT) CNT_ADD(CNT_TALLY, act_add<SMT>(S, sm, tcf, p, ux, uy, dux, duy, dmove, frozen ? p.ciy * S.nx + p.cix : -1));
                        if (p.flags & FL_ABS) {
                            const float wn = p.w * __expf(-__ldg(S.job_abs + size_t(p.job) * S.nz + p.is) * dmove);
                            ACC_ADD(ACC_ATM, double(p.w) - double(wn));
                            if (want_heat) heat_add<SMT>(S, sm, tcf, p.is, tally_col_u(S, ux, uy), double(p.w) - double(wn));
                            p.w = wn;
                        }
                        p.leg += dmove;
                        ux += dux * dmove; uy += duy * dmove;
                        ux -= Lux * floorf(ux * inv_Lux); uy -= Luy * floorf(uy * inv_Luy);
                        ux = (ux >= 0.0f && ux < Lux) ? ux : 0.0f; uy = (uy >= 0.0f && uy < Luy) ? uy : 0.0f;
                        p.tau = fmaxf(0.0f, p.tau - M * dmove);
                        if (!frozen) {
                            p.cix = min(ncx - 1, max(0, __float2int_rd(ux)));
                            p.ciy = min(ncy - 1, max(0, __float2int_rd(uy)));
                        }
                        if (hit) {
                            p.z += dzg * dmove;
                            ev = EV_TENT;
                            p.M = M;
                            p.flags = (p.flags & ~FL_IN3) | FL_EMPTY;
                        } else {
                            p.z = zf;
                            p.flags &= ~FL_STALE;
                            if (want_flux) {
                                const int col = tally_col_u(S, ux, uy);
                                if (!upz && (p.flags & FL_DIRECT)) flux_add<SMT>(S, sm, tcf, 0, p.is, col, p.w);
                                flux_add<SMT>(S, sm, tcf, upz ? 2 : 1, upz ? p.is + 1 : p.is, col, p.w);
                            }
                            const int nis = upz ? p.is + 1 : p.is - 1;
                            if (nis >= S.nslab_z) ev = EV_ESC;
                            else if (nis < 0) ev = EV_SFC;
                            else p.is = nis;
                        }
                    }
                }
                if (!(NO3 && PL && UZ) && have && ev == EV_NONE && !plane) {
                    if (!PL && (UZ || S.uz_ok) && (p.flags & FL_STALE)) {
                        // left a box of several fine slabs sideways: the slab follows from the height
                        p.is = S.uz_s0 + min(S.ncz - 1, max(0, __float2int_rd((p.z - S.uz_z0) * S.uz_inv)));
                        p.flags &= ~FL_STALE;
                    }
                    float4 A = sm.slabA[p.is];                  // zlo, zhi, 1-D majorant, bits: cz | group << 16 (< 0: 1-D slab)
                    int aw = __float_as_int(A.w);
                    bool in3 = aw >= 0;
                    // one look-up gives both the fine-cell majorant and (sign bit) "the enclosing coarse cell is empty"
                    float mj = -1.0f;
                    if (in3) { mj = __ldg(majp + unsigned(((aw & 0xffff) * ncy + p.ciy) * ncx + p.cix)); ++n_cell; }
                    if (!PL && !UZ && mj >= 0.0f && (p.flags & FL_STALE)) {
                        // (3-D layers of unequal thickness only; boxes never span more than one z group then)
                        // entered a non-empty coarse cell sideways: find the fine z slab of the current height
                        const int gw = __float_as_int(sm.grpA[(aw >> 16) & 0x7fff].w);
                        int lo = gw & 0xffff, hi = int(unsigned(gw) >> 16) - 1;
                        while (lo < hi) {
                            const int mid = (lo + hi + 1) >> 1;
                            if (p.z >= sm.slabA[mid].x) lo = mid; else hi = mid - 1;
                        }
                        p.is = lo;
                        A = sm.slabA[lo]; aw = __float_as_int(A.w);
                        mj = fmaxf(0.0f, __ldg(majp + unsigned(((aw & 0xffff) * ncy + p.ciy) * ncx + p.cix)));
                    }
                    const bool empty = mj < 0.0f;                       // 1-D slabs count as empty
                    // empty boxes span the z groups glo ... ghi: the run of empty coarse cells encoded in the look-up
                    // (3-D block), or the slab's own group
                    // (per-level kernels: every slab is a single layer and its own group, coarse cells are fine cells and there
                    // are no runs -- the slab record A is all a step needs, the group look-ups are compiled out)
                    int glo = 0, ghi = 0;
                    float4 G = A, Gh = A;                               // zlo, zhi, 1-D majorant of the group, bits: slo | shi << 16
                    if (!PL) {
                        const int grp = (aw >> 16) & 0x7fff;
                        const int code = (in3 && empty) ? __float2int_rn(-mj) - 1 : (grp | (grp << 12));
                        glo = code & 0xfff; ghi = (code >> 12) & 0xfff;
                        G = sm.grpA[glo]; Gh = sm.grpA[ghi];
                    }
                    // box in cell units: the fine cell, the enclosing coarse cell, or the whole domain (1-D slabs)
                    const int mx = in3 ? ((empty && !PL) ? cmx : 0) : 0x3fffffff, my = in3 ? ((empty && !PL) ? cmy : 0) : 0x3fffffff;
                    const int bxlo = p.cix & ~mx, bylo = p.ciy & ~my;
                    const int fxi = bxlo + ((mx + 1) & upmx), fyi = bylo + ((my + 1) & upmy);    // face index ahead
                    const float fxf = fminf(float(fxi), Lux), fyf = fminf(float(fyi), Luy);
                    const float zf = upz ? (empty ? Gh.y : A.y) : (empty ? G.x : A.x);
                    const float tx = (fxf - ux) * kx, ty = (fyf - uy) * ky, tz = (zf - p.z) * kz;
                    const float M = empty ? (glo == ghi ? G.z : S.maj1d_blk) : A.z + mj;
                    const float dexit = fmaxf(0.0f, fminf(tz, fminf(tx, ty)));
                    const bool hit = p.tau < M * dexit;
                    const float dmove = hit ? __fdividef(p.tau, M) : dexit;
                    const bool zc = !hit && (tz <= tx) && (tz <= ty);
                    const bool xc = !hit && !zc && (tx <= ty);
                    const bool yc = !hit && !zc && !xc;

                    // ---- move
                    if (ACT) CNT_ADD(CNT_TALLY, act_add<SMT>(S, sm, tcf, p, ux, uy, dux, duy, dmove, frozen ? p.ciy * S.nx + p.cix : -1));
                    if (PL && (p.flags & FL_ABS)) {
                        // flux / heating targets: weight must be current at every level (slabs are single layers here)
                        const float wn = p.w * __expf(-__ldg(S.job_abs + size_t(p.job) * S.nz + p.is) * dmove);
                        ACC_ADD(ACC_ATM, double(p.w) - double(wn));
                        if (want_heat) {
                            heat_add<SMT>(S, sm, tcf, p.is, frozen ? p.ciy * S.nx + p.cix : tally_col_u(S, ux, uy), double(p.w) - double(wn));
                        }
                        p.w = wn;
                    }
                    p.leg += dmove;
                    p.z = zc ? zf : p.z + dzg * dmove;
                    ux += dux * dmove; uy += duy * dmove;
                    p.tau = fmaxf(0.0f, p.tau - M * dmove);

                    // ---- new cell: indices follow the position inside the box just traversed; the axis that was
                    //      crossed is set explicitly (periodic wrap included)
                    int cxn = fxi - 1 + ox, cyn = fyi - 1 + oy;
                    float uxn = fxf, uyn = fyf;
                    if (fxi >= ncx) { cxn = 0; uxn = 0.0f; }
                    if (cxn < 0) { cxn = ncx - 1; uxn = Lux; }
                    if (fyi >= ncy) { cyn = 0; uyn = 0.0f; }
                    if (cyn < 0) { cyn = ncy - 1; uyn = Luy; }
                    const int cxi = min(min(p.cix | mx, ncx - 1), max(bxlo, __float2int_rd(ux)));
                    const int cyi = min(min(p.ciy | my, ncy - 1), max(bylo, __float2int_rd(uy)));
                    p.cix = xc ? cxn : cxi; ux = xc ? uxn : ux;
                    p.ciy = yc ? cyn : cyi; uy = yc ? uyn : uy;

                    const int slo = (empty && !PL) ? (__float_as_int(G.w) & 0xffff) : p.is;
                    const int shi = (empty && !PL) ? int(unsigned(__float_as_int(Gh.w)) >> 16) : p.is + 1;
                    int fl = p.flags;
                    if (mj >= 0.0f) fl &= ~FL_STALE;                              // only a non-empty cell resolves staleness
                    if ((xc || yc) && in3 && shi - slo > 1) fl |= FL_STALE;
                    if (hit) {
                        // park at the tentative collision point; RNG, voxel look-up and the layer search happen in the
                        // event phase
                        ev = EV_TENT;
                        p.M = M;
                        fl = (fl & ~(FL_IN3 | FL_EMPTY)) | (in3 ? FL_IN3 : 0) | (empty ? FL_EMPTY : 0);
                    }
                    if (zc) {
                        fl &= ~FL_STALE;
                        if (PL && want_flux) {
                            const int col = frozen ? p.ciy * S.nx + p.cix : tally_col_u(S, ux, uy);
                            if (!upz && (p.flags & FL_DIRECT)) flux_add<SMT>(S, sm, tcf, 0, p.is, col, p.w);
                            flux_add<SMT>(S, sm, tcf, upz ? 2 : 1, upz ? p.is + 1 : p.is, col, p.w);
                        }
                        const int nis = upz ? shi : slo - 1;
                        if (nis >= S.nslab_z) ev = EV_ESC;
                        else if (nis < 0) ev = EV_SFC;
                        else p.is = nis;
                    }
                    p.flags = fl;
                }
                const unsigned flying = __ballot_sync(FULL, have && ev == EV_NONE);
                if (flying == 0u || n - __popc(flying) >= S.event_min) break;
            }
            if (have) {
                p.x = ux; p.y = uy;
                pool_store_flight<NP, PL>(pool, slot, p);
            }
            QPUSH(qF, nF, have && ev == EV_NONE, slot);
            QPUSH(qE, nE, have && (ev == EV_TENT || ev == EV_ESC), slot | (ev << 8));
            QPUSH(qS, nS, have && ev == EV_SFC, slot);
            continue;
        }

        if (phase == 2) {
            // ======================================================= tentative collisions (and escapes)
            const int n = min(nE, 32);
            const bool have = lane < n;
            int ev = EV_NONE, slot = 0;
            if (have) {
                const int e = int(qE[nE - 1 - lane]);
                slot = e & 255; ev = e >> 8;
            }
            nE -= n;
            POP_SYNC();
            if (have) pool_load<NP>(pool, slot, p, S.Sx, S.Sy);
            bool accepted = false, rejected = false;
            float c_apf = 0.0f, c_uz = 0.0f, c_uw = 0.0f, c_s3 = 0.0f;
            if (ev == EV_ESC) {
                if (!PL && (p.flags & FL_ABS)) {
                    const float inv_absdz = p.d.z != 0.0f ? fabsf(1.0f / p.d.z) : RT_INF;
                    float tr;
                    if (KD) tr = KD_LEG(p.z, S.nz - 1, false);
                    else tr = __expf(-abs_tau(S, sm, p.job, p.za, p.iza, p.z, S.nz - 1, p.leg, inv_absdz));
                    const float wn = p.w * tr;
                    ACC_ADD(ACC_ATM, double(p.w) - double(wn));
                    p.w = wn;
                }
                ACC_ADD(ACC_TOA, double(p.w));
            } else if (ev == EV_TENT) {
                const bool frozen = FZ && (p.flags & FL_FROZEN);
                const bool ev_empty = (p.flags & FL_EMPTY) != 0;
                const bool ev_in3 = !NO3 && (p.flags & FL_IN3) != 0;
                float4 u;
                RNG4(u);
                {
                    // layer of the collision point inside the cell the photon parked in (deferred from the flight phase)
                    const bool by_height = !PL && (UZ || S.uz_ok) && ev_empty && ev_in3;     // the box may span several z groups
                    if (by_height) p.is = S.uz_s0 + min(S.ncz - 1, max(0, __float2int_rd((p.z - S.uz_z0) * S.uz_inv)));
                    const int4 sb = sm.slabB[p.is];
                    int l0 = sb.x, l1 = sb.y;
                    if (ev_empty && !by_height) { const int4 gb = sm.grpB[sb.z]; l0 = gb.z; l1 = gb.w; }
                    p.iz = (l1 - l0 > 1) ? find_layer(sm, l0, l1, p.z) : l0;
                }
                const int izn = p.iz;
                float sig = sm.e1tot[izn];
                float s3 = 0.0f;
                int fx = 0, fy = 0;
                unsigned vox = 0;
                if (ev_in3) {
                    if (frozen) { fx = p.cix; fy = p.ciy; }
                    else {
                        const int shx = ev_empty ? S.shx : 0, shy = ev_empty ? S.shy : 0;
                        const int ixlo = (p.cix >> shx) << shx, ixhi = ixlo + (1 << shx);
                        const int iylo = (p.ciy >> shy) << shy, iyhi = iylo + (1 << shy);
                        fx = min(min(S.nx, ixhi * S.svx) - 1, max(ixlo * S.svx, int(p.x * S.inv_dx)));
                        fy = min(min(S.ny, iyhi * S.svy) - 1, max(iylo * S.svy, int(p.y * S.inv_dy)));
                    }
                    vox = unsigned(((izn - S.iz0) * S.ny + fy) * S.nx + fx);
                    if (!ev_empty) { s3 = __ldg(S.ext3tot + vox); sig += s3; CNT_ADD(CNT_TENT, 1u); }
                }
                p.tau = -__logf(u.y);
                float uc = u.x * p.M;
                if (!(uc < sig)) rejected = true;
                else {
                    // ---- real collision: gas absorption of the finished leg, scattering component, implicit capture
                    if (!PL && (p.flags & FL_ABS)) {
                        const float inv_absdz = p.d.z != 0.0f ? fabsf(1.0f / p.d.z) : RT_INF;
                        float tr;
                        if (KD) tr = KD_LEG(p.z, izn, true);
                        else tr = __expf(-abs_tau(S, sm, p.job, p.za, p.iza, p.z, izn, p.leg, inv_absdz));
                        if (JAC) JAC_LEG(p.z, izn);
                        const float wn = p.w * tr;
                        ACC_ADD(ACC_ATM, double(p.w) - double(wn));
                        p.w = wn;
                    }
                    if (PLEN) *plen_state<NP>(S, slot) += p.leg;     // with or without gas absorption
                    float omg = 1.0f, apf = 0.0f;
                    bool found = false;
                    if (uc < s3) {
                        if (S.np3d == 1) {
                            const float2 pr = __ldg(S.prop3 + vox);
                            omg = pr.x; apf = pr.y; found = true;
                        } else {
                            const float2 pr = pick_component3(S.ext3, S.prop3, S.np3d, size_t(S.nz3) * nxy, vox, uc);
                            omg = pr.x; apf = pr.y; found = true;
                        }
                    } else uc -= s3;
                    if (!found) {
                        for (int k = 0; k < S.np1d; ++k) {
                            const float e = sm.e1[k * S.nz + izn];
                            if (uc < e || k == S.np1d - 1) { omg = sm.o1[k * S.nz + izn]; apf = sm.a1[k * S.nz + izn]; break; }
                            uc -= e;
                        }
                    }
                    CNT_ADD(CNT_COLL, 1u);
                    const float wn = p.w * omg;
                    if (wn < p.w) {
                        ACC_ADD(ACC_ATM, double(p.w) - double(wn));
                        if (want_heat) heat_tally<SMT>(S, sm, p, izn, double(p.w) - double(wn));
                    }
                    p.w = wn;
                    p.order++; p.flags &= ~FL_DIRECT;
                    if (p.w > 0.0f) {
                        accepted = true;
                        c_apf = apf; c_uz = u.z; c_uw = u.w; c_s3 = s3;
                        // the fine cell indices follow the collision point (it may lie anywhere in an empty coarse cell);
                        // 0 <= fx < nx, so the quotient is below ncx
                        if (ev_in3 && !frozen) { p.cix = div_exact(fx, S.svx_mul, S.svx_sh); p.ciy = div_exact(fy, S.svy_mul, S.svy_sh); }
                    }
                }
            }
            if (rejected) pool_store_reject<NP>(pool, slot, p);
            if (accepted) pool_store_accept<NP>(pool, slot, p, c_apf, c_uz, c_uw, c_s3);
            QPUSH(qF, nF, rejected, slot);
            QPUSH(qC, nC, accepted, slot);
            QPUSH_DEAD(have && !rejected && !accepted, slot);
            continue;
        }

        // =========================================================== event phase: collisions (phase 3) or surface hits (4)
        // The two kinds come from separate queues, so a warp works on one kind at a time; they share the local estimate,
        // the roulette and the write-back.
        const int evk = phase == 3 ? EV_COLL : EV_SFC;
        int n, slot = 0;
        if (phase == 3) { n = min(nC, 32); if (lane < n) slot = int(qC[nC - 1 - lane]); nC -= n; }
        else { n = min(nS, 32); if (lane < n) slot = int(qS[nS - 1 - lane]); nS -= n; }
        POP_SYNC();
        const bool have = lane < n;
        float c_uw = 0.0f;
        if (have) { pool_load<NP>(pool, slot, p, S.Sx, S.Sy); c_uw = pool[F_AUX * NP + slot]; }
        bool alive = have;
        if (have) do {
            float4 u = make_float4(0.f, 0.f, 0.f, 0.f);
            float3 newd;
            float apf = 0.0f;
            int fx = 0, fy = 0;
            float s3 = 0.0f;
            int sfc_type = 0;
            float prm[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
            const float3 wi = make_float3(-p.d.x, -p.d.y, -p.d.z);
            if (evk == EV_COLL) {
                // ---- hand-over record of the tentative phase (pool_store_accept)
                apf = p.leg; u.z = p.za; u.w = c_uw; s3 = p.M;
                const bool ev_in3 = !NO3 && (p.flags & FL_IN3) != 0;
                if (ev_in3) {
                    if (FZ && (p.flags & FL_FROZEN)) { fx = p.cix; fy = p.ciy; }
                    else {
                        fx = min(min(S.nx, (p.cix + 1) * S.svx) - 1, max(p.cix * S.svx, int(p.x * S.inv_dx)));
                        fy = min(min(S.ny, (p.ciy + 1) * S.svy) - 1, max(p.ciy * S.svy, int(p.y * S.inv_dy)));
                    }
                }
                if (FZ && S.solver == B200RT_SOLVER_PARTIAL_3D && p.order >= S.iso_ss && !(p.flags & FL_FROZEN)) {
                    if (!ev_in3) { p.cix = min(S.nx - 1, int(p.x * S.inv_dx)); p.ciy = min(S.ny - 1, int(p.y * S.inv_dy)); }
                    else { p.cix = fx; p.ciy = fy; }
                    p.x = (float(p.cix) + 0.5f) * S.dx; p.y = (float(p.ciy) + 0.5f) * S.dy;
                    p.flags |= FL_FROZEN;
                }
            } else {
                // ---- surface hit: path-integrated gas absorption of the leg that ends here
                p.iz = 0; p.is = 0; p.z = sm.z[0]; p.flags &= ~FL_STALE;
                if (!PL && (p.flags & FL_ABS)) {
                    const float inv_absdz = p.d.z != 0.0f ? fabsf(1.0f / p.d.z) : RT_INF;
                    float tr;
                    if (KD) tr = KD_LEG(p.z, 0, true);
                    else tr = __expf(-abs_tau(S, sm, p.job, p.za, p.iza, p.z, 0, p.leg, inv_absdz));
                    if (JAC) JAC_LEG(p.z, 0);
                    const float wn = p.w * tr;
                    ACC_ADD(ACC_ATM, double(p.w) - double(wn));
                    p.w = wn;
                }
                if (PLEN) *plen_state<NP>(S, slot) += p.leg;
                CNT_ADD(CNT_SFC, 1u);
                RNG4(u);
                const bool frozen = FZ && (p.flags & FL_FROZEN);
                int sx, sy;
                if (frozen) {
                    sx = min(S.sfc_nx - 1, int((float(p.cix) + 0.5f) / float(S.nx) * float(S.sfc_nx)));
                    sy = min(S.sfc_ny - 1, int((float(p.ciy) + 0.5f) / float(S.ny) * float(S.sfc_ny)));
                } else {
                    sx = min(S.sfc_nx - 1, max(0, int(p.x * S.inv_Lx * float(S.sfc_nx))));
                    sy = min(S.sfc_ny - 1, max(0, int(p.y * S.inv_Ly * float(S.sfc_ny))));
                }
                const int sn = S.sfc_nx * S.sfc_ny, si = sy * S.sfc_nx + sx;
                sfc_type = __ldg(S.sfc_type + si);
#pragma unroll
                for (int q = 0; q < 5; ++q) prm[q] = __ldg(S.sfc_param + q * sn + si);
                if (want_rad && S.nz3 > 0 && S.iz0 == 0) {
                    fx = frozen ? p.cix : min(S.nx - 1, max(0, int(p.x * S.inv_dx)));
                    fy = frozen ? p.ciy : min(S.ny - 1, max(0, int(p.y * S.inv_dy)));
                    s3 = __ldg(S.ext3tot + fy * S.nx + fx);
                }
            }
            p.za = p.z; p.iza = p.iz; p.leg = 0.0f;

            // ---- local estimates toward every sensor (shared by both event kinds)
            if (want_rad) {
                for (int k = 0; k < S.nrad; ++k) {
                    const DevSensor& se = S.sens[k];
                    if (CAM && se.kind == 1) {
                        int pix = 0;
                        unsigned nv = 0;
                        const bool in3 = (S.nz3 > 0) && p.iz >= S.iz0 && p.iz < S.iz0 + S.nz3;
                        const float c = camera_le(S, sm.z, sm.e1tot, sm.e1cum, se, p.x, p.y, p.z, p.iz, p.job, p.flags & FL_ABS, fx, fy, in3, p.d, evk, apf,
                                                  sfc_type, prm[0], prm[1], prm[2], prm[3], prm[4], &pix, &nv);
                        CNT_ADD(CNT_VISIT, nv);
                        if (c > 0.0f) {
                            const DevJob& J = S.jobs[p.job];
                            rad_add<SMT>(S, sm, size_t(J.slab) * S.rad_slab + se.off + pix, double(c * p.w) * J.rad_fac * se.npix);
                            CNT_ADD(CNT_LE, 1u);
                        }
                        continue;
                    }
                    const float dzs = (se.zt - p.z) * se.s.z;
                    if (!(dzs > 0.0f)) continue;
                    float f;
                    if (evk == EV_COLL) {
                        const float cosang = p.d.x * se.s.x + p.d.y * se.s.y + p.d.z * se.s.z;
                        f = phase_eval(S.pt, apf, cosang) * (0.25f / RT_PI);
                    } else {
                        f = se.s.z > 0.0f ? brdf_eval(sfc_type, prm[0], prm[1], prm[2], prm[3], prm[4], wi, se.s) * se.s.z : 0.0f;
                    }
                    if (f > 0.0f)
                        le_deposit<SMT, KD, JAC, PLEN>(S, sm, se, p, f * p.w, fx, fy, s3,
                                                       KD ? kd_state<NP>(S, slot)
                                                          : (JAC ? jac_state<NP>(S, slot) : (PLEN ? plen_state<NP>(S, slot) : nullptr)));
                }
            }

            // ---- new direction
            if (evk == EV_COLL) {
                float xi_tab = 0.5f;
                if (apf >= 1.0f) { float4 v; RNG4(v); xi_tab = v.x; }
                const float mu = phase_sample(S.pt, apf, u.z, xi_tab);
                newd = rotate_dir(p.d, mu, RT_2PI * u.w);
                if (p.order >= S.iso_max) { ACC_ADD(ACC_RR, -(double(p.w))); alive = false; break; }
            } else {
                float3 wo;
                const float fac = surface_sample(sfc_type, prm[0], prm[1], prm[2], prm[3], prm[4], wi, u, &wo);
                const float wn = p.w * fac;
                ACC_ADD(ACC_SFC, double(p.w) - double(wn));
                p.w = wn;
                if (!(p.w > 0.0f)) { alive = false; break; }
                const float nrm = rsqrtf(wo.x * wo.x + wo.y * wo.y + wo.z * wo.z);
                newd = make_float3(wo.x * nrm, wo.y * nrm, wo.z * nrm);
                p.flags &= ~FL_DIRECT; p.order++;
            }
            p.d = newd;
            if (evk == EV_SFC) {
                if (want_flux) flux_tally<SMT>(S, sm, p, 2, 0);
                if (S.nz3 > 0 && S.iz0 == 0 && !(FZ && (p.flags & FL_FROZEN))) {
                    p.cix = min(S.ncx - 1, max(0, int(p.x * S.inv_Sx)));
                    p.ciy = min(S.ncy - 1, max(0, int(p.y * S.inv_Sy)));
                }
                if (FZ && S.solver == B200RT_SOLVER_PARTIAL_3D && p.order >= S.iso_ss && !(p.flags & FL_FROZEN)) {
                    p.cix = min(S.nx - 1, max(0, int(p.x * S.inv_dx))); p.ciy = min(S.ny - 1, max(0, int(p.y * S.inv_dy)));
                    p.x = (float(p.cix) + 0.5f) * S.dx; p.y = (float(p.ciy) + 0.5f) * S.dy;
                    p.flags |= FL_FROZEN;
                }
            }
            // ---- Russian roulette (Pho_wmin / Pho_wfac), shared
            if (p.w < S.wmin) {
                float xi = u.w;
                if (evk == EV_COLL) { float4 v; RNG4(v); xi = v.x; }
                if (xi * S.wfac < p.w) { ACC_ADD(ACC_RR, double(S.wfac) - double(p.w)); p.w = S.wfac; }
                else { ACC_ADD(ACC_RR, -(double(p.w))); CNT_ADD(CNT_KILL, 1u); alive = false; break; }
            }
            if (p.w < 1e-30f) { ACC_ADD(ACC_RR, -(double(p.w))); alive = false; break; }
        } while (0);

        if (have && alive) pool_store<NP>(pool, slot, p, S.inv_Sx, S.inv_Sy);
        QPUSH(qF, nF, have && alive, slot);
        QPUSH_DEAD(have && !alive, slot);
    }
#undef RNG4
#undef KD_LEG
#undef JAC_LEG
#undef QPUSH
#undef QPUSH_DEAD

    // ---- flush the block-private tallies (one global atomic per non-zero entry and block)
    if (SMT && (sm.ftal || sm.htal || sm.rtal || (ACT && sm.atal))) {
        __syncthreads();
        const int nf = sm.ftal ? S.ntal_flux_smem : 0, nh = sm.htal ? S.ntal_heat_smem : 0, nr = S.ntal_rad_smem;
        const int na = ACT && sm.atal ? S.ntal_act_smem : 0;
        const int ntal1 = nf + nh + nr + na;
        const int ncopy = S.tal_per_warp ? int(blockDim.x >> 5) : 1;
        // every warp computed its own `mine`; copy 0 starts where warp 0's (or the block's) copy does
        const double* mine = ACT ? (sm.ftal ? sm.ftal : (sm.htal ? sm.htal : (sm.rtal ? sm.rtal : sm.atal)))
                                 : (sm.ftal ? sm.ftal : (sm.htal ? sm.htal : sm.rtal));
        const double* tal0 = mine - (S.tal_per_warp ? (threadIdx.x >> 5) * ntal1 : 0);
        for (int i = threadIdx.x; i < ntal1; i += blockDim.x) {
            double v = 0.0;
            for (int c = 0; c < ncopy; ++c) v += tal0[c * ntal1 + i];
            if (v != 0.0) {
                if (i < nf) tally_add(S.flux + i, v);
                else if (i < nf + nh) tally_add(S.heat + (i - nf), v);
                else if (ACT && i >= nf + nh + nr) tally_add(S.xt + (i - nf - nh - nr), v);
                else tally_add(S.rad + (i - nf - nh), v);
                CNT_ADD(CNT_TALLY, 1u);
            }
        }
    }
    // ---- flush the event counters and energy sums: the cell counter lives in a register (one atomic per warp), the rest
    //      in the block's per-lane slots (reduced by the first warp once every warp of the block has finished)
    {
        unsigned long long v = n_cell;
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(FULL, v, o);
        if (lane == 0 && v) atomicAdd(reinterpret_cast<unsigned long long*>(S.stats) + 1, v);
        double a = sm.acc_atm[threadIdx.x];
        for (int o = 16; o > 0; o >>= 1) a += __shfl_down_sync(FULL, a, o);
        if (lane == 0) atomicAdd(&S.stats->w_atm, a);
    }
    __syncthreads();
    if (threadIdx.x < 32) {
        // DevStats order: photons, n_cell, n_tent, n_coll, n_sfc, n_le, n_le_visit, n_tally, n_kill
        const int slot_of[8] = {0, 2, 3, 4, 5, 6, 7, 8};     // CNT_PHOT, CNT_TENT, CNT_COLL, CNT_SFC, CNT_LE, CNT_VISIT, CNT_TALLY, CNT_KILL
        unsigned long long* sc = reinterpret_cast<unsigned long long*>(S.stats);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            unsigned long long v = sm.cnt[i * 32 + lane];
            for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(FULL, v, o);
            if (lane == 0 && v) atomicAdd(sc + slot_of[i], v);
        }
        double dsum[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            double v = sm.acc[i * 32 + lane];
            for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(FULL, v, o);
            dsum[i] = v;
        }
        if (lane == 0) {
            atomicAdd(&S.stats->w_toa, dsum[0]); atomicAdd(&S.stats->w_sfc, dsum[1]);
            atomicAdd(&S.stats->w_rr, dsum[3]);
        }
    }
}
#undef ACC_ADD
#undef CNT_ADD

typedef void (*transport_fn)(const DevScene);
template <int NP>
static transport_fn pick_transport_np(bool pl, bool fz, bool cam, bool uz, bool rad, bool no3, int xm) {
    // CAM (all-sky camera sensors present) is its own specialisation: the camera's local estimate is a large cold path
    // whose register pressure must not tax the satellite-view kernels; it needs the 3-D solver (FZ = false).
    // UZ: see the kernel.  RAD = false exists for the per-level kernels only: a pure flux / heating run carries no
    // local-estimate code at all (those kernels are instruction-fetch bound).
    // KD (b200rt_run_kd) and JAC (b200rt_run_jac): radiance kernels with satellite sensors only; the caller has rejected every other case.
    if (xm == XM_KD) {
        if (fz) return uz ? transport_kernel<false, true, NP, false, true, true, false, XM_KD> : transport_kernel<false, true, NP, false, false, true, false, XM_KD>;
        return uz ? transport_kernel<false, false, NP, false, true, true, false, XM_KD> : transport_kernel<false, false, NP, false, false, true, false, XM_KD>;
    }
    // JAC (b200rt_run_jac): the same kernels as KD, carrying the Jacobian tally instead of the terms
    if (xm == XM_JAC) {
        if (fz) return uz ? transport_kernel<false, true, NP, false, true, true, false, XM_JAC> : transport_kernel<false, true, NP, false, false, true, false, XM_JAC>;
        return uz ? transport_kernel<false, false, NP, false, true, true, false, XM_JAC> : transport_kernel<false, false, NP, false, false, true, false, XM_JAC>;
    }
    // PLEN (b200rt_run_plen): the same kernels, carrying the path-length tally
    if (xm == XM_PLEN) {
        if (fz) return uz ? transport_kernel<false, true, NP, false, true, true, false, XM_PLEN> : transport_kernel<false, true, NP, false, false, true, false, XM_PLEN>;
        return uz ? transport_kernel<false, false, NP, false, true, true, false, XM_PLEN> : transport_kernel<false, false, NP, false, false, true, false, XM_PLEN>;
    }
    // ACT (b200rt_run_act): the per-level kernels without radiance, carrying the actinic tally
    if (xm == XM_ACT) {
        if (fz) return uz ? transport_kernel<true, true, NP, false, true, false, false, XM_ACT> : transport_kernel<true, true, NP, false, false, false, false, XM_ACT>;
        if (uz && no3) return transport_kernel<true, false, NP, false, true, false, true, XM_ACT>;
        return uz ? transport_kernel<true, false, NP, false, true, false, false, XM_ACT> : transport_kernel<true, false, NP, false, false, false, false, XM_ACT>;
    }
    if (pl) {
        if (cam) return transport_kernel<true, false, NP, true, false, true, false, XM_NONE>;
        if (rad) {
            if (fz) return uz ? transport_kernel<true, true, NP, false, true, true, false, XM_NONE> : transport_kernel<true, true, NP, false, false, true, false, XM_NONE>;
            return uz ? transport_kernel<true, false, NP, false, true, true, false, XM_NONE> : transport_kernel<true, false, NP, false, false, true, false, XM_NONE>;
        }
        if (fz) return uz ? transport_kernel<true, true, NP, false, true, false, false, XM_NONE> : transport_kernel<true, true, NP, false, false, false, false, XM_NONE>;
        if (uz && no3) return transport_kernel<true, false, NP, false, true, false, true, XM_NONE>;
        return uz ? transport_kernel<true, false, NP, false, true, false, false, XM_NONE> : transport_kernel<true, false, NP, false, false, false, false, XM_NONE>;
    }
    if (cam) return uz ? transport_kernel<false, false, NP, true, true, true, false, XM_NONE> : transport_kernel<false, false, NP, true, false, true, false, XM_NONE>;
    if (fz) return uz ? transport_kernel<false, true, NP, false, true, true, false, XM_NONE> : transport_kernel<false, true, NP, false, false, true, false, XM_NONE>;
    return uz ? transport_kernel<false, false, NP, false, true, true, false, XM_NONE> : transport_kernel<false, false, NP, false, false, true, false, XM_NONE>;
}
static transport_fn pick_transport(bool pl, bool fz, bool cam, bool uz, bool rad, bool no3, int xm, int np) {
    switch (np) {
        case 64: return pick_transport_np<64>(pl, fz, cam, uz, rad, no3, xm);
        case 128: return pick_transport_np<128>(pl, fz, cam, uz, rad, no3, xm);
        default: return pick_transport_np<96>(pl, fz, cam, uz, rad, no3, xm);
    }
}

// ============================================================================ test-hook kernels
__global__ void philox_fill_kernel(unsigned long long seed, unsigned long long first, unsigned c2, unsigned c3, uint4* out,
                                   long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned long long idx = first + (unsigned long long)i;
    out[i] = philox4x32_10(unsigned(idx), unsigned(idx >> 32), c2, c3, unsigned(seed), unsigned(seed >> 32));
}
__global__ void phase_eval_kernel(PhaseTab pt, float apf, const double* mu, double* out, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = double(phase_eval(pt, apf, float(mu[i])));
}
__global__ void phase_sample_kernel(PhaseTab pt, float apf, const double* xi, double* out, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = double(phase_sample(pt, apf, float(xi[i]), 0.999999f));
}
__global__ void brdf_eval_kernel(int type, const float* prm5, const double* din, const double* dout, double* f, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float p[5];
    for (int q = 0; q < 5; ++q) p[q] = prm5[q];
    const float3 wi = make_float3(-float(din[3 * i]), -float(din[3 * i + 1]), -float(din[3 * i + 2]));
    const float3 wo = make_float3(float(dout[3 * i]), float(dout[3 * i + 1]), float(dout[3 * i + 2]));
    f[i] = double(brdf_eval(type, p[0], p[1], p[2], p[3], p[4], wi, wo));
}

// ============================================================================ host side
namespace {

struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
    void release() { if (p) cudaFree(p); p = nullptr; bytes = 0; }
};

struct Handle {
    int device = 0;
    std::string err;
    bool have_scene = false;
    DevScene S{};
    b200rt_options opt{};
    int numSM = 0;
    size_t smem_bytes = 0, smem_tables = 0;
    int pool_slots = 0;
    bool k_pl = false, k_fz = false, k_cam = false;
    int cmz = 1;                 // fine slabs per coarse z cell of the uploaded scene
    // owned device memory
    std::vector<DevBuf*> pool;
    DevBuf zgrd, e1tot, e1cum, e1, o1, a1, slab_lay0, slab_cz, slab_maj1d, slab_cg, group_lo, group_cz, group_maj1d, gz_lo, empty3, runcode;
    DevBuf st_e, st_o, st_a, st_b, f2c;
    DevBuf ext3tot, prop3, ext3, maj, tu3, pmu, pp, pcdf, pgs, pge, sfc_type, sfc_param;
    DevBuf jobs, job_abs, job_cabs, job_fscale, counter, stats, flag;
    DevBuf kd_tab, kd_rf, kd_r;   // spectral runs: per-term tables and the per-slot term state
    DevBuf jac_lev, jac_grp;     // Jacobian runs: group edges, group of every layer
    DevBuf xs, xt;               // Jacobian and path-length runs: per-slot state, per-pixel tally (DevScene::xs, xt);
                                 // actinic runs: the per-layer tally in xt
    size_t nxt = 0;
    int xt_mode = 0;             // XM_JAC / XM_PLEN / XM_ACT: the last run (since the last upload) was such a run and `xt`
                                 // holds its tally; XM_NONE otherwise
    std::vector<double> xt_key;  // its parameters (group edges, or tpmin, tpmax, ntp): what `accumulate` must match
    int ntal_act_smem = 0;       // doubles of an actinic tally that go to the block-private shared tally (DevScene::ntal_act_smem)
    DevBuf flux, rad, heat;
    size_t nflux = 0, nrad = 0, nheat = 0;
    std::vector<float> h_zgrd;
    double src_flx = 1.0;
    cudaStream_t last_stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    b200rt_stats stats_host{};
    bool ran = false;
    bool inflight = false;       // a run has been launched and not yet waited for (one run in flight per handle)
    uint64_t launches = 0;
    void* pin = nullptr;         // page-locked staging of the per-job tables (uploaded with cudaMemcpyAsync on the run's stream)
    size_t pin_bytes = 0;
    const void* attr_set[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // kernels whose smem attribute is set
    size_t attr_smem[8] = {0, 0, 0, 0, 0, 0, 0, 0};
};

// wait for the run in flight (if any) before its inputs, counters or tallies are touched again
static cudaError_t drain(Handle* H) {
    if (!H->inflight) return cudaSuccess;
    H->inflight = false;
    return cudaStreamSynchronize(H->last_stream);
}

// cudaFuncSetAttribute once per (kernel, shared-memory size)
static cudaError_t set_smem_attr(Handle* H, const void* fn, size_t smem) {
    for (int i = 0; i < 8; ++i)
        if (H->attr_set[i] == fn && H->attr_smem[i] >= smem) return cudaSuccess;
    cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e != cudaSuccess) return e;
    for (int i = 0; i < 8; ++i)
        if (H->attr_set[i] == fn || H->attr_set[i] == nullptr) { H->attr_set[i] = fn; H->attr_smem[i] = smem; return cudaSuccess; }
    H->attr_set[0] = fn; H->attr_smem[0] = smem;
    return cudaSuccess;
}

#define CK(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t e_ = (call);                                                                         \
        if (e_ != cudaSuccess) {                                                                         \
            H->err = std::string("CUDA error: ") + cudaGetErrorString(e_) + " at " + #call;              \
            return B200RT_ERR_CUDA;                                                                      \
        }                                                                                                \
    } while (0)

int fail(Handle* H, int code, const std::string& msg) {
    H->err = msg;
    return code;
}

int dev_alloc(Handle* H, DevBuf& b, size_t bytes) {
    if (b.p && b.bytes >= bytes && b.bytes <= 2 * bytes + 4096) return 0;
    b.release();
    if (bytes == 0) bytes = 16;
    cudaError_t e = cudaMalloc(&b.p, bytes);
    if (e != cudaSuccess) {
        H->err = std::string("cudaMalloc failed: ") + cudaGetErrorString(e);
        b.p = nullptr;
        return B200RT_ERR_NOMEM;
    }
    b.bytes = bytes;
    return 0;
}

template <class T>
int upload(Handle* H, DevBuf& b, const std::vector<T>& v) {
    int rc = dev_alloc(H, b, v.size() * sizeof(T));
    if (rc) return rc;
    if (!v.empty()) CK(cudaMemcpy(b.p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
    return 0;
}

// copy `n` elements from a host-or-device pointer into a host vector
template <class T>
int fetch_host(Handle* H, const T* src, size_t n, std::vector<T>& out) {
    out.resize(n);
    if (n == 0) return 0;
    if (!src) return fail(H, B200RT_ERR_ARG, "null pointer in scene");
    CK(cudaMemcpy(out.data(), src, n * sizeof(T), cudaMemcpyDefault));
    return 0;
}

bool is_device_ptr(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

float3 dir_from_angles(double the, double phi) {
    const double t = the * M_PI / 180.0, p = phi * M_PI / 180.0;
    double x = std::sin(t) * std::cos(p), y = std::sin(t) * std::sin(p), z = std::cos(t);
    if (std::fabs(x) < 1e-15) x = 0;
    if (std::fabs(y) < 1e-15) y = 0;
    return make_float3(float(x), float(y), float(z));
}

}  // namespace

extern "C" {

int b200rt_version(void) { return B200RT_VERSION; }

int b200rt_create(void** handle, int device) {
    if (!handle) return B200RT_ERR_ARG;
    *handle = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) return B200RT_ERR_CUDA;
    if (cudaSetDevice(device) != cudaSuccess) return B200RT_ERR_CUDA;
    Handle* H = new Handle();
    H->device = device;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { delete H; return B200RT_ERR_CUDA; }
    H->numSM = prop.multiProcessorCount;
    cudaEventCreate(&H->ev0);
    cudaEventCreate(&H->ev1);
    *handle = H;
    return B200RT_OK;
}

int b200rt_destroy(void* handle) {
    Handle* H = static_cast<Handle*>(handle);
    if (!H) return B200RT_ERR_ARG;
    cudaSetDevice(H->device);
    DevBuf* all[] = {&H->zgrd, &H->e1tot, &H->e1cum, &H->e1, &H->o1, &H->a1, &H->slab_lay0, &H->slab_cz, &H->slab_maj1d,
                     &H->st_e, &H->st_o, &H->st_a, &H->st_b, &H->f2c, &H->slab_cg, &H->group_lo, &H->group_cz, &H->group_maj1d, &H->gz_lo, &H->empty3, &H->runcode,
                     &H->ext3tot, &H->prop3, &H->ext3, &H->maj, &H->tu3, &H->pmu, &H->pp, &H->pcdf, &H->pgs, &H->pge, &H->sfc_type,
                     &H->sfc_param, &H->jobs, &H->job_abs, &H->job_cabs, &H->job_fscale, &H->counter, &H->stats, &H->flag,
                     &H->kd_tab, &H->kd_rf, &H->kd_r, &H->jac_lev, &H->jac_grp, &H->xs, &H->xt, &H->flux, &H->rad, &H->heat};
    for (DevBuf* b : all) b->release();
    if (H->ev0) cudaEventDestroy(H->ev0);
    if (H->ev1) cudaEventDestroy(H->ev1);
    if (H->pin) cudaFreeHost(H->pin);
    delete H;
    return B200RT_OK;
}

const char* b200rt_last_error(void* handle) {
    Handle* H = static_cast<Handle*>(handle);
    return H ? H->err.c_str() : "null handle";
}

// (mul, sh) of div_exact(): x / d == (umulhi(x, mul) + x) >> sh with sh = ceil(log2 d) and mul = ceil(2^(32+sh) / d) - 2^32.
// The error of the 33-bit reciprocal stays below 1/d for every 0 <= x < 2^31; a power of two gives mul = 0, a plain shift.
static void div_magic(int d, unsigned* mul, int* sh) {
    int s = 0;
    while ((1ll << s) < d) ++s;
    *sh = s;
    *mul = unsigned(((1ull << (32 + s)) + unsigned(d) - 1) / unsigned(d) - (1ull << 32));
}
static int div_exact_host(int x, unsigned mul, int sh) {
    return int((unsigned((unsigned long long)unsigned(x) * mul >> 32) + unsigned(x)) >> sh);
}

int b200rt_upload_scene(void* handle, const b200rt_scene* sc, const b200rt_options* opt) {
    Handle* H = static_cast<Handle*>(handle);
    if (!H) return B200RT_ERR_ARG;
    if (!sc || !opt) return fail(H, B200RT_ERR_ARG, "null scene/options");
    CK(cudaSetDevice(H->device));
    CK(drain(H));
    H->have_scene = false;
    // ------------------------------------------------ validate
    if (sc->nx < 1 || sc->ny < 1 || sc->nz < 1 || sc->np1d < 1) return fail(H, B200RT_ERR_ARG, "nx, ny, nz, np1d must be >= 1");
    if (!(sc->dx > 0) || !(sc->dy > 0)) return fail(H, B200RT_ERR_ARG, "dx, dy must be > 0");
    const int nz = sc->nz, nz3 = sc->nz3, iz0 = sc->iz3l - 1;
    if (nz3 < 0 || (nz3 > 0 && (iz0 < 0 || iz0 + nz3 > nz))) return fail(H, B200RT_ERR_ARG, "3-D block [iz3l, iz3l+nz3) exceeds the atmosphere (Atm_iz3l is 1-based)");
    const bool use_cer = nz3 > 0 && sc->cer3d != nullptr;
    if (nz3 > 0 && (sc->np3d < 1 || !sc->ext3d || (!use_cer && (!sc->omg3d || !sc->apf3d)))) return fail(H, B200RT_ERR_ARG, "3-D block without fields");
    if (use_cer) {
        if (sc->np3d != 1) return fail(H, B200RT_ERR_ARG, "cer3d needs exactly one 3-D component");
        if (sc->nref < 2 || sc->nref > CER_MAX || !sc->ref_tab || !sc->ssa_tab || !sc->asy_tab)
            return fail(H, B200RT_ERR_ARG, "cer3d needs ref / ssa / asy tables of 2 ... 64 entries");
        for (int i = 0; i + 1 < sc->nref; ++i)
            if (!(sc->ref_tab[i + 1] > sc->ref_tab[i])) return fail(H, B200RT_ERR_ARG, "ref_tab must be strictly increasing");
    }
    if (sc->nrad < 0 || sc->nrad > MAX_SENS) return fail(H, B200RT_ERR_ARG, "nrad out of range (max 16)");
    if (sc->layout3d != 0 && sc->layout3d != 1) return fail(H, B200RT_ERR_ARG, "layout3d must be 0 or 1");
    if (opt->nslab < 1) return fail(H, B200RT_ERR_ARG, "nslab must be >= 1");
    if (opt->solver < 0 || opt->solver > 2) return fail(H, B200RT_ERR_ARG, "unknown solver mode");
    if (opt->shard_world < 1 || opt->shard_rank < 0 || opt->shard_rank >= opt->shard_world) return fail(H, B200RT_ERR_ARG, "bad shard rank/world");
    if (opt->pool_slots != 0 && opt->pool_slots != 64 && opt->pool_slots != 96 && opt->pool_slots != 128)
        return fail(H, B200RT_ERR_ARG, "pool_slots must be 0 (auto), 64, 96 or 128");
    if (opt->kernel != 0 && opt->kernel != 8)
        return fail(H, B200RT_ERR_ARG, "options.kernel must be 0 (auto) or 8 (the role-specialised kernel 9 was removed)");
    if (sc->sfc_nx < 1 || sc->sfc_ny < 1 || !sc->sfc_type || !sc->sfc_param) return fail(H, B200RT_ERR_ARG, "surface missing");

    std::vector<double> zg, e1, o1, a1;
    int rc;
    if ((rc = fetch_host(H, sc->zgrd, size_t(nz) + 1, zg))) return rc;
    if ((rc = fetch_host(H, sc->ext1d, size_t(sc->np1d) * nz, e1))) return rc;
    if ((rc = fetch_host(H, sc->omg1d, size_t(sc->np1d) * nz, o1))) return rc;
    if ((rc = fetch_host(H, sc->apf1d, size_t(sc->np1d) * nz, a1))) return rc;
    for (int i = 0; i < nz; ++i) if (!(zg[i + 1] > zg[i])) return fail(H, B200RT_ERR_ARG, "Atm_zgrd0 must be strictly increasing");
    for (size_t i = 0; i < e1.size(); ++i)
        if (!(e1[i] >= 0) || !(o1[i] >= 0 && o1[i] <= 1) || !std::isfinite(a1[i])) return fail(H, B200RT_ERR_ARG, "1-D profile out of range (ext >= 0, 0 <= omg <= 1)");

    DevScene& S = H->S;
    std::memset(&S, 0, sizeof(S));
    S.nx = sc->nx; S.ny = sc->ny; S.nz = nz; S.iz0 = nz3 > 0 ? iz0 : 0; S.nz3 = nz3; S.np1d = sc->np1d; S.np3d = nz3 > 0 ? sc->np3d + (sc->abs3d ? 1 : 0) : 0;
    S.dx = float(sc->dx); S.dy = float(sc->dy); S.Lx = float(sc->dx * sc->nx); S.Ly = float(sc->dy * sc->ny);
    S.inv_dx = float(1.0 / sc->dx); S.inv_dy = float(1.0 / sc->dy);
    S.solver = opt->solver; S.target = opt->target;
    S.wmin = float(opt->wmin); S.wfac = float(opt->wfac > 0 ? opt->wfac : 1.0);
    S.iso_ss = opt->iso_ss > 0 ? opt->iso_ss : 1;
    S.iso_max = opt->iso_max > 0 ? std::min(opt->iso_max, (1 << 24) - 1) : 1000000;
    S.shard_rank = opt->shard_rank; S.shard_world = opt->shard_world;

    // ------------------------------------------------ super-voxel grid
    // Tiny radiance tallies (1 x 1-pixel views of plane-parallel / few-column scenes, the columns of an IPA look-up
    // table) are kept block-private in shared memory, which only the per-level kernels do: such scenes take that route
    size_t rad_doubles = 0;
    if ((opt->target & B200RT_TARGET_RADIANCE) && sc->sensors)
        for (int k = 0; k < sc->nrad; ++k) rad_doubles += size_t(std::max(0, sc->sensors[k].nxr)) * size_t(std::max(0, sc->sensors[k].nyr));
    rad_doubles *= size_t(opt->nslab);
    const bool tiny_rad = opt->smem_tally >= 0 && rad_doubles > 0 && rad_doubles <= 512 && (nz3 <= 0 || size_t(sc->nx) * sc->ny <= 64);
    const bool per_level = (opt->target & (B200RT_TARGET_FLUX | B200RT_TARGET_HEATING)) != 0 || tiny_rad;
    // auto sizes: fine cells of 2 x 2 columns and as many layers as make them 0.6 x as high as wide; coarse (empty-space)
    // cells of 4 x 4 fine cells horizontally and about the same physical height (tuned on the config-2 scene,
    // tools/sweep_sv.py; any choice is unbiased, tests/test_gpu_parity.py sweeps several)
    int svx = opt->svx > 0 ? opt->svx : 2, svy = opt->svy > 0 ? opt->svy : 2, svz = opt->svz;
    if (svz <= 0) {
        svz = 1;
        if (nz3 > 1) {
            const double dz_mean = (zg[iz0 + nz3] - zg[iz0]) / nz3;
            svz = std::max(1, int(std::lround(0.6 * svx * sc->dx / dz_mean)));
        }
    }
    if (opt->solver != B200RT_SOLVER_3D) { svx = 1; svy = 1; }     // column-frozen modes need cell == column
    if (per_level) svz = 1;                                       // every z crossing must be a level crossing
    // coarse (emptiness) level: 2^shx x 2^shy fine cells horizontally, cmz fine slabs vertically
    auto log2floor = [](int v) { int s = 0; while ((2 << s) <= v) ++s; return s; };
    int shx = log2floor(std::max(1, opt->cmx > 0 ? opt->cmx : 4)), shy = log2floor(std::max(1, opt->cmy > 0 ? opt->cmy : 4));
    // With vertical runs of empty cells (3-D layers of equal thickness) the finest z granularity is best: a run is crossed
    // in one step however many groups it spans (tools/sweep_sv.py: cmz = 1 gives 19.7 cell steps per photon on config 2
    // against 21.4 for cmz = 5).  Without runs a coarse cell is about as high as it is wide.
    bool uniform3 = nz3 > 0;
    for (int k = 0; k < nz3; ++k)
        if (std::fabs((zg[iz0 + k + 1] - zg[iz0 + k]) - (zg[iz0 + 1] - zg[iz0])) > 1e-5 * (zg[iz0 + 1] - zg[iz0])) uniform3 = false;
    const bool runs_ok = uniform3 && !per_level && opt->empty_runs >= 0;
    int cmz = opt->cmz > 0 ? opt->cmz : (runs_ok ? 1 : 5);
    if (per_level) { shx = 0; shy = 0; cmz = 1; }
    S.flight_steps = opt->flight_steps > 0 ? opt->flight_steps : 16;
    S.event_min = opt->event_min > 0 ? opt->event_min : 12;
    svx = std::min(svx, sc->nx); svy = std::min(svy, sc->ny); svz = std::max(1, std::min(svz, std::max(1, nz3)));
    S.svx = svx; S.svy = svy; S.svz = svz;
    S.ncx = (sc->nx + svx - 1) / svx; S.ncy = (sc->ny + svy - 1) / svy; S.ncz = nz3 > 0 ? (nz3 + svz - 1) / svz : 0;
    div_magic(svx, &S.svx_mul, &S.svx_sh); div_magic(svy, &S.svy_mul, &S.svy_sh);
    for (int x = 0; x < sc->nx; ++x)
        if (div_exact_host(x, S.svx_mul, S.svx_sh) != x / svx) return fail(H, B200RT_ERR_ARG, "no exact reciprocal of the fine-cell width");
    for (int y = 0; y < sc->ny; ++y)
        if (div_exact_host(y, S.svy_mul, S.svy_sh) != y / svy) return fail(H, B200RT_ERR_ARG, "no exact reciprocal of the fine-cell depth");
    // the z-group tables live in shared memory: at most 128 groups in the 3-D block unless the caller chose cmz
    if (opt->cmz <= 0 && !per_level && S.ncz > 128 * cmz) cmz = (S.ncz + 127) / 128;
    H->cmz = cmz;
    S.Sx = float(sc->dx * svx); S.Sy = float(sc->dy * svy); S.inv_Sx = 1.0f / S.Sx; S.inv_Sy = 1.0f / S.Sy;
    S.inv_Lx = 1.0f / S.Lx; S.inv_Ly = 1.0f / S.Ly;
    S.Lux = float(double(sc->nx) / svx); S.Luy = float(double(sc->ny) / svy);
    S.shx = shx; S.shy = shy;
    S.nCx = (S.ncx + (1 << shx) - 1) >> shx; S.nCy = (S.ncy + (1 << shy) - 1) >> shy;

    // ------------------------------------------------ 1-D tables
    std::vector<float> fz(nz + 1), fe1tot(nz, 0.f), fe1cum(nz + 1, 0.f), fe1(e1.size()), fo1(e1.size()), fa1(e1.size());
    std::vector<double> e1tot_d(nz, 0.0);
    for (int i = 0; i <= nz; ++i) fz[i] = float(zg[i]);
    for (int k = 0; k < sc->np1d; ++k)
        for (int i = 0; i < nz; ++i) {
            e1tot_d[i] += e1[size_t(k) * nz + i];
            fe1[size_t(k) * nz + i] = float(e1[size_t(k) * nz + i]);
            fo1[size_t(k) * nz + i] = float(o1[size_t(k) * nz + i]);
            fa1[size_t(k) * nz + i] = float(a1[size_t(k) * nz + i]);
        }
    {
        double acc = 0;
        for (int i = 0; i < nz; ++i) { fe1tot[i] = float(e1tot_d[i]); fe1cum[i] = float(acc); acc += e1tot_d[i] * (zg[i + 1] - zg[i]); }
        fe1cum[nz] = float(acc);
    }
    H->h_zgrd = fz;
    // z slabs: 1-D layers are their own slab; the 3-D block is cut into ncz slabs of svz layers
    std::vector<int> lay0, czv;
    std::vector<float> maj1d;
    for (int i = 0; i < nz;) {
        int n = 1, cz = -1;
        if (nz3 > 0 && i >= iz0 && i < iz0 + nz3) { cz = (i - iz0) / svz; n = std::min(svz, iz0 + nz3 - i); }
        lay0.push_back(i); czv.push_back(cz);
        float m = 0.f;
        for (int q = i; q < i + n; ++q) m = std::max(m, std::nextafter(fe1tot[q], 1e30f));
        maj1d.push_back(m);
        i += n;
    }
    S.nslab_z = int(czv.size());
    lay0.push_back(nz);
    // coarse z groups: runs of 1-D slabs are merged into one group each (unless every level must be visited);
    // the 3-D block is cut into groups of cmz fine slabs.  A group never mixes 1-D and 3-D slabs.
    std::vector<int> cg(S.nslab_z), g_lo, g_cz, gz_lo, f2c(std::max(1, S.ncz), 0);
    std::vector<float> g_maj1d;
    {
        int ncoarse3 = 0;
        for (int s = 0; s < S.nslab_z;) {
            int e = s + 1;
            if (czv[s] < 0) { if (!per_level) while (e < S.nslab_z && czv[e] < 0) ++e; }
            else while (e < S.nslab_z && czv[e] >= 0 && (czv[e] / cmz) == (czv[s] / cmz)) ++e;
            const int gid = int(g_lo.size());
            g_lo.push_back(s);
            if (czv[s] >= 0) { g_cz.push_back(ncoarse3++); gz_lo.push_back(czv[s]); } else g_cz.push_back(-1);
            float m = 0.f;
            for (int q = s; q < e; ++q) { cg[q] = gid; m = std::max(m, maj1d[q]); }
            g_maj1d.push_back(m);
            s = e;
        }
        g_lo.push_back(S.nslab_z);
        gz_lo.push_back(S.ncz);
        for (int K = 0; K + 1 < int(gz_lo.size()); ++K) for (int q = gz_lo[K]; q < gz_lo[K + 1]; ++q) f2c[q] = K;
        S.ngroup = int(g_cz.size());
    }
    // vertical runs of empty coarse cells need "slab from height" in O(1): 3-D layers of equal thickness, targets that do
    // not tally every level, and group numbers that fit the 12-bit run code
    int gid3_0 = 0;
    S.uz_ok = 0; S.uz_s0 = 0; S.uz_z0 = 0.f; S.uz_inv = 0.f; S.maj1d_blk = 0.f;
    if (nz3 > 0) {
        for (int g = 0; g < S.ngroup; ++g) if (g_cz[g] == 0) gid3_0 = g;
        for (int g = 0; g < S.ngroup; ++g) if (g_cz[g] >= 0) S.maj1d_blk = std::max(S.maj1d_blk, g_maj1d[g]);
        const double dz0 = zg[iz0 + 1] - zg[iz0];
        for (int s = 0; s < S.nslab_z; ++s) if (czv[s] == 0) S.uz_s0 = s;
        if (runs_ok) {
            S.uz_ok = 1;
            S.uz_z0 = float(zg[iz0]);
            S.uz_inv = float(1.0 / (dz0 * svz));
        }
    }
    if (S.ngroup > 4095) return fail(H, B200RT_ERR_ARG, "too many z groups for the packed run code (4095)");
    if ((rc = upload(H, H->zgrd, fz)) || (rc = upload(H, H->e1tot, fe1tot)) || (rc = upload(H, H->e1cum, fe1cum)) ||
        (rc = upload(H, H->e1, fe1)) || (rc = upload(H, H->o1, fo1)) || (rc = upload(H, H->a1, fa1)) ||
        (rc = upload(H, H->slab_lay0, lay0)) || (rc = upload(H, H->slab_cz, czv)) || (rc = upload(H, H->slab_maj1d, maj1d)) ||
        (rc = upload(H, H->slab_cg, cg)) || (rc = upload(H, H->group_lo, g_lo)) || (rc = upload(H, H->group_cz, g_cz)) ||
        (rc = upload(H, H->group_maj1d, g_maj1d)) || (rc = upload(H, H->gz_lo, gz_lo)) || (rc = upload(H, H->f2c, f2c)))
        return rc;
    S.slab_cg = (const int*)H->slab_cg.p; S.group_lo = (const int*)H->group_lo.p; S.group_cz = (const int*)H->group_cz.p;
    S.group_maj1d = (const float*)H->group_maj1d.p;
    S.zgrd = (const float*)H->zgrd.p; S.e1tot = (const float*)H->e1tot.p; S.e1cum = (const float*)H->e1cum.p;
    S.e1 = (const float*)H->e1.p; S.o1 = (const float*)H->o1.p; S.a1 = (const float*)H->a1.p;
    S.slab_lay0 = (const int*)H->slab_lay0.p; S.slab_cz = (const int*)H->slab_cz.p; S.slab_maj1d = (const float*)H->slab_maj1d.p;
    H->smem_tables = 16 * (2 * size_t(S.nslab_z) + 2 * size_t(S.ngroup)) + sizeof(float) * (size_t(nz + 1) * 2 + nz + size_t(3) * sc->np1d * nz);
    H->smem_bytes = H->smem_tables + 32 * (4 * 8 + 8 * 4) + 320 * 8;
    if (H->smem_bytes > 120 * 1024) return fail(H, B200RT_ERR_ARG, "1-D tables exceed shared memory (nz * np1d too large)");
    if (S.ncx > 65535 || S.ncy > 65535 || nz > 65535 || S.ncz > 65535 || S.ngroup > 32767)
        return fail(H, B200RT_ERR_ARG, "grid too large for the packed photon record (65535 cells per axis)");

    // ------------------------------------------------ 3-D block
    if (nz3 > 0) {
        const size_t nvox = size_t(nz3) * sc->ny * sc->nx;
        const size_t nall = nvox * sc->np3d;
        const int np3e = S.np3d;                                   // + 1 when Atm_abst3d is present
        if ((rc = dev_alloc(H, H->ext3tot, nvox * 4)) || (rc = dev_alloc(H, H->prop3, nvox * np3e * 8)) ||
            (rc = dev_alloc(H, H->maj, size_t(S.ncx) * S.ncy * S.ncz * 4)) || (rc = dev_alloc(H, H->empty3, size_t(S.nCx) * S.nCy * (gz_lo.size() - 1))) ||
            (rc = dev_alloc(H, H->runcode, size_t(S.nCx) * S.nCy * (gz_lo.size() - 1) * 4)) || (rc = dev_alloc(H, H->tu3, (nvox + size_t(sc->nx) * sc->ny) * 4)) ||
            (rc = dev_alloc(H, H->flag, 16)))
            return rc;
        // stage the caller's arrays on the device when they are host pointers (staging buffers are kept by the handle
        // so that repeated uploads do not pay cudaMalloc/cudaFree)
        const float *de = sc->ext3d, *dom = sc->omg3d, *da = sc->apf3d;
        if (!is_device_ptr(sc->ext3d)) {
            if ((rc = dev_alloc(H, H->st_e, nall * 4))) return rc;
            CK(cudaMemcpy(H->st_e.p, sc->ext3d, nall * 4, cudaMemcpyDefault));
            de = (const float*)H->st_e.p;
        }
        const float* dcer = nullptr;
        CerTab ctab;
        ctab.n = 0;
        if (use_cer) {
            dom = da = nullptr;
            dcer = sc->cer3d;
            if (!is_device_ptr(sc->cer3d)) {
                if ((rc = dev_alloc(H, H->st_o, nall * 4))) return rc;
                CK(cudaMemcpy(H->st_o.p, sc->cer3d, nall * 4, cudaMemcpyDefault));
                dcer = (const float*)H->st_o.p;
            }
            ctab.n = sc->nref;
            for (int i = 0; i < sc->nref; ++i) { ctab.ref[i] = sc->ref_tab[i]; ctab.ssa[i] = sc->ssa_tab[i]; ctab.asy[i] = sc->asy_tab[i]; }
        } else {
            if (!is_device_ptr(sc->omg3d)) {
                if ((rc = dev_alloc(H, H->st_o, nall * 4))) return rc;
                CK(cudaMemcpy(H->st_o.p, sc->omg3d, nall * 4, cudaMemcpyDefault));
                dom = (const float*)H->st_o.p;
            }
            if (!is_device_ptr(sc->apf3d)) {
                if ((rc = dev_alloc(H, H->st_a, nall * 4))) return rc;
                CK(cudaMemcpy(H->st_a.p, sc->apf3d, nall * 4, cudaMemcpyDefault));
                da = (const float*)H->st_a.p;
            }
        }
        const float* dabs = sc->abs3d;
        if (sc->abs3d && !is_device_ptr(sc->abs3d)) {
            if ((rc = dev_alloc(H, H->st_b, nvox * 4))) return rc;
            CK(cudaMemcpy(H->st_b.p, sc->abs3d, nvox * 4, cudaMemcpyDefault));
            dabs = (const float*)H->st_b.p;
        }
        if (np3e > 1) { if ((rc = dev_alloc(H, H->ext3, nvox * np3e * 4))) return rc; }
        CK(cudaMemset(H->flag.p, 0, 16));
        if (sc->layout3d == 1 && np3e == 1 && sc->ny <= 65535 && (sc->nx + 31) / 32 <= 65535) {
            const dim3 tg((nz3 + 31) / 32, (sc->nx + 31) / 32, sc->ny);
            pack_scene_tiled_kernel<<<tg, dim3(32, 8)>>>(de, dom, da, dcer, ctab, sc->nx, sc->ny, nz3, (float*)H->ext3tot.p, (float2*)H->prop3.p,
                                                         (int*)H->flag.p);
        } else {
            const int nb = int(std::min<size_t>((nvox + 255) / 256, size_t(H->numSM) * 16));
            pack_scene_kernel<<<nb, 256>>>(de, dom, da, dabs, dcer, ctab, sc->np3d, sc->nx, sc->ny, nz3, sc->layout3d, (float*)H->ext3tot.p,
                                           (float2*)H->prop3.p, np3e > 1 ? (float*)H->ext3.p : nullptr, (int*)H->flag.p);
        }
        const int ncell = S.ncx * S.ncy * S.ncz;
        majorant_kernel<<<(ncell + 127) / 128, 128>>>((const float*)H->ext3tot.p, sc->nx, sc->ny, nz3, svx, svy, svz, S.ncx, S.ncy, S.ncz, (float*)H->maj.p);
        const int nC = S.nCx * S.nCy * int(gz_lo.size() - 1);
        empty_kernel<<<(nC + 127) / 128, 128>>>((const float*)H->maj.p, S.ncx, S.ncy, shx, shy, S.nCx, S.nCy, int(gz_lo.size() - 1),
                                                 (const int*)H->gz_lo.p, (unsigned char*)H->empty3.p);
        run_kernel<<<(S.nCx * S.nCy + 127) / 128, 128>>>((const unsigned char*)H->empty3.p, S.nCx, S.nCy, int(gz_lo.size() - 1), gid3_0, S.uz_ok,
                                                          (int*)H->runcode.p);
        mark_empty_kernel<<<(ncell + 127) / 128, 128>>>((float*)H->maj.p, S.ncx, S.ncy, S.ncz, shx, shy, S.nCx, S.nCy, (const int*)H->f2c.p,
                                                          (const int*)H->runcode.p);
        const int ncol = sc->nx * sc->ny;
        tau_up_kernel<<<(ncol + 127) / 128, 128>>>((const float*)H->ext3tot.p, S.zgrd, iz0, sc->nx, sc->ny, nz3, (float*)H->tu3.p);
        CK(cudaGetLastError());
        CK(cudaDeviceSynchronize());
        int bad = 0;
        CK(cudaMemcpy(&bad, H->flag.p, sizeof(int), cudaMemcpyDeviceToHost));
        if (bad & 2) return fail(H, B200RT_ERR_ARG, "Atm_abst3d must be finite and >= 0 (a negative absorption perturbation is not supported)");
        if (bad) return fail(H, B200RT_ERR_ARG, "3-D field out of range (need ext >= 0, 0 <= omg <= 1, finite apf)");
        S.ext3tot = (const float*)H->ext3tot.p; S.prop3 = (const float2*)H->prop3.p; S.ext3 = (const float*)H->ext3.p;
        S.maj = (const float*)H->maj.p; S.tu3 = (const float*)H->tu3.p; S.empty3 = (const unsigned char*)H->empty3.p;
    }

    // ------------------------------------------------ phase tables (built in fp64 on the host, stored fp32)
    S.pt.npf = 0; S.pt.nang = 0;
    if (sc->npf > 0) {
        if (sc->nang < 2) return fail(H, B200RT_ERR_ARG, "phase table needs >= 2 angles");
        std::vector<double> ang, pha;
        if ((rc = fetch_host(H, sc->ang, size_t(sc->nang), ang))) return rc;
        if ((rc = fetch_host(H, sc->pha, size_t(sc->npf) * sc->nang, pha))) return rc;
        const int na = sc->nang;
        std::vector<float> fmu(na), fp(size_t(sc->npf) * na), fc(size_t(sc->npf) * na);
        std::vector<double> mu(na);
        for (int j = 0; j < na; ++j) {
            if (j > 0 && !(ang[j] > ang[j - 1])) return fail(H, B200RT_ERR_ARG, "phase-function angles must increase");
            mu[j] = std::cos(ang[j] * M_PI / 180.0);
            if (j == 0 && std::fabs(ang[j]) < 1e-9) mu[j] = 1.0;
            if (j == na - 1 && std::fabs(ang[j] - 180.0) < 1e-9) mu[j] = -1.0;
            fmu[j] = float(mu[j]);
        }
        for (int t = 0; t < sc->npf; ++t) {
            const double* p = pha.data() + size_t(t) * na;
            std::vector<double> cdf(na, 0.0);
            double area = 0;
            for (int j = 1; j < na; ++j) {
                area += 0.5 * (std::max(0.0, p[j]) + std::max(0.0, p[j - 1])) * (mu[j - 1] - mu[j]);
                cdf[j] = area;
            }
            if (!(area > 0)) return fail(H, B200RT_ERR_ARG, "phase function integrates to zero");
            for (int j = 0; j < na; ++j) {
                fp[size_t(t) * na + j] = float(std::max(0.0, p[j]) * 2.0 / area);
                fc[size_t(t) * na + j] = float(cdf[j] / area);
            }
            fc[size_t(t) * na + na - 1] = 1.0f;
        }
        // guide tables (built from the float32 values the kernel compares against)
        if (na > 65535) return fail(H, B200RT_ERR_ARG, "phase table: at most 65535 angles");
        std::vector<unsigned short> gs(size_t(sc->npf) * RT_NGS), ge(RT_NGE);
        for (int t = 0; t < sc->npf; ++t) {
            const float* F = fc.data() + size_t(t) * na;
            int j = 0;
            for (int k = 0; k < RT_NGS; ++k) {
                const float x = float(k) / float(RT_NGS);
                while (j + 1 <= na - 2 && F[j + 1] <= x) ++j;
                gs[size_t(t) * RT_NGS + k] = (unsigned short)j;
            }
        }
        {
            int j = 0;
            for (int k = 0; k < RT_NGE; ++k) {
                const double q = double(k) * (2.0 / RT_NGE);                 // start of bin k: every mu of the bin is <= 1 - q^2 / 2
                const double muk = 1.0 - 0.5 * q * q;
                while (j + 1 <= na - 2 && double(fmu[j + 1]) >= muk) ++j;
                ge[k] = (unsigned short)std::max(0, j - 1);                  // one interval of slack for the rounding of q
            }
        }
        if ((rc = upload(H, H->pmu, fmu)) || (rc = upload(H, H->pp, fp)) || (rc = upload(H, H->pcdf, fc)) || (rc = upload(H, H->pgs, gs)) ||
            (rc = upload(H, H->pge, ge)))
            return rc;
        S.pt.npf = sc->npf; S.pt.nang = na;
        S.pt.mu = (const float*)H->pmu.p; S.pt.p = (const float*)H->pp.p; S.pt.cdf = (const float*)H->pcdf.p;
        S.pt.gs = (const unsigned short*)H->pgs.p; S.pt.ge = (const unsigned short*)H->pge.p;
    }

    // ------------------------------------------------ surface
    {
        const size_t sn = size_t(sc->sfc_nx) * sc->sfc_ny;
        std::vector<int32_t> st;
        std::vector<float> sp;
        if ((rc = fetch_host(H, sc->sfc_type, sn, st))) return rc;
        if ((rc = fetch_host(H, sc->sfc_param, sn * 5, sp))) return rc;
        for (size_t i = 0; i < sn * 5; ++i)
            if (!std::isfinite(sp[i])) return fail(H, B200RT_ERR_ARG, "non-finite surface parameter");
        for (size_t i = 0; i < sn; ++i) {
            if (st[i] != B200RT_SFC_LAMBERT && st[i] != B200RT_SFC_DSM && st[i] != B200RT_SFC_LSRT)
                return fail(H, B200RT_ERR_ARG, "unsupported surface type (1 Lambertian, 2 DSM, 4 LSRT)");
            // parameter ranges (mca_sfc.py:89-133): albedo-like values in [0, 1], slope variance > 0
            if (st[i] == B200RT_SFC_LAMBERT && !(sp[i] >= 0.f && sp[i] <= 1.f)) return fail(H, B200RT_ERR_ARG, "Lambertian albedo outside [0, 1]");
            if (st[i] == B200RT_SFC_DSM) {
                if (!(sp[i] >= 0.f && sp[i] <= 1.f) || !(sp[sn + i] >= 0.f && sp[sn + i] <= 1.f))
                    return fail(H, B200RT_ERR_ARG, "DSM surface: diffuse albedo and diffuse fraction must lie in [0, 1]");
                if (!(sp[4 * sn + i] > 0.f)) return fail(H, B200RT_ERR_ARG, "DSM surface: slope variance must be > 0");
            }
        }
        if ((rc = upload(H, H->sfc_type, st)) || (rc = upload(H, H->sfc_param, sp))) return rc;
        S.sfc_nx = sc->sfc_nx; S.sfc_ny = sc->sfc_ny;
        S.sfc_type = (const int*)H->sfc_type.p; S.sfc_param = (const float*)H->sfc_param.p;
    }

    // ------------------------------------------------ source and sensors
    S.src = dir_from_angles(sc->src_the, sc->src_phi);
    if (!(S.src.z < 0.0f)) return fail(H, B200RT_ERR_ARG, "source must travel downward (Src_the > 90)");
    S.mu0 = float(-std::cos(sc->src_the * M_PI / 180.0));
    S.src_cos_half = float(std::cos(0.5 * sc->src_qmax * M_PI / 180.0));
    H->src_flx = sc->src_flx;
    S.nrad = sc->nrad;
    long long off = 0;
    for (int k = 0; k < sc->nrad; ++k) {
        const b200rt_sensor& q = sc->sensors[k];
        if (q.kind != 2 && q.kind != 1) return fail(H, B200RT_ERR_ARG, "Rad_mrkind must be 1 (all-sky camera) or 2 (satellite)");
        if (q.nxr < 1 || q.nyr < 1) return fail(H, B200RT_ERR_ARG, "sensor pixel grid must be >= 1 x 1");
        const float3 view = dir_from_angles(q.the, q.phi);
        DevSensor& se = S.sens[k];
        se.kind = q.kind;
        if (q.kind == 1) {
            if (opt->solver != B200RT_SOLVER_3D) return fail(H, B200RT_ERR_ARG, "the all-sky camera needs the 3-D solver");
            if (!(q.qmax > 0 && q.qmax <= 360) || !(q.umax > 0) || !(q.vmax > 0)) return fail(H, B200RT_ERR_ARG, "camera: qmax, umax, vmax must be > 0");
            const double t = q.the * M_PI / 180.0, f = q.phi * M_PI / 180.0, ps = q.psi * M_PI / 180.0;
            const double ct = std::cos(t), st = std::sin(t), cf = std::cos(f), sf = std::sin(f), cp = std::cos(ps), sp = std::sin(ps);
            se.s = view;                                                     // the camera looks along its +z axis
            se.ex = make_float3(float(cp * ct * cf - sp * sf), float(cp * ct * sf + sp * cf), float(-cp * st));
            se.ey = make_float3(float(-sp * ct * cf - cp * sf), float(-sp * ct * sf + cp * cf), float(sp * st));
            se.cpos = make_float3(float(q.xpos * sc->dx * sc->nx), float(q.ypos * sc->dy * sc->ny), float(std::min(zg[nz], std::max(zg[0], q.zloc))));
            se.cos_half_fov = float(std::cos(0.5 * std::min(q.qmax, 360.0) * M_PI / 180.0));
            se.u_half = float(0.5 * q.umax * M_PI / 180.0); se.v_half = float(0.5 * q.vmax * M_PI / 180.0);
            se.pix_per_u = float(q.nxr / (q.umax * M_PI / 180.0)); se.pix_per_v = float(q.nyr / (q.vmax * M_PI / 180.0));
            se.ap2 = float(q.apsize * q.apsize);
            se.inv_sz = 1.0f; se.inv_szs = 1.0f; se.zt = se.cpos.z; se.zref = 0.0f; se.lt = 0;
            for (int i = 0; i < nz; ++i) if (se.zt >= fz[i]) se.lt = i;
            se.nxr = q.nxr; se.nyr = q.nyr; se.vertical_up = 0; se.fast_ok = 0;
            se.off = off;
            se.npix = double(sc->dx) * sc->nx * double(sc->dy) * sc->ny;
            off += (long long)q.nxr * q.nyr;
            continue;
        }
        se.s = make_float3(view.x == 0.f ? 0.f : -view.x, view.y == 0.f ? 0.f : -view.y, -view.z);
        if (std::fabs(se.s.z) < 1e-3f) return fail(H, B200RT_ERR_ARG, "horizontal viewing direction is not supported");
        se.inv_sz = 1.0f / std::fabs(se.s.z);
        se.inv_szs = 1.0f / se.s.z;
        se.zt = float(std::min(zg[nz], std::max(zg[0], q.zloc)));
        se.zref = float(q.zref);
        se.lt = 0;
        for (int i = 0; i < nz; ++i) if (se.zt >= fz[i]) se.lt = i;
        se.nxr = q.nxr; se.nyr = q.nyr;
        se.vertical_up = (se.s.x == 0.f && se.s.y == 0.f && se.s.z > 0.f) ? 1 : 0;
        se.fast_ok = (nz3 == 0 || se.zt >= fz[iz0 + nz3]) ? 1 : 0;
        se.off = off;
        se.npix = double(q.nxr) * double(q.nyr);
        off += (long long)q.nxr * q.nyr;
    }
    S.rad_slab = off;

    // ------------------------------------------------ tallies
    const size_t nxy = size_t(sc->nx) * sc->ny;
    H->nflux = (opt->target & B200RT_TARGET_FLUX) ? size_t(opt->nslab) * 3 * (nz + 1) * nxy : 0;
    H->nrad = ((opt->target & B200RT_TARGET_RADIANCE) && sc->nrad > 0) ? size_t(opt->nslab) * size_t(off) : 0;
    H->nheat = (opt->target & B200RT_TARGET_HEATING) ? size_t(opt->nslab) * nz * nxy : 0;
    if ((rc = dev_alloc(H, H->flux, H->nflux * 8)) || (rc = dev_alloc(H, H->rad, H->nrad * 8)) || (rc = dev_alloc(H, H->heat, H->nheat * 8)) ||
        (rc = dev_alloc(H, H->counter, 16)) || (rc = dev_alloc(H, H->stats, sizeof(DevStats))) || (rc = dev_alloc(H, H->flag, 16)))
        return rc;
    CK(cudaMemset(H->flux.p, 0, std::max<size_t>(16, H->nflux * 8)));
    CK(cudaMemset(H->rad.p, 0, std::max<size_t>(16, H->nrad * 8)));
    CK(cudaMemset(H->heat.p, 0, std::max<size_t>(16, H->nheat * 8)));
    S.flux = (double*)H->flux.p; S.rad = (double*)H->rad.p; S.heat = (double*)H->heat.p;
    S.counter = (unsigned long long*)H->counter.p; S.stats = (DevStats*)H->stats.p;

    // block-private tallies when the whole flux + heating tally is small (plane-parallel / few-column scenes)
    // (smem_tally: < 0 off; 0 auto = one copy per block, warp-aggregated shared atomics; 2 = one copy per warp when that
    // fits 24 KB, plain read-modify-write after the aggregation)
    S.ntal_flux_smem = 0; S.ntal_heat_smem = 0; S.ntal_rad_smem = 0; S.tal_per_warp = 0; S.ntal_act_smem = 0;
    H->ntal_act_smem = 0;
    if (opt->smem_tally >= 0 && per_level && (nz3 <= 0 || size_t(sc->nx) * sc->ny <= 64)) {      // the scenes whose kernels hold private tallies
        // two blocks per SM must still fit (pools of 96 slots per warp + tables + accumulators + the private tallies)
        auto fits2 = [&](size_t ntal) {
            const size_t smem = H->smem_tables + 32 * (4 * 8 + 8 * 4) + size_t(RT_TPB) * 8 + size_t(RT_TPB / 32) * size_t(POOL_WORDS(96)) * 4 + 8 * ntal;
            return 2 * (smem + 1024) <= size_t(227) * 1024;
        };
        if (H->nflux + H->nheat <= 2048 && fits2(H->nflux + H->nheat)) { S.ntal_flux_smem = int(H->nflux); S.ntal_heat_smem = int(H->nheat); }
        if (H->nrad > 0 && H->nrad <= 512 && fits2(size_t(S.ntal_flux_smem) + S.ntal_heat_smem + H->nrad)) S.ntal_rad_smem = int(H->nrad);
        const size_t tot = size_t(S.ntal_flux_smem) + S.ntal_heat_smem + S.ntal_rad_smem;
        if (opt->smem_tally == 2 && tot > 0 && tot * 8 * (RT_TPB / 32) <= 24 * 1024) S.tal_per_warp = 1;
        // an actinic run's tally joins them when all of it still fits (same limits, per-warp copies included)
        const size_t nact = 2 * size_t(opt->nslab) * nz * nxy;
        if (tot > 0 && tot == H->nflux + H->nheat + H->nrad && tot + nact <= 2048 && fits2(tot + nact) &&
            (!S.tal_per_warp || (tot + nact) * 8 * (RT_TPB / 32) <= 24 * 1024))
            H->ntal_act_smem = int(nact);
    }
    H->k_pl = per_level; H->k_fz = (opt->solver != B200RT_SOLVER_3D);
    H->k_cam = false;
    for (int k = 0; k < sc->nrad; ++k) if (sc->sensors[k].kind == 1) H->k_cam = true;
    H->pool_slots = opt->pool_slots;
    H->opt = *opt;
    H->have_scene = true;
    H->ran = false;
    H->xt_mode = XM_NONE;
    return B200RT_OK;
}

}  // extern "C"

// what a Jacobian, path-length or actinic run adds to b200rt_run: the kernels' mode and its parameters
struct XtArgs {
    int mode = XM_NONE;                        // XM_NONE, XM_JAC, XM_PLEN or XM_ACT
    const int32_t* edges = nullptr;            // XM_JAC: edges[ngrp+1], the layer groups of the Jacobian tally
    int ngrp = 0;
    double tpmin = 0.0, tpmax = 0.0;           // XM_PLEN: ntp bins on [tpmin, tpmax) metres
    int ntp = 0;
};

// b200rt_run (kd == nullptr, xa.mode = XM_NONE), b200rt_run_kd (kd[njob]: the gas-absorption terms of every job),
// b200rt_run_jac, b200rt_run_plen and b200rt_run_act (xa)
static int run_jobs(Handle* H, const b200rt_job* jobs, const b200rt_kd* kd, const XtArgs& xa, int njob, int accumulate,
                    void* cuda_stream) {
    if (!H->have_scene) return fail(H, B200RT_ERR_STATE, "b200rt_run called before b200rt_upload_scene");
    if (!jobs || njob < 1) return fail(H, B200RT_ERR_ARG, "no jobs");
    if (njob > 65535) return fail(H, B200RT_ERR_ARG, "at most 65535 jobs per run");
    DevScene& S = H->S;
    const int nz = S.nz;
    const bool k_rad = (S.target & B200RT_TARGET_RADIANCE) != 0 && S.nrad > 0;
    int kd_n = 0;
    if (kd) {
        if (H->k_pl)
            return fail(H, B200RT_ERR_ARG, "b200rt_run_kd: radiance targets only (no flux / heating; tiny radiance tallies held in shared memory "
                                           "need options.smem_tally = -1)");
        if (!k_rad) return fail(H, B200RT_ERR_ARG, "b200rt_run_kd: needs the radiance target and at least one sensor");
        if (H->k_cam) return fail(H, B200RT_ERR_ARG, "b200rt_run_kd: the all-sky camera (Rad_mrkind = 1) is not supported");
        for (int j = 0; j < njob; ++j) {
            const b200rt_kd& k = kd[j];
            if (k.nkd < 1 || k.nkd > 32) return fail(H, B200RT_ERR_ARG, "b200rt_run_kd: nkd must be 1 ... 32");
            if (!k.wkd || !k.abs1d || !k.rad_scale) return fail(H, B200RT_ERR_ARG, "b200rt_run_kd: wkd, abs1d and rad_scale are required");
            if (jobs[j].abs1d || jobs[j].flx_scale) return fail(H, B200RT_ERR_ARG, "b200rt_run_kd: job.abs1d and job.flx_scale must be NULL");
            double sw = 0;
            for (int g = 0; g < k.nkd; ++g) {
                if (!(k.wkd[g] >= 0) || !std::isfinite(k.wkd[g]) || !std::isfinite(k.rad_scale[g]))
                    return fail(H, B200RT_ERR_ARG, "b200rt_run_kd: wkd must be finite and >= 0, rad_scale finite");
                sw += k.wkd[g];
            }
            if (!(sw > 0)) return fail(H, B200RT_ERR_ARG, "b200rt_run_kd: the weights wkd sum to zero");
            kd_n = std::max(kd_n, k.nkd);
        }
    }
    const bool plen = xa.mode == XM_PLEN, act = xa.mode == XM_ACT;
    const int32_t* edges = xa.mode == XM_JAC ? xa.edges : nullptr;
    const int jac_n = edges ? xa.ngrp : 0;
    size_t xt_n = 0;              // doubles per radiance pixel of the extra tally (DevScene::xt)
    size_t nxt = 0;               // doubles of the whole extra tally
    std::vector<double> xt_key;
    if (act) {
        const std::string who = "b200rt_run_act: ";
        if (!(S.target & (B200RT_TARGET_FLUX | B200RT_TARGET_HEATING)))
            return fail(H, B200RT_ERR_ARG, who + "needs the flux or heating target");
        if (H->k_cam) return fail(H, B200RT_ERR_ARG, who + "the all-sky camera (Rad_mrkind = 1) is not supported");
        if (k_rad) return fail(H, B200RT_ERR_ARG, who + "no radiance sensors in the same run (drop the radiance target)");
        if (accumulate && H->ran && H->xt_mode != XM_ACT)
            return fail(H, B200RT_ERR_ARG, who + "accumulate needs the previous run to be an actinic run");
        nxt = 2 * size_t(H->opt.nslab) * nz * size_t(S.nx) * size_t(S.ny);
    } else if (xa.mode != XM_NONE) {
        const std::string who = edges ? "b200rt_run_jac: " : "b200rt_run_plen: ";
        if (H->k_pl)
            return fail(H, B200RT_ERR_ARG, who + "radiance targets only (no flux / heating; tiny radiance tallies held in shared memory "
                                                 "need options.smem_tally = -1)");
        if (!k_rad) return fail(H, B200RT_ERR_ARG, who + "needs the radiance target and at least one sensor");
        if (H->k_cam) return fail(H, B200RT_ERR_ARG, who + "the all-sky camera (Rad_mrkind = 1) is not supported");
        if (edges) {
            const int ngrp = xa.ngrp;
            if (ngrp < 1 || ngrp > 64) return fail(H, B200RT_ERR_ARG, who + "ngrp must be 1 ... 64");
            if (edges[0] != 0 || edges[ngrp] != nz)
                return fail(H, B200RT_ERR_ARG, who + "edges must start at layer 0 and end at nz (" + std::to_string(nz) + ")");
            for (int j = 0; j < ngrp; ++j)
                if (!(edges[j + 1] > edges[j])) return fail(H, B200RT_ERR_ARG, who + "edges must be strictly increasing");
            xt_n = size_t(ngrp);
            xt_key.assign(edges, edges + ngrp + 1);
        } else {
            if (xa.ntp < 1 || xa.ntp > 1024) return fail(H, B200RT_ERR_ARG, who + "ntp must be 1 ... 1024");
            // (the kernels bin in fp32: the edges must stay finite and distinct there too)
            if (!std::isfinite(float(xa.tpmin)) || !std::isfinite(float(xa.tpmax)) || !(xa.tpmin >= 0.0) ||
                !(float(xa.tpmax) > float(xa.tpmin)))
                return fail(H, B200RT_ERR_ARG, who + "tpmin and tpmax must be finite with 0 <= tpmin < tpmax");
            xt_n = size_t(xa.ntp) + 3;
            xt_key = {xa.tpmin, xa.tpmax, double(xa.ntp)};
        }
        if (accumulate && H->ran && !(H->xt_mode == xa.mode && H->xt_key == xt_key))
            return fail(H, B200RT_ERR_ARG, who + (edges ? "accumulate needs the previous run to be a Jacobian run with the same edges"
                                                        : "accumulate needs the previous run to be a path-length run with the same binning"));
        nxt = H->nrad * xt_n;
    }
    CK(cudaSetDevice(H->device));
    CK(drain(H));                 // one run in flight per handle: the previous one still reads the job tables and counters
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    // per-job tables (and the per-term tables of a spectral run) are built in page-locked memory and uploaded
    // asynchronously on the caller's stream
    auto al = [](size_t b) { return (b + 15) & ~size_t(15); };
    const size_t b_jobs = size_t(njob) * sizeof(DevJob), b_abs = size_t(njob) * nz * 4, b_cabs = size_t(njob) * (nz + 1) * 4,
                 b_fs = size_t(njob) * (nz + 1) * 8, b_kt = size_t(njob) * (nz + 2) * kd_n * 8, b_kr = size_t(njob) * kd_n * 8,
                 b_jl = edges ? size_t(jac_n + 1) * 4 : 0, b_jg = edges ? size_t(nz) : 0;
    const size_t o_jobs = 0, o_fs = al(b_jobs), o_abs = o_fs + al(b_fs), o_cabs = o_abs + al(b_abs), o_kt = o_cabs + al(b_cabs),
                 o_kr = o_kt + al(b_kt), o_jl = o_kr + al(b_kr), o_jg = o_jl + al(b_jl);
    const size_t need = o_jg + b_jg + 16;
    if (need > H->pin_bytes) {
        if (H->pin) cudaFreeHost(H->pin);
        H->pin = nullptr; H->pin_bytes = 0;
        CK(cudaMallocHost(&H->pin, 2 * need));
        H->pin_bytes = 2 * need;
    }
    char* pin = static_cast<char*>(H->pin);
    DevJob* dj = reinterpret_cast<DevJob*>(pin + o_jobs);
    double* jfs = reinterpret_cast<double*>(pin + o_fs);
    float* jabs = reinterpret_cast<float*>(pin + o_abs);
    float* jcabs = reinterpret_cast<float*>(pin + o_cabs);
    float2* kt = reinterpret_cast<float2*>(pin + o_kt);
    double* kr = reinterpret_cast<double*>(pin + o_kr);
    int* jl = reinterpret_cast<int*>(pin + o_jl);
    unsigned char* jg = reinterpret_cast<unsigned char*>(pin + o_jg);
    for (int j = 0; j < jac_n; ++j) {
        jl[j] = edges[j];
        for (int i = edges[j]; i < edges[j + 1]; ++i) jg[i] = (unsigned char)j;
    }
    if (edges) jl[jac_n] = nz;
    std::memset(jabs, 0, b_abs);
    std::memset(jcabs, 0, b_cabs);
    std::memset(kt, 0, b_kt);                    // terms beyond a job's nkd: no absorption, weight 0, radiance factor 0
    std::memset(kr, 0, b_kr);
    unsigned long long acc = 0;
    for (int j = 0; j < njob; ++j) {
        const b200rt_job& q = jobs[j];
        if (q.nphot < 0) return fail(H, B200RT_ERR_ARG, "negative photon count");
        if (q.slab < 0 || q.slab >= H->opt.nslab) return fail(H, B200RT_ERR_ARG, "job slab out of range");
        DevJob& d = dj[j];
        const long long world = S.shard_world, rank = S.shard_rank;
        const long long cnt = q.nphot > rank ? (q.nphot - rank + world - 1) / world : 0;
        d.first = acc; d.count = (unsigned long long)cnt; acc += d.count;
        d.seed = q.seed;
        d.norm = q.nphot > 0 ? double(S.mu0) * H->src_flx / double(q.nphot) : 0.0;
        d.rad_fac = d.norm * q.rad_scale;
        d.slab = q.slab;
        d.has_abs = 0; d.has_fscale = 0; d._pad = 0;
        if (q.abs1d) {
            double c = 0;
            for (int i = 0; i < nz; ++i) {
                const double a = q.abs1d[i];
                if (!(a >= 0) || !std::isfinite(a)) return fail(H, B200RT_ERR_ARG, "Atm_abs1d must be finite and >= 0");
                if (a > 0) d.has_abs = 1;
                jabs[size_t(j) * nz + i] = float(a);
                jcabs[size_t(j) * (nz + 1) + i] = float(c);
                c += a * (double(H->h_zgrd[i + 1]) - double(H->h_zgrd[i]));
            }
            jcabs[size_t(j) * (nz + 1) + nz] = float(c);
        }
        if (kd) {
            const b200rt_kd& k = kd[j];
            double sw = 0;
            for (int g = 0; g < k.nkd; ++g) sw += k.wkd[g];
            float2* tj = kt + size_t(j) * (nz + 2) * kd_n;
            for (int g = 0; g < k.nkd; ++g) {
                tj[g] = make_float2(float(k.wkd[g] / sw), 0.0f);
                kr[size_t(j) * kd_n + g] = d.rad_fac * k.rad_scale[g];
                double c = 0;
                for (int i = 0; i < nz; ++i) {
                    const double a = k.abs1d[size_t(g) * nz + i];
                    if (!(a >= 0) || !std::isfinite(a)) return fail(H, B200RT_ERR_ARG, "b200rt_run_kd: abs1d must be finite and >= 0");
                    if (a > 0) d.has_abs = 1;
                    tj[size_t(1 + i) * kd_n + g] = make_float2(float(c), float(a));
                    c += a * (double(H->h_zgrd[i + 1]) - double(H->h_zgrd[i]));
                }
                tj[size_t(1 + nz) * kd_n + g] = make_float2(float(c), 0.0f);
            }
        }
        // complete tally scale per level: normalisation x columns in the domain x the caller's per-level factor
        const double nxy_d = double(S.nx) * double(S.ny);
        for (int i = 0; i <= nz; ++i) jfs[size_t(j) * (nz + 1) + i] = d.norm * nxy_d * (q.flx_scale ? q.flx_scale[i] : 1.0);
        if (q.flx_scale) d.has_fscale = 1;
        d.flux_off = (unsigned long long)q.slab * 3ull * (unsigned long long)(nz + 1) * (unsigned long long)(S.nx) * (unsigned long long)(S.ny);
        d.heat_off = (unsigned long long)q.slab * (unsigned long long)nz * (unsigned long long)(S.nx) * (unsigned long long)(S.ny);
    }
    int rc;
    if ((rc = dev_alloc(H, H->jobs, b_jobs)) || (rc = dev_alloc(H, H->job_abs, b_abs)) || (rc = dev_alloc(H, H->job_cabs, b_cabs)) ||
        (rc = dev_alloc(H, H->job_fscale, b_fs)) || (rc = dev_alloc(H, H->kd_tab, b_kt)) ||
        (rc = dev_alloc(H, H->kd_rf, b_kr)))
        return rc;
    CK(cudaMemcpyAsync(H->jobs.p, dj, b_jobs, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(H->job_abs.p, jabs, b_abs, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(H->job_cabs.p, jcabs, b_cabs, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(H->job_fscale.p, jfs, b_fs, cudaMemcpyHostToDevice, st));
    if (kd) {
        CK(cudaMemcpyAsync(H->kd_tab.p, kt, b_kt, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(H->kd_rf.p, kr, b_kr, cudaMemcpyHostToDevice, st));
    }
    if (edges) {
        if ((rc = dev_alloc(H, H->jac_lev, b_jl)) || (rc = dev_alloc(H, H->jac_grp, b_jg))) return rc;
        CK(cudaMemcpyAsync(H->jac_lev.p, jl, b_jl, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(H->jac_grp.p, jg, b_jg, cudaMemcpyHostToDevice, st));
    }
    if (nxt) {
        // `xt` is resized / zeroed from here on: until this run has launched it holds no valid tally (a failure below must
        // not leave b200rt_read_jac / _plen / _act reading the previous run's size out of this buffer)
        H->xt_mode = XM_NONE;
        if ((rc = dev_alloc(H, H->xt, nxt * 8))) return rc;
        // zeroed unless this run adds to the previous run of the same kind (the other tallies are zero after an upload anyway)
        if (!accumulate || !H->ran) CK(cudaMemsetAsync(H->xt.p, 0, nxt * 8, st));
    }
    S.ntal_act_smem = act ? H->ntal_act_smem : 0;
    S.jac_n = jac_n; S.jac_lev = (const int*)H->jac_lev.p; S.jac_grp = (const unsigned char*)H->jac_grp.p; S.xt = (double*)H->xt.p;
    S.pl_ntp = plen ? xa.ntp : 0; S.pl_lo = float(xa.tpmin); S.pl_hi = float(xa.tpmax);
    S.pl_inv_w = plen ? float(double(xa.ntp) / (double(S.pl_hi) - double(S.pl_lo))) : 0.0f;
    S.kd_n = kd_n; S.kd_tab = (const float2*)H->kd_tab.p; S.kd_rf = (const double*)H->kd_rf.p;
    S.njob = njob; S.jobs = (const DevJob*)H->jobs.p; S.job_abs = (const float*)H->job_abs.p;
    S.job_cabs = (const float*)H->job_cabs.p; S.job_fscale = (const double*)H->job_fscale.p;
    S.nphot_local = acc;

    if (!accumulate) {
        if (H->nflux) CK(cudaMemsetAsync(H->flux.p, 0, H->nflux * 8, st));
        if (H->nrad) CK(cudaMemsetAsync(H->rad.p, 0, H->nrad * 8, st));
        if (H->nheat) CK(cudaMemsetAsync(H->heat.p, 0, H->nheat * 8, st));
    }
    CK(cudaMemsetAsync(H->counter.p, 0, 16, st));
    CK(cudaMemsetAsync(H->stats.p, 0, sizeof(DevStats), st));

    // launch shape: the per-warp photon pools decide how many blocks fit on an SM (shared memory), see DESIGN.md
    int tpb = H->opt.threads_per_block > 0 ? H->opt.threads_per_block : RT_TPB;
    tpb = std::min(RT_TPB, std::max(32, (tpb / 32) * 32));
    const int np = H->pool_slots ? H->pool_slots : 96;
    int bps = 0;
    // UZ kernels: equally thick 3-D layers with runs (S.uz_ok) -- or no 3-D block at all (the layer search is dead code then)
    const bool k_uz = H->k_pl ? (S.nz3 <= 0 || size_t(S.nx) * S.ny <= 64) : ((S.uz_ok != 0 && H->cmz == 1) || S.nz3 <= 0);
    transport_fn kern = pick_transport(H->k_pl, H->k_fz, H->k_cam, k_uz, k_rad, S.nz3 <= 0, kd ? XM_KD : xa.mode, np);
    const size_t smem = H->smem_tables + 32 * (4 * 8 + 8 * 4) + size_t(tpb) * 8 + size_t(tpb / 32) * size_t(POOL_WORDS(np)) * 4 +
                        8 * size_t(S.ntal_flux_smem + S.ntal_heat_smem + S.ntal_rad_smem + S.ntal_act_smem) * size_t(S.tal_per_warp ? RT_TPB / 32 : 1);
    if (smem > 227 * 1024) return fail(H, B200RT_ERR_ARG, "photon pools + 1-D tables exceed shared memory; lower threads_per_block or pool_slots");
    CK(set_smem_attr(H, (const void*)kern, smem));
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, kern, tpb, smem));
    if (bps < 1) return fail(H, B200RT_ERR_CUDA, "transport kernel does not fit on an SM");
    if (H->opt.blocks_per_sm > 0) bps = std::min(bps, H->opt.blocks_per_sm);
    unsigned long long want = (acc + tpb - 1) / tpb;
    int grid = int(std::min<unsigned long long>((unsigned long long)H->numSM * bps, std::max<unsigned long long>(1, want)));
    if (kd) {
        // per-term state of every pool slot of the launch: [block][warp][slot][kd_n]
        if ((rc = dev_alloc(H, H->kd_r, size_t(grid) * (tpb / 32) * np * kd_n * 4))) return rc;
        S.kd_r = (float*)H->kd_r.p;
    }
    if (xt_n) {     // (JAC, PLEN)
        // per-slot state of every pool slot of the launch: [block][warp][slot][jac_n] per-group paths, or [block][warp][slot] path
        if ((rc = dev_alloc(H, H->xs, size_t(grid) * (tpb / 32) * np * (edges ? jac_n : 1) * 4))) return rc;
        S.xs = (float*)H->xs.p;
    }
    CK(cudaEventRecord(H->ev0, st));
    kern<<<grid, tpb, smem, st>>>(S);
    CK(cudaGetLastError());
    CK(cudaEventRecord(H->ev1, st));
    H->last_stream = st;
    H->ran = true;
    H->inflight = true;
    H->launches = 1;
    H->xt_mode = xa.mode;
    if (nxt) {
        H->xt_key = xt_key;
        H->nxt = nxt;
    }
    return B200RT_OK;
}

extern "C" {

int b200rt_run(void* handle, const b200rt_job* jobs, int njob, int accumulate, void* cuda_stream) {
    Handle* H = static_cast<Handle*>(handle);
    if (!H) return B200RT_ERR_ARG;
    return run_jobs(H, jobs, nullptr, XtArgs(), njob, accumulate, cuda_stream);
}

int b200rt_run_kd(void* handle, const b200rt_job* jobs, const b200rt_kd* kd, int njob, int accumulate, void* cuda_stream) {
    Handle* H = static_cast<Handle*>(handle);
    if (!H) return B200RT_ERR_ARG;
    if (!kd) return fail(H, B200RT_ERR_ARG, "b200rt_run_kd: kd is NULL");
    return run_jobs(H, jobs, kd, XtArgs(), njob, accumulate, cuda_stream);
}

int b200rt_run_jac(void* handle, const b200rt_job* jobs, int njob, const int32_t* edges, int ngrp, int accumulate, void* cuda_stream) {
    Handle* H = static_cast<Handle*>(handle);
    if (!H) return B200RT_ERR_ARG;
    if (!edges) return fail(H, B200RT_ERR_ARG, "b200rt_run_jac: edges is NULL");
    XtArgs xa;
    xa.mode = XM_JAC; xa.edges = edges; xa.ngrp = ngrp;
    return run_jobs(H, jobs, nullptr, xa, njob, accumulate, cuda_stream);
}

int b200rt_run_plen(void* handle, const b200rt_job* jobs, int njob, double tpmin, double tpmax, int ntp, int accumulate,
                    void* cuda_stream) {
    Handle* H = static_cast<Handle*>(handle);
    if (!H) return B200RT_ERR_ARG;
    XtArgs xa;
    xa.mode = XM_PLEN; xa.tpmin = tpmin; xa.tpmax = tpmax; xa.ntp = ntp;
    return run_jobs(H, jobs, nullptr, xa, njob, accumulate, cuda_stream);
}

int b200rt_run_act(void* handle, const b200rt_job* jobs, int njob, int accumulate, void* cuda_stream) {
    Handle* H = static_cast<Handle*>(handle);
    if (!H) return B200RT_ERR_ARG;
    XtArgs xa;
    xa.mode = XM_ACT;
    return run_jobs(H, jobs, nullptr, xa, njob, accumulate, cuda_stream);
}

int b200rt_sync(void* handle) {
    Handle* H = static_cast<Handle*>(handle);
    if (!H) return B200RT_ERR_ARG;
    if (!H->ran) return fail(H, B200RT_ERR_STATE, "nothing has been run");
    CK(cudaSetDevice(H->device));
    cudaStream_t st = H->last_stream;
    CK(cudaMemsetAsync(H->flag.p, 0, 16, st));
    const int nb = H->numSM * 4;
    if (H->nflux) check_finite_kernel<<<nb, 256, 0, st>>>((const double*)H->flux.p, H->nflux, (int*)H->flag.p);
    if (H->nrad) check_finite_kernel<<<nb, 256, 0, st>>>((const double*)H->rad.p, H->nrad, (int*)H->flag.p);
    if (H->nheat) check_finite_kernel<<<nb, 256, 0, st>>>((const double*)H->heat.p, H->nheat, (int*)H->flag.p);
    const bool xt = H->xt_mode != XM_NONE && H->nxt > 0;
    if (xt) check_finite_kernel<<<nb, 256, 0, st>>>((const double*)H->xt.p, H->nxt, (int*)H->flag.p);
    H->launches = 1 + (H->nflux ? 1 : 0) + (H->nrad ? 1 : 0) + (H->nheat ? 1 : 0) + (xt ? 1 : 0);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(st));
    H->inflight = false;
    int bad = 0;
    CK(cudaMemcpy(&bad, H->flag.p, sizeof(int), cudaMemcpyDeviceToHost));
    DevStats ds;
    CK(cudaMemcpy(&ds, H->stats.p, sizeof(ds), cudaMemcpyDeviceToHost));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, H->ev0, H->ev1));
    b200rt_stats& o = H->stats_host;
    std::memset(&o, 0, sizeof(o));
    o.photons = ds.photons; o.n_cell = ds.n_cell; o.n_tent = ds.n_tent; o.n_coll = ds.n_coll; o.n_sfc = ds.n_sfc;
    o.n_le = ds.n_le; o.n_le_visit = ds.n_le_visit; o.n_tally = ds.n_tally; o.n_roulette_kill = ds.n_kill;
    o.w_toa_up = ds.w_toa; o.w_sfc_abs = ds.w_sfc; o.w_atm_abs = ds.w_atm; o.w_roulette = ds.w_rr;
    o.elapsed_ms = ms;
    o.bytes_alg = 4.0 * double(ds.n_cell) + 4.0 * double(ds.n_tent) + 8.0 * double(ds.n_coll) + 4.0 * double(ds.n_le_visit) +
                  8.0 * double(ds.n_tally) + 2.0 * 8.0 * double(H->nflux + H->nrad + H->nheat);
    o.launches = H->launches;
    if (bad) return fail(H, B200RT_ERR_NUMERIC, "NaN/Inf found in tallies");
    return B200RT_OK;
}

static int read_any(Handle* H, const DevBuf& b, size_t n, double* dst, int64_t count, const char* what) {
    if (!H->ran) return fail(H, B200RT_ERR_STATE, "nothing has been run");
    if (n == 0) return fail(H, B200RT_ERR_STATE, std::string(what) + " was not part of the target");
    if (!dst || count < 0 || size_t(count) < n) return fail(H, B200RT_ERR_ARG, std::string("destination too small for ") + what);
    CK(cudaSetDevice(H->device));
    CK(drain(H));
    CK(cudaMemcpy(dst, b.p, n * 8, cudaMemcpyDefault));
    return B200RT_OK;
}

int b200rt_read_flux(void* handle, double* dst, int64_t count) {
    Handle* H = static_cast<Handle*>(handle);
    if (!H) return B200RT_ERR_ARG;
    return read_any(H, H->flux, H->nflux, dst, count, "flux");
}
int b200rt_read_rad(void* handle, double* dst, int64_t count) {
    Handle* H = static_cast<Handle*>(handle);
    if (!H) return B200RT_ERR_ARG;
    return read_any(H, H->rad, H->nrad, dst, count, "radiance");
}
int b200rt_read_heat(void* handle, double* dst, int64_t count) {
    Handle* H = static_cast<Handle*>(handle);
    if (!H) return B200RT_ERR_ARG;
    return read_any(H, H->heat, H->nheat, dst, count, "heating");
}

// the extra tally of the last run, which must have been a run of kind `mode` (XM_JAC, XM_PLEN or XM_ACT)
static int check_xt(Handle* H, int mode) {
    if (!H->ran || H->xt_mode != mode)
        return fail(H, B200RT_ERR_STATE, mode == XM_JAC    ? "the last run was not a Jacobian run (b200rt_run_jac)"
                                         : mode == XM_PLEN ? "the last run was not a path-length run (b200rt_run_plen)"
                                                           : "the last run was not an actinic run (b200rt_run_act)");
    return B200RT_OK;
}
static int read_xt(void* handle, int mode, double* dst, int64_t count) {
    Handle* H = static_cast<Handle*>(handle);
    if (!H) return B200RT_ERR_ARG;
    if (int rc = check_xt(H, mode)) return rc;
    return read_any(H, H->xt, H->nxt, dst, count, mode == XM_JAC ? "Jacobian" : (mode == XM_PLEN ? "path-length tally" : "actinic flux"));
}
static int xt_ptr(void* handle, int mode, double** p, int64_t* n) {
    Handle* H = static_cast<Handle*>(handle);
    if (!H) return B200RT_ERR_ARG;
    if (int rc = check_xt(H, mode)) return rc;
    if (p) *p = (double*)H->xt.p;
    if (n) *n = int64_t(H->nxt);
    return B200RT_OK;
}

int b200rt_read_jac(void* handle, double* dst, int64_t count) { return read_xt(handle, XM_JAC, dst, count); }
int b200rt_jac_ptr(void* handle, double** p, int64_t* n) { return xt_ptr(handle, XM_JAC, p, n); }
int b200rt_read_plen(void* handle, double* dst, int64_t count) { return read_xt(handle, XM_PLEN, dst, count); }
int b200rt_plen_ptr(void* handle, double** p, int64_t* n) { return xt_ptr(handle, XM_PLEN, p, n); }
int b200rt_read_act(void* handle, double* dst, int64_t count) { return read_xt(handle, XM_ACT, dst, count); }
int b200rt_act_ptr(void* handle, double** p, int64_t* n) { return xt_ptr(handle, XM_ACT, p, n); }

int b200rt_tally_ptrs(void* handle, double** flux, int64_t* nflux, double** rad, int64_t* nrad, double** heat, int64_t* nheat) {
    Handle* H = static_cast<Handle*>(handle);
    if (!H) return B200RT_ERR_ARG;
    if (!H->have_scene) return fail(H, B200RT_ERR_STATE, "no scene");
    if (flux) *flux = H->nflux ? (double*)H->flux.p : nullptr;
    if (nflux) *nflux = int64_t(H->nflux);
    if (rad) *rad = H->nrad ? (double*)H->rad.p : nullptr;
    if (nrad) *nrad = int64_t(H->nrad);
    if (heat) *heat = H->nheat ? (double*)H->heat.p : nullptr;
    if (nheat) *nheat = int64_t(H->nheat);
    return B200RT_OK;
}

int b200rt_stats_get(void* handle, b200rt_stats* out) {
    Handle* H = static_cast<Handle*>(handle);
    if (!H || !out) return B200RT_ERR_ARG;
    *out = H->stats_host;
    return B200RT_OK;
}

int b200rt_philox_fill(void* handle, uint64_t seed, uint64_t first, uint32_t c2, uint32_t c3, uint32_t* out_host, int64_t n) {
    Handle* H = static_cast<Handle*>(handle);
    if (!H) return B200RT_ERR_ARG;
    if (!out_host || n < 0) return fail(H, B200RT_ERR_ARG, "bad output buffer");
    if (n == 0) return B200RT_OK;
    CK(cudaSetDevice(H->device));
    DevBuf tmp;
    int rc = dev_alloc(H, tmp, size_t(n) * 16);
    if (rc) return rc;
    philox_fill_kernel<<<unsigned((n + 255) / 256), 256>>>(seed, first, c2, c3, (uint4*)tmp.p, n);
    cudaError_t e = cudaMemcpy(out_host, tmp.p, size_t(n) * 16, cudaMemcpyDefault);
    tmp.release();
    if (e != cudaSuccess) return fail(H, B200RT_ERR_CUDA, cudaGetErrorString(e));
    return B200RT_OK;
}

static int map_kernel_io(Handle* H, const double* in, size_t nin, double* out, size_t nout, DevBuf& din, DevBuf& dout) {
    int rc;
    if ((rc = dev_alloc(H, din, nin * 8)) || (rc = dev_alloc(H, dout, nout * 8))) return rc;
    CK(cudaMemcpy(din.p, in, nin * 8, cudaMemcpyDefault));
    (void)out;
    return 0;
}

int b200rt_phase_eval(void* handle, double apf, const double* mu, double* p_out, int64_t n) {
    Handle* H = static_cast<Handle*>(handle);
    if (!H) return B200RT_ERR_ARG;
    if (!H->have_scene) return fail(H, B200RT_ERR_STATE, "no scene");
    if (n <= 0) return B200RT_OK;
    CK(cudaSetDevice(H->device));
    DevBuf a, b;
    int rc = map_kernel_io(H, mu, n, p_out, n, a, b);
    if (rc) return rc;
    phase_eval_kernel<<<unsigned((n + 255) / 256), 256>>>(H->S.pt, float(apf), (const double*)a.p, (double*)b.p, n);
    cudaError_t e = cudaMemcpy(p_out, b.p, size_t(n) * 8, cudaMemcpyDefault);
    a.release(); b.release();
    if (e != cudaSuccess) return fail(H, B200RT_ERR_CUDA, cudaGetErrorString(e));
    return B200RT_OK;
}

int b200rt_phase_sample(void* handle, double apf, const double* xi, double* mu_out, int64_t n) {
    Handle* H = static_cast<Handle*>(handle);
    if (!H) return B200RT_ERR_ARG;
    if (!H->have_scene) return fail(H, B200RT_ERR_STATE, "no scene");
    if (n <= 0) return B200RT_OK;
    CK(cudaSetDevice(H->device));
    DevBuf a, b;
    int rc = map_kernel_io(H, xi, n, mu_out, n, a, b);
    if (rc) return rc;
    phase_sample_kernel<<<unsigned((n + 255) / 256), 256>>>(H->S.pt, float(apf), (const double*)a.p, (double*)b.p, n);
    cudaError_t e = cudaMemcpy(mu_out, b.p, size_t(n) * 8, cudaMemcpyDefault);
    a.release(); b.release();
    if (e != cudaSuccess) return fail(H, B200RT_ERR_CUDA, cudaGetErrorString(e));
    return B200RT_OK;
}

int b200rt_brdf_eval(void* handle, int32_t type, const float* param5, const double* dir_in3, const double* dir_out3,
                     double* f_out, int64_t n) {
    Handle* H = static_cast<Handle*>(handle);
    if (!H) return B200RT_ERR_ARG;
    if (n <= 0) return B200RT_OK;
    CK(cudaSetDevice(H->device));
    DevBuf a, b, c, d;
    int rc;
    if ((rc = dev_alloc(H, a, 5 * 4)) || (rc = dev_alloc(H, b, size_t(n) * 24)) || (rc = dev_alloc(H, c, size_t(n) * 24)) ||
        (rc = dev_alloc(H, d, size_t(n) * 8)))
        return rc;
    CK(cudaMemcpy(a.p, param5, 20, cudaMemcpyDefault));
    CK(cudaMemcpy(b.p, dir_in3, size_t(n) * 24, cudaMemcpyDefault));
    CK(cudaMemcpy(c.p, dir_out3, size_t(n) * 24, cudaMemcpyDefault));
    brdf_eval_kernel<<<unsigned((n + 255) / 256), 256>>>(type, (const float*)a.p, (const double*)b.p, (const double*)c.p, (double*)d.p, n);
    cudaError_t e = cudaMemcpy(f_out, d.p, size_t(n) * 8, cudaMemcpyDefault);
    a.release(); b.release(); c.release(); d.release();
    if (e != cudaSuccess) return fail(H, B200RT_ERR_CUDA, cudaGetErrorString(e));
    return B200RT_OK;
}

}  // extern "C"
