/* rtb200.h -- C-ABI of the B200-native transport kernels for razoumov/radiativeTransfer (FTTE).
 *
 * The reference has NO plugin / FFI interface for its hot path: the diffuse sweep is inline in
 * `program pointTransfer` (equiSources.f90:1372-1808) and the point-source caster is a set of internal
 * procedures (equiSources.f90:3120-3385), both reading and writing `zoneType` fields through Fortran
 * pointers.  This header therefore DEFINES the drop-in boundary: each entry point names the reference block it
 * replaces.  All arrays are plain host pointers unless the name ends in `_device`; per-leaf arrays are in the
 * reference's own flattened leaf order (`writeCell` pre-order, equiSources.f90:4044-4079 driven by the
 * i/j/k loops at :4830-4836: base cells i outer, j, k inner; children i, j, k), the order of the
 * `cellArrayNNNN.h4` datasets.  Every function returns 0 on success or an RTB200_ERR_* code where the
 * reference would `write(*,*) ...; stop`; the Fortran shim (radiativetransfer_b200/fortran/rtb200_shim.f90)
 * turns a non-zero status into the same `stop`.  There is no CPU fallback: without a CUDA device
 * rtb200_create fails with RTB200_ERR_CUDA.
 */
#ifndef RTB200_H
#define RTB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RTB200_VERSION 100

enum rtb200_status {
  RTB200_OK = 0,
  RTB200_ERR_PHI = 1,             /* equiSources.f90:1413 'error in phi' */
  RTB200_ERR_THETA = 2,           /* equiSources.f90:1426 'error in theta' */
  RTB200_ERR_THETA_OR_PHI = 3,    /* equiSources.f90:1449 */
  RTB200_ERR_PATTERN_RANGE = 4,   /* transportRoutinesModule.f90:33,60,183; equiSources.f90:1523 */
  RTB200_ERR_TOP_SELECTOR = 5,    /* 'error in xyTop/xzTop/yzTop': equiSources.f90:1605,1672,1741; transportRoutinesModule.f90:609 */
  RTB200_ERR_RAY_INACTIVE = 6,    /* 'Error: xzRay should be active': equiSources.f90:1679 ... */
  RTB200_ERR_INTENSITY_GUARD = 7, /* transportRoutinesModule.f90:680-688 */
  RTB200_ERR_ANGLE_LARGE = 8,     /* equiSources.f90:2224 */
  RTB200_ERR_LEVELS = 9,          /* readCellArray.f90:181 'error in levels' */
  RTB200_ERR_CHECKPOINT = 10,     /* equiSources.f90:2962 checkPoint */
  RTB200_ERR_IDEPTH = 11,         /* equiSources.f90:4196 'error in idepth123' */
  RTB200_ERR_ARG = 12,            /* bad argument (null pointer, size mismatch, grid not set ...) */
  RTB200_ERR_CUDA = 13,           /* CUDA runtime failure or no device: no CPU fallback exists */
  RTB200_ERR_NOMEM = 14,
  RTB200_ERR_CHEMISTRY = 15       /* equiSources.f90:3634-3655: ionisation fraction outside [0,1] (the reference prints and stops) */
};

/* arithmetic mode of the per-segment update (transportRoutinesModule.f90:651-698, 1036-1054) */
enum rtb200_math {
  RTB200_MATH_FAST = 0,     /* J_seg = Iin*(1-exp(-tau))/tau: the same quantity without the exp->log round trip */
  RTB200_MATH_FAITHFUL = 1  /* J_seg = (Iin-Iout)/log(Iin/Iout), operation for operation as the reference */
};

typedef struct rtb200_ctx rtb200_ctx;

int rtb200_version(void);
const char* rtb200_status_string(int status);

/* One context for one GPU.  `device` is the CUDA ordinal. */
int rtb200_create(int device, rtb200_ctx** ctx);
int rtb200_destroy(rtb200_ctx* ctx);

/* Device groups: ONE handle for all GPUs of a node, accepted by every call below that takes a context.
 *   rtb200_create_multi    one process drives `ngpus` devices (devices = NULL: 0..ngpus-1): what the reference's serial
 *                          driver needs (the "init(ngpus)" entry SURVEY.md 8b proposes): rtbSetGrid / rtbDiffuse / rtbPoint of the
 *                          Fortran shim are unchanged, the directions and sources are sharded inside the library.
 *   rtb200_create_rank     the same group with one process per GPU (torchrun): every process passes the 128-byte id
 *                          that rank 0 obtained from rtb200_comm_unique_id (broadcast by the launcher) and calls every
 *                          function collectively.  Per-leaf host arrays are then read and written SLAB-WISE: rank r
 *                          touches leaves [r*slab, (r+1)*slab) of the caller's arrays only (rtb200_multi_info).
 * Data path (csrc/multi.cu): slab H2D + NVLink all-gather of the species, direction / source shards on full grids,
 * reduce-scatter of the per-leaf sums (a peer-memory kernel of this library with the photo-rate epilogue fused, or
 * NCCL: set_tuning "multi_reduce" 1 / 0), slab D2H.  NCCL (libnccl.so.2) is loaded with dlopen when a group of more
 * than one device is created (RTB200_NCCL_LIB overrides the search path).  RTB200_TIMING=1 in the environment makes rank 0
 * print the host wall time of every phase of the host-buffer calls (slab copies, all-gather, sweep, reduce-scatter).  Results are bit-identical from run to run
 * and independent of multi_reduce only in mode 1 (fixed summation order rank 0, 1, ...). */
int rtb200_comm_unique_id(char* id128);
int rtb200_create_multi(int ngpus, const int* devices, rtb200_ctx** ctx);
int rtb200_create_rank(int device, int nranks, int rank, const char* id128, rtb200_ctx** ctx);
/* nranks, devices of this process, first global rank of this process, leaves per slab, active reduction (1 peer kernel,
 * 0 NCCL, -1 single device); any output may be NULL */
int rtb200_multi_info(rtb200_ctx* ctx, int32_t* nranks, int32_t* nlocal, int32_t* firstRank, int64_t* slab,
                      int32_t* reduceMode);
/* the direction shard of a rank (HEALPix NESTED pixel numbers; whole zones, longest-processing-time-first on segment
 * counts x "zone_cost_x/y/z" tuning factors); host only */
int rtb200_multi_shard(rtb200_ctx* ctx, int nAngularLevel, int rank, int32_t* rays, int32_t cap, int32_t* nrays);
/* the same rule without a handle (zoneCost3 = NULL: the library's measured defaults): what a one-process-per-GPU caller of the single-GPU entry
 * points (rays = its shard) would use */
int rtb200_shard_directions(int nranks, int nAngularLevel, int nx, const double* zoneCost3, int rank, int32_t* rays,
                            int32_t cap, int32_t* nrays);
/* Resident steps of a device group (results stay in the library's slab buffers, asynchronous; streams[i] = cudaStream_t
 * of local device i, NULL = internal streams):
 *   rtb200_multi_diffuse_resident  computeOpacities + sweep of each rank's direction shard + reduce-scatter of Jmean1..3
 *                                  [+ diffuse photo-rates into K when ksi6 = {ksi24[3], ksi25, ksi26[2]} is given]
 *                                  [+ solveRateEquations on the slab + all-gather of HI, HeI, HeII when chemistry != 0;
 *                                  uses the point-source rates of a preceding rtb200_multi_point_resident]
 *   rtb200_multi_point_resident    setZeroRates + ray casting of each rank's sources + reduce-scatter of the 6 rate fields
 *   rtb200_multi_slab              this process's slab of local device `local`: leaves [offset, offset + count), device
 *                                  pointers J [3][slab], K [3][slab] (krate24, krate25, krate26), R [6][slab]
 *   rtb200_multi_sync              waits for all devices of the group; returns a pending device-side status */
int rtb200_multi_diffuse_resident(rtb200_ctx* ctx, int nAngularLevel, const double* uvb, const double* beta,
                                  const double* ksi6, int chemistry, void* const* streams, int64_t* nseg);
int rtb200_multi_point_resident(rtb200_ctx* ctx, int nWave, const double* wavelength, const double* lum,
                                const double* metallicity, double coefSpectrum, const double* aDust, int dustApproximation,
                                int maxPixelLevel, int32_t nsrc, const int32_t* srcLeaf, const int32_t* srcWeight,
                                void* const* streams, double* ndotRemaining, double* ndotBoundary, double* ndotDust,
                                double* ndotSpectrum, int32_t* highestPixelLevel, int64_t* nseg);
int rtb200_multi_slab(rtb200_ctx* ctx, int local, int64_t* offset, int64_t* count, double** J_device, double** K_device,
                      double** R_device);
int rtb200_multi_sync(rtb200_ctx* ctx);
/* copies of the slab buffers of local device `local` to the host after a synchronisation: J3 [3][slab], K3 [3][slab],
 * R6 [6][slab] (any may be NULL); entries beyond the slab's leaf count are padding */
int rtb200_multi_slab_get(rtb200_ctx* ctx, int local, double* J3, double* K3, double* R6);

int rtb200_set_math(rtb200_ctx* ctx, int math_mode);
/* Launch tuning knobs; results do not depend on them (tests/test_diffuse_gpu.py, test_point_gpu.py).  Keys:
 *   uniform sweep  "slots" (zone tasks per launch, 0 = all), "graph" (CUDA graph replay, 1), "dirs_per_task" (0 = chosen
 *                  from a wave model), "cells" (cells of a layer per thread: 1, 2, or 0 = by grid size and zone tasks per
 *                  launch; an emissive sweep always runs one-cell threads), "block_warps" (warps per block 8 / 4 / 2,
 *                  at most 4 for two-cell threads, 0 = by the number of blocks a launch has), "transpose_z" (z-major copy for
 *                  the zones sweeping along the contiguous axis, 1), "pdl" (programmatic dependent launch of layer
 *                  l+1 on layer l, also used by the nested-grid waves, 1), "l2_mb"
 *   nested grids   "force_amr" (general octree path on a uniform grid), "amr_batch" (directions per batch, 0 = as many
 *                  as fit in memory), "amr_stream" (2:1-balanced grids: 1 = the whole sweep as one launch whose work items wait
 *                  for their upstream intensity records, 0 = one launch per wave, -1 = by the size of the waves, the default;
 *                  identical bits), "amr_order" (waves of the sweep: -1 = centre-sum key on 2:1-balanced grids and the leaf's depth in the dependency
 *                  graph elsewhere, 1 = depth always, 0 = centre-sum key with per-leaf flags and a deferred list on grids that
 *                  are not balanced: the round-1 scheme; identical bits), "amr_slots" (per-item arrays
 *                  in wave order, 1), "amr_thin" (thin segments with the reference's operation sequence, 1), "amr_min_blocks"
 *                  (register cap of the wave kernel: 6 or 8 blocks per SM, 0 = by the size of the waves)
 *   device groups  "multi_reduce" (1 = peer-memory reduce-scatter kernel, 0 = NCCL), "zone_cost_x" / "_y" / "_z"
 *                  (relative time per segment of zones sweeping along x / y / z, for the direction sharding)
 *   point sources  "point_batch" (sources per batch), "point_min_blocks" (register cap of the march kernel, 5),
 *                  "point_deposit" (atomic-free and reproducible: 2 = planned, the default -- the (leaf, ray, segment) sort is done
 *                  once per grid and source list, later passes write every deposit to its cached leaf-ordered slot and add up
 *                  each leaf's run; 1 = records + sort + segmented reduction every pass (what 2 falls back to with dust);
 *                  0 = fp64 RED.ADD, the ablation: fastest, summation order not fixed), "point_record_cap",
 *                  "point_refill" (lane refill on the last pixel level, 0)
 * "portable_math" (default 1) selects, for the FAITHFUL point-source path, exp/log built from IEEE +,*,/,fma
 * (csrc/portable_math.h) instead of CUDA libm, so that a host build of the same header reproduces it bit for bit. */
int rtb200_set_tuning(rtb200_ctx* ctx, const char* key, double value);
/* status raised by a device-side guard during an asynchronous (*_device) call since the last query; clears it */
int rtb200_device_error(rtb200_ctx* ctx);

/* Replaces the pointer-linked octree (definitionsModule.f90:163-182; built at equiSources.f90:1870-1974) with
 * structure-of-arrays device buffers plus a linear octree rebuilt from `level` alone, exactly as
 * readCellArray.f90:154-187 does.  nx = ny = nz (equiSources.f90:427-436 requires a cubic level-1 grid).
 * HeI / HeII may be NULL (taken as zero: a hydrogen-only grid); rho and abun2 may be NULL when only the diffuse path is
 * used -- rtb200_point*, rtb200_chemistry_device and rtb200_compute_mass then return RTB200_ERR_ARG.  Arrays are copied. */
int rtb200_grid_set(rtb200_ctx* ctx, int nx, int64_t nleaf, const int8_t* level, const double* HI,
                    const double* HeI, const double* HeII, const double* rho, const double* abun2,
                    double physicalBoxSize);

/* New absorber densities after a chemistry step (solveRateEquations writes back HI, HeI, HeII only:
 * equiSources.f90:3671-3673).  NULL keeps the current array.  Ordering: the call first waits for ALL work queued on the
 * context's device (including what *_device calls put on the caller's streams), then copies, then returns when the
 * copies are complete -- work issued afterwards on any stream sees the new arrays. */
int rtb200_grid_update_species(rtb200_ctx* ctx, const double* HI, const double* HeI, const double* HeII);

/* Emission (an extension without a reference value, DESIGN.md 4.6): per leaf and frequency group an emission
 * coefficient eta >= 0 in the units of uvb per cm, [3][nleaf] in the leaf order of rtb200_grid_set.  A segment of path
 * dpath and optical depth tau = kappa dpath then leaves with
 *     Iout = Iin e^-tau + eta t,   t = (1 - e^-tau) / kappa  if tau > (double)1.e-10f,  else dpath
 * (the reference's `nemi` slot, transportRoutinesModule.f90:673-678, with nemi = eta dpath) and contributes to Jmean
 *     J_seg = L(Iin) + eta dpath phi(tau),   phi(tau) = (tau - 1 + e^-tau) / tau^2,  phi(0) = 1/2,
 * L(Iin) being what the math mode computes today for the attenuated part; J_seg is the exact path average.  With eta = 0
 * every result is bit for bit the emission-free one.  rtb200_diffuse, rtb200_diffuse_device, the device-group host call
 * and rtb200_multi_diffuse_resident honour the emission; the point-source path does not.  rtb200_grid_set clears it,
 * rtb200_grid_update_species leaves it alone.  The intensity guard of refined leaves (status 7) still applies.
 *   rtb200_grid_set_emission         eta = host [3][nleaf], copied; NULL clears the emission.  Ordering as
 *                                    rtb200_grid_update_species.  A device group reads the array slab-wise in rank mode
 *                                    (all-gathered on the devices, as the species) and every rank returns the same status.
 *   rtb200_grid_set_emission_device  eta_device = device [3][nleaf], copied on `stream` (a cudaStream_t) and checked there;
 *                                    returns after synchronising that stream.  Single contexts only (a group: ERR_ARG).
 * An entry that is negative, NaN or Inf refuses the call with RTB200_ERR_ARG and the previous emission stays: the streamed
 * nested-grid sweep marks its intensity records with the sign bit, which needs intensities >= 0 (DESIGN.md 4.4). */
int rtb200_grid_set_emission(rtb200_ctx* ctx, const double* eta);
int rtb200_grid_set_emission_device(rtb200_ctx* ctx, const double* eta_device, void* stream);

/* Scattering (an extension without a reference value, DESIGN.md 4.7): per leaf and frequency group a scattering
 * coefficient sigma >= 0 in the units of kappa (1/cm), [3][nleaf] in the leaf order of rtb200_grid_set; coherent within a
 * group and isotropic.  The sweep then uses the extinction kappa_ext = kappa_abs + sigma (sigma added last, rounded
 * once) and solves by source iteration: sweep k runs with the emission coefficient
 *     eta_k = eta_th + sigma * J_{k-1}     (two roundings, no FMA),   J_0 = 0,
 * eta_th being the emission of rtb200_grid_set_emission (0 if none) and J the full Jmean of the previous sweep.  The
 * residual of sweep k is r_k = max over (group, leaf) of |J_k - J_{k-1}| / J_k (0 where J_k == J_{k-1}, +inf where
 * J_k == 0 != J_{k-1}); with tolerance > 0 the solve stops after the first k with r_k <= tolerance or at maxIterations,
 * with tolerance == 0 it runs exactly maxIterations sweeps without reading anything back in between (so it stays
 * asynchronous on the stream of the *_device calls).  Not converging is not an error: the call returns J_k.
 * rtb200_diffuse, rtb200_diffuse_device, the device-group host call and rtb200_multi_diffuse_resident (whose photo-rates
 * are those of the last iteration, its chemistry runs once after it) solve this way; a direction subset (rays != NULL)
 * returns RTB200_ERR_ARG, because a shard's J is not the mean intensity.  The point-source path ignores scattering.
 * nseg and rtb200_last_stats count all sweeps of the call (algorithmic bytes 96 B per leaf, direction and iteration; the
 * device time covers the whole call, the sweep time is the last sweep's).  sigma = 0 gives the results of no scattering
 * bit for bit (with tolerance > 0 after 2 sweeps, residual 0).  rtb200_grid_set clears the scattering,
 * rtb200_grid_update_species keeps it; a device group reads sigma slab-wise as the emission.
 *   rtb200_grid_set_scattering  sigma = host [3][nleaf], copied (NULL clears); maxIterations >= 1; tolerance >= 0 and
 *                               finite.  A negative, NaN or Inf entry or a bad count or tolerance is refused with
 *                               RTB200_ERR_ARG and the previous state stays.  Queued work completes before the copy.
 *   rtb200_last_scattering      sweeps done and the last residual of the latest diffuse call (0 / 0 without scattering). */
int rtb200_grid_set_scattering(rtb200_ctx* ctx, const double* sigma, int32_t maxIterations, double tolerance);
int rtb200_last_scattering(rtb200_ctx* ctx, int32_t* iterations, double* residual);

/* Dust in the diffuse sweep (an extension without a reference value, DESIGN.md 4.8): the dust model of the point-source
 * path (dustModule.f90:30-73) as an opacity of the diffuse field.  betaDust[3] is a band-mean dust cross-section per
 * frequency group in cm^2 per H (rtb200_uvb_dust_beta).  Per leaf and group the diffuse calls compute, on the device
 * and from the current species of every call (no FMA, every step rounded):
 *     mode 1:  kd_g = ((HI * betaDust[g]) * abun2) / (double)0.2f
 *     mode 2:  kd_g = (((((double)0.76f * rho) / (double)1.6726231e-24f) * betaDust[g]) * abun2) / (double)0.2f
 * (the dust column of the point path, point_source.cu), the extinction kappa_g = kappa_abs,g + kd_g (rounded once; a
 * per-leaf sigma of rtb200_grid_set_scattering is added after it) and, while albedo[g] > 0, the scattering source
 * sigma_g = albedo[g] * kd_g of the source iteration of rtb200_grid_set_scattering (same residual, stopping rule, stats
 * and rtb200_last_scattering), with this call's maxIterations / tolerance.  Mode 0 is no dust.  One scattering medium at
 * a time: dust with an albedo > 0 is refused while a per-leaf sigma is set, and rtb200_grid_set_scattering(sigma !=
 * NULL) is refused while dust scatters; dust that only absorbs combines with emission and a per-leaf sigma.  A direction
 * subset is refused while dust scatters.  The point-source path ignores this setting (it has its own dustApproximation).
 * rtb200_grid_set clears the dust, rtb200_grid_update_species keeps it (the next call follows the new HI).  A device
 * group stores the scalars on every member; each computes the dust of the whole grid from its complete species.
 *   rtb200_grid_set_dust  mode 0..2; betaDust[3] >= 0 and finite; albedo[3] in [0, 1] (both may be NULL for mode 0);
 *                         mode 1 needs abun2, mode 2 rho and abun2 in rtb200_grid_set; with an albedo > 0,
 *                         maxIterations >= 1 and tolerance >= 0 and finite.  Anything else, or a conflict above, is
 *                         refused with RTB200_ERR_ARG and the previous state stays.  Queued work completes first. */
int rtb200_grid_set_dust(rtb200_ctx* ctx, int dustApproximation, const double* betaDust3, const double* albedo3,
                         int32_t maxIterations, double tolerance);

/* Acceleration of the source iteration (DESIGN.md 4.9), for whichever medium scatters (a per-leaf sigma or dust with an
 * albedo > 0).  In a diffuse call, x_{k-1} is the J that forms the source of sweep k (eta_k = eta_th + sigma * x_{k-1})
 * and y_k the J that sweep k returns; the residual is r_k = maxrel(y_k, x_{k-1}) as above, the stopping rule is
 * unchanged, and the call returns y_k (a sweep output, never an extrapolated J).  Flags 0 is plain source iteration.
 *   RTB200_SCATTER_WARM_START  x_0 = the J the previous diffuse call of this context returned, if that call completed a
 *                              scattering solve; else x_0 = 0.  The stored J survives rtb200_grid_update_species, new
 *                              emission, sigma, dust and iteration settings (it is only a starting guess); it is dropped
 *                              by rtb200_grid_set, by clearing every scattering medium and by a call that fails.
 *   RTB200_SCATTER_NG          Ng extrapolation of order 2 (Auer 1987).  After every fourth sweep counted from the call's
 *                              start or from the last attempted extrapolation, except on the sweep that stops the call,
 *                              with I0..I3 = y_k .. y_{k-3}: w = 1/I0 where I0 > 0 (else 0), d0 = (I0-I1) w,
 *                              d1 = (I1-I2) w, d2 = (I2-I3) w, q1 = d0-d1, q2 = d0-d2, the sums over (group, leaf)
 *                              A11 = <q1,q1>, A12 = <q1,q2>, A22 = <q2,q2>, c1 = <d0,q1>, c2 = <d0,q2>,
 *                              det = A11 A22 - A12^2, a = (c1 A22 - c2 A12) / det, b = (c2 A11 - c1 A12) / det; if
 *                              det > 1e-14 A11 A22 and a, b are finite, x_k = max(0, (1-a-b) I0 + a I1 + b I2), else
 *                              the step is skipped (x_k = y_k).  The sums are taken in a fixed order (bit-identical
 *                              from run to run; a device group sums its ranks' partials in rank order, so all ranks
 *                              take the same step) and stay on the device: no host round trip is added.  While set, the
 *                              history costs three more [3][nleaf] fields (a device group: [3][slab] per rank).
 *   rtb200_grid_set_scattering_acceleration  flags = a combination of the two (0 = none); unknown bits are refused with
 *                              RTB200_ERR_ARG and the previous flags stay.  Queued work completes first.  A device
 *                              group calls it collectively (every rank returns the same status).  rtb200_grid_set
 *                              resets it to 0.
 *   rtb200_last_scattering_acceleration  extrapolations the latest diffuse call applied (skipped ones not counted) and
 *                              whether it started warm (1) or from J = 0 (0). */
#define RTB200_SCATTER_NG 1
#define RTB200_SCATTER_WARM_START 2
int rtb200_grid_set_scattering_acceleration(rtb200_ctx* ctx, int32_t flags);
int rtb200_last_scattering_acceleration(rtb200_ctx* ctx, int32_t* extrapolations, int32_t* warmStarted);

/* Photo-heating and dust absorption of the diffuse field (an extension without a reference value, DESIGN.md 4.10).
 * While heating is set, every diffuse call ends with one pass over the J it returns (for a scattering solve the J of
 * the last sweep) that fills five per-leaf fields [5][nleaf] in leaf order.  With t_g = fourPi * J_g (fourPi = 4 * pi
 * as in the diffuse photo-rates) and every operation rounded on its own (no FMA):
 *   f = 0, 1, 2  Gamma_s = ((t_1 * gamma[1][s]) + (t_2 * gamma[2][s])) + (t_3 * gamma[3][s])   photo-heating per
 *                absorber HI, HeI, HeII [erg/s]; gamma[g][s] = gammaHI, gammaHeI, gammaHeII of group g (table57)
 *   f = 3        H_gas  = ((HI * Gamma_HI) + (HeI * Gamma_HeI)) + (HeII * Gamma_HeII)   [erg/s/cm^3], with the
 *                species the call's sweep used (a resident call with chemistry: those before chemistry)
 *   f = 4        H_dust = (u_1 + u_2) + u_3,  u_g = ((1 - albedo_g) * kd_g) * (t_g * W_g)   [erg/s/cm^3]: the power
 *                the dust of rtb200_grid_set_dust absorbs (kd_g its opacity, exactly as the sweep used it); 0 without
 *                dust.  W_g is the band width in Hz of rtb200_uvb_band_width, so betaDust_g * W_g is the band integral
 *                of (nu/nu_g)^-alpha_g sigma_d(nu) d nu and 4 pi kd_g W_g J_g the power absorbed from the power-law band.
 * Every field is linear in J: the fields of a direction subset are that shard's share, and the shares add up.
 *   rtb200_grid_set_heating  gamma9 = [group][gammaHI, gammaHeI, gammaHeII] (NULL clears the setting and frees the
 *                            buffer), width3 = band widths [Hz].  An entry that is negative, NaN or Inf is refused with
 *                            RTB200_ERR_ARG and the previous state stays.  Queued work completes first.  rtb200_grid_set
 *                            clears it; rtb200_grid_update_species, emission, scattering, dust and the acceleration keep
 *                            it.  A device group calls it collectively and stores it on every member.
 *   rtb200_last_heating      heat5 = host [5][nleaf]: the fields of the latest diffuse call (a device group in rank mode
 *                            writes its slab only, as the J of the host call).  RTB200_ERR_ARG while heating is not set,
 *                            when no diffuse call has completed since the setting or the grid changed, or after a
 *                            failed call.
 *   rtb200_heating_device    the library's device buffer [5][stride]: offset 0, count = stride = nleaf for a single
 *                            context (local 0); leaves [offset, offset + count) of local device `local` of a group, as
 *                            rtb200_multi_slab.  Valid until the next diffuse call or setting change; ERR_ARG while
 *                            heating is not set.
 * rtb200_diffuse reads its J, rtb200_diffuse_device the caller's J_device on the caller's stream, the group calls every
 * member's reduced slab of J (once, after a source iteration).  rtb200_last_stats counts the pass in launches and the
 * device time; the sweep figures stay the sweep's. */
int rtb200_grid_set_heating(rtb200_ctx* ctx, const double* gamma9, const double* width3);
int rtb200_last_heating(rtb200_ctx* ctx, double* heat5);
int rtb200_heating_device(rtb200_ctx* ctx, int local, int64_t* offset, int64_t* count, int64_t* stride,
                          double** H_device);

/* Diffuse (UV background) sweep: replaces equiSources.f90:1372-1808 (computeOpacities :4956, the loop over
 * 12*4**(nAngularLevel-1) HEALPix directions, pattern set-up, neighbour threading, transport).
 *   uvb[3]      boundary intensities uvb1..3 (definitionsModule.f90:53)
 *   beta[9]     group cross-sections, [group g=1..3][beta24, beta26, beta25] (uvbBetaTable.f90:262-296)
 *   rays/nrays  HEALPix NESTED pixel numbers to sweep (direction sharding across GPUs); NULL/0 = all
 *   Jmean1..3   caller-allocated [nleaf], OVERWRITTEN with the sum over the swept directions (Jmean is zeroed
 *               by computeOpacities in the reference); a multi-GPU caller sums the per-rank results
 *   nseg        optional: number of ray-cell segment updates performed (the benchmark's unit)               */
int rtb200_diffuse(rtb200_ctx* ctx, int nAngularLevel, const double* uvb, const double* beta,
                   const int32_t* rays, int32_t nrays, double* Jmean1, double* Jmean2, double* Jmean3,
                   int64_t* nseg);

/* Same sweep with the result left on the GPU: J_device is a device pointer to [3][nleaf] doubles (Jmean1, then
 * Jmean2, then Jmean3), `stream` a cudaStream_t (NULL = default stream).  Asynchronous with respect to the host
 * except for plan building on first use.  Used for the NCCL all-reduce and the resident-data benchmark. */
int rtb200_diffuse_device(rtb200_ctx* ctx, int nAngularLevel, const double* uvb, const double* beta,
                          const int32_t* rays, int32_t nrays, double* J_device, void* stream, int64_t* nseg);

/* Diffuse contribution to the photo-rates (equiSources.f90:3546-3553), fused after the (all-reduced) J:
 *   krate24 += 4*pi*(J1*ksi24[0] + J2*ksi24[1] + J3*ksi24[2]);  krate25 += 4*pi*J3*ksi25;
 *   krate26 += 4*pi*(J2*ksi26[0] + J3*ksi26[1]).   All pointers are device pointers, k* accumulate. */
int rtb200_diffuse_rates_device(rtb200_ctx* ctx, const double* J_device, const double* ksi24, const double* ksi25,
                                const double* ksi26, double* k24_device, double* k25_device, double* k26_device,
                                void* stream);

/* UV-background tables that feed the sweep (host only, no device needed): the band amplitudes uvb1..3 with the
 * effective slopes alpha(3) (equiSources.f90:198-246 + powerSpectrumIndex :4985-5043) and uvbBetaTable.f90:31-296.
 *   rtb200_uvb_amplitudes   uvb[3], alpha[3] for a redshift and the `uvbCoefficient` of inputParameters
 *   rtb200_uvb_beta_table   table57 = [group 1..3][beta24, beta25, beta26, beta27..31, ksi24, ksi25, ksi26, ksi27..31,
 *                           gammaHI, gammaHeI, gammaHeII] (the fields of group1..3, definitionsModule.f90)
 *   rtb200_uvb_background   both, returned in the shapes the calls above take: beta[9] = [group][beta24, beta26,
 *                           beta25], ksi24[3], ksi25[1] (group 3), ksi26[2] (groups 2, 3); any output may be NULL.
 * nfreq = nfbins = 400, freqdel = frequencyBinWidth = (double)0.02f in the reference (definitionsModule.f90:239-241).
 * Returns RTB200_ERR_ARG where powerSpectrumIndex prints 'wrong sign' and stops.
 *   rtb200_uvb_dust_beta    betaDust3[g] = band mean of the dust cross-section over group g with the weights of beta24:
 *                           sum over the in-band bins i >= 1 of dt * sD(e_i) / (shape_g * nu_g), dt = (e_i/nu_g)^-alpha_g
 *                           * (e_i - e_{i-1}), sD = the 7-term fit of aDust[7][5] (dustModule.f90:30-73) at the bin's
 *                           wavelength, as the point path evaluates it.  Group 3 runs to wavelengths below the fit's
 *                           range (down to ~1e-4 A at nfreq 400); the fit is extrapolated there as in the point tables.
 *                           Input to rtb200_grid_set_dust.  ERR_ARG for NULL pointers or nfreq < 2.
 *   rtb200_uvb_band_width   width3[g] = shape_g * nu_g * eVtoHz, the band width in Hz of group g (shape_g the band
 *                           integral of the beta24 normalisation): betaDust3[g] * width3[g] is the band integral of the
 *                           dust cross-section.  Input to rtb200_grid_set_heating.  ERR_ARG for NULL pointers. */
int rtb200_uvb_band_width(const double* alpha, double* width3);
int rtb200_uvb_dust_beta(int nfreq, double freqdel, const double* alpha, const double* aDust, double* betaDust3);
int rtb200_uvb_amplitudes(double currentRedshift, double uvbCoefficient, double* uvb, double* alpha);
int rtb200_uvb_beta_table(int nfreq, double freqdel, const double* alpha, double* table57);
int rtb200_uvb_background(double currentRedshift, double uvbCoefficient, int nfreq, double freqdel, double* uvb,
                          double* alpha, double* beta, double* ksi24, double* ksi25, double* ksi26, double* table57);

/* Point-source pass: replaces the source loop equiSources.f90:1256-1370 with its internal procedures
 * startNewLongRay (:3120-3385), drawSegment (:2412-2595), find/zoom??Neighbour (:2647-2960),
 * getRatesHydrogenHelium (:4157-4311) and the per-source table build stellarBetaTable.f90 (+ stellarPopulationModule.f90,
 * dustModule.f90).  None of the reference's data files ship with it, so what it reads from disk is passed in:
 *   nWave, wavelength[nWave]    wavelength grid of the population-synthesis spectra [cm], increasing (equiSources.f90:851-892)
 *   lum[5][2][nWave]            log10 specific luminosity [erg/s/A]: metallicity m, time slices iSpectrum / iSpectrum+1
 *   metallicity[5]              log10 Z of the five spectra;  coefSpectrum: time interpolation weight (:1241-1242)
 *   aDust[7][5]                 rows of smc_dust_parameters.dat (dustModule.f90:15-24)
 *   dustApproximation           0 noDust, 1 completeSublimation, 2 noSublimation (definitionsModule.f90:254)
 *   maxPixelLevel               HEALPix level at which rays stop splitting (6 in the reference, 1..8 here)
 *   srcLeaf[nsrc], srcWeight[nsrc]  host leaf (leaf order of rtb200_grid_set) and multiplicity of every merged source
 *                               (star%hostCell / star%weight, :1169-1206); weight <= 0 is skipped (:1264).  Source
 *                               sharding across GPUs = each rank passes its own subset, the caller sums the rates.
 *   krate24,25,26, crate24,25,26 [nleaf]   ACCUMULATED (+=) like the reference's cell fields (zeroed by setZeroRates)
 *   ndotRemaining[nsrc][7], ndotBoundary[nsrc][7], ndotDust[nsrc], ndotSpectrum[nsrc][300]  per-source escape
 *                               diagnostics (:3198-3233); each may be NULL
 *   highestPixelLevel[nsrc]     deepest HEALPix level a split of the source has opened (:1266, :3316; 0 = no ray
 *                               split), the fourth column of the driver's 'src:' line (:1353-1357); may be NULL
 *   nseg                        optional: ray-cell segment updates performed (iterations of the loop at :3168)
 * rtb200_set_math: RTB200_MATH_FAITHFUL evaluates every table lookup with the reference's operation sequence;
 * RTB200_MATH_FAST evaluates the same interpolant without the R(d) - R(d+tau) cancellation.                        */
int rtb200_point(rtb200_ctx* ctx, int nWave, const double* wavelength, const double* lum, const double* metallicity,
                 double coefSpectrum, const double* aDust, int dustApproximation, int maxPixelLevel, int32_t nsrc,
                 const int32_t* srcLeaf, const int32_t* srcWeight, double* krate24, double* krate25, double* krate26,
                 double* crate24, double* crate25, double* crate26, double* ndotRemaining, double* ndotBoundary,
                 double* ndotDust, double* ndotSpectrum, int32_t* highestPixelLevel, int64_t* nseg);

/* Same pass with the rates left on the GPU: rates_device = device pointer to [6][nleaf] doubles in the order krate24,
 * krate25, krate26, crate24, crate25, crate26 (accumulated); the diagnostics are host pointers (NULL = not wanted). */
int rtb200_point_device(rtb200_ctx* ctx, int nWave, const double* wavelength, const double* lum,
                        const double* metallicity, double coefSpectrum, const double* aDust, int dustApproximation,
                        int maxPixelLevel, int32_t nsrc, const int32_t* srcLeaf, const int32_t* srcWeight,
                        double* rates_device, void* stream, double* ndotRemaining, double* ndotBoundary,
                        double* ndotDust, double* ndotSpectrum, int32_t* highestPixelLevel, int64_t* nseg);

/* Ionisation equilibrium per leaf: replaces solveRateEquations (equiSources.f90:3459-3677), the consumer of the
 * transport results, so that the outer transport <-> chemistry iteration can stay on the GPU.
 *   rtb200_chemistry_tables       k1a..k6a of calc_rates.f (nratec bins in log T from logtem0 to logtem9, :174-190)
 *   rtb200_chemistry_temperature  tgas per leaf (held fixed by the driver, :3671-3673); log(tgas) is taken here, with libm
 *   rtb200_chemistry_device       rates_device [6][nleaf] as rtb200_point_device leaves them (NULL = no point sources);
 *                                 J_device [3][nleaf] of rtb200_diffuse_device with ksi = {ksi24 of groups 1..3, ksi25
 *                                 of group 3, ksi26 of groups 2, 3} (:3546-3553), or J_device = NULL and uniform =
 *                                 {add24, add25, add26, selfShieldingThreshold [cm]} for the uniform background with the
 *                                 mean-free-path switch (:3555-3562; addXX = 4 pi (uniformQuasar quasar%ksiXX +
 *                                 uniformStellar stellar%ksiXX)).  Updates the context's HI, HeI, HeII in place;
 *                                 maxChange (host, optional; forces a synchronisation) = largest change of a species
 *                                 fraction, the quantity the reference computes as `tmp` (:3665-3669).
 *   rtb200_grid_get_species       HI, HeI, HeII back to the host (any may be NULL)
 *   rtb200_compute_mass           neutral and total hydrogen mass in solar masses from the context's current HI and
 *                                 rho: replaces the computeMass recursion (equiSources.f90:4369-4393) the driver runs
 *                                 after every chemistry pass (:1018, :1828) to print neutralHydrogenMass /
 *                                 totalHydrogenMass.  Per-leaf terms in the reference's operation order; the sum is
 *                                 a fixed-order tree (reproducible; differs from the serial sum by rounding only). */
int rtb200_chemistry_tables(rtb200_ctx* ctx, int nratec, double logtem0, double logtem9, double dlogtem, const double* k1a,
                            const double* k2a, const double* k3a, const double* k4a, const double* k5a,
                            const double* k6a);
int rtb200_chemistry_temperature(rtb200_ctx* ctx, const double* tgas);
int rtb200_chemistry_device(rtb200_ctx* ctx, const double* rates_device, const double* J_device, const double* ksi,
                            const double* uniform, double* maxChange, void* stream);
int rtb200_grid_get_species(rtb200_ctx* ctx, double* HI, double* HeI, double* HeII);
int rtb200_compute_mass(rtb200_ctx* ctx, double* neutralHydrogenMass, double* totalHydrogenMass, void* stream);

/* Octree build on the device: from the per-level cell lists of the driver's input grid (equiSources.f90:316-423: pos
 * [ncell][3] in kpc, lT, lnH, lx, and the second abundance abun(:,2) or NULL, all real*4, level 1 first with exactly n^3
 * cells) to the leaf arrays in writeCell order that rtb200_grid_set takes.  Replaces the driver's cell-by-cell tree
 * construction for the data path (box :455-489, level-1 abundance smoothing :527-578, placement with inheritance
 * :580-618 + :1870-1974) with sorted key sets (csrc/octree_build.cu).
 *   rtb200_octree_build  builds on `device`; returns the leaf count, nx, physicalBoxSize [cm] and a handle
 *   rtb200_octree_get    copies level[nleaf] and HI, HeI, HeII, rho, abun2, tgas [nleaf] (any may be NULL) to the host
 *   rtb200_octree_free   releases the handle */
int rtb200_octree_build(int device, int nlevels, const int64_t* ncell, const float* const* pos, const float* const* lT,
                        const float* const* lnH, const float* const* lx, const float* const* abun2, int64_t* nleaf,
                        int32_t* nx, double* physicalBoxSize, void** handle);
int rtb200_octree_get(void* handle, int8_t* level, double* HI, double* HeI, double* HeII, double* rho, double* abun2,
                      double* tgas);
int rtb200_octree_free(void* handle);

/* --- debugging / parity exports (bit-exact traversal checks) ------------------------------------------- */
/* point-source pass that also records every ray-cell segment: trace[2*i] = leaf<<32 | pixelLevel<<28 | pixel<<8 | exit
 * face (2*plane + side; 0 = the ray split inside the cell), trace[2*i+1] = source<<52 | pixelLevel<<48 | pixel<<24 |
 * index of the segment along its ray (a sort key: rays run concurrently).  rates6 = host [6][nleaf], accumulated. */
int rtb200_point_trace(rtb200_ctx* ctx, int nWave, const double* wavelength, const double* lum,
                       const double* metallicity, double coefSpectrum, const double* aDust, int dustApproximation,
                       int maxPixelLevel, int32_t nsrc, const int32_t* srcLeaf, const int32_t* srcWeight,
                       double* rates6, int64_t* nseg, int64_t* trace, int64_t traceCap, int64_t* traceLen);
/* the six (0:10)^4 tables of stellarBetaTable.f90:217-285 for one metallicity bracket, [6][11^4] in Fortran element
 * order: reactionRate1..3, energyRate1..3 */
int rtb200_point_tables(rtb200_ctx* ctx, int nWave, const double* wavelength, const double* lum,
                        const double* metallicity, double coefSpectrum, const double* aDust, int iMetal,
                        double coefMetal, double* tables);
/* zone number (1..24) and local angles of one direction: equiSources.f90:1391-1454 */
int rtb200_direction(int nAngularLevel, int64_t iray, int32_t* izone, double* phi, double* theta);
/* base-layer pattern table of one direction, [nx][12] = xy(x0,y0,len) xz(x0,z0,len) yz(y0,z0,len) xyTop xzTop yzTop */
int rtb200_patterns(int nAngularLevel, int64_t iray, int nx, double* out);
/* upstream leaf of every leaf for one direction, [3][nleaf] = xy, yz, xz; -1 boundary, -2 ray inactive
 * (transportRoutinesModule.f90:264-418) */
int rtb200_neighbours(rtb200_ctx* ctx, int nAngularLevel, int64_t iray, int32_t* nb);
/* wave of every leaf in the nested-grid sweep order of that direction, [nleaf], and the number of waves: every upstream
 * leaf rtb200_neighbours reports must lie in an earlier wave (centre-sum key on 2:1-balanced grids, dependency depth
 * elsewhere; set_tuning "amr_order") -- the property tests/test_diffuse_amr_gpu.py checks at sizes no oracle run reaches */
int rtb200_debug_waves(rtb200_ctx* ctx, int nAngularLevel, int64_t iray, int32_t* waveOfLeaf, int32_t* nwaves);

/* exp / log of csrc/portable_math.h evaluated on the device for n host values (bit-identity with a host build of the
 * same header is what makes the FAITHFUL point-source deposits comparable bit for bit, tests/test_portable_math.py) */
int rtb200_debug_portable_math(rtb200_ctx* ctx, int64_t n, const double* x, double* expOut, double* logOut);

/* the FAST arithmetic's exponential of the diffuse sweeps (csrc/segment_math.cuh: 64-entry table, degree-4 polynomial)
 * evaluated on the device for n host values tau >= 0: e^-tau and 1 - e^-tau (the latter without cancellation).  Its
 * truncation error is part of FAST mode's error budget (DESIGN.md 4.1); tests/test_diffuse_gpu.py holds it to 1e-11. */
int rtb200_debug_fast_exp(rtb200_ctx* ctx, int64_t n, const double* tau, double* expOut, double* oneMinusOut);

/* timing of the last rtb200_diffuse* call, from CUDA events on the launch stream: device milliseconds of the whole
 * call (opacities + sweep + merge) and of the sweep kernels alone, kernel launches issued (all / sweep kernel), and
 * the algorithmic bytes of the call (72 B per leaf per direction, SURVEY.md 8d; 96 B while emission is set). */
int rtb200_last_stats(rtb200_ctx* ctx, double* device_ms, double* sweep_ms, int64_t* launches,
                      int64_t* sweep_launches, double* algorithmic_bytes);

#ifdef __cplusplus
}
#endif
#endif /* RTB200_H */
