/*
 * libemagls_cuda -- C ABI of the B200-native eMagLS filter-design / binaural-render engine.
 *
 * The reference (thomasdeppisch/eMagLS @ d204b49) is pure MATLAB and has no FFI; its boundary
 * is the set of MATLAB function signatures below.  Each entry point here is what a MEX drop-in
 * of the same name binds (see INTEGRATION.md and mex/).  All matrices are column-major
 * ("MATLAB layout"), all reals are IEEE double, all angles are radians (azimuth, zenith).
 * Host pointers unless the function name ends in _dev.  Every function returns 0 on success or
 * a negative emagls_status; emagls_last_error() gives the message (the MEX shim turns it into
 * mexErrMsgIdAndTxt, mirroring the reference's assert()/error() behaviour).
 *
 * Batched extension (not in the reference API): `num_sets` HRTF sets (pages of hL/hR) times
 * `num_orient` head orientations (3x3 rotations R_o, row-major; world direction of HRIR-grid
 * direction u is R_o u, which equals one reference call with the rotated grid angles).
 * Outputs are [len x channels x (num_sets*num_orient)], orientation fastest.
 */
#ifndef EMAGLS_CUDA_H
#define EMAGLS_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct emagls_ctx* emagls_handle;

typedef enum {
  EMAGLS_OK = 0,
  EMAGLS_ERR_INVALID = -1,      /* bad argument; reference: assert(len >= size(hL,1)) etc.   */
  EMAGLS_ERR_CUDA = -2,         /* CUDA runtime / cuFFT failure                                */
  EMAGLS_ERR_UNSUPPORTED = -3,  /* valid in the reference but outside this build's hot path    */
  EMAGLS_ERR_NUMERIC = -4       /* e.g. HRIR grid too sparse for the simulation order          */
} emagls_status;

typedef enum { EMAGLS_BASIS_REAL = 0, EMAGLS_BASIS_COMPLEX = 1 } emagls_basis;
typedef enum { EMAGLS_ARRAY_RIGID = 0, EMAGLS_ARRAY_OPEN = 1 } emagls_array_type;
/* FP64 (default): every result within the FP64 tolerances of the parity tests.  FP32: the optional
 * reduced-precision path of the model-based designers -- the two direction-grid contractions of the
 * MagLS recursion carry 32 instead of 48 bits (4 instead of 6 int8 slices: 10 instead of 21 tensor-core
 * products); the factorisations stay FP64, because FP32 cannot represent the clipped subspace.
 * Filters agree with the FP64 path to ~1e-7 (bound asserted in the tests: 1e-4 relative, 0.05 dB).     */
typedef enum { EMAGLS_PRECISION_FP64 = 0, EMAGLS_PRECISION_FP32 = 1 } emagls_precision;

/* Constants that sit at the top of every reference function
 * (lib/getEMagLs2Filters.m:35-39, dependencies/getSMAIRMatrix.m:86). */
typedef struct {
  int nfft_max_len;      /* NFFT_MAX_LEN    = 2048 */
  double f_cut_min;      /* F_CUT_MIN_FREQ  = 1e3  */
  double svd_regul;      /* SVD_REGUL_CONST = 0.01 */
  double speed_of_sound; /* C               = 343  */
  int array_type;        /* SIMULATION_ARRAY_TYPE = 'rigid' */
  int basis;             /* shDefinition: 'real' (default) or 'complex' */
  int precision;         /* emagls_precision (default FP64) */
  int diffuseness_const; /* EXTENSION, default 0: diffuse-field covariance constraint ("applyDiffusenessConst" of
                          * earlier reference versions, removed before the surveyed commit: CHANGELOG.md:10-18) applied
                          * to the per-bin solutions of getEMagLsFilters / getEMagLs2Filters before the DC bin is set;
                          * real SH basis only, as in the reference (CHANGELOG.md:18) */
  int reserved[4];
} emagls_config;

/* A handle owns one CUDA stream and one private stream-ordered memory pool on `device` (scratch stays cached in
 * it between calls and is returned to the device by emagls_destroy; the device's default pool is not touched).
 * A handle is NOT thread-safe: calls on one handle must not overlap (error text, plans and profiler state are per
 * handle).  Different handles may be used from different host threads concurrently.                          */
int emagls_create(int device, emagls_handle* out);
int emagls_destroy(emagls_handle h);
const char* emagls_last_error(emagls_handle h);
void emagls_config_default(emagls_config* cfg);
/* Number of kernels launched by this handle since creation (bench.py's gpu_launches). */
long long emagls_launch_count(emagls_handle h);
/* Built-in CUDA-event profiler: when enabled, every kernel class of the design / render paths is
 * bracketed by an event pair on the handle's stream.  emagls_profile_read() synchronises, fills
 * ms[i] / counts[i] (accumulated milliseconds and spans per class, i < EMAGLS_PROF_CLASSES) and
 * returns the number of classes.  Class order: setup, factor, chain_fwd, gemm_fwd, gemm_bwd,
 * chain_bwd, tail, render_mac, render_fft, render_stage, gram, jacobi.                          */
#define EMAGLS_PROF_CLASSES 12
int emagls_profile_enable(emagls_handle h, int on);
int emagls_profile_read(emagls_handle h, double* ms, long long* counts, int reset);
/* Work statistics of the design calls since creation / the last reset (bench.py's roofline accounting):
 * out[0] = (problem, bin) pairs factorised on the TSQR + Jacobi route, out[1] = pairs solved on the Gram route,
 * out[2] = Jacobi problems, out[3] = Jacobi sweeps summed over them.  Synchronises the handle's stream.      */
int emagls_stats_read(emagls_handle h, long long* out, int reset);
/* Stream all work of this handle is enqueued on (cudaStream_t as void*), for event timing. */
void* emagls_stream(emagls_handle h);

/* ---- getEMagLs2Filters (lib/getEMagLs2Filters.m:1-2) ---------------------------------------
 * [wMlsL, wMlsR] = getEMagLs2Filters(hL, hR, hrirGridAziRad, hrirGridZenRad, micRadius,
 *                                    micGridAziRad, micGridZenRad, order, fs, len)
 * hL,hR: [num_samples x num_dirs x num_sets]; wL,wR: [len x num_mics x (num_sets*num_orient)].
 * rotations: [num_orient x 9] row-major 3x3, or NULL (num_orient must then be 1: identity,
 * i.e. exactly the reference call).  spectra (optional, may be NULL) receives the
 * positive-frequency solutions W_MLS as interleaved complex [K x num_mics x batch x 2 ears]
 * (what the reference holds at lib/getEMagLs2Filters.m:110) for per-bin parity tests.          */
int emagls_design_emagls2(emagls_handle h, const emagls_config* cfg,
                          const double* hL, const double* hR, int num_samples, int num_dirs,
                          const double* grid_azi, const double* grid_zen,
                          double mic_radius, const double* mic_azi, const double* mic_zen,
                          int num_mics, int order, double fs, int len,
                          int num_sets, int num_orient, const double* rotations,
                          double* wL, double* wR, double* spectra);

/* Same, but every array argument is a device pointer on the handle's device: no bulk host <-> device
 * copies; all kernels run on emagls_stream(h) (bench.py's device-resident `value`).  The call is NOT
 * fully asynchronous: it waits on the stream for four small read-backs that decide what is launched next
 * (the group delays, whose median is taken on the host; the conditioning flag of the grid basis; per
 * 128-bin group the bins admitted to the Gram route) and returns with the remaining work enqueued.       */
int emagls_design_emagls2_dev(emagls_handle h, const emagls_config* cfg,
                              const double* hL, const double* hR, int num_samples, int num_dirs,
                              const double* grid_azi, const double* grid_zen,
                              double mic_radius, const double* mic_azi, const double* mic_zen,
                              int num_mics, int order, double fs, int len,
                              int num_sets, int num_orient, const double* rotations,
                              double* wL, double* wR, double* spectra);

/* ---- custom shFunction handles (lib/getEMagLs2Filters.m:32, lib/getEMagLsFilters.m:32; example at
 * verifyEMagLs.m:356-368) ---------------------------------------------------------------------
 * A CUDA library cannot call back into MATLAB: the MEX shim evaluates a non-default handle on the host and
 * passes the two basis matrices down (SURVEY.md H8).  Both are evaluated at the SIMULATION order
 * simN = max(order, ceil(fs pi micRadius / c)) (getSMAIRMatrix.m:95), num_harmonics = (simN+1)^2:
 *   Y_hrir = shFunction(simN, [hrirGridAziRad hrirGridZenRad], 'real')       [num_dirs x num_harmonics], column-major
 *   Y_mic  = shFunction(simN, [micGridAziRad  micGridZenRad ], 'real')       [num_mics x num_harmonics x num_orient]
 * (one page of Y_mic per head orientation: the basis at the microphone positions seen from that orientation).
 * sh_domain = 0: getEMagLs2Filters (outputs [len x num_mics x P]); 1: getEMagLsFilters (outputs
 * [len x (order+1)^2 x P], Y_lo = the leading (order+1)^2 columns of the first page of Y_mic).  Real bases only. */
int emagls_design_sma_basis(emagls_handle h, const emagls_config* cfg, int sh_domain, const double* hL, const double* hR,
                            int num_samples, int num_dirs, const double* Y_hrir, int num_harmonics, double mic_radius,
                            const double* Y_mic, int num_mics, int order, double fs, int len, int num_sets,
                            int num_orient, double* wL, double* wR, double* spectra);

/* ---- getEMagLsFilters (lib/getEMagLsFilters.m:1-2): SH-domain output, (order+1)^2 channels.
 * For cfg->basis == COMPLEX the outputs are interleaved complex [len x nsh x batch].           */
int emagls_design_emagls(emagls_handle h, const emagls_config* cfg,
                         const double* hL, const double* hR, int num_samples, int num_dirs,
                         const double* grid_azi, const double* grid_zen,
                         double mic_radius, const double* mic_azi, const double* mic_zen,
                         int num_mics, int order, double fs, int len,
                         int num_sets, int num_orient, const double* rotations,
                         double* wL, double* wR, double* spectra);

/* ---- getMagLsFilters (lib/getMagLsFilters.m:1-2) and getLsFilters (lib/getLsFilters.m:1-2) */
int emagls_design_magls(emagls_handle h, const emagls_config* cfg,
                        const double* hL, const double* hR, int num_samples, int num_dirs,
                        const double* grid_azi, const double* grid_zen,
                        int order, double fs, int len, double* wL, double* wR, double* spectra);
/* Batched extension (not in the reference API): hL, hR [num_samples x num_dirs x num_sets]; the one pinv(Y)
 * serves every HRTF set; outputs [len x (order+1)^2 x num_sets], spectra [K x (order+1)^2 x num_sets x 2].   */
int emagls_design_magls_batch(emagls_handle h, const emagls_config* cfg,
                              const double* hL, const double* hR, int num_samples, int num_dirs,
                              const double* grid_azi, const double* grid_zen,
                              int order, double fs, int len, int num_sets, double* wL, double* wR, double* spectra);
int emagls_design_ls(emagls_handle h, const emagls_config* cfg,
                     const double* hL, const double* hR, int num_samples, int num_dirs,
                     const double* grid_azi, const double* grid_zen, int order,
                     double* wL, double* wR);

/* ---- getEMagLsFiltersFromAtf (lib/getEMagLsFiltersFromAtf.m:1) ------------------------------
 * hrir_grid: [num_dirs x 2] (azi, zen) column-major; atf_irs: [atf_samples x num_mics x atf_dirs];
 * atf_grid: [atf_dirs x 2].  mean_grid_dev_deg (optional) receives the value the reference
 * prints at lib/getEMagLsFiltersFromAtf.m:96.                                                  */
int emagls_design_from_atf(emagls_handle h, const emagls_config* cfg,
                           const double* hL, const double* hR, int num_samples, int num_dirs,
                           const double* hrir_grid, const double* atf_irs, int atf_samples,
                           int num_mics, int atf_dirs, const double* atf_grid,
                           double fs, int filter_len, double f_trans,
                           double* wL, double* wR, double* spectra, double* mean_grid_dev_deg);
/* Batched extension (not in the reference API): rotations [num_orient x 9] row-major; orientation b sees
 * HRIR-grid direction u at R_b u, so page b equals one reference call with hrirGridAziZenRad rotated by R_b.
 * wL, wR: [filter_len x num_mics x num_orient]; spectra (optional): [K x num_mics x num_orient x 2];
 * mean_grid_dev_deg (optional): [num_orient].  When the ATF grid is the smaller one (BASELINE config 3) the
 * per-bin factorisations are shared by the whole batch (lib/getEMagLsFiltersFromAtf.m:72-75,82-95).
 * _dev: all pointers on the device, enqueued on the handle's stream.                                         */
int emagls_design_from_atf_batch(emagls_handle h, const emagls_config* cfg,
                                 const double* hL, const double* hR, int num_samples, int num_dirs,
                                 const double* hrir_grid, const double* atf_irs, int atf_samples,
                                 int num_mics, int atf_dirs, const double* atf_grid,
                                 double fs, int filter_len, double f_trans, int num_orient, const double* rotations,
                                 double* wL, double* wR, double* spectra, double* mean_grid_dev_deg);
int emagls_design_from_atf_batch_dev(emagls_handle h, const emagls_config* cfg,
                                     const double* hL, const double* hR, int num_samples, int num_dirs,
                                     const double* hrir_grid, const double* atf_irs, int atf_samples,
                                     int num_mics, int atf_dirs, const double* atf_grid,
                                     double fs, int filter_len, double f_trans, int num_orient, const double* rotations,
                                     double* wL, double* wR, double* spectra);

/* ---- getEMagLsFiltersEMAinCH / EMAinSH (lib/getEMagLsFiltersEMAinCH.m:1-2, ...EMAinSH.m:1-2) */
int emagls_design_ema_ch(emagls_handle h, const emagls_config* cfg,
                         const double* hL, const double* hR, int num_samples, int num_dirs,
                         const double* grid_azi, const double* grid_zen,
                         double mic_radius, const double* mic_azi, int num_mics,
                         int order, double fs, int len, double* wL, double* wR, double* spectra);
/* Batched extension (not in the reference API), as for getEMagLs2Filters: hL, hR [num_samples x num_dirs x num_sets],
 * rotations [num_orient x 9] row-major (page b = one reference call with the HRIR grid rotated by R_b),
 * outputs [len x (2 order + 1) x (num_sets * num_orient)].                                                          */
int emagls_design_ema_ch_batch(emagls_handle h, const emagls_config* cfg,
                               const double* hL, const double* hR, int num_samples, int num_dirs,
                               const double* grid_azi, const double* grid_zen,
                               double mic_radius, const double* mic_azi, int num_mics,
                               int order, double fs, int len, int num_sets, int num_orient, const double* rotations,
                               double* wL, double* wR, double* spectra);
int emagls_design_ema_sh(emagls_handle h, const emagls_config* cfg,
                         const double* hL, const double* hR, int num_samples, int num_dirs,
                         const double* grid_azi, const double* grid_zen,
                         double mic_radius, const double* mic_azi, int num_mics,
                         int order, double fs, int len, double* wL, double* wR, double* spectra);

/* ---- getSMAIRMatrix (dependencies/getSMAIRMatrix.m:1) ---------------------------------------
 * The `params` struct fields that are read on the hot path, flattened.  out: interleaved complex
 * [rows x (simN+1)^2 x (nfft/2+1)], rows = num_mics if return_raw_mic_sigs else (order+1)^2.
 * sim_order_out (optional) receives simulationOrder (getSMAIRMatrix.m:95).
 * Call with out == NULL to query sim_order_out only.                                           */
int emagls_smair_matrix(emagls_handle h, const emagls_config* cfg,
                        const double* mic_azi, const double* mic_zen, int num_mics,
                        int order, double fs, double sma_radius, int nfft,
                        int return_raw_mic_sigs, double* out, int* sim_order_out);

/* ---- binauralDecode (dependencies/binauralDecode.m:1-2) -------------------------------------
 * in: [num_samples x num_ch]; wL,wR: [len x num_ch]; out: [out_rows x 2] with
 * out_rows = num_samples (compensate_delay == 0) or num_samples - len/2 + 1.                   */
int emagls_binaural_decode(emagls_handle h, const double* in, long long num_samples, int num_ch,
                           const double* wL, const double* wR, int len, int compensate_delay,
                           double* out);
int emagls_binaural_decode_dev(emagls_handle h, const double* in, long long num_samples,
                               int num_ch, const double* wL, const double* wR, int len,
                               int compensate_delay, double* out);

/* ---- head-tracked binauralDecode (not in the reference API) ---------------------------------------------------
 * Renders `in` [num_samples x num_ch] with a filter bank wL, wR [len x num_ch x num_pages] (column-major, the layout
 * the designers return: page = set * num_orient + orient) while a head tracker picks the page: track[f] (0-based, int32,
 * num_frames entries) is the page of frame f, which covers samples [f hop, (f + 1) hop) of the track's time axis, and
 * in[0] sits at first_sample on that axis (so that consecutive pieces of a stream, or time shards, compose).  With
 * y_p = binauralDecode with page p, t = first_sample + n, f = t / hop, i = t - f hop, c = track[f],
 * a = track[max(f - 1, 0)] and g = (i < fade) ? (i + 0.5) / fade : 1:
 *     out[n] = (1 - g) y_a[n] + g y_c[n]       (a == c: exactly y_c[n])
 * a linear equal-amplitude crossfade over the first `fade` samples of every frame (fade = 0: hard switch).
 * compensate_delay as in emagls_binaural_decode (output row r holds sample r + len/2 - 1; the frame timing refers to the
 * input sample n).  EMAGLS_ERR_INVALID, checked on the host before anything is launched: a null pointer, hop < 1, fade
 * outside [0, hop], first_sample < 0, num_frames < (first_sample + num_samples - 1) / hop + 1, a used track entry
 * outside [0, num_pages), an odd len with compensate_delay.
 * _dev: in, wL, wR and out are device pointers; `track` is HOST memory in both variants (the launch geometry is derived
 * from it on the host), the one exception to the _dev convention.  The call returns with the work enqueued on
 * emagls_stream(h) after the upload of its tables.                                                                  */
int emagls_binaural_decode_tracked(emagls_handle h, const double* in, long long num_samples, int num_ch,
                                   const double* wL, const double* wR, int len, int num_pages,
                                   const int32_t* track, long long num_frames, int hop, int fade,
                                   long long first_sample, int compensate_delay, double* out);
int emagls_binaural_decode_tracked_dev(emagls_handle h, const double* in, long long num_samples, int num_ch,
                                       const double* wL, const double* wR, int len, int num_pages,
                                       const int32_t* track, long long num_frames, int hop, int fade,
                                       long long first_sample, int compensate_delay, double* out);

/* ======================================================================================================
 * Callers either side of the hot path (SURVEY.md section 8-f): radial filters, SH/CH encoding and
 * rotation of the recording in front of the render, the remaining lib/ designers.
 * ====================================================================================================== */
typedef enum {
  EMAGLS_RADIAL_NONE = 0,       /* 'none'      (getRadialFilter.m:29-33)  */
  EMAGLS_RADIAL_TIKHONOV = 1,   /* 'tikhonov'  (:45-52), the default      */
  EMAGLS_RADIAL_SOFTLIMIT = 2,  /* 'softlimit' (:54-59)                   */
  EMAGLS_RADIAL_FULL = 3        /* 'full'      (:61-62)                   */
} emagls_radial_kind;

/* The fields of the reference `params` struct that getRadialFilter reads (getRadialFilter.m:9-23,48-56). */
typedef struct {
  int kind;              /* emagls_radial_kind; anything else -> EMAGLS_ERR_INVALID ("Unkown radialFilter") */
  double regul_const;    /* params.regulConst  (default 1e-2)  */
  double noise_gain_db;  /* params.noiseGainDb (softlimit)     */
  int array_type;        /* emagls_array_type ('directional' is not built) */
} emagls_radial_params;
void emagls_radial_params_default(emagls_radial_params* rp);

/* radFilts = getRadialFilter(params) (dependencies/getRadialFilter.m:1): out interleaved complex
 * [nfft/2+1 x (order+1)] column-major, nfft = oversamplingFactor * irLen.  NaN entries (e.g. softlimit
 * at kr = 0) are returned as NaN, exactly as the reference does.                                      */
int emagls_radial_filter(emagls_handle h, const emagls_config* cfg, const emagls_radial_params* rp,
                         int order, double fs, double sma_radius, int nfft, double* out);

/* sigFiltered = applyRadialFilter(inSig, params) (dependencies/applyRadialFilter.m:1):
 * in [num_samples x (order+1)^2]; out [emagls_apply_radial_filter_rows(num_samples, nfft) x (order+1)^2]
 * (= max(num_samples, nfft) - nfft/2 rows: zero padding of short signals, filter delay removed).     */
long long emagls_apply_radial_filter_rows(long long num_samples, int nfft);
int emagls_apply_radial_filter(emagls_handle h, const emagls_config* cfg, const emagls_radial_params* rp,
                               const double* in, long long num_samples, int order, double fs,
                               double sma_radius, int nfft, double* out);
int emagls_apply_radial_filter_dev(emagls_handle h, const emagls_config* cfg,
                                   const emagls_radial_params* rp, const double* in,
                                   long long num_samples, int order, double fs, double sma_radius,
                                   int nfft, double* out);

/* getSMAIRMatrix with params.radialFilter ~= 'none' (dependencies/getSMAIRMatrix.m:129-139, SH-domain
 * output only; includes the reference's double application of real(BnTi) at the Nyquist bin).       */
int emagls_smair_matrix_radial(emagls_handle h, const emagls_config* cfg, const emagls_radial_params* rp,
                               const double* mic_azi, const double* mic_zen, int num_mics, int order,
                               double fs, double sma_radius, int nfft, double* out, int* sim_order_out);

/* shRecording = smaRecording * pinv(getSH(order, mics, shDefinition).') (verifyEMagLs.m:235-236,
 * testEMagLs.m:98): in [num_samples x num_mics]; out [num_samples x (order+1)^2], interleaved complex
 * for cfg->basis == COMPLEX.  emagls_ch_encode: the same with getCH(order, mic_azi) (testEMagLs.m:99-102),
 * out [num_samples x (2*order+1)].                                                                   */
int emagls_sh_encode(emagls_handle h, const emagls_config* cfg, const double* in, long long num_samples,
                     int num_mics, const double* mic_azi, const double* mic_zen, int order, double* out);
int emagls_sh_encode_dev(emagls_handle h, const emagls_config* cfg, const double* in,
                         long long num_samples, int num_mics, const double* mic_azi,
                         const double* mic_zen, int order, double* out);
int emagls_ch_encode(emagls_handle h, const emagls_config* cfg, const double* in, long long num_samples,
                     int num_mics, const double* mic_azi, int order, double* out);

/* Rotation of a real-SH-domain signal, the rotateHOA_N3D(in, yaw, pitch, roll) call of
 * dependencies/binauralDecode.m:26-30 (angles in radians here): out = in * getSHrotMtx(
 * euler2rotationMatrix(-yaw, -pitch, roll, 'zyx'), order, 'real').'; in/out [num_samples x (order+1)^2]. */
int emagls_rotate_sh(emagls_handle h, const double* in, long long num_samples, int order,
                     double yaw_rad, double pitch_rad, double roll_rad, double* out);
int emagls_rotate_sh_dev(emagls_handle h, const double* in, long long num_samples, int order,
                         double yaw_rad, double pitch_rad, double roll_rad, double* out);

/* [wMlsL, wMlsR] = getMagLsFilters2D(hLHor, hRHor, horHrirGridAziRad, order, fs, len, chDefinition)
 * (lib/getMagLsFilters2D.m:1): outputs [len x (2*order+1)], interleaved complex for COMPLEX;
 * spectra (optional) complex [K x (2*order+1) x 2 ears].                                             */
int emagls_design_magls_2d(emagls_handle h, const emagls_config* cfg, const double* hL, const double* hR,
                           int num_samples, int num_dirs, const double* grid_azi, int order, double fs,
                           int len, double* wL, double* wR, double* spectra);

/* [wShf, W_Shf] = getMagLsSphericalHeadFilter(micRadius, order, fs, len)
 * (lib/getMagLsSphericalHeadFilter.m:1): w [len]; W_full (optional) [min(nfft_max_len, 2 len)] real.  */
int emagls_spherical_head_filter(emagls_handle h, const emagls_config* cfg, double mic_radius, int order,
                                 double fs, int len, double* w, double* W_full);
/* wAdf = getMagLsArrayDiffuseFilter(micRadius, micGridAziRad, micGridZenRad, order, fs, len, shDefinition)
 * (lib/getMagLsArrayDiffuseFilter.m:1): w [len]; shDefinition = cfg->basis (the result depends on it). */
int emagls_array_diffuse_filter(emagls_handle h, const emagls_config* cfg, double mic_radius,
                                const double* mic_azi, const double* mic_zen, int num_mics, int order,
                                double fs, int len, double* w);

/* ---- building blocks exposed for parity tests (each mirrors one reference function) --------- */
/* getSH(N, [azi zen], basis) (dependencies/Spherical-Harmonic-Transform/getSH.m:1):
 * out [num_dirs x (N+1)^2] column-major; interleaved complex for COMPLEX.                      */
int emagls_get_sh(emagls_handle h, int order, const double* azi, const double* zen, int num_dirs,
                  int basis, double* out);
/* grpdelay(sum(h, 2), 1, f, fs) with f = linspace(0, fs/2, num_freqs), and its median: the group delay the
 * designers remove from an HRIR set (lib/getEMagLs2Filters.m:72-75).  hrir [taps x num_dirs] column-major
 * on the host; gd [num_freqs] and median_out may be NULL.                                          */
int emagls_group_delay(emagls_handle h, const double* hrir, int taps, int num_dirs, int num_freqs,
                       double fs, double* gd, double* median_out);
/* sphModalCoeffs(N, kr, arrayType) (dependencies/Array-Response-Simulator/sphModalCoeffs.m:1):
 * out interleaved complex [num_kr x (N+1)] column-major.                                       */
int emagls_sph_modal_coeffs(emagls_handle h, int order, const double* kr, int num_kr,
                            int array_type, double* out);
/* Per-bin regularised inverse applied to targets (lib/getEMagLs2Filters.m:87-94):
 * pw: interleaved complex [num_ch x num_dirs] column-major, targets: complex [num_t x num_dirs];
 * out: complex [num_t x num_ch] = targets * Y_reg_inv.                                         */
int emagls_regularized_apply(emagls_handle h, const double* pw, int num_ch, int num_dirs,
                             const double* targets, int num_t, double svd_regul, double* out);

#ifdef __cplusplus
}
#endif
#endif /* EMAGLS_CUDA_H */
