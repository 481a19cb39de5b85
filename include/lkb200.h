/* lkb200.h - C ABI of the B200-native periodogram-and-detrending engine.
 *
 * The reference (lightkurve, pure Python) has no FFI: its de-facto boundary is
 * five Python call sites into astropy/scipy/numpy (SURVEY.md 8b).  Each entry
 * point below replaces one of those call sites; the ctypes stub a lightkurve
 * maintainer would add is shown in INTEGRATION.md.
 *
 * Conventions
 *  - every function returns an int status: 0 = LKB_OK, < 0 = error; a
 *    thread-local message is available from lkb_last_error().
 *  - all buffers are caller-allocated and caller-owned.  `mem` says where they
 *    live: LKB_MEM_HOST (plain host pointers; the call stages through the
 *    library's device workspace and is synchronous) or LKB_MEM_DEVICE (device
 *    pointers on the current device; the call is asynchronous on `stream`).
 *  - `stream` is a cudaStream_t passed as void* (NULL = the legacy default
 *    stream).  No torch types anywhere.
 *  - ragged batches are CSR: int64 offsets[B+1] into the concatenated arrays.
 *  - there is NO CPU fallback: without a CUDA device every compute entry point
 *    returns LKB_E_CUDA.
 */
#ifndef LKB200_H
#define LKB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LKB_OK             0
#define LKB_E_ARG         -1   /* bad argument */
#define LKB_E_CUDA        -2   /* CUDA runtime error / no device */
#define LKB_E_OOM         -3   /* device allocation failed */
#define LKB_E_SINGULAR    -4   /* normal equations singular (numpy LinAlgError analogue) */
#define LKB_E_UNSUPPORTED -5   /* shape outside what the kernels support / optional component absent */
#define LKB_E_NCCL        -6   /* NCCL call failed */
#define LKB_E_VERIFY      -7   /* a kernel's built-in self-check (LKB_NUFFT_VERIFY=1) found a wrong result */

#define LKB_MEM_HOST   0
#define LKB_MEM_DEVICE 1

#define LKB_DTYPE_F32 0
#define LKB_DTYPE_F64 1

/* Lomb-Scargle output normalisation (periodogram.py:969-975) */
#define LKB_LS_NORM_PSD_RAW   0  /* astropy normalization="psd": 0.5*N*(YC^2/CC+YS^2/SS)   */
#define LKB_LS_NORM_PSD_SCALE 1  /* raw * norm_scale[b]   (lightkurve "psd": 2/(N*oversample*fs)) */
#define LKB_LS_NORM_AMPLITUDE 2  /* sqrt(raw)*sqrt(4/N)   (lightkurve "amplitude")          */

/* shared-grid Lomb-Scargle contraction algorithm */
#define LKB_LS_ALGO_AUTO     0   /* NUFFT when the grid allows it and the job is large (regular f_k = (k0 + k) df,
                                    integer k0, df * baseline <= 1, ascending times); else tcgen05 / direct sums */
#define LKB_LS_ALGO_SIMT     1   /* exact direct sums on the CUDA cores (K1: ls_direct_kernel, K2: tiled contraction):
                                    what the shim maps ls_method="slow" to */
#define LKB_LS_ALGO_TCGEN05  2   /* K2 only: split-fp16 tcgen05.mma, fp32 TMEM accumulators */
#define LKB_LS_ALGO_NUFFT    3   /* type-1 NUFFT (spread + FFT): the algorithm behind the reference's optional
                                    ls_method="fastnifty" (periodogram.py:917-946); LKB_E_UNSUPPORTED when the
                                    grid / times do not qualify */

/* BLS objective (astropy BoxLeastSquares.power objective=) */
#define LKB_BLS_LIKELIHOOD 0
#define LKB_BLS_SNR        1

/* ---- library management ------------------------------------------------ */
const char* lkb_last_error(void);
int lkb_version(void);                 /* 1000*major + minor */
int lkb_device_count(void);            /* number of visible CUDA devices (0 if none) */
int lkb_init(int device);              /* bind the calling process to `device`, create the workspace pool */
int lkb_shutdown(void);                /* free the workspace pool */
int lkb_sm_count(void);                /* multiprocessor count of the bound device */
/* counters: number of kernels this library launched since init (bench gpu_launches) */
int64_t lkb_launch_count(void);
/* kernel family (LKB_LS_ALGO_SIMT / _TCGEN05 / _NUFFT) the most recent lkb_ls_power* call actually ran; -1 before
 * the first call.  Lets a caller (bench.py, tests) see what LKB_LS_ALGO_AUTO resolved to. */
int lkb_ls_last_algo(void);
/* light curves of the most recent shared-grid NUFFT call that were transformed a second time in double precision
 * (precision escalation: flux excursion > LKB_NUFFT_ESCALATE [250] x the in-band peak amplitude; DESIGN.md section 2) */
int lkb_ls_last_escalated(void);
/* Measurement hooks (bench.py roofline): when enabled, every compute call records CUDA events on
 * its stream around its DOMINANT kernel (LS contraction / BLS search / flatten / Gram accumulation).
 * lkb_profile_read synchronises, writes up to max_n durations [ms] in call order, resets the ring
 * and returns how many were written (< 0 on error). */
int lkb_profile_enable(int on);
/* Diagnostic (not part of the drop-in boundary): read back `bytes` bytes at `offset` of one of the library's
 * internal workspace buffers (slot numbering: enum Slot in lightkurve_b200/csrc/common.cuh) after the last call -
 * used by tools/nufft_gpu_check.py to compare intermediate results stage by stage with the CPU harness. */
int lkb_ws_read(int slot, int64_t offset, int64_t bytes, void* out);
int lkb_profile_read(double* ms_out, int max_n);

/* ---- Lomb-Scargle ------------------------------------------------------- */
/* K1: ragged batch, one (time, flux) pair per light curve; replaces
 *   LombScargle(time, flux, normalization="psd").power(frequency, method)
 * at /root/reference/src/lightkurve/periodogram.py:961-964 plus the rescale at
 * :969-975.  Computes the exact floating-mean sums (astropy "slow" math).
 *   t            [offsets[B]] fp64 days (any origin; shifted internally)
 *   y            [offsets[B]] flux, y_dtype F32 or F64; no NaNs (caller drops
 *                them as periodogram.py:785-790 does)
 *   freq         fp64 cycles/day.  freq_offsets == NULL: one grid of F bins
 *                shared by all light curves; else CSR [B+1] per-LC grids.
 *   norm_scale   [B] or NULL (required for LKB_LS_NORM_PSD_SCALE)
 *   power        fp32, [B,F] (shared grid) or CSR like freq.
 */
int lkb_ls_power(const double* t, const void* y, int y_dtype, const int64_t* offsets, int B,
                 const double* freq, const int64_t* freq_offsets, int64_t F,
                 int normalization, const double* norm_scale,
                 float* power, int mem, void* stream);
/* The same with the kernel family chosen by the caller (`method=` of LombScargle.power at
 * periodogram.py:964): LKB_LS_ALGO_AUTO (what lkb_ls_power does), LKB_LS_ALGO_SIMT (direct sums, "slow") or
 * LKB_LS_ALGO_NUFFT ("fastnifty": one shared regular host-visible grid, sorted times). */
int lkb_ls_power_ex(const double* t, const void* y, int y_dtype, const int64_t* offsets, int B,
                    const double* freq, const int64_t* freq_offsets, int64_t F,
                    int normalization, const double* norm_scale,
                    float* power, int mem, void* stream, int algo);

/* K1n: multi-term ("chi2") periodogram = LombScargle(time, flux, nterms=n, normalization="psd")
 * .power(frequency, method="chi2"|"fastchi2"), the call lightkurve makes for nterms > 1
 * (periodogram.py:948-964): P = 0.5 XTy^T (XTX)^-1 XTy with X = [1, sin(k w t), cos(k w t)], k <= n.
 * Same ragged layout as lkb_ls_power; nterms in [1, 4].  theta (nullable) receives the
 * 2n+1 fitted parameters per (light curve, frequency) [same order as power, (2n+1) doubles each]:
 * the maximum-likelihood model LombScargle.model evaluates (periodogram.py:1010), for times
 * measured from the light curve's first cadence and flux centred on its mean. */
int lkb_ls_power_chi2(const double* t, const void* y, int y_dtype, const int64_t* offsets, int B,
                      const double* freq, const int64_t* freq_offsets, int64_t F, int nterms,
                      int normalization, const double* norm_scale, float* power, double* theta,
                      int mem, void* stream);

/* K2: batch sharing ONE cadence grid (BASELINE config 2); same math, but the
 * sin/cos design matrix is synthesised once per (frequency, cadence) tile and
 * contracted against all B light curves.
 *   t [N] fp64, y [B,N] row-major (y_dtype), freq [F] fp64, power [B,F] fp32.
 *   norm_scale: scalar pointer (one value, all LCs share N) or NULL.
 */
int lkb_ls_power_shared(const double* t, const void* y, int y_dtype, int B, int64_t N,
                        const double* freq, int64_t F,
                        int normalization, const double* norm_scale,
                        float* power, int mem, void* stream, int algo);

/* ---- Box Least Squares --------------------------------------------------- */
/* K3: replaces BoxLeastSquares(t, y, dy).power(period, duration, objective,
 * method="fast", oversample) at periodogram.py:1161-1169.  Inputs are the RAW
 * time/flux (the call subtracts min(t) and median(y) itself like astropy's
 * core.py); dy == NULL means unit weights.  period [P] ascending or not,
 * duration [D]; outputs fp64 [B,P] each; transit_time is absolute (t_ref added).
 * best_bins (nullable) int32 [B,P,2] = (start bin n, duration in bins) of the
 * winning box - the quantity the parity tests require bit-exact.
 */
int lkb_bls_power(const double* t, const double* y, const double* dy, const int64_t* offsets, int B,
                  const double* period, int64_t P, const double* duration, int D,
                  int oversample, int objective,
                  double* power, double* depth, double* depth_err, double* duration_out,
                  double* transit_time, double* depth_snr, double* log_likelihood,
                  int32_t* best_bins, int mem, void* stream);

/* K3s: the exact, unbinned search BoxLeastSquares(t, y, dy).power(period, duration,
 * objective, method="slow", oversample) - lightkurve passes `method=` of
 * to_periodogram("bls", ...) through to that call (periodogram.py:1169).  For each
 * duration d, the transit epochs are t0_i = i*d/oversample (i < ceil((P + d/oversample)
 * / (d/oversample))), a cadence is in the box when |((x - t0 + P/2) % P) - P/2| < d/2
 * (x = t - min(t), numpy float semantics), and the FIRST strict maximum of the
 * objective in (duration, t0) order with depth > 0 is kept.  duration_out is the
 * trial duration itself.  Same arguments and layouts as lkb_bls_power, except:
 *   times must be ascending within each light curve (else LKB_E_UNSUPPORTED);
 *   best_index (nullable) int32 [B,P,3] = (duration index, t0 index, number of
 *   in-box cadences) of the winning box.
 * A period where no box has depth > 0 gets power = -inf, depth = depth_err =
 * depth_snr = log_likelihood = duration = 0, transit_time = min(t), best_index =
 * (-1, -1, 0); astropy raises there instead.
 */
int lkb_bls_power_slow(const double* t, const double* y, const double* dy, const int64_t* offsets, int B,
                       const double* period, int64_t P, const double* duration, int D,
                       int oversample, int objective,
                       double* power, double* depth, double* depth_err, double* duration_out,
                       double* transit_time, double* depth_snr, double* log_likelihood,
                       int32_t* best_index, int mem, void* stream);

/* Debug/parity entry: the per-sample bin index of bls.c for ONE period,
 * ind[n] = (int)(fabs(fmod(t[n]-min_t, period))/bin_duration)+1, evaluated by the
 * same device function the search kernel uses. */
int lkb_bls_bin_index(const double* t_rel, int64_t N, double min_t, double period,
                      double bin_duration, int32_t* ind, int mem, void* stream);

/* ---- flatten (Savitzky-Golay detrend) ------------------------------------ */
/* K4: replaces the body of LightCurve.flatten, lightcurve.py:996-1070
 * (scipy savgol_filter :1040 + interp1d :1053 + the sigma-clip loop).
 *   time, flux, flux_err  [offsets[B]] fp64 (flux_err may be NULL)
 *   exclude_mask          uint8 [offsets[B]] or NULL; 1 = do not use (mask=True in lightkurve)
 *   break_tolerance       NaN disables gap splitting (break_tolerance=None)
 *   outputs flat, flat_err, trend  fp64 [offsets[B]]  (flat_err may be NULL)
 */
int lkb_flatten(const double* time, const double* flux, const double* flux_err,
                const uint8_t* exclude_mask, const int64_t* offsets, int B,
                int window_length, int polyorder, double break_tolerance, int niters, double sigma,
                double* flat, double* flat_err, double* trend, int mem, void* stream);

/* Host-only helper (no GPU needed): the Savitzky-Golay tables lkb_flatten uploads -
 * coeffs[w] = scipy.signal.savgol_coeffs(w, p) (symmetric FIR) and edge[w*(w/2)] with
 * edge[j*(w/2)+i] = weight of x[j] in the degree-p polynomial fit of the first w samples
 * evaluated at position i (scipy _fit_edges_polyfit).  Exposed so CPU tests can pin them. */
int lkb_savgol_tables(int window_length, int polyorder, double* coeffs, double* edge);

/* ---- RegressionCorrector -------------------------------------------------- */
/* K5: replaces _fit_coefficients + the correct() loop,
 * correctors/regressioncorrector.py:127-189,244-279 (dense branch).
 *   X            [N,K] row-major fp64, shared by the batch (x_batched=0) or [B,N,K] (x_batched=1)
 *   y            [B,N] fp64;  flux_err [B,N] or NULL (NULL = ones, :157-160)
 *   cadence_mask uint8 [B,N] or NULL (1 = use)
 *   prior_mu, prior_sigma [K] fp64 (sigma may be +inf) or both NULL
 *   outputs: coeff [B,K], model [B,N] (median-subtracted, :278-279),
 *            outlier_mask uint8 [B,N]; status_out int32 [B] (0 or LKB_E_SINGULAR per LC, nullable);
 *            coeff_cov [B,K,K] (nullable) = (X^T W X + diag(1/prior_sigma^2))^-1 of the last fit, the
 *            np.linalg.inv(sigma_w_inv) of propagate_errors=True (:185)
 */
int lkb_regress(const double* X, int x_batched, const double* y, const double* flux_err,
                const uint8_t* cadence_mask, const double* prior_mu, const double* prior_sigma,
                int B, int64_t N, int K, double clip_sigma, int niters,
                double* coeff, double* model, uint8_t* outlier_mask, int32_t* status_out, double* coeff_cov,
                int mem, void* stream);

/* ---- batched order statistics (K6) ---------------------------------------- */
/* nanmedian and nanstd (ddof=0) per light curve: np.nanmedian / np.nanstd as used by
 * normalize (lightcurve.py:1253-1254) and flatten (:1003-1005). out_median/out_std [B]. */
int lkb_nanmedian_std(const double* x, const int64_t* offsets, int B,
                      double* out_median, double* out_std, int mem, void* stream);

/* ---- periodogram background (the step after Lomb-Scargle) -------------------- */
/* Periodogram.smooth(method="logmedian") (periodogram.py:260-284), the background that
 * Periodogram.flatten (:381-429) divides by, for B periodograms on one frequency grid:
 *   background[b, i] = mean over the windows w covering bin i of nanmedian(power[b, lo_w:hi_w]) / corr_factor.
 * win_lo/win_hi [W] (HOST, int32, ordered) are the half-open bin ranges of the reference's moving window
 * (|log10 f - x0| < filter_width, x0 advancing by filter_width / 2), built by the caller from the grid.
 * power/background [B, F] fp64 (host or device per `mem`).  Bins covered by no window get NaN (0/0). */
int lkb_pg_logmedian(const double* power, int B, int64_t F, const int32_t* win_lo, const int32_t* win_hi, int W,
                     double corr_factor, double* background, int mem, void* stream);

/* ---- multi-GPU: the one exchange step of the path (SURVEY.md 8e) ------------------ */
/* A LightCurveCollection is sharded BY TARGET over one process per GPU; the only data exchange is the
 * reassembly of the fp32 power array [B, F] from the per-rank blocks (the reference has no counterpart: it
 * loops over light curves in one Python process, collections.py:145-276).  NCCL is bound at run time
 * (dlopen), so single-GPU use needs no NCCL.  Bootstrap: rank 0 fills a 128-byte id with
 * lkb_nccl_unique_id, the host program carries it to the other ranks (torch.distributed store, MPI, a
 * pipe ...), then EVERY rank calls lkb_nccl_init(rank, world_size, id) after lkb_init(device) - collectively,
 * like ncclCommInitRank.  lkb_allgather_f32 gathers `n_local` floats from every rank into
 * global[world_size * n_local] (rank-major) - DEVICE pointers, asynchronous on `stream` (0 = default
 * stream), one ncclAllGather over NVLink/NVSwitch.  Ragged shards are padded to a common n_local by the
 * caller (lightkurve_b200/dist.py).  Errors: LKB_E_UNSUPPORTED if no NCCL library can be loaded,
 * LKB_E_NCCL if an NCCL call fails, LKB_E_ARG without a communicator. */
#define LKB_NCCL_ID_BYTES 128
int lkb_nccl_version(void);            /* NCCL_VERSION_CODE of the bound library, 0 if none */
int lkb_nccl_unique_id(void* id_out /* [LKB_NCCL_ID_BYTES] */);
int lkb_nccl_init(int rank, int world_size, const void* id /* [LKB_NCCL_ID_BYTES] */);
int lkb_nccl_shutdown(void);
int lkb_nccl_rank(void);               /* -1 without a communicator */
int lkb_nccl_world_size(void);         /* 0 without a communicator */
int lkb_allgather_f32(const float* local, int64_t n_local, float* global, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LKB200_H */
