/*
 * bdlm.h -- C ABI of libbdlm.so: the B200-native Kalman hot path of bayesian_dlms.
 *
 * The reference (jonnylaw/bayesian_dlms, pure Scala) has no FFI seam of its own; the
 * "operator API" for this path is its public Scala surface.  Every entry point below
 * names the reference function(s) it replaces (paths relative to
 * core/src/main/scala/dlm/model/ of the reference).  INTEGRATION.md shows the Scala
 * (Panama / JNI) binding a maintainer would add on the reference side.
 *
 * Conventions
 *  - fp64 everywhere.  Matrices are column-major inside a row (Breeze DenseMatrix.data).
 *  - F is n x p (enters as F^T x, Dlm.scala:264), G is n x n, V p x p, W n x n.
 *  - A missing observation (None in DenseVector[Option[Double]], Dlm.scala:94) is NaN.
 *  - "rows" = T + keep_init.  keep_init = 1 reproduces KalmanFilter(adv).filter
 *    (Filter.scala:41-45: the initial state is kept, row 0, with f,Q = NaN for None);
 *    keep_init = 0 reproduces filterDlm / filterTraverse / filterArray (Filter.scala:32-62).
 *  - Per-step arrays (y, z, every output) are addressed through `layout`:
 *      BDLM_TIME_MAJOR   [rows][k][B]  (device-native: a warp of 32 series touches 256
 *                                       contiguous bytes per scalar field per step)
 *      BDLM_SERIES_MAJOR [B][rows][k]  (the order a Vector[KfState] per series flattens to)
 *    y has T rows (never the extra initial row), z and all outputs have `rows` rows
 *    (FFBS always T+1).
 *  - Per-series parameters (V, W, m0, C0) are either shared by the whole batch
 *    (host pointers, tiny) or given per series, [k][B] for TIME_MAJOR and [B][k] for
 *    SERIES_MAJOR, in the same memory space as the data.
 *  - F, G, times are model-assembly products evaluated from the Scala closures
 *    mod.f(time_t), mod.g(dt_t) on the host: HOST pointers shared by the batch, unless the
 *    BDLM_PS_TIMES / BDLM_PS_F / BDLM_PS_G bits of per_series say they are given per series.
 *    g_tv / f_tv = 1 when they vary with t: G[T][n*n] with G[t] = g(times[t]-times[t-1]),
 *    times[-1] := min(times) - 1 (KalmanFilter.initialiseState, KalmanFilter.scala:112-118).
 *    times == NULL means the regular grid 1..T (every dt = 1).
 *  - mem = BDLM_DEVICE: y/z/outputs/per-series params/status are device pointers on the
 *    context's GPU and the call only enqueues work on the context's stream (call
 *    bdlm_sync or synchronise the stream yourself).  mem = BDLM_HOST: they are host
 *    pointers (pinned for full PCIe speed); the library stages slabs of series through
 *    device memory, overlapping H2D, kernels and D2H, and returns when the outputs are
 *    in host memory.
 *  - Ownership: the caller owns every buffer it passes; the library owns only the
 *    context and its internal workspace (freed by bdlm_destroy).
 *  - Return value: 0 ok; < 0 API misuse (BDLM_E_*), nothing was launched, message in
 *    bdlm_last_error.  Numerical failures never abort the batch: they are reported per
 *    series in status[b] (bit mask BDLM_ST_*), mirroring the exceptions the reference
 *    would throw for that series.  No C++ exception crosses this ABI.
 *  - Threading: a context is single-threaded-at-a-time and owns one CUDA stream;
 *    distinct contexts are fully concurrent (one per GPU for multi-GPU use).
 *  - There is no CPU fallback: without a CUDA device bdlm_create fails.
 */
#ifndef BDLM_H
#define BDLM_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define BDLM_API __attribute__((visibility("default")))
#else
#define BDLM_API
#endif

#define BDLM_VERSION 100

#define BDLM_MAX_N 48 /* state dimension (n and p together must fit one SM's 227 KB)     */
#define BDLM_MAX_P 32 /* observation dimension                                          */
#define BDLM_COMM_ID_BYTES 128  /* opaque rendezvous id of a multi-process communicator     */
#define BDLM_COMM_MAX_WORLD 64  /* ranks (GPUs) per communicator                            */

enum { BDLM_TIME_MAJOR = 0, BDLM_SERIES_MAJOR = 1 };
enum { BDLM_DEVICE = 0, BDLM_HOST = 1 };

/* error codes (return values < 0) */
enum {
  BDLM_E_ARG = -1,       /* null pointer / bad dims / unsupported n,p / bad flag  */
  BDLM_E_EMPTY = -2,     /* T == 0: NoSuchElementException (KalmanFilter.scala:116-117) */
  BDLM_E_CUDA = -3,      /* CUDA runtime error, see bdlm_last_error                */
  BDLM_E_NODEVICE = -4,  /* no usable CUDA device: there is no CPU fallback        */
  BDLM_E_NCCL = -5       /* NCCL could not be loaded or a collective failed        */
};

/* per-series status bits */
enum {
  BDLM_ST_SINGULAR = 1,     /* zero pivot in `\`  (Breeze MatrixSingularException)    */
  BDLM_ST_NOTCONVERGED = 2, /* Jacobi sweep cap   (Breeze NotConvergedException)      */
  BDLM_ST_NOTPD = 4,        /* Cholesky failed    (MultivariateGaussian on W*dt)      */
  BDLM_ST_NONFINITE = 8,    /* NaN/Inf in the final state                             */
  BDLM_ST_TIMEOUT = 16      /* time-sharded scan: a peer's aggregate never arrived    */
};

/* compat flags: default 0 = reference-verbatim behaviour (what parity is judged on) */
enum {
  BDLM_TEXTBOOK_SMOOTHER = 1, /* S = C - B (R-S) B^T instead of Smoothing.scala:44's ... B */
  BDLM_SVD_CONSISTENT_W = 2,  /* SVD time update stacks W^{1/2} sqrt(dt) (DlmFsv.scala:213-217)
                                 instead of the raw W the filterDlm/ffbsDlm/Gibbs closures hold */
  BDLM_PARALLEL_IN_TIME = 4   /* ONE long series may run through the associative-scan kernels
                                 instead of T dependent steps of ~0.3 us each, at 1e-9 relative
                                 instead of bit-for-bit agreement with the sequential recursion --
                                 hence opt-in.  Eligible: B = 1, T >= 4096, p = 1, n <= 4, regular
                                 grid, time-invariant model (no f_tv, g_tv, v_tv, w_tv), shared
                                 parameters, device or host buffers; then
                                   bdlm_kf_filter_smooth  runs bdlm_scan_filter_smooth when also
                                                          n = 1 or BDLM_TEXTBOOK_SMOOTHER;
                                   bdlm_loglik,
                                   bdlm_kf_filter_last    run bdlm_scan_loglik (any n <= 4);
                                   bdlm_ffbs              runs bdlm_scan_ffbs when also
                                                          keep_init = 1 (any n <= 4; same
                                                          normals as the sequential kernel for
                                                          the same z or bdlm_set_rng).
                                 Ignored (sequential kernel, bit for bit) when the problem is not
                                 eligible. */
};

/* which params are per series (bit mask for bdlm_problem.per_series) */
enum { BDLM_PS_V = 1, BDLM_PS_W = 2, BDLM_PS_M0 = 4, BDLM_PS_C0 = 8,
       /* Data(time, observation) is per series in the reference (Dlm.scala:94): a batch whose
        * series sit on DIFFERENT (irregular) grids or carry different covariates runs as one call.
        *  BDLM_PS_TIMES: `times` is a per-step per-series array laid out like y with k = 1, in the
        *                 data's memory space; every series starts from its own min(times) - 1
        *                 (KalmanFilter.scala:112-118) unless t_init is given.  Needs a
        *                 dt-independent G (g_tv = 0: polynomial, regression, autoregressive) or
        *                 BDLM_PS_G.
        *  BDLM_PS_F:     F (with f_tv = 1) is laid out like y with k = n*p -- mod.f(time_t) of each
        *                 series, e.g. Dlm.regression's F_t = (1, x_t) (Dlm.scala:159-169).
        *  BDLM_PS_G:     G (with g_tv = 1) is laid out like y with k = n*n -- mod.g(dt_t) of each
        *                 series (seasonal models on per-series irregular grids,
        *                 AqMeshExample.scala:86-127).
        * Ragged batches (filter, smoother, innovations likelihood): pad a short series at the END
        * with NaN observations at its last time (dt = 0: advState passes the state through, an
        * all-missing update leaves it unchanged, the smoother's recursion is the identity there).
        * The backward SAMPLER and the transition-form likelihood are not padding-invariant. */
       BDLM_PS_TIMES = 16, BDLM_PS_F = 32, BDLM_PS_G = 64 };

typedef struct bdlm_ctx bdlm_ctx;

/* One batch of independent series / chains sharing a model (Dlm.scala:14-15) and a
 * time grid.  Dlm.f/g closures arrive materialised (see header comment). */
typedef struct bdlm_problem {
  int64_t B;          /* series or chains                                   */
  int32_t T;          /* observations per series                            */
  int32_t n, p;       /* state / observation dimension                      */
  int32_t layout;     /* BDLM_TIME_MAJOR | BDLM_SERIES_MAJOR                */
  int32_t mem;        /* BDLM_DEVICE | BDLM_HOST                            */
  int32_t keep_init;  /* see "rows" above                                   */
  int32_t f_tv, g_tv; /* F / G vary with t                                  */
  int32_t per_series; /* BDLM_PS_* mask                                     */
  int32_t compat;     /* BDLM_TEXTBOOK_* / BDLM_SVD_* mask                  */
  const double *F;    /* host [n*p] or [T][n*p]   (or per series: BDLM_PS_F)  */
  const double *G;    /* host [n*n] or [T][n*n]   (or per series: BDLM_PS_G)  */
  const double *times;/* host [T] or NULL (regular grid) (or BDLM_PS_TIMES)   */
  const double *V;    /* DlmParameters.v  (Dlm.scala:36)                    */
  const double *W;    /* DlmParameters.w                                    */
  const double *m0;   /* DlmParameters.m0                                   */
  const double *C0;   /* DlmParameters.c0                                   */
  const double *y;    /* observations, T rows, k = p                        */
  int32_t v_tv;       /* next row f2 (StudentTGibbs.filter, StudentTGibbs.scala:100-119;
                         DlmFsv.ffbsSvd, DlmFsv.scala:208-229): V varies with t.  V then
                         holds T matrices: host [T][p*p] when shared, or, with BDLM_PS_V, a
                         per-step array laid out like y with k = p*p.  Served by the
                         warp-per-series kernels.                               */
  int32_t w_tv;       /* W varies with t (DlmFsvSystem.ffbs, DlmFsvSystem.scala:137-167): W holds T
                         matrices, W[t] driving the transition INTO observation t; same layout
                         rules as v_tv with BDLM_PS_W and k = n*n.                  */
  const double *t_init; /* host scalar or NULL.  NULL: the state (m0, C0) sits at min(times) - 1
                         (KalmanFilter.initialiseState).  Non-NULL: it sits at *t_init, i.e.
                         the call RESUMES a filter from a saved state -- folding
                         KalmanFilter.step over later data (NoModel.scala:153-155) or starting
                         Dlm.forecast (Dlm.scala:322-338, first dt = 0).  Ignored when times is
                         NULL (unit grid).                                        */
} bdlm_problem;

/* KfState fields (KalmanFilter.scala:22-30), `rows` rows each; NULL = not wanted. */
typedef struct bdlm_kf_out {
  double *m, *C; /* mt, ct : k = n, n*n */
  double *a, *R; /* at, rt : k = n, n*n */
  double *f, *Q; /* ft, qt : k = p, p*p */
} bdlm_kf_out;

/* SmoothingState mean / covariance (Smoothing.scala:18-22); at1, rt1 are KfState a, R. */
typedef struct bdlm_smooth_out {
  double *s; /* k = n   */
  double *S; /* k = n*n (full: Smoothing.scala:44 makes it non-symmetric for n > 1) */
} bdlm_smooth_out;

/* SvdState fields (SvdFilter.scala:7-14), `rows` rows each; NULL = not wanted. */
typedef struct bdlm_svd_out {
  double *m, *dc, *uc; /* mt, dc, uc : k = n, n, n*n */
  double *a, *dr, *ur; /* at, dr, ur : k = n, n, n*n */
  double *f;           /* ft         : k = p         */
} bdlm_svd_out;

/* Gibbs sufficient statistics per chain (one row per chain: [k][B] or [B][k]).
 * GibbsSampling.sampleObservationMatrix (Gibbs.scala:29-43): ssy[p], ny[p];
 * sampleSystemMatrix (Gibbs.scala:63-73): ssw[n];
 * GibbsWishart.sampleSystemMatrix (GibbsWishart.scala:22-29): scatter[n*n]. NULL = skip. */
typedef struct bdlm_gibbs_stats {
  double *ssy, *ny, *ssw, *scatter;
} bdlm_gibbs_stats;

/* ---- context ---------------------------------------------------------------------- */
BDLM_API int bdlm_create(int device, bdlm_ctx **out);
BDLM_API void bdlm_destroy(bdlm_ctx *ctx);
BDLM_API const char *bdlm_last_error(bdlm_ctx *ctx); /* ctx may be NULL: last create error */
BDLM_API int bdlm_version(void);
/* Adopt a caller-owned cudaStream_t (e.g. torch's current stream).  The handle is used
 * as given: NULL is the legacy default stream.  use_own != 0 ignores the handle and
 * restores the context's own (non-blocking) stream. */
BDLM_API int bdlm_set_stream(bdlm_ctx *ctx, void *cuda_stream, int use_own);
BDLM_API int bdlm_sync(bdlm_ctx *ctx);
/* On-device RNG mode of bdlm_ffbs / bdlm_svd_ffbs: when their `z` argument is NULL the kernels
 * draw the N(0,1) values themselves -- Philox4x32-10 keyed by `seed`, one subsequence per series
 * / chain (first_series + index within the call: ranks that shard a batch pass the global index
 * of their first series), offset by (sweep, row, component), so a draw depends only on (seed,
 * sweep, global series, row, component), not on the batch split, kernel variant or layout.
 * Callers advance `sweep` once per Gibbs iteration.  Bit-for-bit parity with the reference
 * needs injected `z`. */
BDLM_API int bdlm_set_rng(bdlm_ctx *ctx, uint64_t seed, uint64_t sweep, int64_t first_series);
/* Kernel launches issued by this context since creation (bench.py's gpu_launches). */
BDLM_API int64_t bdlm_launch_count(bdlm_ctx *ctx);
/* Cap on the device bytes a mem = BDLM_HOST call may use for staging (default 8 GiB). */
BDLM_API int bdlm_set_staging_bytes(bdlm_ctx *ctx, int64_t bytes);
/* Series that exactly fill the GPU once ("one wave") for the fused filter+smoother kernel
 * of a model with these dimensions on a regular grid: resident blocks per SM x SM count x
 * threads per block.  Every series of a launch takes the same time, so batches (or slabs)
 * that are a multiple of this number leave no partially filled last wave.  Returns
 * BDLM_E_ARG for dimensions served by the warp-per-series kernels (wave = resident warps). */
BDLM_API int64_t bdlm_wave_series(bdlm_ctx *ctx, int32_t n, int32_t p);
/* Measured FP64 pipe peak of the context's GPU in TFLOP/s (DFMA microbenchmark, 2 flops per
 * DFMA): the roofline denominator for the FP64-bound kernels (FFBS, SVD).  The numerical
 * kernels never fuse multiply-add (parity contract), so their attainable rate is half of it. */
BDLM_API int bdlm_fp64_peak_tflops(bdlm_ctx *ctx, double *tflops);

/* ---- forward filter ----------------------------------------------------------------
 * KalmanFilter.filterDlm (KalmanFilter.scala:291-294) / KalmanFilter(adv).filter
 * (Filter.scala:41-45) with adv = KalmanFilter.advanceState (:262-286), step (:99-107),
 * missing-data aware Joseph update (:64-94), one-step forecast (:311-321).
 * status: int32[B] or NULL. */
BDLM_API int bdlm_kf_filter(bdlm_ctx *ctx, const bdlm_problem *prob, const bdlm_kf_out *out,
                   int32_t *status);

/* ---- RTS smoother --------------------------------------------------------------------
 * Smoothing.backwardsSmoother (Smoothing.scala:57-64) on filtered states previously
 * produced by bdlm_kf_filter with the same problem: filt->m, filt->C are read;
 * a_{t+1}, R_{t+1} are read from filt->a, filt->R when given, else recomputed from
 * (m_t, C_t) exactly as the forward pass did. */
BDLM_API int bdlm_rts_smooth(bdlm_ctx *ctx, const bdlm_problem *prob, const bdlm_kf_out *filt,
                    const bdlm_smooth_out *out, int32_t *status);

/* ---- fused filter + smoother ---------------------------------------------------------
 * KalmanFilter(adv).filter followed by Smoothing.backwardsSmoother in one launch per
 * slab: forward pass writes the requested KfState fields, backward pass re-reads (m, C)
 * and writes (s, S).  If kf->m / kf->C are NULL the spill goes to context workspace. */
BDLM_API int bdlm_kf_filter_smooth(bdlm_ctx *ctx, const bdlm_problem *prob, const bdlm_kf_out *kf,
                          const bdlm_smooth_out *sm, int32_t *status);

/* ---- log-likelihoods -----------------------------------------------------------------
 * transition[b] : KalmanFilter.likelihood (KalmanFilter.scala:299-306) = sum_t log
 *                 N(m_t; G m_{t-1}, W dt) over the filtered means (the quantity
 *                 Metropolis.dlm / MetropolisHastings.dlm evaluate per proposal,
 *                 MetropolisHastings.scala:126-137,199-209);
 * innovations[b]: sum_t KalmanFilter.conditionalLikelihood (:138-153), the textbook
 *                 prediction-error decomposition.  Either may be NULL.  [B] doubles. */
BDLM_API int bdlm_loglik(bdlm_ctx *ctx, const bdlm_problem *prob, double *transition,
                double *innovations, int32_t *status);

/* ---- last filtered state only ----------------------------------------------------------
 * `data.foldLeft(init)(kf.step(mod, p))` (NoModel.scala:153-155): the filter without any
 * per-step store.  m_last [n] / C_last [n*n] per series ([k][B] or [B][k]) receive the state
 * after the last observation; the two log-likelihoods of bdlm_loglik come for free.  Any output
 * may be NULL.  Together with bdlm_problem.t_init this is the streaming pattern: keep the last
 * state, resume when more data arrive. */
BDLM_API int bdlm_kf_filter_last(bdlm_ctx *ctx, const bdlm_problem *prob, double *m_last,
                                 double *C_last, double *transition, double *innovations,
                                 int32_t *status);

/* ---- FFBS ----------------------------------------------------------------------------
 * Smoothing.ffbs / ffbsDlm (Smoothing.scala:151-180): filter keeping the initial state,
 * then Smoothing.sample (:114-122) with Smoothing.step (:74-103) and
 * MultivariateGaussianSvd.draw (MultivariateGaussianSvd.scala:13-22).
 * prob->keep_init must be 1.  z: injected N(0,1) values, rows x n per series, z[row]
 * being the n values consumed when drawing theta[row] (the reference draws the last
 * row first, index 0..n-1 within a row); NULL = draw them on the device (bdlm_set_rng).
 * theta: rows x n.  kf (optional) receives
 * the SamplingState's filter moments; stats (optional) the Gibbs sufficient statistics
 * of the drawn path (Gibbs.scala:29-43,63-73; GibbsWishart.scala:22-29). */
BDLM_API int bdlm_ffbs(bdlm_ctx *ctx, const bdlm_problem *prob, const double *z, double *theta,
              const bdlm_kf_out *kf, const bdlm_gibbs_stats *stats, int32_t *status);

/* ---- SVD filter ----------------------------------------------------------------------
 * SvdFilter.filterDlm / filter (SvdFilter.scala:100-119,158-161): parameters are
 * transformed on the device (transformParams :232-236), the advance closure holds the
 * RAW W unless BDLM_SVD_CONSISTENT_W is set. */
BDLM_API int bdlm_svd_filter(bdlm_ctx *ctx, const bdlm_problem *prob, const bdlm_svd_out *out,
                    int32_t *status);

/* ---- SVD FFBS ------------------------------------------------------------------------
 * SvdSampler.ffbs / ffbsDlm (SvdSampler.scala:66-82) as used by GibbsSampling.stepSvd
 * (Gibbs.scala:182-198): filterDecomp on transformed params, then SvdSampler.sample
 * (:54-60) with step (:15-36) and rnorm (:94-102).  z / theta / stats as bdlm_ffbs. */
BDLM_API int bdlm_svd_ffbs(bdlm_ctx *ctx, const bdlm_problem *prob, const double *z, double *theta,
                  const bdlm_svd_out *filt, const bdlm_gibbs_stats *stats,
                  int32_t *status);

/* ---- Gibbs sufficient statistics of a given path ------------------------------------
 * Same statistics as the `stats` argument above for a caller-supplied theta (rows =
 * T + 1). */
BDLM_API int bdlm_gibbs_suffstats(bdlm_ctx *ctx, const bdlm_problem *prob, const double *theta,
                         const bdlm_gibbs_stats *stats);

/* ---- parallel-in-time filter + smoother for ONE long series ---------------------------
 * Not in the reference (its recursion is strictly sequential, Filter.scala:41-62; BASELINE
 * config 5).  Temporal parallelisation by associative scan (Sarkka & Garcia-Fernandez 2021).
 * Restrictions: B = 1, p = 1, n <= 4, regular grid (times = NULL), time-invariant F and G,
 * shared parameters, mem = BDLM_DEVICE.  Results equal bdlm_kf_filter_smooth with
 * BDLM_TEXTBOOK_SMOOTHER to 1e-9 relative (for n = 1 that is the reference itself).
 *
 * Single GPU: bdlm_scan_filter_smooth.  Several GPUs, each owning a contiguous time chunk:
 * bdlm_comm_scan_filter_smooth, or, for hosts that bring their own transport, the bdlm_scan_dist_*
 * sequence.  There the chunk aggregate stays in device memory, the caller all-gathers it (NCCL,
 * or a copy through the host and back) on the context's stream (aggs_dev =
 * [world][bdlm_scan_elem_doubles] doubles), and the carry is folded by a one-thread kernel inside
 * the finish call.  Per rank: forward_local -> all-gather -> forward_finish -> backward_local ->
 * all-gather -> backward_finish; nothing synchronises with the host.  prob describes the rank's
 * chunk (keep_init = 1 on rank 0 only); kf->m and kf->C are required; the context's workspace
 * must not be used by other calls between a local and its finish phase.
 * Elements are laid out [A | b | C | eta | J] (forward) and [E | g | L] (backward), matrices
 * column-major. */
BDLM_API int bdlm_scan_filter_smooth(bdlm_ctx *ctx, const bdlm_problem *prob,
                                     const bdlm_kf_out *kf, const bdlm_smooth_out *sm,
                                     int32_t *status);
/* Log-likelihoods and last filtered state of ONE long series by the scan's forward pass alone:
 * arguments as bdlm_kf_filter_last (any output may be NULL, not all; status int32[1]), same
 * restrictions as bdlm_scan_filter_smooth, any T >= 1, keep_init ignored (the state (m0, C0) sits
 * before the first observation, as in bdlm_loglik).  Nothing is stored per time step; the sums are
 * reduced in a fixed order (same bits on every call) and agree with bdlm_loglik to 1e-9 of
 * sum_t |term_t|.  Enqueue-only: no host synchronisation. */
BDLM_API int bdlm_scan_loglik(bdlm_ctx *ctx, const bdlm_problem *prob, double *m_last,
                              double *C_last, double *transition, double *innovations,
                              int32_t *status);
/* FFBS of ONE long series by the associative scan: forward pass, then the backward sampler as a
 * scan of the affine maps theta_r = B_r theta_{r+1} + c_r, with the Gibbs statistics of the drawn
 * path summed in the same sweep.  Arguments as bdlm_ffbs (z NULL = Philox normals of
 * bdlm_set_rng, the same values the sequential kernel consumes; kf, stats and any of their fields
 * may be NULL; status int32[1]); same restrictions as bdlm_scan_filter_smooth plus keep_init = 1,
 * any T >= 1.  Each draw uses the eigen basis of the sequential kernel (same z, same path to 1e-9
 * of each row's largest entry where H_r's eigenvalues are well separated); the statistics are
 * reduced in a fixed order (same bits on every call).  Enqueue-only: no host synchronisation. */
BDLM_API int bdlm_scan_ffbs(bdlm_ctx *ctx, const bdlm_problem *prob, const double *z, double *theta,
                            const bdlm_kf_out *kf, const bdlm_gibbs_stats *stats, int32_t *status);
BDLM_API int bdlm_scan_elem_doubles(int32_t n, int32_t backward);
BDLM_API int bdlm_scan_dist_forward_local(bdlm_ctx *ctx, const bdlm_problem *prob, int32_t rank,
                                          int32_t world, double *agg_dev);
BDLM_API int bdlm_scan_dist_forward_finish(bdlm_ctx *ctx, const bdlm_problem *prob, int32_t rank,
                                           int32_t world, const double *aggs_dev,
                                           const bdlm_kf_out *kf, int32_t *status);
BDLM_API int bdlm_scan_dist_backward_local(bdlm_ctx *ctx, const bdlm_problem *prob, int32_t rank,
                                           int32_t world, const bdlm_kf_out *filt,
                                           const bdlm_smooth_out *sm, double *agg_dev);
BDLM_API int bdlm_scan_dist_backward_finish(bdlm_ctx *ctx, const bdlm_problem *prob, int32_t rank,
                                            int32_t world, const double *aggs_dev,
                                            const bdlm_kf_out *filt, const bdlm_smooth_out *sm,
                                            int32_t *status);
/* out = earlier (x) later on the host: the host build of the combine the scan kernels inline. */
BDLM_API int bdlm_scan_combine(int32_t n, int32_t backward, const double *earlier,
                               const double *later, double *out);

/* ======================================================================================
 * Multi-GPU communicator (SURVEY.md 8b "Threading", 8e): one context per device, NCCL behind
 * one object.  Series and chains are independent -- the reference fits one model per sensor
 * (UoModel.scala:69-104) and its only parallel driver maps chains over futures
 * (Streaming.scala:162-173) -- so batches are cut into contiguous blocks of series, one per GPU,
 * with NO data-path collective; the only inter-GPU traffic is an ncclAllReduce of summed
 * log-likelihoods / pooled Gibbs statistics, and the chunk aggregates of the time-sharded scan.
 * NCCL is dlopen'ed (libnccl.so.2; BDLM_NCCL_LIB overrides): libbdlm.so does not link it.
 *
 *  single process, n GPUs (a JVM host):  bdlm_comm_create(devs, n, 0, n, NULL, &comm)
 *  one process per GPU (rank r of w):    rank 0: bdlm_comm_unique_id(id), broadcast id, then
 *                                        every rank: bdlm_comm_create(&dev, 1, r, w, id, &comm)
 *
 * Sharded calls take the problem of THIS PROCESS (prob->B = the series it owns): host buffers
 * (mem = BDLM_HOST) are cut over the process's devices and run concurrently, one host thread and
 * one slab pipeline per device; device buffers need one device per process.  Results are those
 * of one bdlm_* call on the whole batch (status, per-series parameters and the Philox
 * subsequences are indexed by the position in the call; bdlm_set_rng(first_series) on each
 * context makes them global across processes).
 * ==================================================================================== */
typedef struct bdlm_comm bdlm_comm;
BDLM_API int bdlm_comm_unique_id(void *id /* BDLM_COMM_ID_BYTES */);
BDLM_API int bdlm_comm_create(const int32_t *devices, int32_t n_local, int32_t first_rank,
                              int32_t world, const void *id, bdlm_comm **out);
BDLM_API void bdlm_comm_destroy(bdlm_comm *comm);
BDLM_API const char *bdlm_comm_last_error(bdlm_comm *comm); /* NULL: last create error */
BDLM_API int32_t bdlm_comm_size(bdlm_comm *comm);           /* ranks of the whole job      */
BDLM_API int32_t bdlm_comm_local_size(bdlm_comm *comm);     /* devices driven by this process */
BDLM_API bdlm_ctx *bdlm_comm_ctx(bdlm_comm *comm, int32_t local_index); /* owned by the comm */
BDLM_API int bdlm_comm_sync(bdlm_comm *comm);               /* bdlm_sync on every local context */
/* 1 when the time-sharded scan exchanges its aggregates through peer mailboxes (direct NVLink
 * stores + flag, single-process communicators with full peer access) instead of NCCL. */
BDLM_API int32_t bdlm_comm_uses_peer_exchange(bdlm_comm *comm);
/* values[count] (host) <- sum over all PROCESSES of their values (ncclAllReduce, fp64). */
BDLM_API int bdlm_comm_allreduce_sum(bdlm_comm *comm, double *values, int32_t count);
/* Same on device memory of a one-device-per-process communicator; enqueue-only. */
BDLM_API int bdlm_comm_allreduce_sum_device(bdlm_comm *comm, double *values_dev, int32_t count);
/* bdlm_kf_filter / bdlm_svd_filter / bdlm_kf_filter_smooth over the communicator's devices. */
BDLM_API int bdlm_comm_kf_filter(bdlm_comm *comm, const bdlm_problem *prob, const bdlm_kf_out *out,
                                 int32_t *status);
BDLM_API int bdlm_comm_svd_filter(bdlm_comm *comm, const bdlm_problem *prob, const bdlm_svd_out *out,
                                  int32_t *status);
BDLM_API int bdlm_comm_kf_filter_smooth(bdlm_comm *comm, const bdlm_problem *prob,
                                        const bdlm_kf_out *kf, const bdlm_smooth_out *sm,
                                        int32_t *status);
/* bdlm_loglik over the devices; sums (host [2], optional) receives Sum_b transition[b] and
 * Sum_b innovations[b] over every series of EVERY rank -- the pooled log-likelihood a
 * Metropolis step over shared parameters evaluates (MetropolisHastings.scala:126-137). */
BDLM_API int bdlm_comm_loglik(bdlm_comm *comm, const bdlm_problem *prob, double *transition,
                              double *innovations, int32_t *status, double *sums);
/* bdlm_ffbs / bdlm_svd_ffbs over the devices; pooled (host arrays ssy[p], ny[p], ssw[n],
 * scatter[n*n], any may be NULL) receives the sufficient statistics summed over the chains of
 * every rank (needs the per-chain `stats` arrays). */
BDLM_API int bdlm_comm_ffbs(bdlm_comm *comm, const bdlm_problem *prob, const double *z, double *theta,
                            const bdlm_kf_out *kf, const bdlm_gibbs_stats *stats, int32_t *status,
                            const bdlm_gibbs_stats *pooled);
BDLM_API int bdlm_comm_svd_ffbs(bdlm_comm *comm, const bdlm_problem *prob, const double *z,
                                double *theta, const bdlm_svd_out *filt,
                                const bdlm_gibbs_stats *stats, int32_t *status,
                                const bdlm_gibbs_stats *pooled);
/* ONE long series cut along time over the ranks (BASELINE config 5): the six-phase protocol of
 * bdlm_scan_dist_* behind one call.  probs / kfs / sms / status have one entry per LOCAL device
 * (rank order) describing that rank's contiguous time chunk in that device's memory; keep_init =
 * 1 on global rank 0 only; kf->m and kf->C are required.  Enqueue-only (bdlm_comm_sync). */
BDLM_API int bdlm_comm_scan_filter_smooth(bdlm_comm *comm, const bdlm_problem *probs,
                                          const bdlm_kf_out *kfs, const bdlm_smooth_out *sms,
                                          int32_t *const *status);

/* ======================================================================================
 * "Next" rows (SURVEY.md section 8f): the callers and neighbours of the hot path.
 * ==================================================================================== */

/* ---- scalar AR(1) / Ornstein-Uhlenbeck state: filter and backward sampler ---------------
 * FilterAr.filterUnivariate / univariateSample / ffbs (FilterAr.scala:15-83) and
 * FilterOu.filterUnivariate / univariateSample / ffbs (FilterOu.scala:7-79): the inner loop of
 * the reference's stochastic-volatility samplers.  SvParameters(phi, mu, sigmaEta) are host
 * scalars ([1]) or, with per_series = 1, [B] arrays in the data's memory space.  v holds the
 * observation variances (`vs: Vector[Double]`): one host scalar, a host [T] array shared by the
 * batch, or one value per series and step laid out like y.  times: host [T] or NULL (1..T); only
 * the OU process reads it.  All per-step arrays have k = 1; outputs, z and theta have T + 1 rows
 * (row 0 = the stationary prior), z[row] is the N(0,1) value consumed when drawing theta[row]. */
enum { BDLM_AR1 = 0, BDLM_OU = 1 };
enum { BDLM_V_SCALAR = 0, BDLM_V_PER_STEP = 1, BDLM_V_PER_SERIES_STEP = 2 };
typedef struct bdlm_ar_problem {
  int64_t B;
  int32_t T;
  int32_t layout, mem;    /* as bdlm_problem */
  int32_t process;        /* BDLM_AR1 | BDLM_OU */
  int32_t per_series;     /* phi, mu, sigma_eta are [B] arrays */
  int32_t v_mode;         /* BDLM_V_* */
  const double *phi, *mu, *sigma_eta;
  const double *times;
  const double *v;
  const double *y;        /* T rows, NaN = None */
} bdlm_ar_problem;
/* FilterAr.FilterState fields (FilterAr.scala:9-13); NULL = not wanted. */
typedef struct bdlm_ar_out {
  double *m, *C, *a, *R;
} bdlm_ar_out;
BDLM_API int bdlm_ar_filter(bdlm_ctx *ctx, const bdlm_ar_problem *prob, const bdlm_ar_out *out);
BDLM_API int bdlm_ar_ffbs(bdlm_ctx *ctx, const bdlm_ar_problem *prob, const double *z,
                          double *theta, const bdlm_ar_out *filt /* optional */);

/* ---- conjugate filter: unknown observation variance ---------------------------------------
 * ConjugateFilter(prior, ConjugateFilter.advanceState(p, g)).filter (ConjugateFilter.scala:
 * 17-112): Kalman filter with V replaced by the running mean of an InverseGamma(shape, scale)
 * posterior that is updated at every step.  p = 1, n <= 4, time-invariant F and G, keep_init = 1;
 * prob->V is ignored.  shape / scale: T + 1 rows, k = 1 (row 0 = the prior). */
BDLM_API int bdlm_conjugate_filter(bdlm_ctx *ctx, const bdlm_problem *prob, double prior_shape,
                                   double prior_scale, const bdlm_kf_out *out, double *shape,
                                   double *scale, int32_t *status);

/* ---- conjugate draws of V and W from the Gibbs sufficient statistics ----------------------
 * The second half of GibbsSampling.dinvGammaStep / stepSvd (Gibbs.scala:134-151,182-198) and of
 * GibbsWishart.wishartStep (GibbsWishart.scala:40-53), on the device, so that a sweep
 * (bdlm_ffbs / bdlm_svd_ffbs with `stats`, then this call, then the next sweep with
 * per_series = BDLM_PS_V | BDLM_PS_W) never leaves the GPU.
 *   V_out [p*p] per chain: diag(InverseGamma(v_shape + ny_i / 2, v_scale + ssy_i / 2).draw)
 *   W_out [n*n] per chain: w_psi == NULL: diag(InverseGamma(w_shape + T / 2, w_scale + ssw_i / 2))
 *                          w_psi != NULL (host n*n): InverseWishart(w_nu + T, w_psi + scatter).draw
 * prob supplies B, T, n, p, layout, mem (stats and outputs are one row per chain: [k][B] or
 * [B][k]).  Randomness: Philox4x32-10 keyed by (seed, chain, element), advanced by `sweep`;
 * or injected variates for bit-exact checks: gamma_v [p] / gamma_w [n] standard Gamma(shape, 1)
 * values per chain, bartlett [n*n] the lower-triangular Bartlett factor (Wishart.scala:34-43).
 * v_shape_rate [2p] / w_shape_rate [2n] (optional) receive the posterior shapes then rates. */
typedef struct bdlm_gibbs_prior {
  double v_shape, v_scale; /* InverseGamma prior on diag(V) */
  double w_shape, w_scale; /* InverseGamma prior on diag(W) */
  double w_nu;             /* InverseWishart(w_nu, w_psi) prior on W */
  const double *w_psi;
} bdlm_gibbs_prior;
typedef struct bdlm_gibbs_rng {
  uint64_t seed, sweep;
  const double *gamma_v, *gamma_w, *bartlett; /* NULL = generate on the device */
} bdlm_gibbs_rng;
BDLM_API int bdlm_gibbs_draw(bdlm_ctx *ctx, const bdlm_problem *prob, const bdlm_gibbs_stats *stats,
                             const bdlm_gibbs_prior *prior, const bdlm_gibbs_rng *rng,
                             double *V_out, double *W_out, double *v_shape_rate,
                             double *w_shape_rate, int32_t *status);

#ifdef __cplusplus
}
#endif
#endif /* BDLM_H */
