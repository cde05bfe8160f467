// launch.h -- host-callable launchers implemented in the .cu files.
#pragma once
#include "common.cuh"

namespace bdlm {

// kf_small.cu: thread-per-series register kernels (n <= 4, p = 1).
bool small_supported(int n, int p);
cudaError_t launch_kf_small(const Batch &bt, const double *hG, const double *hF,
                            const KfViews &kf, const View &sv, const View &Sv,
                            bool do_filter, bool do_smooth, cudaStream_t stream,
                            int *wave_series = nullptr);  // non-null: occupancy query only

// kf_warp.cu: warp-per-series shared-memory kernels (n <= 48, p <= 32).
struct SvdViews {
  View m, dc, uc, a, dr, ur, f;
};
struct StatViews {  // one row per chain: element (b, k) at ptr[b*sb + k*sk]
  View ssy, ny, ssw, scatter;
};
enum WarpOp {
  kOpFilter = 0,       // forward Kalman filter
  kOpSmooth = 1,       // RTS smoother from stored (m, C[, a, R])
  kOpFilterSmooth = 2, // fused
  kOpFfbs = 3,         // filter + backward sampling (+ Gibbs statistics)
  kOpLoglik = 4,       // filter + both log-likelihoods
  kOpSvdFilter = 5,
  kOpSvdFfbs = 6,
  kOpStats = 7         // Gibbs statistics of a given theta
};
struct WarpArgs {
  Batch bt;
  KfViews kf;          // user-visible KfState outputs (any may be null)
  View s, S;           // smoother outputs
  CView z;             // injected normals, rows x n; ptr == nullptr: generate them (rng)
  unsigned long long rng_seed, rng_sweep;  // Philox key of the on-device RNG mode
  long long rng_base;  // global index of series 0 of this launch (subsequence = rng_base + b)
  View theta;          // sampled path, rows x n (input for kOpStats)
  SvdViews svd;
  StatViews stats;
  double *ll_transition, *ll_innov;  // [B]
  View last_m, last_C;               // kOpLoglik: final filtered state, one row per series
  double *spill;       // series-major workspace [B][rows][spill_k] or nullptr
  int64_t spill_k;
};
size_t warp_spill_doubles_per_row(int op, int n, int p);
size_t warp_smem_bytes(int op, int n, int p);  // one warp's shared-memory workspace (<= 227 KB to launch)
cudaError_t launch_warp(int op, const WarpArgs &wa, cudaStream_t stream);

// ffbs_small.cu: FFBS with one thread per chain (n <= 4, p = 1, time-invariant F, G).
struct FfbsSmallArgs {
  Batch bt;
  KfViews kf;          // optional a, R, f, Q outputs (m, C travel through sm / sC)
  View sm, sC;         // (m, C) spill, rows x k: the caller's m / C arrays or workspace
  CView z;             // injected normals or ptr == nullptr (Philox)
  View theta;
  StatViews stats;
  unsigned long long rng_seed, rng_sweep;
  long long rng_base;
};
bool ffbs_small_supported(const Batch &bt);
cudaError_t launch_ffbs_small(const FfbsSmallArgs &a, const double *hG, const double *hF,
                              cudaStream_t stream);

// kf_group.cu: two series per warp, compile-time n, p = 1 (FFBS / filter, n in {7, 13}).
bool group_supported(int op, int n, int p, int keep_init);
cudaError_t launch_group(int op, const WarpArgs &wa, cudaStream_t stream);

// transpose.cu: [R][C] -> [C][R] for doubles (layout conversion of staged slabs).
cudaError_t launch_transpose(const double *in, double *out, int64_t rows, int64_t cols,
                             cudaStream_t stream);

// transpose.cu: dt[b][t] from per-series observation times (element (b, t) at base[b*sb + t*sr]).
cudaError_t launch_dt_from_times(const double *times, int64_t tsb, int64_t tsr, double *dt,
                                 int64_t dsb, int64_t dsr, int64_t B, int T, const double *t_init,
                                 cudaStream_t stream);

// scan.cu: parallel-in-time filter / smoother for one long series (n <= 4, p = 1, regular
// grid, time-invariant G, V, W; F time-invariant or given per step).
enum { kScanApply = 0,
       // time-sharded run over several GPUs: local = level-1 + scan with an identity carry, chunk
       // aggregate left in DEVICE memory for the all-gather; finish = fold the gathered aggregates
       // of the other ranks on the device and apply
       kScanDistLocal = 1, kScanDistFinish = 2 };
// Peer mailboxes of a single-process communicator (comm.cu): box[r] / flag[r] live in rank r's
// device memory and are mapped into every other device (cudaDeviceEnablePeerAccess).  A rank
// PUBLISHES its chunk aggregate by storing it into slot [its rank] of every peer's box over
// NVLink, followed by a system-scope release of flag[r][its rank] = epoch; the carry-folding
// thread of the finish phase spins on its own flags.  world == 0: not in use (NCCL all-gather).
struct ScanPeers {
  int world;
  double *box[BDLM_COMM_MAX_WORLD];
  unsigned long long *flag[BDLM_COMM_MAX_WORLD];
};

struct ScanArgs {
  int n;
  int64_t T;           // observations in this chunk
  int keep_init;       // rows = T + keep_init
  int backward;        // 0 = filter pass, 1 = smoother pass
  int phase;           // kScanApply: whole series on one GPU; kScanDist*: one rank's chunk
  int has_successor;   // backward: another chunk follows this one in time
  const double *G, *F, *W;  // host, column-major; F = nullptr with a per-step F (f_tv)
  double V;
  const double *y;     // device [T]
  const double *Fd;    // f_tv: device [T][n], F of each observation of the chunk; else nullptr
  const double *start; // host [n + n*n]: the prior (m0, C0) of the series (forward apply / finish)
  KfViews kf;          // forward: outputs; backward: filtered (m, C) inputs
  View s, S;           // backward outputs
  int32_t *status;     // device, one int, OR-ed
  void *workspace;     // device, scan_workspace_bytes(n, T)
  void *fuse_sagg;     // forward apply / finish: also write the smoother's level-1 aggregates
                       // here (the backward workspace of the call that follows, which has no
                       // other source of them), or nullptr
  double *agg_dev;     // dist local: device [elem doubles], this rank's chunk aggregate (out)
  const double *aggs_dev;  // dist finish: device [world][elem doubles], all ranks' aggregates
  int rank, world;     // dist phases
  ScanPeers peers;     // dist phases: peer mailboxes instead of agg_dev + all-gather (world > 0)
  const unsigned long long *epoch_dev;  // device: this rank's call counter = the value its flags take
  void *table;         // device, scan_table_bytes(): y-independent parts of the level-1 aggregates
  int table_upload;    // 1 = (re)build the table for this model before the forward pass
};
cudaError_t launch_epoch_bump(unsigned long long *epoch_dev, cudaStream_t stream);
size_t scan_table_bytes();
size_t scan_workspace_bytes(int n, int64_t T);
int scan_forward_elem_doubles(int n);
int scan_backward_elem_doubles(int n);
cudaError_t launch_scan(const ScanArgs &a, cudaStream_t stream, int64_t *launches);
// Log-likelihoods + last filtered state of one series (forward pass only, nothing stored per row):
// a = a forward kScanApply pass with keep_init = 1 (a.kf unused).  Outputs are device pointers,
// any may be null; status (one int) is written, not OR-ed.
struct ScanLoglikOut {
  double *transition, *innovations;  // [1]
  double *m_last, *C_last;           // [n], [n*n]
  int32_t *status;
  void *parts;                       // device, scan_loglik_bytes(n, T): block partials
  double *part_vec;                  // time-sharded: the rank's [transition, innovations, status] (out)
};
size_t scan_loglik_bytes(int n, int64_t T);
cudaError_t launch_scan_loglik(const ScanArgs &a, const ScanLoglikOut &o, cudaStream_t stream,
                               int64_t *launches);
// Time-sharded log-likelihoods, one rank's chunk after the all-gather of the forward aggregates:
// a = the forward finish phase's arguments (aggs_dev, rank, world, start = the prior, workspace =
// that of the local phase); o.transition / o.innovations / o.status unused, o.m_last / o.C_last
// written on rank world - 1.  Then the rank-order sum of the gathered partial vectors [world][3].
cudaError_t launch_scan_dist_loglik(const ScanArgs &a, const ScanLoglikOut &o, cudaStream_t stream,
                                    int64_t *launches);
cudaError_t launch_scan_dist_loglik_finish(const double *parts, int world, double *transition, double *innovations,
                                           int32_t *status, cudaStream_t stream, int64_t *launches);
// FFBS + Gibbs statistics of one series: a = a forward kScanApply pass with keep_init = 1 whose a.kf
// has (m, C) (the caller's arrays or workspace) and any of a, R, f, Q; a.status is OR-ed (the caller
// zeroes it).  Statistics pointers may be null.
struct ScanFfbsOut {
  CView z;             // injected normals, rows x n, or ptr == nullptr (Philox)
  unsigned long long rng_seed, rng_sweep;
  long long rng_base;
  View theta;          // rows x n
  StatViews stats;
  void *workspace;     // device, scan_workspace_bytes(n, T): the sampler's level-2 elements
  double *parts;       // device, scan_ffbs_parts_bytes(n, T): block partials of the statistics
  long long total_rows, first_row;  // Philox offsets: rows of the whole series (T + 1), global row of row 0
  double *agg_dev;           // time-sharded local: this rank's sampler aggregate (out)
  const double *aggs_dev;    // time-sharded finish: [world][n*n + n] gathered aggregates
  double *part_vec;          // time-sharded finish: [ssy, ny, ssw, scatter, status] of the chunk (out)
};
size_t scan_ffbs_parts_bytes(int n, int64_t T);
cudaError_t launch_scan_ffbs(const ScanArgs &a, const ScanFfbsOut &o, cudaStream_t stream, int64_t *launches);
// Time-sharded FFBS, one rank's chunk: a = the forward finish phase's arguments with a.kf (m, C)
// required and fuse_sagg = nullptr, has_successor = rank < world - 1.  finish = false: forward finish
// + the sampler's level 1 and 2, aggregate into o.agg_dev; finish = true: carry, apply, partial vector.
cudaError_t launch_scan_dist_ffbs(const ScanArgs &a, const ScanFfbsOut &o, bool finish, cudaStream_t stream,
                                  int64_t *launches);
cudaError_t launch_scan_dist_ffbs_stats_finish(int n, const double *parts, int world, const StatViews &sv,
                                               int32_t *status, cudaStream_t stream, int64_t *launches);
int scan_sampler_elem_doubles(int n);
void scan_combine_host(int n, bool backward, const double *ei, const double *ej, double *out);

// scalar_filters.cu: scalar AR(1) / OU filter + backward sampler (FilterAr.scala, FilterOu.scala)
// and the conjugate (unknown observation variance) filter (ConjugateFilter.scala), one thread
// per series.  Views here address element (series b, row r) at ptr[b*sb + r*sr].
struct ArArgs {
  int64_t B;
  int T;
  int ou;                   // 0 = AR(1) on the unit grid, 1 = Ornstein-Uhlenbeck on dt[]
  int ffbs;                 // 0 = filter only, 1 = filter + backward sample
  PView phi, mu, sigma;     // per series (ptr != nullptr) ...
  double phi_s, mu_s, sigma_s;  // ... or shared scalars
  const double *dt;         // device [T] (OU): dt[0] = 0, dt[t] = times[t] - times[t-1]
  View v;                   // per-series per-step variances (T rows) or ptr == nullptr
  const double *v_shared;   // device [T] shared by the batch, or nullptr
  double v_s;               // one variance for every step
  View y;                   // T rows
  View m, C, a, R;          // T + 1 rows, any may be null (filter mode)
  View sm, sC;              // ffbs mode: where (m, C) are spilled (user m, C or workspace)
  View z, theta;            // T + 1 rows
};
cudaError_t launch_ar(const ArArgs &a, cudaStream_t stream);

struct ConjArgs {
  Batch bt;                 // V unused; F, G time-invariant (passed on the host side)
  double prior_shape, prior_scale;
  KfViews kf;
  View shape, scale;        // T + 1 rows, k = 1
};
bool conjugate_supported(int n, int p);
// both log-likelihoods, one thread per series (n <= 4, p = 1, time-invariant model)
bool loglik_small_supported(const Batch &bt);
cudaError_t launch_loglik_small(const Batch &bt, const double *hG, const double *hF,
                                double *ll_transition, double *ll_innov, const View &last_m,
                                const View &last_C, cudaStream_t stream);
cudaError_t launch_conjugate(const ConjArgs &a, const double *hG, const double *hF,
                             cudaStream_t stream);

// gibbs_draw.cu: conjugate draws of V and W from the Gibbs sufficient statistics.
struct GibbsDrawArgs {
  int64_t B;
  int n, p, T;
  int wishart;              // 0: diagonal W ~ d-inverse-gamma; 1: full W ~ inverse Wishart
  double v_shape, v_scale, w_shape, w_scale, w_nu;
  const double *psi;        // device n*n (wishart)
  StatViews stats;          // inputs (sb, sk strides)
  View gv, gw, bart;        // injected standard-gamma variates [p], [n] / Bartlett factor [n*n]
  unsigned long long seed, sweep;
  long long base;           // global index of chain 0 of this launch (Philox subsequences)
  View V, W;                // outputs: per-chain p*p and n*n (column-major), either may be null
  View v_shape_rate, w_shape_rate;  // optional outputs [2p], [2n]: posterior shapes | rates
  int32_t *status;          // [B] or nullptr (OR-ed)
};
cudaError_t launch_gibbs_draw(const GibbsDrawArgs &a, cudaStream_t stream, int64_t *launches);

// peak.cu: DFMA throughput microbenchmark (TFLOP/s at 2 flops per DFMA).
cudaError_t measure_fp64_peak(cudaStream_t stream, double *scratch, double *tflops);

}  // namespace bdlm
