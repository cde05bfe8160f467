// kf_warp.cu -- generic-dimension kernels (n <= 48, p <= 32): ONE WARP PER SERIES / CHAIN.
//
// Covers every function of the hot path for any model shape: forward Kalman filter with
// partially-missing observations, RTS smoother, FFBS with the Jacobi eigen draw, both
// log-likelihoods, the SVD filter / sampler and the Gibbs sufficient statistics.  These
// configurations (n = 13 FFBS, n = p = 8 SVD) are FP64-/shared-memory-bound, not HBM
// bound (SURVEY.md section 8d): the state matrices of a series live in the warp's slice
// of shared memory, lanes split the output elements of each small matrix operation
// (warp_linalg.cuh), and HBM is touched once per row for inputs, outputs and the
// forward->backward spill, which is kept series-major ([B][rows][k], contiguous per
// series) so every spill access of a warp is a run of full 128-byte lines.
//
// Arithmetic mirrors oracle/bdlm_oracle.c operation for operation; citations there.
#include "common.cuh"
#include "launch.h"
#include "rng.cuh"
#include "warp_linalg.cuh"

namespace bdlm {

namespace {

__host__ __device__ inline int imax(int a, int b) { return a > b ? a : b; }

// Per-warp shared-memory carve-up; the same arithmetic runs on the host (size only).
struct Ws {
  double *G, *F, *W, *V, *Wsq;
  double *m, *C, *a, *R, *f, *Q, *dcv, *drv, *th, *Sm;
  double *t1, *t2, *t3, *t4, *t5, *t6, *stk;
  double *v1, *v2, *v3, *v4, *yrow;
  double *scr;
  int *iscr;
  size_t total;  // doubles

  __host__ __device__ Ws() {}

  // svd4_kernel layout: the temporaries and the (batch-shared) model matrices exist ONCE per
  // warp, only what must survive from one phase to the next is kept per series.  Four full
  // workspaces (41.7 KB) allow 5 warps per SM; this layout (23.6 KB) allows 9, which is what
  // hides the serial rotation-parameter chain of the joint SVDs.
  // shared_params: V, W (and their square-root factors) are the same for every series of the
  // batch (BASELINE config 4 as a filter / sampler; not inside a Gibbs sweep with per-series
  // draws): one copy per warp instead of four.
  static __host__ __device__ size_t svd4_shared_doubles(int n, int p, bool shared_params) {
    const int L = imax(n, p), LL = L * L;
    const bool scr_in_t = 2 * LL >= kScrDoubles;  // the Jacobi scratch of the (cold) generic SVDs
    return (size_t)n * n + (size_t)n * p + 6 * (size_t)LL + 4 * (size_t)L + p +
           (scr_in_t ? 0 : kScrDoubles) + kIscrInts / 2 +
           (shared_params ? 2 * (size_t)n * n + (size_t)p * p : 0);
  }
  static __host__ __device__ size_t svd4_series_doubles(int n, int p, bool shared_params) {
    const int nn = n * n, L = imax(n, p);
    return (shared_params ? 0 : 2 * (size_t)nn + (size_t)p * p) + 3 * (size_t)n + 2 * (size_t)nn + p +
           2 * (size_t)n + (size_t)imax((n + L) * n, L * L) + n;
  }
  static __device__ Ws svd4(double *shared, double *series, int n, int p, bool shared_params,
                            double *&sV, double *&sS) {
    Ws w;
    const int nn = n * n, L = imax(n, p), LL = L * L;
    double *o = shared;
    auto take = [&](size_t cnt) { double *ptr = o; o += cnt; return ptr; };
    w.G = take(nn); w.F = take((size_t)n * p);
    w.t1 = take(LL); w.t2 = take(LL); w.t3 = take(LL); w.t4 = take(LL); w.t5 = take(LL); w.t6 = take(LL);
    w.v1 = take(L); w.v2 = take(L); w.v3 = take(L); w.v4 = take(L); w.yrow = take(p);
    // w_jacobi_svd (initial state / per-step parameter transforms) works in t3, t4, t5 only:
    // its dot-product scratch can sit in t1 | t2 when they are large enough
    w.scr = (2 * LL >= kScrDoubles) ? w.t1 : take(kScrDoubles);
    w.iscr = reinterpret_cast<int *>(take(kIscrInts / 2));
    if (shared_params) { w.W = take(nn); w.Wsq = take(nn); w.V = take((size_t)p * p); }
    o = series;
    if (!shared_params) { w.W = take(nn); w.Wsq = take(nn); w.V = take((size_t)p * p); }
    w.m = take(n); w.a = take(n); w.th = take(n);
    w.C = take(nn); w.R = take(nn); w.f = take(p);
    w.dcv = take(n); w.drv = take(n);
    w.stk = take((size_t)imax((n + L) * n, LL));
    // right singular vectors of the joint SVDs: written after every lane of the octet has pulled
    // its column of the stack into registers, so they can overwrite the stack
    sV = w.stk; sS = take(n);
    w.Q = nullptr; w.Sm = nullptr;
    w.total = 0;
    return w;
  }

  __host__ __device__ Ws(double *base, int n, int p, int op) {
    const int nn = n * n, L = imax(n, p), LL = L * L;
    size_t o = 0;
    auto take = [&](size_t cnt) { double *ptr = base ? base + o : nullptr; o += cnt; return ptr; };
    const bool svd = (op == kOpSvdFilter || op == kOpSvdFfbs);
    G = take(nn); F = take((size_t)n * p); W = take(nn); V = take((size_t)p * p);
    Wsq = svd ? take(nn) : nullptr;
    m = take(n); C = take(nn); a = take(n); R = take(nn); f = take(p);
    // The SVD operations never form Q or the smoothed covariance, and their sixth temporary is
    // only live while t1 is dead (svd_update: the gain after Fm is consumed; SvdSampler.step:
    // (du^T du) gWinv after G^T sqrtW^T is consumed) -- so t6 shares t1's storage there.  That is
    // what lets n = 48 (12 n^2 + stack doubles) fit the 227 KB of one SM.
    Q = svd ? nullptr : take((size_t)p * p);
    dcv = svd ? take(n) : nullptr; drv = svd ? take(n) : nullptr;
    th = take(n); Sm = svd ? nullptr : take(nn);
    t1 = take(LL); t2 = take(LL); t3 = take(LL); t4 = take(LL); t5 = take(LL);
    t6 = svd ? t1 : take(LL);
    stk = svd ? take((size_t)imax((n + L) * n, LL)) : nullptr;
    v1 = take(L); v2 = take(L); v3 = take(L); v4 = take(L); yrow = take(p);
    scr = take(kScrDoubles);
    iscr = reinterpret_cast<int *>(take(kIscrInts / 2));
    total = o;
  }
};

struct Lane {
  int lane;
  int64_t b;
};

__device__ __forceinline__ void load_pview(int lane, const PView &v, int64_t b, int cnt,
                                           double *dst) {
  const double *p = v.ptr + b * v.sb;
  for (int k = lane; k < cnt; k += 32) dst[k] = p[k * v.sk];
}

__device__ __forceinline__ void store_view(int lane, const View &v, int64_t b, int64_t row,
                                           int cnt, const double *src) {
  if (v.ptr == nullptr) return;
  double *p = v.ptr + b * v.sb + row * v.sr;
  for (int k = lane; k < cnt; k += 32) st_stream(p + k * v.sk, src[k]);
}

__device__ __forceinline__ void store_view_const(int lane, const View &v, int64_t b,
                                                 int64_t row, int cnt, double val) {
  if (v.ptr == nullptr) return;
  double *p = v.ptr + b * v.sb + row * v.sr;
  for (int k = lane; k < cnt; k += 32) st_stream(p + k * v.sk, val);
}

__device__ __forceinline__ void load_view(int lane, const View &v, int64_t b, int64_t row,
                                          int cnt, double *dst) {
  const double *p = v.ptr + b * v.sb + row * v.sr;
  for (int k = lane; k < cnt; k += 32) dst[k] = p[k * v.sk];
}

__device__ __forceinline__ void load_cview(int lane, const CView &v, int64_t b, int64_t row,
                                           int cnt, double *dst) {
  const double *p = v.ptr + b * v.sb + row * v.sr;
  for (int k = lane; k < cnt; k += 32) dst[k] = p[k * v.sk];
}

// The n normals consumed when drawing theta[row]: injected, or generated (rng.cuh).
__device__ __forceinline__ void load_z(int lane, const WarpArgs &wa, int64_t b, int64_t row, int rows,
                                       int n, double *dst) {
  if (wa.z.ptr) { load_cview(lane, wa.z, b, row, n, dst); return; }
  const RngKey key{wa.rng_seed, wa.rng_sweep};
  for (int k = lane; k < n; k += 32) dst[k] = philox_normal(key, wa.rng_base + b, rows, (int)row, n, k);
}

// Model matrices for observation t of series b into the warp's G / F slots.
__device__ __forceinline__ void load_model(int lane, const Batch &bt, const Ws &ws, int64_t b, int t,
                                           bool first) {
  const int n = bt.n, p = bt.p;
  if (bt.g_tv || first) {
    const double *g = bt.G + b * bt.G_sb + (int64_t)t * bt.G_sr;
    for (int k = lane; k < n * n; k += 32) ws.G[k] = g[k * bt.G_sk];
  }
  if (bt.f_tv || first) {
    const double *f = bt.F + b * bt.F_sb + (int64_t)t * bt.F_sr;
    for (int k = lane; k < n * p; k += 32) ws.F[k] = f[k * bt.F_sk];
  }
  __syncwarp();
}

// Observed-component list of the row in ws.yrow: returns po, fills obs[] (ints).
__device__ __forceinline__ int observed(int lane, int p, const double *yrow, int *obs) {
  const bool ok = lane < p && !isnan(yrow[lane]);
  const unsigned mask = __ballot_sync(FULL, ok);
  const int po = __popc(mask);
  if (lane < po) obs[lane] = __fns(mask, 0, lane + 1);
  __syncwarp();
  return po;
}

// KalmanFilter.advState (KalmanFilter.scala:273-286): (m, C) -> (a, R)
__device__ __forceinline__ void kf_advance(int lane, int n, const Ws &ws, double dt,
                                           const double *m, const double *C, double *a,
                                           double *R) {
  if (dt == 0.0) {
    for (int k = lane; k < n; k += 32) a[k] = m[k];
    for (int k = lane; k < n * n; k += 32) R[k] = C[k];
    __syncwarp();
    return;
  }
  w_mv(lane, n, n, ws.G, n, false, m, a);
  w_mm(lane, n, n, n, ws.G, n, false, C, n, false, ws.t1, n);
  w_mm(lane, n, n, n, ws.t1, n, false, ws.G, n, true, R, n);
  for (int k = lane; k < n * n; k += 32) R[k] = R[k] + ws.W[k] * dt;
  __syncwarp();
}

// oneStepPrediction (:311-321) + updateState (:64-94).  Reads ws.a, ws.R, ws.yrow;
// writes ws.f, ws.Q, ws.m, ws.C.
__device__ __forceinline__ int kf_update(int lane, int n, int p, const Ws &ws) {
  int st = 0;
  w_mv(lane, p, n, ws.F, n, true, ws.a, ws.f);
  w_mm(lane, p, n, n, ws.F, n, true, ws.R, n, false, ws.t1, p);
  w_mm(lane, p, n, p, ws.t1, p, false, ws.F, n, false, ws.Q, p);
  for (int k = lane; k < p * p; k += 32) ws.Q[k] = ws.Q[k] + ws.V[k];
  __syncwarp();
  int *obs = ws.iscr + kObsOff;
  const int po = observed(lane, p, ws.yrow, obs);
  if (po == 0) {
    for (int k = lane; k < n; k += 32) ws.m[k] = ws.a[k];
    for (int k = lane; k < n * n; k += 32) ws.C[k] = ws.R[k];
    __syncwarp();
    return st;
  }
  double *Fm = ws.t2, *Vm = ws.t3, *Qm = ws.t4, *fm = ws.v1, *e = ws.v2;
  for (ElemIter it(lane, n, po); it.ok(); it.next()) Fm[it.i + it.j * n] = ws.F[it.i + obs[it.j] * n];
  for (ElemIter it(lane, po, po); it.ok(); it.next())
    Vm[it.i + it.j * po] = ws.V[obs[it.i] + obs[it.j] * p];
  __syncwarp();
  w_mv(lane, po, n, Fm, n, true, ws.a, fm);
  w_mm(lane, po, n, n, Fm, n, true, ws.R, n, false, ws.t1, po);
  w_mm(lane, po, n, po, ws.t1, po, false, Fm, n, false, Qm, po);
  for (int k = lane; k < po * po; k += 32) Qm[k] = Qm[k] + Vm[k];
  if (lane < po) e[lane] = ws.yrow[obs[lane]] - fm[lane];
  __syncwarp();
  // K = (Qm^T \ (Fm^T R^T))^T
  w_mm(lane, po, n, n, Fm, n, true, ws.R, n, true, ws.t1, po);
  w_transpose(lane, po, Qm, ws.t5);
  st |= w_lu_solve(lane, po, ws.t5, n, ws.t1);
  double *K = ws.t6;
  for (ElemIter it(lane, n, po); it.ok(); it.next()) K[it.i + it.j * n] = ws.t1[it.j + it.i * po];
  __syncwarp();
  w_mv(lane, n, po, K, n, false, e, ws.v3);
  for (int k = lane; k < n; k += 32) ws.m[k] = ws.a[k] + ws.v3[k];
  // D = I - K Fm^T
  w_mm(lane, n, po, n, K, n, false, Fm, n, true, ws.t1, n);
  for (ElemIter it(lane, n, n); it.ok(); it.next())
    ws.t1[it.i + it.j * n] = ((it.i == it.j) ? 1.0 : 0.0) - ws.t1[it.i + it.j * n];
  __syncwarp();
  w_mm(lane, n, n, n, ws.t1, n, false, ws.R, n, false, ws.t5, n);
  w_mm(lane, n, n, n, ws.t5, n, false, ws.t1, n, true, ws.C, n);
  w_mm(lane, n, po, po, K, n, false, Vm, po, false, ws.t4, n);
  w_mm(lane, n, po, n, ws.t4, n, false, K, n, true, ws.t5, n);
  for (int k = lane; k < n * n; k += 32) ws.C[k] = ws.C[k] + ws.t5[k];
  __syncwarp();
  return st;
}

// B = (R1^T \ (G C^T))^T into ws.t3  (Smoothing.scala:41 and :85)
__device__ __forceinline__ int smoothing_gain(int lane, int n, const Ws &ws, const double *C,
                                              const double *R1) {
  w_mm(lane, n, n, n, ws.G, n, false, C, n, true, ws.t1, n);
  w_transpose(lane, n, R1, ws.t2);
  const int st = w_lu_solve(lane, n, ws.t2, n, ws.t1);
  w_transpose(lane, n, ws.t1, ws.t3);
  return st;
}

// MultivariateGaussianSvd(mu, cov).draw with injected normals z -> out (n).
// cov must not alias t2, t3, t6; uses t2, t3, t6, v1, v2, scr, iscr.
__device__ __forceinline__ int mvn_eig_draw(int lane, int n, const Ws &ws, const double *mu,
                                            const double *cov, const double *z, double *out) {
  const int st = w_jacobi_eigsym(lane, n, cov, ws.t2, ws.t3, ws.scr, ws.iscr, ws.v1, ws.t6);
  for (ElemIter it(lane, n, n); it.ok(); it.next())
    ws.t2[it.i + it.j * n] = ws.t6[it.i + it.j * n] * sqrt(ws.v1[it.j]);
  __syncwarp();
  w_mv(lane, n, n, ws.t2, n, false, z, ws.v2);
  for (int k = lane; k < n; k += 32) out[k] = mu[k] + ws.v2[k];
  __syncwarp();
  return st;
}

// sum(log(diag(cholesky(S)))) -- oracle chol_logdet; L workspace n*n.  All lanes get it.
__device__ __forceinline__ int w_chol_logdet(int lane, int n, const double *S, double *L,
                                             double &sumlog) {
  int st = 0;
  for (int k = lane; k < n * n; k += 32) L[k] = S[k];
  __syncwarp();
  double acc = 0.0;
  for (int j = 0; j < n; ++j) {
    double d = L[j + j * n];
    for (int k = 0; k < j; ++k) d = d - L[j + k * n] * L[j + k * n];
    if (!(d > 0.0)) st = BDLM_ST_NOTPD;
    d = sqrt(d);
    __syncwarp();
    if (lane == 0) L[j + j * n] = d;
    for (int i = j + 1 + lane; i < n; i += 32) {
      double v = L[i + j * n];
      for (int k = 0; k < j; ++k) v = v - L[i + k * n] * L[j + k * n];
      L[i + j * n] = v / d;
    }
    __syncwarp();
    acc = acc + log(d);
  }
  sumlog = acc;
  return st;
}

constexpr double kLog2Pi = 1.8378770664093453;

// breeze MultivariateGaussian(mu, S).logPdf(x); uses t1 (S copy / L), t2, v1, v2.
__device__ __forceinline__ int w_mvn_logpdf(int lane, int n, const Ws &ws, const double *x,
                                            const double *mu, const double *S, double &out) {
  int st = 0;
  for (int k = lane; k < n; k += 32) { ws.v1[k] = x[k] - mu[k]; ws.v2[k] = ws.v1[k]; }
  for (int k = lane; k < n * n; k += 32) ws.t1[k] = S[k];
  __syncwarp();
  st |= w_lu_solve(lane, n, ws.t1, 1, ws.v2);
  double dot = 0.0;
  for (int i = 0; i < n; ++i) {
    const double prod = ws.v2[i] * ws.v1[i];
    dot = (i == 0) ? prod : dot + prod;
  }
  double ld;
  st |= w_chol_logdet(lane, n, S, ws.t2, ld);
  out = -dot / 2.0 - (n / 2.0 * kLog2Pi + ld);
  return st;
}

// SvdFilter.sqrtInvSvd (inv) / sqrtSvd: out = diag(g(s)) V^T of svd(M); M n x n.
__device__ __forceinline__ int w_sqrt_svd(int lane, int n, const Ws &ws, const double *M,
                                          bool inv, double *out) {
  for (int k = lane; k < n * n; k += 32) ws.stk[k] = M[k];
  __syncwarp();
  const int st = w_jacobi_svd(lane, n, n, ws.stk, ws.t3, ws.scr, ws.iscr, ws.v1, ws.t4);
  for (ElemIter it(lane, n, n); it.ok(); it.next()) {
    const double s = ws.v1[it.i];
    const double d = inv ? 1.0 / sqrt(s) : sqrt(s);
    out[it.i + it.j * n] = d * ws.t4[it.j + it.i * n];
  }
  __syncwarp();
  return st;
}

// Next row f2 on the SVD path: the parameters of observation t, transformed as the reference
// transforms them at every step -- ps = vs.map(vi => transformParams(p.copy(v = vi)))
// (DlmFsv.scala:213, DlmFsvSystem.scala:182): ws.V <- sqrtInvSvd(V_t), ws.Wsq <- sqrtSvd(W_t) and
// ws.W <- the advance closure's factor (raw W_t, or sqrtSvd(W_t) with BDLM_SVD_CONSISTENT_W, which
// is what those two callers use).  Clobbers stk, t3, t4, t5, v1, scr, iscr.
__device__ __forceinline__ int svd_load_params_tv(int lane, const Batch &bt, const Ws &ws,
                                               int64_t b, int t, bool want_v) {
  int st = 0;
  const int n = bt.n, p = bt.p;
  if (bt.v_tv && want_v) {
    PView vt = bt.V;
    vt.ptr += (int64_t)t * bt.V_sr;
    load_pview(lane, vt, b, p * p, ws.V);
    __syncwarp();
    st |= w_sqrt_svd(lane, p, ws, ws.V, true, ws.t5);
    w_copy(lane, p * p, ws.t5, ws.V);
  }
  if (bt.w_tv) {
    PView wt = bt.W;
    wt.ptr += (int64_t)t * bt.W_sr;
    load_pview(lane, wt, b, n * n, ws.W);
    __syncwarp();
    st |= w_sqrt_svd(lane, n, ws, ws.W, false, ws.Wsq);
    if (bt.compat & BDLM_SVD_CONSISTENT_W) w_copy(lane, n * n, ws.Wsq, ws.W);
  }
  return st;
}

// SvdFilter.advState (SvdFilter.scala:183-202): (m, dcv, C=uc) -> (a, drv, R=ur);
// ws.W holds the advance closure's W factor.
__device__ __forceinline__ int svd_advance(int lane, int n, const Ws &ws, double dt) {
  if (dt == 0.0) {
    for (int k = lane; k < n; k += 32) { ws.a[k] = ws.m[k]; ws.drv[k] = ws.dcv[k]; }
    for (int k = lane; k < n * n; k += 32) ws.R[k] = ws.C[k];
    __syncwarp();
    return 0;
  }
  w_mv(lane, n, n, ws.G, n, false, ws.m, ws.a);
  for (ElemIter it(lane, n, n); it.ok(); it.next())
    ws.t1[it.i + it.j * n] = ws.dcv[it.i] * ws.C[it.j + it.i * n];
  __syncwarp();
  w_mm(lane, n, n, n, ws.t1, n, false, ws.G, n, true, ws.t2, n);
  const double sq = sqrt(dt);
  for (ElemIter it(lane, n, n); it.ok(); it.next()) {
    ws.stk[it.i + it.j * 2 * n] = ws.t2[it.i + it.j * n];
    ws.stk[n + it.i + it.j * 2 * n] = ws.W[it.i + it.j * n] * sq;
  }
  __syncwarp();
  return w_jacobi_svd(lane, 2 * n, n, ws.stk, ws.t3, ws.scr, ws.iscr, ws.drv, ws.R);
}

// SvdFilter.updateState (SvdFilter.scala:38-68); ws.V holds V^{-1/2}.
__device__ __forceinline__ int svd_update(int lane, int n, int p, const Ws &ws) {
  int st = 0;
  int *obs = ws.iscr + kObsOff;
  const int po = observed(lane, p, ws.yrow, obs);
  if (po == 0) {
    for (int k = lane; k < n; k += 32) { ws.m[k] = ws.a[k]; ws.dcv[k] = ws.drv[k]; }
    for (int k = lane; k < n * n; k += 32) ws.C[k] = ws.R[k];
    __syncwarp();
    return st;
  }
  double *Fm = ws.t1, *Vm = ws.t2;
  for (ElemIter it(lane, n, po); it.ok(); it.next()) Fm[it.i + it.j * n] = ws.F[it.i + obs[it.j] * n];
  for (ElemIter it(lane, po, po); it.ok(); it.next())
    Vm[it.i + it.j * po] = ws.V[obs[it.i] + obs[it.j] * p];
  __syncwarp();
  w_mv(lane, po, n, Fm, n, true, ws.a, ws.v1);  // fm
  w_mm(lane, po, po, n, Vm, po, false, Fm, n, true, ws.t3, po);
  w_mm(lane, po, n, n, ws.t3, po, false, ws.R, n, false, ws.t4, po);
  const int r = po + n;
  for (ElemIter it(lane, r, n); it.ok(); it.next()) {
    const int i = it.i, j = it.j;
    ws.stk[i + j * r] = (i < po) ? ws.t4[i + j * po]
                                 : ((i - po == j) ? 1.0 / ws.drv[j] : 0.0);
  }
  if (lane < po) ws.v1[lane] = ws.yrow[obs[lane]] - ws.v1[lane];  // e
  __syncwarp();
  st |= w_jacobi_svd(lane, r, n, ws.stk, ws.t3, ws.scr, ws.iscr, ws.v2, ws.t5);
  w_mm(lane, n, n, n, ws.R, n, false, ws.t5, n, false, ws.C, n);  // uc = ur * V
  w_mm(lane, n, po, po, Fm, n, false, Vm, po, true, ws.t3, n);
  w_mm(lane, n, po, po, ws.t3, n, false, Vm, po, false, ws.t4, n);  // fv
  for (int k = lane; k < n; k += 32) ws.dcv[k] = 1.0 / ws.v2[k];
  __syncwarp();
  for (ElemIter it(lane, n, n); it.ok(); it.next())
    ws.t3[it.i + it.j * n] = ws.dcv[it.i] * ws.C[it.j + it.i * n];  // X = diag(dc) uc^T
  __syncwarp();
  w_mm(lane, n, n, n, ws.t3, n, true, ws.t3, n, false, ws.t5, n);
  w_mm(lane, n, n, po, ws.t5, n, false, ws.t4, n, false, ws.t6, n);  // gain
  w_mv(lane, n, po, ws.t6, n, false, ws.v1, ws.v3);
  for (int k = lane; k < n; k += 32) ws.m[k] = ws.a[k] + ws.v3[k];
  __syncwarp();
  return st;
}

// Gibbs sufficient statistics of the path in `theta` (rows = T + 1), accumulated in the
// reference's (ascending-time) order: Gibbs.scala:29-43, :63-73, GibbsWishart.scala:22-29.
// Lane i owns ssy[i] / ssw[i]; scatter elements are split over lanes.
__device__ __forceinline__ void gibbs_stats(int lane, const Batch &bt, const Ws &ws,
                                            const View &theta, const StatViews &sv,
                                            int64_t b) {
  const int n = bt.n, p = bt.p, T = bt.T;
  double ssy = 0.0, ny = 0.0, ssw = 0.0, ssw_hi = 0.0;  // ssw_hi: component lane + 32 (n > 32)
  double sc[72];  // scatter elements idx = lane + 32 * q, q < 72 (n*n <= 48*48)
  const int nsc = (n * n + 31) / 32;
  const bool want_sc = sv.scatter.ptr != nullptr;
  double tprev = 0.0;
  load_view(lane, theta, b, 0, n, ws.th);  // theta_0
  __syncwarp();
  for (int t = 0; t < T; ++t) {
    load_model(lane, bt, ws, b, t, t == 0);
    load_view(lane, theta, b, t + 1, n, ws.v4);
    load_cview(lane, bt.y, b, t, p, ws.yrow);
    __syncwarp();
    w_mv(lane, p, n, ws.F, n, true, ws.v4, ws.v1);
    if (lane < p) {
      const double yi = ws.yrow[lane];
      double res = 0.0;
      if (!isnan(yi)) { const double d = yi - ws.v1[lane]; res = d * d; ny += 1.0; }
      ssy = (t == 0) ? res : ssy + res;
    }
    const double dt = dt_at(bt, b, t);
    w_mv(lane, n, n, ws.G, n, false, ws.th, ws.v2);
    for (int k = lane; k < n; k += 32) ws.v3[k] = ws.v4[k] - ws.v2[k];
    __syncwarp();
    if (lane < n) {
      const double v = (ws.v3[lane] * ws.v3[lane]) / dt;
      ssw = (t == 0) ? v : ssw + v;
    }
    if (lane + 32 < n) {
      const double v = (ws.v3[lane + 32] * ws.v3[lane + 32]) / dt;
      ssw_hi = (t == 0) ? v : ssw_hi + v;
    }
    if (want_sc) {
#pragma unroll 4
      for (int q = 0; q < nsc; ++q) {
        const int idx = lane + 32 * q;
        if (idx < n * n) {
          const int j = idx / n, i = idx - j * n;
          const double v = (ws.v3[i] * ws.v3[j]) / dt;
          sc[q] = (t == 0) ? v : sc[q] + v;
        }
      }
    }
    for (int k = lane; k < n; k += 32) ws.th[k] = ws.v4[k];
    __syncwarp();
    (void)tprev;
  }
  if (sv.ssy.ptr && lane < p) sv.ssy.ptr[b * sv.ssy.sb + lane * sv.ssy.sk] = ssy;
  if (sv.ny.ptr && lane < p) sv.ny.ptr[b * sv.ny.sb + lane * sv.ny.sk] = ny;
  if (sv.ssw.ptr && lane < n) sv.ssw.ptr[b * sv.ssw.sb + lane * sv.ssw.sk] = ssw;
  if (sv.ssw.ptr && lane + 32 < n) sv.ssw.ptr[b * sv.ssw.sb + (lane + 32) * sv.ssw.sk] = ssw_hi;
  if (want_sc)
    for (int q = 0; q < nsc; ++q) {
      const int idx = lane + 32 * q;
      if (idx < n * n) sv.scatter.ptr[b * sv.scatter.sb + idx * sv.scatter.sk] = sc[q];
    }
}

template <int OP, int NT, int PT>
__global__ void __launch_bounds__(64)
warp_kernel(const WarpArgs wa, const int ws_doubles) {
  extern __shared__ double smem[];
  const Batch &bt = wa.bt;
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int64_t b = (int64_t)blockIdx.x * (blockDim.x >> 5) + wib;
  if (b >= bt.B) return;
  // NT, PT > 0: dimensions known at compile time (hot shapes; loops unroll, index math folds)
  const int n = NT > 0 ? NT : bt.n, p = PT > 0 ? PT : bt.p;
  const int nn = n * n, T = bt.T, ki = bt.keep_init, rows = T + ki;
  Ws ws(smem + (size_t)wib * ws_doubles, n, p, OP);
  int st = 0;

  constexpr bool kSvd = (OP == kOpSvdFilter || OP == kOpSvdFfbs);
  constexpr bool kForward = (OP != kOpSmooth && OP != kOpStats);
  constexpr bool kSpill = (OP == kOpFilterSmooth || OP == kOpFfbs || OP == kOpSvdFfbs);

  if (OP == kOpStats) {
    gibbs_stats(lane, bt, ws, wa.theta, wa.stats, b);
    return;
  }

  load_pview(lane, bt.W, b, nn, ws.W);
  load_pview(lane, bt.V, b, p * p, ws.V);
  __syncwarp();
  double *spill = kSpill ? wa.spill + (size_t)b * rows * wa.spill_k : nullptr;
  const double nanv = __longlong_as_double(0x7ff8000000000000LL);
  double ll_tr = 0.0, ll_in = 0.0;

  if (kForward) {
    load_pview(lane, bt.m0, b, n, ws.m);
    load_pview(lane, bt.C0, b, nn, ws.C);
    __syncwarp();
    load_model(lane, bt, ws, b, 0, true);
    if (kSvd) {
      // transformParams (SvdFilter.scala:232-236) + initialiseState (:83-95)
      st |= w_sqrt_svd(lane, p, ws, ws.V, true, ws.t5);
      w_copy(lane, p * p, ws.t5, ws.V);
      st |= w_sqrt_svd(lane, n, ws, ws.W, false, ws.Wsq);
      if (bt.compat & BDLM_SVD_CONSISTENT_W) w_copy(lane, nn, ws.Wsq, ws.W);
      w_copy(lane, nn, ws.C, ws.stk);
      st |= w_jacobi_svd(lane, n, n, ws.stk, ws.t3, ws.scr, ws.iscr, ws.v1, ws.t4);
      for (int k = lane; k < n; k += 32) ws.dcv[k] = sqrt(ws.v1[k]);
      w_copy(lane, nn, ws.t4, ws.C);
      if (ki) {
        w_mv(lane, p, n, ws.F, n, true, ws.m, ws.f);
        store_view(lane, wa.svd.m, b, 0, n, ws.m);
        store_view(lane, wa.svd.a, b, 0, n, ws.m);
        store_view(lane, wa.svd.dc, b, 0, n, ws.dcv);
        store_view(lane, wa.svd.dr, b, 0, n, ws.dcv);
        store_view(lane, wa.svd.uc, b, 0, nn, ws.C);
        store_view(lane, wa.svd.ur, b, 0, nn, ws.C);
        store_view(lane, wa.svd.f, b, 0, p, ws.f);
        if (kSpill) {  // [m, dc, uc, a]
          for (int k = lane; k < n; k += 32) {
            spill[k] = ws.m[k]; spill[n + k] = ws.dcv[k]; spill[2 * n + nn + k] = ws.m[k];
          }
          for (int k = lane; k < nn; k += 32) spill[2 * n + k] = ws.C[k];
        }
      }
    } else if (ki) {
      store_view(lane, wa.kf.m, b, 0, n, ws.m);
      store_view(lane, wa.kf.a, b, 0, n, ws.m);
      store_view(lane, wa.kf.C, b, 0, nn, ws.C);
      store_view(lane, wa.kf.R, b, 0, nn, ws.C);
      store_view_const(lane, wa.kf.f, b, 0, p, nanv);
      store_view_const(lane, wa.kf.Q, b, 0, p * p, nanv);
      if (kSpill) {  // [m, C, a, R]
        for (int k = lane; k < n; k += 32) { spill[k] = ws.m[k]; spill[n + nn + k] = ws.m[k]; }
        for (int k = lane; k < nn; k += 32) { spill[n + k] = ws.C[k]; spill[2 * n + nn + k] = ws.C[k]; }
      }
    }
    __syncwarp();

    for (int t = 0; t < T; ++t) {
      const int64_t row = t + ki;
      load_model(lane, bt, ws, b, t, false);
      load_cview(lane, bt.y, b, t, p, ws.yrow);
      const double dt = dt_at(bt, b, t);
      if (!kSvd && bt.v_tv) {  // V_t: params.copy(v = V_t) at every step (StudentTGibbs.scala:105-118)
        PView vt = bt.V;
        vt.ptr += (int64_t)t * bt.V_sr;
        load_pview(lane, vt, b, p * p, ws.V);
      }
      if (!kSvd && bt.w_tv) {  // W_t: params.copy(w = W_t) (DlmFsvSystem.scala:142-153)
        PView wt = bt.W;
        wt.ptr += (int64_t)t * bt.W_sr;
        load_pview(lane, wt, b, nn, ws.W);
      }
      __syncwarp();
      if (kSvd) {
        if (bt.v_tv || bt.w_tv) st |= svd_load_params_tv(lane, bt, ws, b, t, true);
        st |= svd_advance(lane, n, ws, dt);
        w_mv(lane, p, n, ws.F, n, true, ws.a, ws.f);
        st |= svd_update(lane, n, p, ws);
        store_view(lane, wa.svd.m, b, row, n, ws.m);
        store_view(lane, wa.svd.a, b, row, n, ws.a);
        store_view(lane, wa.svd.dc, b, row, n, ws.dcv);
        store_view(lane, wa.svd.dr, b, row, n, ws.drv);
        store_view(lane, wa.svd.uc, b, row, nn, ws.C);
        store_view(lane, wa.svd.ur, b, row, nn, ws.R);
        store_view(lane, wa.svd.f, b, row, p, ws.f);
        if (kSpill) {
          double *sp = spill + (size_t)row * wa.spill_k;
          for (int k = lane; k < n; k += 32) {
            sp[k] = ws.m[k]; sp[n + k] = ws.dcv[k]; sp[2 * n + nn + k] = ws.a[k];
          }
          for (int k = lane; k < nn; k += 32) sp[2 * n + k] = ws.C[k];
        }
      } else {
        if (OP == kOpLoglik) w_copy(lane, n, ws.m, ws.th);  // m_{t-1}
        kf_advance(lane, n, ws, dt, ws.m, ws.C, ws.a, ws.R);
        st |= kf_update(lane, n, p, ws);
        store_view(lane, wa.kf.a, b, row, n, ws.a);
        store_view(lane, wa.kf.R, b, row, nn, ws.R);
        store_view(lane, wa.kf.f, b, row, p, ws.f);
        store_view(lane, wa.kf.Q, b, row, p * p, ws.Q);
        store_view(lane, wa.kf.m, b, row, n, ws.m);
        store_view(lane, wa.kf.C, b, row, nn, ws.C);
        if (kSpill) {
          double *sp = spill + (size_t)row * wa.spill_k;
          for (int k = lane; k < n; k += 32) { sp[k] = ws.m[k]; sp[n + nn + k] = ws.a[k]; }
          for (int k = lane; k < nn; k += 32) { sp[n + k] = ws.C[k]; sp[2 * n + nn + k] = ws.R[k]; }
        }
        if (OP == kOpLoglik) {
          // KalmanFilter.logLikelihood (KalmanFilter.scala:175-183): N(m_t; G m_{t-1}, W dt)
          double v;
          if (wa.ll_transition) {  // only when asked for: a rank-deficient W is fine otherwise
            w_mv(lane, n, n, ws.G, n, false, ws.th, ws.v3);
            for (int k = lane; k < nn; k += 32) ws.t3[k] = ws.W[k] * dt;
            __syncwarp();
            st |= w_mvn_logpdf(lane, n, ws, ws.m, ws.v3, ws.t3, v);
            ll_tr = (t == 0) ? v : ll_tr + v;
          }
          // conditionalLikelihood (:138-153)
          int *obs = ws.iscr + kObsOff;
          const int po = observed(lane, p, ws.yrow, obs);
          if (po == 1) {
            const int o = obs[0];
            const double sd = sqrt(ws.Q[o + o * p]);
            const double dd = (ws.yrow[o] - ws.f[o]) / sd;
            ll_in += -dd * dd / 2.0 - log(sqrt(2.0 * 3.141592653589793) * sd);
          } else if (po > 1) {
            if (lane < po) { ws.v3[lane] = ws.f[obs[lane]]; ws.v4[lane] = ws.yrow[obs[lane]]; }
            for (ElemIter it(lane, po, po); it.ok(); it.next())
              ws.t3[it.i + it.j * po] = ws.Q[obs[it.i] + obs[it.j] * p];
            __syncwarp();
            st |= w_mvn_logpdf(lane, po, ws, ws.v4, ws.v3, ws.t3, v);
            ll_in += v;
          }
          __syncwarp();
        }
      }
      __syncwarp();
    }
  }

  if (OP == kOpLoglik) {
    if (lane == 0) {
      if (wa.ll_transition) wa.ll_transition[b] = ll_tr;
      if (wa.ll_innov) wa.ll_innov[b] = ll_in;
    }
    {  // last filtered state only (bdlm_kf_filter_last): one row per series
      store_view(lane, wa.last_m, b, 0, n, ws.m);
      store_view(lane, wa.last_C, b, 0, nn, ws.C);
    }
  }

  // ------------------------------------------------------------------ backward passes
  if (OP == kOpSmooth || OP == kOpFilterSmooth) {
    // Smoothing.backwardsSmoother (Smoothing.scala:57-64)
    if (OP == kOpSmooth) {
      load_model(lane, bt, ws, b, 0, true);  // no forward pass ran: G, F are not in smem yet
      load_view(lane, wa.kf.m, b, rows - 1, n, ws.m);
      load_view(lane, wa.kf.C, b, rows - 1, nn, ws.C);
      __syncwarp();
    }
    w_copy(lane, n, ws.m, ws.th);
    w_copy(lane, nn, ws.C, ws.Sm);
    store_view(lane, wa.s, b, rows - 1, n, ws.th);
    store_view(lane, wa.S, b, rows - 1, nn, ws.Sm);
    const bool textbook = (bt.compat & BDLM_TEXTBOOK_SMOOTHER) != 0;
    for (int r = rows - 2; r >= 0; --r) {
      const int tobs = r + 1 - ki;
      load_model(lane, bt, ws, b, tobs, false);
      if (OP == kOpFilterSmooth) {
        const double *sp = spill + (size_t)r * wa.spill_k, *sp1 = sp + wa.spill_k;
        for (int k = lane; k < n; k += 32) { ws.m[k] = sp[k]; ws.a[k] = sp1[n + nn + k]; }
        for (int k = lane; k < nn; k += 32) { ws.C[k] = sp[n + k]; ws.R[k] = sp1[2 * n + nn + k]; }
        __syncwarp();
      } else {
        load_view(lane, wa.kf.m, b, r, n, ws.m);
        load_view(lane, wa.kf.C, b, r, nn, ws.C);
        if (wa.kf.a.ptr && wa.kf.R.ptr) {
          load_view(lane, wa.kf.a, b, r + 1, n, ws.a);
          load_view(lane, wa.kf.R, b, r + 1, nn, ws.R);
          __syncwarp();
        } else {
          __syncwarp();
          const double dt = dt_at(bt, b, tobs);
          kf_advance(lane, n, ws, dt, ws.m, ws.C, ws.a, ws.R);
        }
      }
      st |= smoothing_gain(lane, n, ws, ws.C, ws.R);  // B in t3
      for (int k = lane; k < n; k += 32) ws.v1[k] = ws.th[k] - ws.a[k];
      for (int k = lane; k < nn; k += 32) ws.t1[k] = ws.R[k] - ws.Sm[k];
      __syncwarp();
      w_mv(lane, n, n, ws.t3, n, false, ws.v1, ws.v2);
      w_mm(lane, n, n, n, ws.t3, n, false, ws.t1, n, false, ws.t2, n);
      w_mm(lane, n, n, n, ws.t2, n, false, ws.t3, n, textbook, ws.t4, n);
      for (int k = lane; k < n; k += 32) ws.th[k] = ws.m[k] + ws.v2[k];
      for (int k = lane; k < nn; k += 32) ws.Sm[k] = ws.C[k] - ws.t4[k];
      __syncwarp();
      store_view(lane, wa.s, b, r, n, ws.th);
      store_view(lane, wa.S, b, r, nn, ws.Sm);
    }
  }

  if (OP == kOpFfbs) {
    // Smoothing.sample (Smoothing.scala:114-122), initialise (:105-109), step (:74-103)
    load_z(lane, wa, b, rows - 1, rows, n, ws.v3);
    __syncwarp();
    st |= mvn_eig_draw(lane, n, ws, ws.m, ws.C, ws.v3, ws.th);
    store_view(lane, wa.theta, b, rows - 1, n, ws.th);
    for (int r = rows - 2; r >= 0; --r) {
      const int tobs = r + 1 - ki;
      load_model(lane, bt, ws, b, tobs, false);
      const double dt = dt_at(bt, b, tobs);
      const double *sp = spill + (size_t)r * wa.spill_k, *sp1 = sp + wa.spill_k;
      for (int k = lane; k < n; k += 32) { ws.m[k] = sp[k]; ws.a[k] = sp1[n + nn + k]; }
      for (int k = lane; k < nn; k += 32) { ws.C[k] = sp[n + k]; ws.R[k] = sp1[2 * n + nn + k]; }
      load_z(lane, wa, b, r, rows, n, ws.v3);
      if (bt.w_tv) {  // W of the transition r -> r + 1 (DlmFsvSystem.scala:155-163)
        PView wt = bt.W;
        wt.ptr += (int64_t)tobs * bt.W_sr;
        load_pview(lane, wt, b, nn, ws.W);
      }
      __syncwarp();
      st |= smoothing_gain(lane, n, ws, ws.C, ws.R);  // B in t3
      for (int k = lane; k < n; k += 32) ws.v1[k] = ws.th[k] - ws.a[k];
      __syncwarp();
      w_mv(lane, n, n, ws.t3, n, false, ws.v1, ws.v2);
      for (int k = lane; k < n; k += 32) ws.a[k] = ws.m[k] + ws.v2[k];  // h (a is free now)
      // diff = I - B G ; cov = (diff C) diff^T + ((B W) dt) B^T  (:93-94)
      w_mm(lane, n, n, n, ws.t3, n, false, ws.G, n, false, ws.t1, n);
      for (ElemIter it(lane, n, n); it.ok(); it.next())
        ws.t1[it.i + it.j * n] = ((it.i == it.j) ? 1.0 : 0.0) - ws.t1[it.i + it.j * n];
      __syncwarp();
      w_mm(lane, n, n, n, ws.t1, n, false, ws.C, n, false, ws.t2, n);
      w_mm(lane, n, n, n, ws.t2, n, false, ws.t1, n, true, ws.t4, n);
      w_mm(lane, n, n, n, ws.t3, n, false, ws.W, n, false, ws.t2, n);
      for (int k = lane; k < nn; k += 32) ws.t2[k] = ws.t2[k] * dt;
      __syncwarp();
      w_mm(lane, n, n, n, ws.t2, n, false, ws.t3, n, true, ws.t5, n);
      for (int k = lane; k < nn; k += 32) ws.t4[k] = ws.t4[k] + ws.t5[k];
      __syncwarp();
      for (ElemIter it(lane, n, n); it.ok(); it.next())  // (cov + cov^T) / 2  (:95)
        ws.R[it.i + it.j * n] = (ws.t4[it.i + it.j * n] + ws.t4[it.j + it.i * n]) / 2.0;
      __syncwarp();
      st |= mvn_eig_draw(lane, n, ws, ws.a, ws.R, ws.v3, ws.th);
      store_view(lane, wa.theta, b, r, n, ws.th);
    }
  }

  if (OP == kOpSvdFfbs) {
    // SvdSampler.sample (SvdSampler.scala:54-60), initialise (:38-45), step (:15-36)
    load_z(lane, wa, b, rows - 1, rows, n, ws.v3);
    for (ElemIter it(lane, n, n); it.ok(); it.next())
      ws.t1[it.i + it.j * n] = ws.C[it.i + it.j * n] * ws.dcv[it.j];
    __syncwarp();
    w_mv(lane, n, n, ws.t1, n, false, ws.v3, ws.v2);
    for (int k = lane; k < n; k += 32) ws.th[k] = ws.m[k] + ws.v2[k];
    __syncwarp();
    store_view(lane, wa.theta, b, rows - 1, n, ws.th);
    for (int r = rows - 2; r >= 0; --r) {
      const int tobs = r + 1 - ki;
      load_model(lane, bt, ws, b, tobs, false);
      const double *sp = spill + (size_t)r * wa.spill_k, *sp1 = sp + wa.spill_k;
      for (int k = lane; k < n; k += 32) {
        ws.m[k] = sp[k]; ws.dcv[k] = sp[n + k]; ws.a[k] = sp1[2 * n + nn + k];
      }
      for (int k = lane; k < nn; k += 32) ws.C[k] = sp[2 * n + k];
      load_z(lane, wa, b, r, rows, n, ws.v3);
      __syncwarp();
      // W_t: the state of row r is stepped with sqrtSvd(W) of observation r (DlmFsvSystem.scala:193-201)
      if (bt.w_tv) st |= svd_load_params_tv(lane, bt, ws, b, tobs, false);
      w_mm(lane, n, n, n, ws.Wsq, n, false, ws.G, n, false, ws.t1, n);
      w_mm(lane, n, n, n, ws.t1, n, false, ws.C, n, false, ws.t2, n);
      for (ElemIter it(lane, n, n); it.ok(); it.next()) {
        ws.stk[it.i + it.j * 2 * n] = ws.t2[it.i + it.j * n];
        ws.stk[n + it.i + it.j * 2 * n] = (it.i == it.j) ? 1.0 / ws.dcv[it.i] : 0.0;
      }
      __syncwarp();
      st |= w_jacobi_svd(lane, 2 * n, n, ws.stk, ws.t3, ws.scr, ws.iscr, ws.v1, ws.t4);
      w_mm(lane, n, n, n, ws.C, n, false, ws.t4, n, false, ws.t5, n);  // uh
      for (int k = lane; k < n; k += 32) ws.v1[k] = 1.0 / ws.v1[k];    // dh
      __syncwarp();
      w_mm(lane, n, n, n, ws.G, n, true, ws.Wsq, n, true, ws.t1, n);
      w_mm(lane, n, n, n, ws.t1, n, false, ws.Wsq, n, false, ws.t2, n);  // gWinv
      for (ElemIter it(lane, n, n); it.ok(); it.next())
        ws.t3[it.i + it.j * n] = ws.v1[it.i] * ws.t5[it.j + it.i * n];  // du
      __syncwarp();
      w_mm(lane, n, n, n, ws.t3, n, true, ws.t3, n, false, ws.t4, n);
      w_mm(lane, n, n, n, ws.t4, n, false, ws.t2, n, false, ws.t6, n);
      for (int k = lane; k < n; k += 32) ws.v2[k] = ws.th[k] - ws.a[k];
      __syncwarp();
      w_mv(lane, n, n, ws.t6, n, false, ws.v2, ws.v4);
      for (int k = lane; k < n; k += 32) ws.v4[k] = ws.m[k] + ws.v4[k];  // h
      for (ElemIter it(lane, n, n); it.ok(); it.next())
        ws.t1[it.i + it.j * n] = ws.t5[it.i + it.j * n] * ws.v1[it.j];
      __syncwarp();
      w_mv(lane, n, n, ws.t1, n, false, ws.v3, ws.v2);
      for (int k = lane; k < n; k += 32) ws.th[k] = ws.v4[k] + ws.v2[k];
      __syncwarp();
      store_view(lane, wa.theta, b, r, n, ws.th);
    }
  }

  if ((OP == kOpFfbs || OP == kOpSvdFfbs) &&
      (wa.stats.ssy.ptr || wa.stats.ny.ptr || wa.stats.ssw.ptr || wa.stats.scatter.ptr)) {
    __threadfence_block();
    __syncwarp();
    gibbs_stats(lane, bt, ws, wa.theta, wa.stats, b);
  }

  if (bt.status && lane == 0) {
    const double *chk =
        (OP == kOpFilter || OP == kOpLoglik || OP == kOpSvdFilter) ? ws.m : ws.th;
    bool finite = true;
    for (int k = 0; k < n; ++k) finite = finite && isfinite(chk[k]);
    if (!finite) st |= BDLM_ST_NONFINITE;
    bt.status[b] = st;
  }
}

// =====================================================================================
// FOUR SERIES PER WARP for the SVD path with n, p <= 8 (BASELINE config 4: n = p = 8).
//
// ncu on warp_kernel<kOpSvdFfbs, 8, 8> (profiles/r1_warp_svd_ffbs_full.txt): 7.8 warps per
// issue-active cycle wait on shared memory (short scoreboard), FP64 pipe 12 % busy.  The time
// goes into the three one-sided Jacobi SVDs per step (stacks of <= 16 x 8): their dot products
// are 16-long serial chains through shared memory on 12 of 32 lanes, with four __syncwarp per
// round.  Here a warp owns FOUR series: everything around the SVDs still runs one series after
// the other on all 32 lanes (the same code as above, so bit-identical), but the SVDs of the
// four series run TOGETHER, one octet of lanes per series, lane j holding column j of U
// (16 rows) and of V (8 rows) in registers; partners exchange columns with width-8 shuffles.
// No shared-memory traffic and no barrier inside a sweep, all 32 lanes busy.

constexpr int kQuad = 4;     // series per warp
__host__ __device__ inline bool svd4_shared_params(const Batch &bt) {
  return bt.V.sb == 0 && bt.W.sb == 0 && !bt.v_tv && !bt.w_tv;
}
constexpr int kOctRows = 16; // max rows of a stacked matrix: (p + n) or 2n with n, p <= 8
constexpr int kOctN = 8;

// One-sided Jacobi SVD (oracle jacobi_svd) of this octet's r x n matrix U (column-major, leading
// dimension r; nullptr = nothing to do for this series).  Results to shared memory: sv[n]
// descending, Vout (n x n) ordered + sign-normalised right singular vectors.  All 32 lanes must
// call it; returns the octet's status (uniform within the octet).  Rows r..15 are zero padding:
// they add exact zeros to the sums, which leaves every partial sum bit-identical.
__device__ __noinline__ int oct_jacobi_svd(int lane, int n, int r, const double *U, double *sv,
                                           double *Vout) {
  const int j = lane & 7;
  const bool col = U != nullptr && j < n;
  double u[kOctRows], v[kOctN];
#pragma unroll
  for (int i = 0; i < kOctRows; ++i) u[i] = (col && i < r) ? U[i + j * r] : 0.0;
#pragma unroll
  for (int i = 0; i < kOctN; ++i) v[i] = (i == j) ? 1.0 : 0.0;
  const unsigned octmask = 0xffu << (lane & 24);
  const int m = (n + 1) & ~1;
  bool conv = (n == 1) || U == nullptr;
  for (int sweep = 0; sweep < kJacobiMaxSweeps && n > 1; ++sweep) {
    bool rotated = false;
    for (int round = 0; round < m - 1; ++round) {
      const int q = col ? rr_partner(n, round, j) : -1;
      const int src = q < 0 ? j : q;
      const bool low = j < src;  // this lane holds column p (the smaller index) of the pair
      // every lane: |own column|^2 and own . partner; the partner's norm arrives by shuffle
      // (it sums the same squares in the same order, so alpha / beta are the oracle's bits)
      double own = 0.0, gamma = 0.0;
      double w[kOctRows], vw[kOctN];
#pragma unroll
      for (int i = 0; i < kOctRows; ++i) {
        w[i] = __shfl_sync(FULL, u[i], src, 8);
        const double sq = u[i] * u[i], pq = u[i] * w[i];
        own = (i == 0) ? sq : own + sq;
        gamma = (i == 0) ? pq : gamma + pq;
      }
      const double other = __shfl_sync(FULL, own, src, 8);
      const double alpha = low ? own : other, beta = low ? other : own;
#pragma unroll
      for (int i = 0; i < kOctN; ++i) vw[i] = __shfl_sync(FULL, v[i], src, 8);
      const bool rot = q >= 0 && (gamma * gamma > kJacobiThr2 * (alpha * beta));
      if (rot) {
        double c, sn;
        sym_rot(alpha, beta, gamma, c, sn);
        // lower-index lane: c*up - s*uq; higher: s*up + c*uq.  Both are own' = c*own + s'*partner
        // with s' = -+s (a - b == a + (-b) and (-s)*w == -(s*w) exactly; + commutes), so the two
        // lanes of a pair run ONE instruction stream instead of two divergent ones.
        const double sp = low ? -sn : sn;
#pragma unroll
        for (int i = 0; i < kOctRows; ++i) u[i] = c * u[i] + sp * w[i];
#pragma unroll
        for (int i = 0; i < kOctN; ++i) v[i] = c * v[i] + sp * vw[i];
      }
      rotated = rotated || rot;
    }
    const unsigned ball = __ballot_sync(FULL, rotated);
    if ((ball & octmask) == 0) conv = true;  // this series saw a sweep without a rotation
    if (ball == 0) break;                    // every series of the warp has converged
  }
  // singular values = column norms, stable descending order; sign rule of order_and_sign
  double acc = 0.0;
#pragma unroll
  for (int i = 0; i < kOctRows; ++i) {
    const double sq = u[i] * u[i];
    acc = (i == 0) ? sq : acc + sq;
  }
  const double nrm = sqrt(acc);
  int rank = 0;
#pragma unroll
  for (int k = 0; k < kOctN; ++k) {
    const double nk = __shfl_sync(FULL, nrm, k, 8);
    if (k < n) rank += ((nk > nrm) || (nk == nrm && k < j)) ? 1 : 0;
  }
  if (col) {
    int im = 0;
    double best = fabs(v[0]);
#pragma unroll
    for (int i = 1; i < kOctN; ++i) {
      const double a = fabs(v[i]);
      if (i < n && a > best) { best = a; im = i; }
    }
    double vim = v[0];
#pragma unroll
    for (int i = 1; i < kOctN; ++i) vim = (im == i) ? v[i] : vim;
    const bool flip = vim < 0.0;
    sv[rank] = nrm;
#pragma unroll
    for (int i = 0; i < kOctN; ++i)
      if (i < n) Vout[i + rank * n] = flip ? -v[i] : v[i];
  }
  __syncwarp();
  return conv ? 0 : BDLM_ST_NOTCONVERGED;
}

// svd_advance split around its SVD: pre builds the stack, the joint SVD writes (drv, R).
__device__ __forceinline__ void svd_advance_pre(int lane, int n, const Ws &ws, double dt) {
  if (dt == 0.0) {
    for (int k = lane; k < n; k += 32) { ws.a[k] = ws.m[k]; ws.drv[k] = ws.dcv[k]; }
    for (int k = lane; k < n * n; k += 32) ws.R[k] = ws.C[k];
    __syncwarp();
    return;
  }
  w_mv(lane, n, n, ws.G, n, false, ws.m, ws.a);
  for (ElemIter it(lane, n, n); it.ok(); it.next())
    ws.t1[it.i + it.j * n] = ws.dcv[it.i] * ws.C[it.j + it.i * n];
  __syncwarp();
  w_mm(lane, n, n, n, ws.t1, n, false, ws.G, n, true, ws.t2, n);
  const double sq = sqrt(dt);
  for (ElemIter it(lane, n, n); it.ok(); it.next()) {
    ws.stk[it.i + it.j * 2 * n] = ws.t2[it.i + it.j * n];
    ws.stk[n + it.i + it.j * 2 * n] = ws.W[it.i + it.j * n] * sq;
  }
  __syncwarp();
}

// svd_update split around its SVD.  pre returns po (0 = all missing: state copied, no SVD).
__device__ __forceinline__ int svd_update_pre(int lane, int n, int p, const Ws &ws) {
  int *obs = ws.iscr + kObsOff;
  const int po = observed(lane, p, ws.yrow, obs);
  if (po == 0) {
    for (int k = lane; k < n; k += 32) { ws.m[k] = ws.a[k]; ws.dcv[k] = ws.drv[k]; }
    for (int k = lane; k < n * n; k += 32) ws.C[k] = ws.R[k];
    __syncwarp();
    return 0;
  }
  double *Fm = ws.t1, *Vm = ws.t2;
  for (ElemIter it(lane, n, po); it.ok(); it.next()) Fm[it.i + it.j * n] = ws.F[it.i + obs[it.j] * n];
  for (ElemIter it(lane, po, po); it.ok(); it.next())
    Vm[it.i + it.j * po] = ws.V[obs[it.i] + obs[it.j] * p];
  __syncwarp();
  w_mv(lane, po, n, Fm, n, true, ws.a, ws.v1);  // fm
  w_mm(lane, po, po, n, Vm, po, false, Fm, n, true, ws.t3, po);
  w_mm(lane, po, n, n, ws.t3, po, false, ws.R, n, false, ws.t4, po);
  const int r = po + n;
  for (ElemIter it(lane, r, n); it.ok(); it.next()) {
    const int i = it.i, j = it.j;
    ws.stk[i + j * r] = (i < po) ? ws.t4[i + j * po]
                                 : ((i - po == j) ? 1.0 / ws.drv[j] : 0.0);
  }
  if (lane < po) ws.v1[lane] = ws.yrow[obs[lane]] - ws.v1[lane];  // e
  __syncwarp();
  return po;
}

// Second half of svd_update.  The shared temporaries were overwritten by the other series'
// phases in between, so the observed-component selection (Fm, Vm) and the innovation e are
// rebuilt -- the same operations on the same inputs, hence the same bits.  sS / sV: singular
// values and right vectors the joint SVD left for this series.
__device__ __forceinline__ void svd_update_post(int lane, int n, int p, const Ws &ws,
                                                const double *sS, const double *sV) {
  int *obs = ws.iscr + kObsOff;
  const int po = observed(lane, p, ws.yrow, obs);
  double *Fm = ws.t1, *Vm = ws.t2;
  for (ElemIter it(lane, n, po); it.ok(); it.next()) Fm[it.i + it.j * n] = ws.F[it.i + obs[it.j] * n];
  for (ElemIter it(lane, po, po); it.ok(); it.next())
    Vm[it.i + it.j * po] = ws.V[obs[it.i] + obs[it.j] * p];
  __syncwarp();
  w_mv(lane, po, n, Fm, n, true, ws.a, ws.v1);  // fm
  if (lane < po) ws.v1[lane] = ws.yrow[obs[lane]] - ws.v1[lane];  // e
  __syncwarp();
  w_mm(lane, n, n, n, ws.R, n, false, sV, n, false, ws.C, n);  // uc = ur * V
  w_mm(lane, n, po, po, Fm, n, false, Vm, po, true, ws.t3, n);
  w_mm(lane, n, po, po, ws.t3, n, false, Vm, po, false, ws.t4, n);  // fv
  for (int k = lane; k < n; k += 32) ws.dcv[k] = 1.0 / sS[k];
  __syncwarp();
  for (ElemIter it(lane, n, n); it.ok(); it.next())
    ws.t3[it.i + it.j * n] = ws.dcv[it.i] * ws.C[it.j + it.i * n];  // X = diag(dc) uc^T
  __syncwarp();
  w_mm(lane, n, n, n, ws.t3, n, true, ws.t3, n, false, ws.t5, n);
  w_mm(lane, n, n, po, ws.t5, n, false, ws.t4, n, false, ws.t6, n);  // gain
  w_mv(lane, n, po, ws.t6, n, false, ws.v1, ws.v3);
  for (int k = lane; k < n; k += 32) ws.m[k] = ws.a[k] + ws.v3[k];
  __syncwarp();
}

// NP > 0: n = p = NP known at compile time (BASELINE config 4 is n = p = 8): the element loops of
// the per-series phases fold their index arithmetic (they were 3/4 integer instructions).
template <int OP, int NP>
__global__ void __launch_bounds__(32)  // (32, 9) caps ptxas at 168 registers -> spills, 16 % slower
svd4_kernel(const WarpArgs wa, const int shared_doubles, const int series_doubles) {
  extern __shared__ double smem[];
  const Batch &bt = wa.bt;
  const int lane = threadIdx.x;
  const int64_t b0 = (int64_t)blockIdx.x * kQuad;
  if (b0 >= bt.B) return;
  const int n = NP > 0 ? NP : bt.n, p = NP > 0 ? NP : bt.p;
  const int nn = n * n, T = bt.T, ki = bt.keep_init, rows = T + ki;
  const int oct = lane >> 3;
  constexpr bool kSpill = OP == kOpSvdFfbs;
  const bool shared_params = svd4_shared_params(bt);
  // series s of this warp: shared temporaries + its own state slice; series past the end of the
  // batch are skipped
  struct Slot { Ws ws; double *sV, *sS; };
  auto slot = [&](int s) {
    Slot q;
    q.ws = Ws::svd4(smem, smem + shared_doubles + (size_t)s * series_doubles, n, p, shared_params, q.sV, q.sS);
    return q;
  };
  auto live = [&](int s) { return b0 + s < bt.B; };
  const Slot mine = slot(oct);
  const bool mine_live = live(oct);
  // The series loops are run-time loops on purpose: unrolled four times (with the SVD inlined at
  // its three call sites) the kernel was 87.7 k SASS instructions and ncu showed 1.8 warps per
  // issue-active cycle stalled on instruction fetch.  Status bits are kept per octet (st_mine =
  // the status of this lane's own series).
  int st_mine = 0;
  auto fold_status = [&](int so) { st_mine |= so; };
  auto add_status = [&](int s, int bits) { if (oct == s) st_mine |= bits; };
  {  // the model is shared by the batch: one copy per warp
    const Ws ws = mine.ws;
    load_model(lane, bt, ws, b0, 0, true);  // (svd4 is only chosen for batch-shared F, G, dt)
  }

  // ---- initial state: transformParams (SvdFilter.scala:232-236) + initialiseState (:83-95);
  // once per series, generic routines
#pragma unroll 1
  for (int s = 0; s < kQuad; ++s) {
    if (!live(s)) continue;
    const Ws ws = slot(s).ws;
    const int64_t b = b0 + s;
    load_pview(lane, bt.W, b, nn, ws.W);
    load_pview(lane, bt.V, b, p * p, ws.V);
    load_pview(lane, bt.m0, b, n, ws.m);
    load_pview(lane, bt.C0, b, nn, ws.C);
    __syncwarp();
    add_status(s, w_sqrt_svd(lane, p, ws, ws.V, true, ws.t5));
    w_copy(lane, p * p, ws.t5, ws.V);
    add_status(s, w_sqrt_svd(lane, n, ws, ws.W, false, ws.Wsq));
    if (bt.compat & BDLM_SVD_CONSISTENT_W) w_copy(lane, nn, ws.Wsq, ws.W);
    w_copy(lane, nn, ws.C, ws.stk);
    add_status(s, w_jacobi_svd(lane, n, n, ws.stk, ws.t3, ws.scr, ws.iscr, ws.v1, ws.t4));
    for (int k = lane; k < n; k += 32) ws.dcv[k] = sqrt(ws.v1[k]);
    w_copy(lane, nn, ws.t4, ws.C);
    if (ki) {
      w_mv(lane, p, n, ws.F, n, true, ws.m, ws.f);
      store_view(lane, wa.svd.m, b, 0, n, ws.m);
      store_view(lane, wa.svd.a, b, 0, n, ws.m);
      store_view(lane, wa.svd.dc, b, 0, n, ws.dcv);
      store_view(lane, wa.svd.dr, b, 0, n, ws.dcv);
      store_view(lane, wa.svd.uc, b, 0, nn, ws.C);
      store_view(lane, wa.svd.ur, b, 0, nn, ws.C);
      store_view(lane, wa.svd.f, b, 0, p, ws.f);
      if (kSpill) {  // [m, dc, uc, a]
        double *spill = wa.spill + (size_t)b * rows * wa.spill_k;
        for (int k = lane; k < n; k += 32) {
          spill[k] = ws.m[k]; spill[n + k] = ws.dcv[k]; spill[2 * n + nn + k] = ws.m[k];
        }
        for (int k = lane; k < nn; k += 32) spill[2 * n + k] = ws.C[k];
      }
    }
    __syncwarp();
  }

  // ---- forward filter
  for (int t = 0; t < T; ++t) {
    const int64_t row = t + ki;
    const double dt = dt_at(bt, b0, t);
    load_model(lane, bt, mine.ws, b0, t, false);  // no-op unless F or G vary with t
#pragma unroll 1
    for (int s = 0; s < kQuad; ++s)
      if (live(s)) {
        if (bt.v_tv || bt.w_tv) add_status(s, svd_load_params_tv(lane, bt, slot(s).ws, b0 + s, t, true));
        svd_advance_pre(lane, n, slot(s).ws, dt);
      }
    if (dt != 0.0)  // the four time updates' SVDs together: stack (2n x n) -> (drv, R)
      fold_status(oct_jacobi_svd(lane, n, 2 * n, mine_live ? mine.ws.stk : nullptr, mine.ws.drv,
                                 mine.ws.R));
    int po_mine = 0;
#pragma unroll 1
    for (int s = 0; s < kQuad; ++s) {
      if (!live(s)) continue;
      const Ws ws = slot(s).ws;
      load_cview(lane, bt.y, b0 + s, t, p, ws.yrow);
      __syncwarp();
      w_mv(lane, p, n, ws.F, n, true, ws.a, ws.f);
      const int po = svd_update_pre(lane, n, p, ws);
      if (oct == s) po_mine = po;
    }
    // the four measurement updates' SVDs: stack ((po + n) x n) -> (sS, sV)
    fold_status(oct_jacobi_svd(lane, n, po_mine + n, po_mine > 0 ? mine.ws.stk : nullptr, mine.sS,
                               mine.sV));
#pragma unroll 1
    for (int s = 0; s < kQuad; ++s) {
      if (!live(s)) continue;
      const Slot q = slot(s);
      const Ws &ws = q.ws;
      const int64_t b = b0 + s;
      const int po = __shfl_sync(FULL, po_mine, s * 8);
      if (po > 0) {
        load_cview(lane, bt.y, b, t, p, ws.yrow);
        __syncwarp();
        svd_update_post(lane, n, p, ws, q.sS, q.sV);
      }
      store_view(lane, wa.svd.m, b, row, n, ws.m);
      store_view(lane, wa.svd.a, b, row, n, ws.a);
      store_view(lane, wa.svd.dc, b, row, n, ws.dcv);
      store_view(lane, wa.svd.dr, b, row, n, ws.drv);
      store_view(lane, wa.svd.uc, b, row, nn, ws.C);
      store_view(lane, wa.svd.ur, b, row, nn, ws.R);
      store_view(lane, wa.svd.f, b, row, p, ws.f);
      if (kSpill) {
        double *sp = wa.spill + ((size_t)b * rows + row) * wa.spill_k;
        for (int k = lane; k < n; k += 32) {
          sp[k] = ws.m[k]; sp[n + k] = ws.dcv[k]; sp[2 * n + nn + k] = ws.a[k];
        }
        for (int k = lane; k < nn; k += 32) sp[2 * n + k] = ws.C[k];
      }
      __syncwarp();
    }
  }

  // ---- backward sampler: SvdSampler.sample (SvdSampler.scala:54-60), initialise (:38-45),
  // step (:15-36)
  if (OP == kOpSvdFfbs) {
#pragma unroll 1
    for (int s = 0; s < kQuad; ++s) {
      if (!live(s)) continue;
      const Ws ws = slot(s).ws;
      const int64_t b = b0 + s;
      load_z(lane, wa, b, rows - 1, rows, n, ws.v3);
      for (ElemIter it(lane, n, n); it.ok(); it.next())
        ws.t1[it.i + it.j * n] = ws.C[it.i + it.j * n] * ws.dcv[it.j];
      __syncwarp();
      w_mv(lane, n, n, ws.t1, n, false, ws.v3, ws.v2);
      for (int k = lane; k < n; k += 32) ws.th[k] = ws.m[k] + ws.v2[k];
      __syncwarp();
      store_view(lane, wa.theta, b, rows - 1, n, ws.th);
      __syncwarp();
    }
    for (int r = rows - 2; r >= 0; --r) {
      const int tobs = r + 1 - ki;
      load_model(lane, bt, mine.ws, b0, tobs, false);
#pragma unroll 1
      for (int s = 0; s < kQuad; ++s) {
        if (!live(s)) continue;
        const Ws ws = slot(s).ws;
        const int64_t b = b0 + s;
        const double *sp = wa.spill + ((size_t)b * rows + r) * wa.spill_k, *sp1 = sp + wa.spill_k;
        for (int k = lane; k < n; k += 32) {
          ws.m[k] = sp[k]; ws.dcv[k] = sp[n + k]; ws.a[k] = sp1[2 * n + nn + k];
        }
        for (int k = lane; k < nn; k += 32) ws.C[k] = sp[2 * n + k];
        __syncwarp();
        if (bt.w_tv) add_status(s, svd_load_params_tv(lane, bt, ws, b, tobs, false));
        w_mm(lane, n, n, n, ws.Wsq, n, false, ws.G, n, false, ws.t1, n);
        w_mm(lane, n, n, n, ws.t1, n, false, ws.C, n, false, ws.t2, n);
        for (ElemIter it(lane, n, n); it.ok(); it.next()) {
          ws.stk[it.i + it.j * 2 * n] = ws.t2[it.i + it.j * n];
          ws.stk[n + it.i + it.j * 2 * n] = (it.i == it.j) ? 1.0 / ws.dcv[it.i] : 0.0;
        }
        __syncwarp();
      }
      fold_status(oct_jacobi_svd(lane, n, 2 * n, mine_live ? mine.ws.stk : nullptr, mine.sS, mine.sV));
#pragma unroll 1
      for (int s = 0; s < kQuad; ++s) {
        if (!live(s)) continue;
        const Slot q = slot(s);
        const Ws &ws = q.ws;
        load_z(lane, wa, b0 + s, r, rows, n, ws.v3);
        w_mm(lane, n, n, n, ws.C, n, false, q.sV, n, false, ws.t5, n);  // uh
        for (int k = lane; k < n; k += 32) ws.v1[k] = 1.0 / q.sS[k];    // dh
        __syncwarp();
        w_mm(lane, n, n, n, ws.G, n, true, ws.Wsq, n, true, ws.t1, n);
        w_mm(lane, n, n, n, ws.t1, n, false, ws.Wsq, n, false, ws.t2, n);  // gWinv
        for (ElemIter it(lane, n, n); it.ok(); it.next())
          ws.t3[it.i + it.j * n] = ws.v1[it.i] * ws.t5[it.j + it.i * n];  // du
        __syncwarp();
        w_mm(lane, n, n, n, ws.t3, n, true, ws.t3, n, false, ws.t4, n);
        w_mm(lane, n, n, n, ws.t4, n, false, ws.t2, n, false, ws.t6, n);
        for (int k = lane; k < n; k += 32) ws.v2[k] = ws.th[k] - ws.a[k];
        __syncwarp();
        w_mv(lane, n, n, ws.t6, n, false, ws.v2, ws.v4);
        for (int k = lane; k < n; k += 32) ws.v4[k] = ws.m[k] + ws.v4[k];  // h
        for (ElemIter it(lane, n, n); it.ok(); it.next())
          ws.t1[it.i + it.j * n] = ws.t5[it.i + it.j * n] * ws.v1[it.j];
        __syncwarp();
        w_mv(lane, n, n, ws.t1, n, false, ws.v3, ws.v2);
        for (int k = lane; k < n; k += 32) ws.th[k] = ws.v4[k] + ws.v2[k];
        __syncwarp();
        store_view(lane, wa.theta, b0 + s, r, n, ws.th);
        __syncwarp();
      }
    }
    if (wa.stats.ssy.ptr || wa.stats.ny.ptr || wa.stats.ssw.ptr || wa.stats.scatter.ptr) {
      __threadfence_block();
      __syncwarp();
#pragma unroll 1
      for (int s = 0; s < kQuad; ++s)
        if (live(s)) gibbs_stats(lane, bt, slot(s).ws, wa.theta, wa.stats, b0 + s);
    }
  }

  if (bt.status && mine_live && (lane & 7) == 0) {  // first lane of each octet: its own series
    const double *chk = (OP == kOpSvdFilter) ? mine.ws.m : mine.ws.th;
    bool finite = true;
    for (int k = 0; k < n; ++k) finite = finite && isfinite(chk[k]);
    bt.status[b0 + oct] = st_mine | (finite ? 0 : BDLM_ST_NONFINITE);
  }
}

bool svd4_supported(int op, const Batch &bt) {
  // one copy of F, G and one dt per warp: per-series grids / models go to the warp-per-series kernel
  return (op == kOpSvdFilter || op == kOpSvdFfbs) && bt.n <= kOctN && bt.p <= kOctN &&
         !bt.ps_model && bt.dt_sb == 0;
}

template <int OP, int NP>
cudaError_t launch_svd4_np(const WarpArgs &wa, cudaStream_t stream) {
  const int n = wa.bt.n, p = wa.bt.p;
  const bool sp = svd4_shared_params(wa.bt);
  const int shared_doubles = (int)((Ws::svd4_shared_doubles(n, p, sp) + 1) & ~(size_t)1);
  const int series_doubles = (int)((Ws::svd4_series_doubles(n, p, sp) + 1) & ~(size_t)1);
  const size_t smem = ((size_t)shared_doubles + (size_t)kQuad * series_doubles) * sizeof(double);
  cudaError_t e = cudaFuncSetAttribute(svd4_kernel<OP, NP>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)smem);
  if (e != cudaSuccess) return e;
  const int64_t blocks = (wa.bt.B + kQuad - 1) / kQuad;
  if (blocks <= 0) return cudaSuccess;
  svd4_kernel<OP, NP><<<(unsigned)blocks, 32, smem, stream>>>(wa, shared_doubles, series_doubles);
  return cudaGetLastError();
}
template <int OP>
cudaError_t launch_svd4(const WarpArgs &wa, cudaStream_t stream) {
  if (wa.bt.n == 8 && wa.bt.p == 8) return launch_svd4_np<OP, 8>(wa, stream);
  return launch_svd4_np<OP, 0>(wa, stream);
}

template <int OP, int NT, int PT>
cudaError_t launch_dims(const WarpArgs &wa, cudaStream_t stream) {
  Ws sz(nullptr, wa.bt.n, wa.bt.p, OP);
  const int ws_doubles = (int)((sz.total + 1) & ~(size_t)1);
  // two warps per block unless their workspaces would not fit one SM's shared memory (n or p
  // close to 32: a single workspace is > 100 KB)
  const int wpb = ((size_t)2 * ws_doubles * sizeof(double) <= (size_t)200 * 1024) ? 2 : 1;
  const size_t smem = (size_t)wpb * ws_doubles * sizeof(double);
  cudaError_t e = cudaFuncSetAttribute(warp_kernel<OP, NT, PT>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  const int64_t blocks = (wa.bt.B + wpb - 1) / wpb;
  if (blocks <= 0) return cudaSuccess;
  warp_kernel<OP, NT, PT><<<(unsigned)blocks, wpb * 32, smem, stream>>>(wa, ws_doubles);
  return cudaGetLastError();
}

// Hot shapes get compile-time dimensions: (13, 1) = polynomial(1) |+| seasonal(24, 6)
// (BASELINE config 3) and (8, 8) = 8-fold outer sum of polynomial(1) (config 4).
template <int OP>
cudaError_t launch_op(const WarpArgs &wa, cudaStream_t stream) {
  constexpr bool kHot = (OP == kOpFilter || OP == kOpFilterSmooth || OP == kOpFfbs ||
                         OP == kOpSvdFilter || OP == kOpSvdFfbs);
  if (kHot && wa.bt.n == 13 && wa.bt.p == 1) return launch_dims<OP, kHot ? 13 : 0, kHot ? 1 : 0>(wa, stream);
  if (kHot && wa.bt.n == 8 && wa.bt.p == 8) return launch_dims<OP, kHot ? 8 : 0, kHot ? 8 : 0>(wa, stream);
  return launch_dims<OP, 0, 0>(wa, stream);
}

}  // namespace

size_t warp_spill_doubles_per_row(int op, int n, int p) {
  (void)p;
  if (op == kOpFilterSmooth || op == kOpFfbs) return (size_t)2 * n + 2 * n * n;
  if (op == kOpSvdFfbs) return (size_t)3 * n + n * n;
  return 0;
}

size_t warp_smem_bytes(int op, int n, int p) {
  Ws sz(nullptr, n, p, op);
  return ((sz.total + 1) & ~(size_t)1) * sizeof(double);
}

cudaError_t launch_warp(int op, const WarpArgs &wa, cudaStream_t stream) {
  if (svd4_supported(op, wa.bt))
    return op == kOpSvdFilter ? launch_svd4<kOpSvdFilter>(wa, stream)
                              : launch_svd4<kOpSvdFfbs>(wa, stream);
  switch (op) {
    case kOpFilter: return launch_op<kOpFilter>(wa, stream);
    case kOpSmooth: return launch_op<kOpSmooth>(wa, stream);
    case kOpFilterSmooth: return launch_op<kOpFilterSmooth>(wa, stream);
    case kOpFfbs: return launch_op<kOpFfbs>(wa, stream);
    case kOpLoglik: return launch_op<kOpLoglik>(wa, stream);
    case kOpSvdFilter: return launch_op<kOpSvdFilter>(wa, stream);
    case kOpSvdFfbs: return launch_op<kOpSvdFfbs>(wa, stream);
    case kOpStats: return launch_op<kOpStats>(wa, stream);
    default: return cudaErrorInvalidValue;
  }
}

}  // namespace bdlm
