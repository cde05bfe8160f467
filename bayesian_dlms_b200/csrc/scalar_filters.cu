// scalar_filters.cu -- "next" rows of SURVEY.md section 8(f), thread-per-series kernels:
//
//   ar_kernel         scalar AR(1) / Ornstein-Uhlenbeck Kalman filter and backward sampler, the
//                     inner loop of the reference's stochastic-volatility models
//                     (FilterAr.scala:15-75, FilterOu.scala:7-71; per-step observation
//                     variances v_t).  HBM-bound: y, v in; m, C, a, R out; the sampler re-reads
//                     (m, C) and recomputes (a, R)_{t+1} from them exactly as the forward pass
//                     did, so the backward sweep moves 8*(2 + 1 + 1) bytes per step.
//   conjugate_kernel  Kalman filter with unknown scalar observation variance under an
//                     inverse-gamma prior (ConjugateFilter.scala:23-94), n <= 4, p = 1.
//
// Same arithmetic contract as the other bit-exact kernels (common.cuh): the reference's
// operations in the reference's order, no FMA.  OU needs exp(): device exp() and the JVM's
// differ in the last place, so OU parity is 1e-9 relative, AR(1) is bit exact.
#include "common.cuh"
#include "launch.h"
#include "small_steps.cuh"

namespace bdlm {

namespace {

__device__ __forceinline__ double ldv(const View &v, int64_t b, int64_t r) {
  return v.ptr[b * v.sb + r * v.sr];
}
__device__ __forceinline__ void stv(const View &v, int64_t b, int64_t r, double x) {
  if (v.ptr) st_stream(v.ptr + b * v.sb + r * v.sr, x);
}

// One-step prediction of the scalar state (FilterAr.scala:19-20, FilterOu.scala:12-16).
template <bool OU>
__device__ __forceinline__ void ar_predict(double phi, double mu, double sigma, double dt,
                                           double m, double C, double &at, double &rt) {
  if (OU) {
    const double variance = ((sigma * sigma) * (1 - exp(-2 * phi * dt))) / (2 * phi);
    at = mu + exp(-phi * dt) * (m - mu);
    rt = exp(-2 * phi * dt) * C + variance;
  } else {
    at = mu + phi * (m - mu);
    rt = phi * phi * C + sigma * sigma;
  }
}

// 8 resident blocks per SM and one step of y, v (and m, C, z on the way back) in flight per
// thread: occupancy beats per-thread prefetch depth (profiles/r1_tuning.txt, "AR(1) filter /
// FFBS": FFBS 13.1 ms at depth 1 with 8 blocks/SM asked of ptxas, 21.5 ms at depth 8 with 1).
template <bool OU, bool FFBS>
__global__ void __launch_bounds__(128, 8)
ar_kernel(const ArArgs a) {
  const int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (b >= a.B) return;
  const double phi = a.phi.ptr ? a.phi.ptr[b * a.phi.sb] : a.phi_s;
  const double mu = a.mu.ptr ? a.mu.ptr[b * a.mu.sb] : a.mu_s;
  const double sigma = a.sigma.ptr ? a.sigma.ptr[b * a.sigma.sb] : a.sigma_s;
  const int T = a.T;
  // filterUnivariate: m0 = mu, c0 = stationary variance (FilterAr.scala:40-43; the OU
  // expression is the reference's own, FilterOu.scala:36)
  double m = mu;
  double C = OU ? sigma * sigma / phi * phi : sigma * sigma / (1 - phi * phi);
  const View &om = FFBS ? a.sm : a.m, &oC = FFBS ? a.sC : a.C;
  stv(om, b, 0, m); stv(oC, b, 0, C); stv(a.a, b, 0, m); stv(a.R, b, 0, C);
  // y (and v) do not depend on the recursion: load step t + 1 before computing step t
  double ynext = (0 < T) ? ld_stream(a.y.ptr + b * a.y.sb) : 0.0;
  double vnext = (0 < T && a.v.ptr) ? ld_stream(a.v.ptr + b * a.v.sb) : 0.0;
  for (int t = 0; t < T; ++t) {
    const double y = ynext;
    const double v = a.v.ptr ? vnext : (a.v_shared ? a.v_shared[t] : a.v_s);
    const int tn = t + 1;
    if (tn < T) {
      ynext = ld_stream(a.y.ptr + b * a.y.sb + tn * a.y.sr);
      if (a.v.ptr) vnext = ld_stream(a.v.ptr + b * a.v.sb + tn * a.v.sr);
    }
    double at, rt;
    ar_predict<OU>(phi, mu, sigma, OU ? a.dt[t] : 1.0, m, C, at, rt);
    if (isnan(y)) {  // None: (at, rt, at, rt)
      m = at; C = rt;
    } else {
      const double kt = rt / (rt + v);
      const double et = y - at;
      m = at + kt * et;
      C = kt * v;
    }
    if (FFBS) {
      // spill with default policy: re-read by this thread on the way back
      a.sm.ptr[b * a.sm.sb + (t + 1) * a.sm.sr] = m;
      a.sC.ptr[b * a.sC.sb + (t + 1) * a.sC.sr] = C;
    } else {
      stv(a.m, b, t + 1, m); stv(a.C, b, t + 1, C);
    }
    stv(a.a, b, t + 1, at); stv(a.R, b, t + 1, rt);
  }
  if (!FFBS) return;
  // univariateSample: theta_T ~ N(m_T, C_T), then backStepUni down to row 0
  double th = m + sqrt(C) * ld_stream(a.z.ptr + b * a.z.sb + (int64_t)T * a.z.sr);
  stv(a.theta, b, T, th);
  const int tl = T - 1;
  double mnext = tl >= 0 ? ldv(a.sm, b, tl) : 0.0;
  double cnext = tl >= 0 ? ldv(a.sC, b, tl) : 0.0;
  double znext = tl >= 0 ? ld_stream(a.z.ptr + b * a.z.sb + tl * a.z.sr) : 0.0;
  for (int t = tl; t >= 0; --t) {
    const double mt = mnext, ct = cnext, z = znext;
    const int tn = t - 1;
    if (tn >= 0) {
      mnext = ldv(a.sm, b, tn); cnext = ldv(a.sC, b, tn);
      znext = ld_stream(a.z.ptr + b * a.z.sb + tn * a.z.sr);
    }
    const double dt = OU ? a.dt[t] : 1.0;
    double a1, r1;
    ar_predict<OU>(phi, mu, sigma, dt, mt, ct, a1, r1);  // == the forward (a, R) of row t + 1
    const double ph = OU ? exp(-phi * dt) : phi;
    const double mean = mt + (ct * ph / r1) * (th - a1);
    const double cov = ct - ((ct * ct) * (ph * ph)) / r1;
    th = mean + sqrt(cov) * z;
    stv(a.theta, b, t, th);
  }
}

// ---- conjugate filter ---------------------------------------------------------------------

template <int N>
struct ConjModel {
  double G[N * N], F[N];
};

template <int N>
__global__ void __launch_bounds__(128)
conjugate_kernel(const ConjModel<N> md, const ConjArgs a) {
  using namespace small;
  const int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (b >= a.bt.B) return;
  const Batch &bt = a.bt;
  double m[N], C[N * N], W[N * N];
#pragma unroll
  for (int k = 0; k < N; ++k) m[k] = bt.m0.ptr[b * bt.m0.sb + k * bt.m0.sk];
#pragma unroll
  for (int k = 0; k < N * N; ++k) {
    C[k] = bt.C0.ptr[b * bt.C0.sb + k * bt.C0.sk];
    W[k] = bt.W.ptr[b * bt.W.sb + k * bt.W.sk];
  }
  double shape = a.prior_shape, scale = a.prior_scale;
  int st = 0;
  auto store = [&](const View &v, int64_t row, const double *x, int K) {
    if (!v.ptr) return;
    for (int k = 0; k < K; ++k) st_stream(v.ptr + b * v.sb + row * v.sr + k * v.sk, x[k]);
  };
  // initialiseState (ConjugateFilter.scala:23-31): row 0 = (m0, C0, m0, C0, None, None), prior
  const double nanv = __longlong_as_double(0x7ff8000000000000LL);
  store(a.kf.m, 0, m, N); store(a.kf.C, 0, C, N * N);
  store(a.kf.a, 0, m, N); store(a.kf.R, 0, C, N * N);
  store(a.kf.f, 0, &nanv, 1); store(a.kf.Q, 0, &nanv, 1);
  store(a.shape, 0, &shape, 1); store(a.scale, 0, &scale, 1);
  for (int t = 0; t < bt.T; ++t) {
    const double dt = dt_at(bt, b, t);
    const double y = ld_stream(bt.y.ptr + b * bt.y.sb + t * bt.y.sr);
    double av[N], R[N * N];
    advance<N, false>(md.G, W, dt, m, C, av, R);
    const double v = scale / (shape - 1);  // meanVariance (:50-52): InverseGamma.mean
    double ft, qt, fr[N], rhs[N], K[N], D[N * N], t1[N * N], C1[N * N], kv[N], C2[N * N];
    smm<1, N, 1, true, false>(md.F, av, &ft);
    smm<1, N, N, true, false>(md.F, R, fr);
    smm<1, N, 1, false, false>(fr, md.F, &qt);
    qt = qt + v;
    const double e = y - ft;
    smm<1, N, N, true, true>(md.F, R, rhs);  // f.t * rt.t
    if (qt == 0.0) st |= BDLM_ST_SINGULAR;
#pragma unroll
    for (int i = 0; i < N; ++i) K[i] = rhs[i] / qt;
    // updateStats (:39-48)
    const double nscale = scale + (v * (e * e)) / qt;
    shape = shape + 1;
    scale = nscale;
#pragma unroll
    for (int j = 0; j < N; ++j)
#pragma unroll
      for (int i = 0; i < N; ++i) D[i + j * N] = ((i == j) ? 1.0 : 0.0) - K[i] * md.F[j];
    smm<N, N, N, false, false>(D, R, t1);
    smm<N, N, N, false, true>(t1, D, C1);
#pragma unroll
    for (int i = 0; i < N; ++i) kv[i] = K[i] * v;
    smm<N, 1, N, false, true>(kv, K, C2);
#pragma unroll
    for (int k = 0; k < N * N; ++k) C[k] = C1[k] + C2[k];
#pragma unroll
    for (int i = 0; i < N; ++i) m[i] = m[i] + K[i] * e;  // sic: previous mt, not at (:83)
    store(a.kf.a, t + 1, av, N); store(a.kf.R, t + 1, R, N * N);
    store(a.kf.f, t + 1, &ft, 1); store(a.kf.Q, t + 1, &qt, 1);
    store(a.kf.m, t + 1, m, N); store(a.kf.C, t + 1, C, N * N);
    store(a.shape, t + 1, &shape, 1); store(a.scale, t + 1, &scale, 1);
  }
  if (bt.status && st) bt.status[b] = st;
}

// ---- log-likelihoods, thread per series ------------------------------------------------------
// KalmanFilter.likelihood (transition form, KalmanFilter.scala:299-306 with logLikelihood
// :175-183) and the innovations form (conditionalLikelihood :138-153) for n <= 4, p = 1 and a
// time-invariant F, G: what Metropolis / MetropolisHastings.dlm evaluate per proposal
// (MetropolisHastings.scala:126-137,199-209).  Nothing is stored per step: the kernel reads y
// (8 B / series-step) and is bound by FP64 issue; the warp-per-series kernel it replaces for
// these shapes needs a whole warp and shared-memory round trips per series.
// Operation order = oracle_loglik / mvn_logpdf / chol_logdet (dgesv solve, dpotrf log-determinant);
// the transition density goes through small::MvnPrepared (small_steps.cuh).
template <int N>
__global__ void __launch_bounds__(128)
loglik_small_kernel(const ConjModel<N> md, const Batch bt, double *ll_transition, double *ll_innov,
                    const View last_m, const View last_C) {
  using namespace small;
  const int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (b >= bt.B) return;
  double m[N], C[N * N], W[N * N];
#pragma unroll
  for (int k = 0; k < N; ++k) m[k] = bt.m0.ptr[b * bt.m0.sb + k * bt.m0.sk];
#pragma unroll
  for (int k = 0; k < N * N; ++k) {
    C[k] = bt.C0.ptr[b * bt.C0.sb + k * bt.C0.sk];
    W[k] = bt.W.ptr[b * bt.W.sb + k * bt.W.sk];
  }
  const double V = bt.V.ptr[b * bt.V.sb];
  int st = 0;
  double ll = 0.0, li = 0.0;
  // regular grid: S = W * 1.0 at every step -> factorise once
  MvnPrepared<N> mvn;
  const bool regular = bt.dt == nullptr;
  // the transition density N(m_t; G m_{t-1}, W dt) -- and the singular / not-PD status bits a
  // rank-deficient W raises in it -- only when the caller asked for it (bdlm_kf_filter_last and
  // innovations-only calls are valid for W = diag(s2, 0))
  const bool want_tr = ll_transition != nullptr;
  if (regular && want_tr) {
    double S[N * N];
#pragma unroll
    for (int k = 0; k < N * N; ++k) S[k] = W[k] * 1.0;
    mvn.prepare(S);
  }
  double ynext = ld_stream(bt.y.ptr + b * bt.y.sb);
  for (int t = 0; t < bt.T; ++t) {
    const double y = ynext;
    if (t + 1 < bt.T) ynext = ld_stream(bt.y.ptr + b * bt.y.sb + (int64_t)(t + 1) * bt.y.sr);
    const double dt = dt_at(bt, b, t);
    double a[N], R[N * N], mu[N], f, Q;
    smm<N, N, 1, false, false>(md.G, m, mu);  // G m_{t-1}
    advance<N, false>(md.G, W, dt, m, C, a, R);
    update<N>(md.F, V, y, a, R, f, Q, m, C, st);
    if (want_tr) {
      if (!regular) {
        double S[N * N];
#pragma unroll
        for (int k = 0; k < N * N; ++k) S[k] = W[k] * dt;
        mvn.prepare(S);
      }
      st |= mvn.st;
      const double v = mvn.eval(m, mu);
      ll = (t == 0) ? v : ll + v;
    }
    if (!isnan(y)) {
      const double sd = sqrt(Q);
      const double dd = (y - f) / sd;
      li += -dd * dd / 2.0 - log(sqrt(2.0 * 3.141592653589793) * sd);
    }
  }
  if (ll_transition) ll_transition[b] = ll;
  if (ll_innov) ll_innov[b] = li;
  if (last_m.ptr)  // final filtered state (bdlm_kf_filter_last)
    for (int k = 0; k < N; ++k) last_m.ptr[b * last_m.sb + k * last_m.sk] = m[k];
  if (last_C.ptr)
    for (int k = 0; k < N * N; ++k) last_C.ptr[b * last_C.sb + k * last_C.sk] = C[k];
  if (bt.status) {
    bool finite = true;
#pragma unroll
    for (int k = 0; k < N; ++k) finite = finite && isfinite(m[k]);
    bt.status[b] = st | (finite ? 0 : BDLM_ST_NONFINITE);
  }
}

template <int N>
cudaError_t launch_ll(const Batch &bt, const double *hG, const double *hF, double *tr, double *in,
                      const View &lm, const View &lC, cudaStream_t s) {
  ConjModel<N> md;
  for (int k = 0; k < N * N; ++k) md.G[k] = hG[k];
  for (int k = 0; k < N; ++k) md.F[k] = hF[k];
  loglik_small_kernel<N><<<(unsigned)((bt.B + 127) / 128), 128, 0, s>>>(md, bt, tr, in, lm, lC);
  return cudaGetLastError();
}

template <int N>
cudaError_t launch_conj(const ConjArgs &a, const double *hG, const double *hF, cudaStream_t s) {
  ConjModel<N> md;
  for (int k = 0; k < N * N; ++k) md.G[k] = hG[k];
  for (int k = 0; k < N; ++k) md.F[k] = hF[k];
  const unsigned blocks = (unsigned)((a.bt.B + 127) / 128);
  conjugate_kernel<N><<<blocks, 128, 0, s>>>(md, a);
  return cudaGetLastError();
}

}  // namespace

cudaError_t launch_ar(const ArArgs &a, cudaStream_t stream) {
  if (a.B == 0) return cudaSuccess;
  const unsigned blocks = (unsigned)((a.B + 127) / 128);
  if (a.ou) {
    if (a.ffbs) ar_kernel<true, true><<<blocks, 128, 0, stream>>>(a);
    else ar_kernel<true, false><<<blocks, 128, 0, stream>>>(a);
  } else {
    if (a.ffbs) ar_kernel<false, true><<<blocks, 128, 0, stream>>>(a);
    else ar_kernel<false, false><<<blocks, 128, 0, stream>>>(a);
  }
  return cudaGetLastError();
}

bool loglik_small_supported(const Batch &bt) {
  return bt.p == 1 && bt.n >= 1 && bt.n <= 4 && !bt.f_tv && !bt.g_tv && !bt.v_tv && !bt.w_tv && !bt.ps_model;
}

cudaError_t launch_loglik_small(const Batch &bt, const double *hG, const double *hF,
                                double *ll_transition, double *ll_innov, const View &last_m,
                                const View &last_C, cudaStream_t stream) {
  if (bt.B == 0) return cudaSuccess;
  switch (bt.n) {
    case 1: return launch_ll<1>(bt, hG, hF, ll_transition, ll_innov, last_m, last_C, stream);
    case 2: return launch_ll<2>(bt, hG, hF, ll_transition, ll_innov, last_m, last_C, stream);
    case 3: return launch_ll<3>(bt, hG, hF, ll_transition, ll_innov, last_m, last_C, stream);
    case 4: return launch_ll<4>(bt, hG, hF, ll_transition, ll_innov, last_m, last_C, stream);
    default: return cudaErrorInvalidValue;
  }
}

bool conjugate_supported(int n, int p) { return p == 1 && n >= 1 && n <= 4; }

cudaError_t launch_conjugate(const ConjArgs &a, const double *hG, const double *hF,
                             cudaStream_t stream) {
  if (a.bt.B == 0) return cudaSuccess;
  switch (a.bt.n) {
    case 1: return launch_conj<1>(a, hG, hF, stream);
    case 2: return launch_conj<2>(a, hG, hF, stream);
    case 3: return launch_conj<3>(a, hG, hF, stream);
    case 4: return launch_conj<4>(a, hG, hF, stream);
    default: return cudaErrorInvalidValue;
  }
}

}  // namespace bdlm
