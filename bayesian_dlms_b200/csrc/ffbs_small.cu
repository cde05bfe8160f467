// ffbs_small.cu -- forward filtering backward sampling, ONE THREAD PER CHAIN, for the small models
// the reference's own Gibbs examples run (first / second order DLMs: FirstOrderDlm.scala:79-118,
// SecondOrder.scala:53-97): n <= 4, p = 1, time-invariant F and G.
//
// Smoothing.ffbs / ffbsDlm (Smoothing.scala:151-180) = KalmanFilter(adv).filter, then
// Smoothing.sample (:114-122) with Smoothing.step (:74-103) and MultivariateGaussianSvd.draw
// (MultivariateGaussianSvd.scala:13-22), plus the Gibbs sufficient statistics of the drawn path
// (Gibbs.scala:29-43,63-73; GibbsWishart.scala:22-29).  The warp-per-chain kernel (kf_warp.cu)
// spends a whole warp and shared-memory round trips on 2 x 2 matrices; here everything lives in
// registers, the Jacobi rounds are unrolled (static partner indices), and HBM sees y, z in and
// theta out plus one (m, C) spill written forwards and re-read backwards -- (a, R)_{t+1} are
// recomputed from (m_t, C_t), bit-identical to the forward values.
//
// Arithmetic mirrors oracle/bdlm_oracle.c operation for operation (jacobi_eigsym, mvn_eig_draw,
// smoothing_gain, backward_sample_impl, oracle_gibbs_stats): results are bit-identical.
#include "common.cuh"
#include "launch.h"
#include "rng.cuh"
#include "small_steps.cuh"

namespace bdlm {

namespace {

using namespace small;

template <int N>
struct FfbsModel {
  double G[N * N], F[N];
};

template <int N>
__global__ void __launch_bounds__(128)
ffbs_small_kernel(const FfbsModel<N> md, const FfbsSmallArgs a) {
  const Batch &bt = a.bt;
  const int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (b >= bt.B) return;
  const int T = bt.T, rows = T + 1;
  double m[N], C[N * N], W[N * N];
#pragma unroll
  for (int k = 0; k < N; ++k) m[k] = bt.m0.ptr[b * bt.m0.sb + k * bt.m0.sk];
#pragma unroll
  for (int k = 0; k < N * N; ++k) {
    C[k] = bt.C0.ptr[b * bt.C0.sb + k * bt.C0.sk];
    W[k] = bt.W.ptr[b * bt.W.sb + k * bt.W.sk];
  }
  double V = bt.V.ptr[b * bt.V.sb];
  // time-varying V_t / W_t (StudentTGibbs.sampleState, DlmFsvSystem.ffbs): row t of the arrays
  auto load_vw = [&](int t) {
    if (bt.v_tv) V = bt.V.ptr[b * bt.V.sb + (int64_t)t * bt.V_sr];
    if (bt.w_tv) {
      const double *wp = bt.W.ptr + b * bt.W.sb + (int64_t)t * bt.W_sr;
#pragma unroll
      for (int k = 0; k < N * N; ++k) W[k] = wp[k * bt.W.sk];
    }
  };
  int st = 0;
  auto put = [&](const View &v, int64_t row, const double *x, int K, bool stream) {
    if (!v.ptr) return;
    double *p = v.ptr + b * v.sb + row * v.sr;
    for (int k = 0; k < K; ++k) {
      if (stream) st_stream(p + k * v.sk, x[k]);
      else p[k * v.sk] = x[k];
    }
  };
  auto get = [&](const View &v, int64_t row, double *x, int K) {
    const double *p = v.ptr + b * v.sb + row * v.sr;
    for (int k = 0; k < K; ++k) x[k] = p[k * v.sk];
  };
  const double nanv = __longlong_as_double(0x7ff8000000000000LL);

  // ---- forward filter, keeping the initial state (Filter.scala:41-45)
  put(a.sm, 0, m, N, false); put(a.sC, 0, C, N * N, false);
  put(a.kf.a, 0, m, N, true); put(a.kf.R, 0, C, N * N, true);
  put(a.kf.f, 0, &nanv, 1, true); put(a.kf.Q, 0, &nanv, 1, true);
  double ynext = ld_stream(bt.y.ptr + b * bt.y.sb);
  for (int t = 0; t < T; ++t) {
    const double y = ynext;
    if (t + 1 < T) ynext = ld_stream(bt.y.ptr + b * bt.y.sb + (int64_t)(t + 1) * bt.y.sr);
    const double dt = dt_at(bt, b, t);
    double av[N], R[N * N], f, Q;
    load_vw(t);
    advance<N, false>(md.G, W, dt, m, C, av, R);
    update<N>(md.F, V, y, av, R, f, Q, m, C, st);
    put(a.sm, t + 1, m, N, false); put(a.sC, t + 1, C, N * N, false);
    put(a.kf.a, t + 1, av, N, true); put(a.kf.R, t + 1, R, N * N, true);
    put(a.kf.f, t + 1, &f, 1, true); put(a.kf.Q, t + 1, &Q, 1, true);
  }

  // ---- backward sampler: Smoothing.initialise (:105-109), then Smoothing.step (:74-103)
  auto normals = [&](int64_t row, double (&z)[N]) {
    if (a.z.ptr) {
      const double *p = a.z.ptr + b * a.z.sb + row * a.z.sr;
#pragma unroll
      for (int k = 0; k < N; ++k) z[k] = ld_stream(p + k * a.z.sk);
    } else {
      const RngKey key{a.rng_seed, a.rng_sweep};
#pragma unroll
      for (int k = 0; k < N; ++k) z[k] = philox_normal(key, a.rng_base + b, rows, (int)row, N, k);
    }
  };
  double th[N], z[N];
  normals(T, z);
  st |= eig_draw_small<N>(m, C, z, th);
  put(a.theta, T, th, N, false);
  for (int r = T - 1; r >= 0; --r) {
    const double dt = dt_at(bt, b, r);  // transition r -> r + 1 = the step into observation r
    double mr[N], Cr[N * N], a1[N], R1[N * N];
    get(a.sm, r, mr, N); get(a.sC, r, Cr, N * N);
    normals(r, z);
    load_vw(r);  // W of the transition r -> r + 1 (DlmFsvSystem.scala:155-163)
    advance<N, false>(md.G, W, dt, mr, Cr, a1, R1);  // == the forward (a, R) of row r + 1
    // smoothing_gain: B = (R1^T \ (G C^T))^T
    double rhs[N * N], At[N * N], Bg[N * N], d[N], t1[N * N], t2[N * N], h[N], D[N * N],
        Hm[N * N], Hs[N * N], tv[N];
    smm<N, N, N, false, true>(md.G, Cr, rhs);
#pragma unroll
    for (int j = 0; j < N; ++j)
#pragma unroll
      for (int i = 0; i < N; ++i) At[i + j * N] = R1[j + i * N];
    st |= lu_solve<N, N>(At, rhs);
#pragma unroll
    for (int j = 0; j < N; ++j)
#pragma unroll
      for (int i = 0; i < N; ++i) Bg[i + j * N] = rhs[j + i * N];
#pragma unroll
    for (int i = 0; i < N; ++i) d[i] = th[i] - a1[i];
    smm<N, N, 1, false, false>(Bg, d, tv);
#pragma unroll
    for (int i = 0; i < N; ++i) h[i] = mr[i] + tv[i];
    // diff = I - B G ; cov = (diff C) diff^T + ((B W) dt) B^T ; symmetrised (:93-95)
    smm<N, N, N, false, false>(Bg, md.G, D);
#pragma unroll
    for (int j = 0; j < N; ++j)
#pragma unroll
      for (int i = 0; i < N; ++i) D[i + j * N] = ((i == j) ? 1.0 : 0.0) - D[i + j * N];
    smm<N, N, N, false, false>(D, Cr, t1);
    smm<N, N, N, false, true>(t1, D, Hm);
    smm<N, N, N, false, false>(Bg, W, t1);
#pragma unroll
    for (int k = 0; k < N * N; ++k) t1[k] = t1[k] * dt;
    smm<N, N, N, false, true>(t1, Bg, t2);
#pragma unroll
    for (int k = 0; k < N * N; ++k) Hm[k] = Hm[k] + t2[k];
#pragma unroll
    for (int j = 0; j < N; ++j)
#pragma unroll
      for (int i = 0; i < N; ++i) Hs[i + j * N] = (Hm[i + j * N] + Hm[j + i * N]) / 2.0;
    st |= eig_draw_small<N>(h, Hs, z, th);
    put(a.theta, r, th, N, false);
  }

  // ---- Gibbs sufficient statistics of the drawn path, ascending time (oracle_gibbs_stats)
  const StatViews &sv = a.stats;
  if (sv.ssy.ptr || sv.ny.ptr || sv.ssw.ptr || sv.scatter.ptr) {
    double ssy = 0.0, ny = 0.0, ssw[N], sc[N * N], prev[N], cur[N];
#pragma unroll
    for (int k = 0; k < N; ++k) ssw[k] = 0.0;
#pragma unroll
    for (int k = 0; k < N * N; ++k) sc[k] = 0.0;
    get(a.theta, 0, prev, N);
    for (int t = 0; t < T; ++t) {
      get(a.theta, t + 1, cur, N);
      const double y = bt.y.ptr[b * bt.y.sb + (int64_t)t * bt.y.sr];
      double ft;
      smm<1, N, 1, true, false>(md.F, cur, &ft);
      double res = 0.0;
      if (!isnan(y)) { res = (y - ft) * (y - ft); ny += 1.0; }
      ssy = (t == 0) ? res : ssy + res;
      const double dt = dt_at(bt, b, t);
      double gx[N], diff[N];
      smm<N, N, 1, false, false>(md.G, prev, gx);
#pragma unroll
      for (int i = 0; i < N; ++i) diff[i] = cur[i] - gx[i];
#pragma unroll
      for (int i = 0; i < N; ++i) {
        const double v = (diff[i] * diff[i]) / dt;
        ssw[i] = (t == 0) ? v : ssw[i] + v;
      }
#pragma unroll
      for (int j = 0; j < N; ++j)
#pragma unroll
        for (int i = 0; i < N; ++i) {
          const double v = (diff[i] * diff[j]) / dt;
          sc[i + j * N] = (t == 0) ? v : sc[i + j * N] + v;
        }
#pragma unroll
      for (int i = 0; i < N; ++i) prev[i] = cur[i];
    }
    if (sv.ssy.ptr) sv.ssy.ptr[b * sv.ssy.sb] = ssy;
    if (sv.ny.ptr) sv.ny.ptr[b * sv.ny.sb] = ny;
    if (sv.ssw.ptr)
      for (int k = 0; k < N; ++k) sv.ssw.ptr[b * sv.ssw.sb + k * sv.ssw.sk] = ssw[k];
    if (sv.scatter.ptr)
      for (int k = 0; k < N * N; ++k) sv.scatter.ptr[b * sv.scatter.sb + k * sv.scatter.sk] = sc[k];
  }

  if (bt.status) {
    bool finite = true;
#pragma unroll
    for (int k = 0; k < N; ++k) finite = finite && isfinite(th[k]);
    bt.status[b] = st | (finite ? 0 : BDLM_ST_NONFINITE);
  }
}

template <int N>
cudaError_t launch_n(const FfbsSmallArgs &a, const double *hG, const double *hF, cudaStream_t s) {
  FfbsModel<N> md;
  for (int k = 0; k < N * N; ++k) md.G[k] = hG[k];
  for (int k = 0; k < N; ++k) md.F[k] = hF[k];
  ffbs_small_kernel<N><<<(unsigned)((a.bt.B + 127) / 128), 128, 0, s>>>(md, a);
  return cudaGetLastError();
}

}  // namespace

bool ffbs_small_supported(const Batch &bt) {
  return bt.p == 1 && bt.n >= 1 && bt.n <= 4 && bt.keep_init && !bt.f_tv && !bt.g_tv && !bt.ps_model;
}

cudaError_t launch_ffbs_small(const FfbsSmallArgs &a, const double *hG, const double *hF,
                              cudaStream_t stream) {
  if (a.bt.B == 0) return cudaSuccess;
  switch (a.bt.n) {
    case 1: return launch_n<1>(a, hG, hF, stream);
    case 2: return launch_n<2>(a, hG, hF, stream);
    case 3: return launch_n<3>(a, hG, hF, stream);
    case 4: return launch_n<4>(a, hG, hF, stream);
    default: return cudaErrorInvalidValue;
  }
}

}  // namespace bdlm
