// small_steps.cuh -- register-level building blocks shared by the thread-per-series kernels
// (kf_small.cu, ffbs_small.cu) and the parallel-in-time scan kernels (scan.cu): unrolled small
// matrix products, the dgesv restatement, the Kalman / RTS steps for p = 1 and the eigSym draw of
// the backward sampler.
//
// Arithmetic mirrors oracle/bdlm_oracle.c operation for operation (see common.cuh);
// reference citations: KalmanFilter.scala:64-107,273-321 and Smoothing.scala:31-64.
#pragma once
#include "common.cuh"
#include "warp_linalg.cuh"  // rr_partner, sym_rot

namespace bdlm {
namespace small {

// out(AR x BC) = A(AR x AC) * B(AC x BC), column-major, TA/TB = operand stored
// transposed.  Products summed in increasing inner index, first product initialises.
template <int AR, int AC, int BC, bool TA, bool TB>
__host__ __device__ __forceinline__ void smm(const double *A, const double *B, double *out) {
#pragma unroll
  for (int j = 0; j < BC; ++j)
#pragma unroll
    for (int i = 0; i < AR; ++i) {
      double acc = 0.0;
#pragma unroll
      for (int k = 0; k < AC; ++k) {
        const double a = TA ? A[k + i * AC] : A[i + k * AR];
        const double b = TB ? B[j + k * BC] : B[k + j * AC];
        const double prod = a * b;
        acc = (k == 0) ? prod : acc + prod;
      }
      out[i + j * AR] = acc;
    }
}

// dgesv restatement (see oracle lu_solve): A is N x N (destroyed), Bm is N x NR.
template <int N, int NR>
__host__ __device__ __forceinline__ int lu_solve(double (&A)[N * N], double (&Bm)[N * NR]) {
  int st = 0;
#pragma unroll
  for (int j = 0; j < N; ++j) {
    int jp = j;
    double best = fabs(A[j + j * N]);
#pragma unroll
    for (int i = j + 1; i < N; ++i) {
      const double v = fabs(A[i + j * N]);
      if (v > best) { best = v; jp = i; }
    }
    double pv = A[j + j * N];
#pragma unroll
    for (int i = j + 1; i < N; ++i)
      if (jp == i) pv = A[i + j * N];
    if (pv != 0.0) {
#pragma unroll
      for (int i = j + 1; i < N; ++i)
        if (jp == i) {
#pragma unroll
          for (int c = 0; c < N; ++c) {
            const double t = A[j + c * N]; A[j + c * N] = A[i + c * N]; A[i + c * N] = t;
          }
#pragma unroll
          for (int c = 0; c < NR; ++c) {
            const double t = Bm[j + c * N]; Bm[j + c * N] = Bm[i + c * N]; Bm[i + c * N] = t;
          }
        }
      const double r = 1.0 / A[j + j * N];
#pragma unroll
      for (int i = j + 1; i < N; ++i) A[i + j * N] = A[i + j * N] * r;
    } else {
      st = BDLM_ST_SINGULAR;
    }
#pragma unroll
    for (int c = j + 1; c < N; ++c)
#pragma unroll
      for (int i = j + 1; i < N; ++i)
        A[i + c * N] = A[i + c * N] - A[i + j * N] * A[j + c * N];
  }
#pragma unroll
  for (int c = 0; c < NR; ++c) {
#pragma unroll
    for (int k = 0; k < N; ++k)
#pragma unroll
      for (int i = k + 1; i < N; ++i)
        Bm[i + c * N] = Bm[i + c * N] - Bm[k + c * N] * A[i + k * N];
#pragma unroll
    for (int k = N - 1; k >= 0; --k) {
      Bm[k + c * N] = Bm[k + c * N] / A[k + k * N];
#pragma unroll
      for (int i = 0; i < k; ++i)
        Bm[i + c * N] = Bm[i + c * N] - Bm[k + c * N] * A[i + k * N];
    }
  }
  return st;
}

// KalmanFilter.advState (KalmanFilter.scala:273-286)
template <int N, bool REG>
__host__ __device__ __forceinline__ void advance(const double *G, const double (&W)[N * N],
                                        double dt, const double (&m)[N],
                                        const double (&C)[N * N], double (&a)[N],
                                        double (&R)[N * N]) {
  if (!REG && dt == 0.0) {
#pragma unroll
    for (int i = 0; i < N; ++i) a[i] = m[i];
#pragma unroll
    for (int k = 0; k < N * N; ++k) R[k] = C[k];
    return;
  }
  double t1[N * N];
  smm<N, N, 1, false, false>(G, m, a);
  smm<N, N, N, false, false>(G, C, t1);
  smm<N, N, N, false, true>(t1, G, R);
#pragma unroll
  for (int k = 0; k < N * N; ++k) R[k] = R[k] + (REG ? W[k] : W[k] * dt);  // W * 1.0 == W
}

// oneStepPrediction (:311-321) + updateState (:64-94) for p = 1.
// RECIP (parallel-in-time scan only, 1e-9 contract): one reciprocal of Q instead of N divisions.
template <int N, bool RECIP = false>
__host__ __device__ __forceinline__ void update(const double *F, double V, double y,
                                       const double (&a)[N], const double (&R)[N * N],
                                       double &f, double &Q, double (&m)[N],
                                       double (&C)[N * N], int &st) {
  double fr[N];
  smm<1, N, 1, true, false>(F, a, &f);
  smm<1, N, N, true, false>(F, R, fr);
  smm<1, N, 1, false, false>(fr, F, &Q);
  Q = Q + V;
  if (isnan(y)) {  // all missing (:74-75)
#pragma unroll
    for (int i = 0; i < N; ++i) m[i] = a[i];
#pragma unroll
    for (int k = 0; k < N * N; ++k) C[k] = R[k];
    return;
  }
  // oneStepMissing (:44-53) on the full F, V repeats the same operations: reuse f, Q.
  const double e = y - f;
  double rhs[N], K[N], D[N * N], t1[N * N], t2[N], C2[N * N];
  smm<1, N, N, true, true>(F, R, rhs);  // F^T R^T
  if (Q == 0.0) st |= BDLM_ST_SINGULAR;
  if (RECIP) {
    const double rq = 1.0 / Q;
#pragma unroll
    for (int i = 0; i < N; ++i) K[i] = rhs[i] * rq;
  } else {
#pragma unroll
    for (int i = 0; i < N; ++i) K[i] = rhs[i] / Q;  // (Q^T \ (F^T R^T))^T  (:83)
  }
#pragma unroll
  for (int i = 0; i < N; ++i) m[i] = a[i] + K[i] * e;
  smm<N, 1, N, false, true>(K, F, D);  // K F^T
#pragma unroll
  for (int j = 0; j < N; ++j)
#pragma unroll
    for (int i = 0; i < N; ++i) D[i + j * N] = ((i == j) ? 1.0 : 0.0) - D[i + j * N];
  smm<N, N, N, false, false>(D, R, t1);
  smm<N, N, N, false, true>(t1, D, C);
#pragma unroll
  for (int i = 0; i < N; ++i) t2[i] = K[i] * V;
  smm<N, 1, N, false, true>(t2, K, C2);
#pragma unroll
  for (int k = 0; k < N * N; ++k) C[k] = C[k] + C2[k];
}

// Smoothing.smoothStep (Smoothing.scala:31-47)
template <int N>
__host__ __device__ __forceinline__ void rts_step(const double *G, const double (&m)[N],
                                         const double (&C)[N * N], const double (&a1)[N],
                                         const double (&R1)[N * N], bool textbook,
                                         double (&s)[N], double (&S)[N * N], int &st) {
  double rhs[N * N], At[N * N], Bg[N * N], d[N], t[N], Dm[N * N], t1[N * N], t2[N * N];
  smm<N, N, N, false, true>(G, C, rhs);  // G C^T
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
  for (int i = 0; i < N; ++i) d[i] = s[i] - a1[i];
  smm<N, N, 1, false, false>(Bg, d, t);
#pragma unroll
  for (int k = 0; k < N * N; ++k) Dm[k] = R1[k] - S[k];
  smm<N, N, N, false, false>(Bg, Dm, t1);
  if (textbook) smm<N, N, N, false, true>(t1, Bg, t2);
  else smm<N, N, N, false, false>(t1, Bg, t2);  // Smoothing.scala:44 (no transpose)
#pragma unroll
  for (int i = 0; i < N; ++i) s[i] = m[i] + t[i];
#pragma unroll
  for (int k = 0; k < N * N; ++k) S[k] = C[k] - t2[k];
}

// breeze MultivariateGaussian(mu, S).logPdf(x) (oracle mvn_logpdf), split so that the part that
// depends on S alone -- the dgesv factorisation (dgetf2) and sum(log(diag(cholesky(S)))) -- can be
// hoisted out of the time loop when S = W dt is the same at every step (regular grid).  prepare()
// followed by eval() performs exactly the operations of lu_solve + chol_logdet in the oracle's
// order, so hoisting does not change a bit.  Used by the thread-per-series log-likelihood
// (scalar_filters.cu) and the parallel-in-time log-likelihood sweep (scan.cu).
template <int N>
struct MvnPrepared {
  double LU[N * N];  // unit-lower multipliers below the diagonal, U on and above it
  int piv[N];        // row exchanged with row j at step j (j = no exchange)
  bool singular[N];  // zero pivot at step j: dgetf2 skips the scaling (info > 0)
  double ld;         // sum log diag chol(S)
  int st;

  __device__ __forceinline__ void prepare(const double (&S)[N * N]) {
    st = 0;
#pragma unroll
    for (int k = 0; k < N * N; ++k) LU[k] = S[k];
#pragma unroll
    for (int j = 0; j < N; ++j) {
      int jp = j;
      double best = fabs(LU[j + j * N]);
#pragma unroll
      for (int i = j + 1; i < N; ++i) {
        const double v = fabs(LU[i + j * N]);
        if (v > best) { best = v; jp = i; }
      }
      double pv = LU[j + j * N];
#pragma unroll
      for (int i = j + 1; i < N; ++i)
        if (jp == i) pv = LU[i + j * N];
      piv[j] = j;
      singular[j] = !(pv != 0.0);
      if (pv != 0.0) {
#pragma unroll
        for (int i = j + 1; i < N; ++i)
          if (jp == i) {
            piv[j] = i;
#pragma unroll
            for (int c = 0; c < N; ++c) {
              const double t = LU[j + c * N]; LU[j + c * N] = LU[i + c * N]; LU[i + c * N] = t;
            }
          }
        const double r = 1.0 / LU[j + j * N];
#pragma unroll
        for (int i = j + 1; i < N; ++i) LU[i + j * N] = LU[i + j * N] * r;
      } else {
        st = BDLM_ST_SINGULAR;
      }
#pragma unroll
      for (int c = j + 1; c < N; ++c)
#pragma unroll
        for (int i = j + 1; i < N; ++i)
          LU[i + c * N] = LU[i + c * N] - LU[i + j * N] * LU[j + c * N];
    }
    double L[N * N];
#pragma unroll
    for (int k = 0; k < N * N; ++k) L[k] = S[k];
    ld = 0.0;
#pragma unroll
    for (int j = 0; j < N; ++j) {
      double d = L[j + j * N];
#pragma unroll
      for (int k = 0; k < j; ++k) d = d - L[j + k * N] * L[j + k * N];
      if (!(d > 0.0)) st |= BDLM_ST_NOTPD;
      d = sqrt(d);
      L[j + j * N] = d;
#pragma unroll
      for (int i = j + 1; i < N; ++i) {
        double v = L[i + j * N];
#pragma unroll
        for (int k = 0; k < j; ++k) v = v - L[i + k * N] * L[j + k * N];
        L[i + j * N] = v / d;
      }
      ld = ld + log(d);
    }
  }

  __device__ __forceinline__ double eval(const double (&x)[N], const double (&mu)[N]) const {
    double c[N], slv[N];
#pragma unroll
    for (int i = 0; i < N; ++i) { c[i] = x[i] - mu[i]; slv[i] = c[i]; }
    // the row exchanges dgetf2 applied to the right-hand side as it went (same order)
#pragma unroll
    for (int j = 0; j < N; ++j)
      if (!singular[j]) {
#pragma unroll
        for (int i = j + 1; i < N; ++i)
          if (piv[j] == i) { const double t = slv[j]; slv[j] = slv[i]; slv[i] = t; }
      }
#pragma unroll
    for (int k = 0; k < N; ++k)
#pragma unroll
      for (int i = k + 1; i < N; ++i) slv[i] = slv[i] - slv[k] * LU[i + k * N];
#pragma unroll
    for (int k = N - 1; k >= 0; --k) {
      slv[k] = slv[k] / LU[k + k * N];
#pragma unroll
      for (int i = 0; i < k; ++i) slv[i] = slv[i] - slv[k] * LU[i + k * N];
    }
    double dot = 0.0;
#pragma unroll
    for (int i = 0; i < N; ++i) {
      const double prod = slv[i] * c[i];
      dot = (i == 0) ? prod : dot + prod;
    }
    return -dot / 2.0 - (N / 2.0 * 1.8378770664093453 + ld);
  }
};

// eigSym restatement (oracle jacobi_eigsym): one-sided Jacobi on the columns of U = A (lower
// triangle of Ain read) with V accumulated from I; lam_j = sign(v_j . u_j) |u_j| ascending, Vout
// columns = sign-normalised eigenvectors.  All indices are compile-time after unrolling.
template <int N>
__device__ __forceinline__ int jacobi_eigsym_small(const double (&Ain)[N * N], double (&lam)[N],
                                                   double (&Vout)[N * N]) {
  double A[N * N], V[N * N];
#pragma unroll
  for (int j = 0; j < N; ++j)
#pragma unroll
    for (int i = 0; i < N; ++i) {
      A[i + j * N] = (i >= j) ? Ain[i + j * N] : Ain[j + i * N];
      V[i + j * N] = (i == j) ? 1.0 : 0.0;
    }
  constexpr int M = (N + 1) & ~1;
  int st = (N == 1) ? 0 : BDLM_ST_NOTCONVERGED;
  for (int sweep = 0; sweep < kJacobiMaxSweeps && N > 1; ++sweep) {
    bool rotated = false;
#pragma unroll
    for (int round = 0; round < M - 1; ++round) {
#pragma unroll
      for (int p = 0; p < N; ++p) {
        const int q = rr_partner(N, round, p);
        if (q < 0 || q < p) continue;   // compile-time after unrolling
        double alpha = 0.0, beta = 0.0, gamma = 0.0;
#pragma unroll
        for (int i = 0; i < N; ++i) {
          const double up = A[i + p * N], uq = A[i + q * N];
          const double pp = up * up, qq = uq * uq, pq = up * uq;
          alpha = (i == 0) ? pp : alpha + pp;
          beta = (i == 0) ? qq : beta + qq;
          gamma = (i == 0) ? pq : gamma + pq;
        }
        if (gamma * gamma > kJacobiThr2 * (alpha * beta)) {
          rotated = true;
          double c, s;
          sym_rot(alpha, beta, gamma, c, s);
#pragma unroll
          for (int i = 0; i < N; ++i) {
            const double up = A[i + p * N], uq = A[i + q * N];
            A[i + p * N] = c * up - s * uq;
            A[i + q * N] = s * up + c * uq;
            const double vp = V[i + p * N], vq = V[i + q * N];
            V[i + p * N] = c * vp - s * vq;
            V[i + q * N] = s * vp + c * vq;
          }
        }
      }
    }
    if (!rotated) { st = 0; break; }
  }
  double d[N];
#pragma unroll
  for (int j = 0; j < N; ++j) {
    double nn = 0.0, dot = 0.0;
#pragma unroll
    for (int i = 0; i < N; ++i) {
      const double u = A[i + j * N];
      const double sq = u * u, vu = V[i + j * N] * u;
      nn = (i == 0) ? sq : nn + sq;
      dot = (i == 0) ? vu : dot + vu;
    }
    const double nrm = sqrt(nn);
    d[j] = (dot < 0.0) ? -nrm : nrm;
  }
  // eigenvalues ascending (stable), sign rule: largest-|component| (first such) positive
#pragma unroll
  for (int k = 0; k < N; ++k) {
    int rank = 0;
#pragma unroll
    for (int j = 0; j < N; ++j) rank += ((d[j] < d[k]) || (d[j] == d[k] && j < k)) ? 1 : 0;
    int im = 0;
    double best = fabs(V[0 + k * N]);
#pragma unroll
    for (int i = 1; i < N; ++i) {
      const double a = fabs(V[i + k * N]);
      if (a > best) { best = a; im = i; }
    }
    double vim = V[0 + k * N];
#pragma unroll
    for (int i = 1; i < N; ++i) vim = (im == i) ? V[i + k * N] : vim;
    const bool flip = vim < 0.0;
#pragma unroll
    for (int r = 0; r < N; ++r)
      if (rank == r) {
        lam[r] = d[k];
#pragma unroll
        for (int i = 0; i < N; ++i) Vout[i + r * N] = flip ? -V[i + k * N] : V[i + k * N];
      }
  }
  return st;
}

// MultivariateGaussianSvd(mu, cov).draw with injected normals z (oracle mvn_eig_draw)
template <int N>
__device__ __forceinline__ int eig_draw_small(const double (&mu)[N], const double (&cov)[N * N],
                                              const double (&z)[N], double (&out)[N]) {
  double lam[N], V[N * N], Mx[N * N], x[N];
  const int st = jacobi_eigsym_small<N>(cov, lam, V);
#pragma unroll
  for (int j = 0; j < N; ++j) {
    const double sq = sqrt(lam[j]);
#pragma unroll
    for (int i = 0; i < N; ++i) Mx[i + j * N] = V[i + j * N] * sq;
  }
  smm<N, N, 1, false, false>(Mx, z, x);
#pragma unroll
  for (int i = 0; i < N; ++i) out[i] = mu[i] + x[i];
  return st;
}

}  // namespace small
}  // namespace bdlm
